"""Helpers for the -m gpu parity tests: every call goes through the C ABI."""
import ctypes as C

import numpy as np

from squeezedet_b200 import _lib
from squeezedet_b200._lib import DeviceBuffer


def conv2d_gpu(x, w, b=None, stride=1, padding='SAME', relu=True, scale=None, shift=None,
               y_cstride=None, y_coff=0, math_mode=0, device=0, y_init=None):
  lib = _lib.load()
  B, H, W, Cin = x.shape
  k, _, _, Cout = w.shape
  import oracle
  Ho = oracle.conv_geometry(H, k, stride, padding)[0]
  Wo = oracle.conv_geometry(W, k, stride, padding)[0]
  cs = y_cstride or Cout
  dx = DeviceBuffer.from_numpy(x.astype(np.float32), device)
  dw = DeviceBuffer.from_numpy(w.astype(np.float32), device)
  db = DeviceBuffer.from_numpy(b.astype(np.float32), device) if b is not None else None
  dsc = DeviceBuffer.from_numpy(scale.astype(np.float32), device) if scale is not None else None
  dsh = DeviceBuffer.from_numpy(shift.astype(np.float32), device) if shift is not None else None
  y0 = y_init if y_init is not None else np.full((B, Ho, Wo, cs), np.nan, np.float32)
  dy = DeviceBuffer.from_numpy(y0, device)
  _lib.check(lib.sqdet_conv2d(dx.ptr, dw.ptr, db.ptr if db else None, dsc.ptr if dsc else None,
                              dsh.ptr if dsh else None, dy.ptr, B, H, W, Cin, Cout, k, stride,
                              _lib.pad_code(padding), int(relu), cs, y_coff, math_mode, None))
  _lib.check(lib.sqdet_stream_sync(device, None))
  return dy.to_numpy(np.float32, (B, Ho, Wo, cs))


def maxpool_gpu(x, k, stride, padding, device=0):
  lib = _lib.load()
  import oracle
  B, H, W, Cc = x.shape
  Ho = oracle.conv_geometry(H, k, stride, padding)[0]
  Wo = oracle.conv_geometry(W, k, stride, padding)[0]
  dx = DeviceBuffer.from_numpy(x.astype(np.float32), device)
  dy = DeviceBuffer(B * Ho * Wo * Cc * 4, device)
  _lib.check(lib.sqdet_maxpool_nhwc(dx.ptr, dy.ptr, B, H, W, Cc, k, stride,
                                    _lib.pad_code(padding), None))
  return dy.to_numpy(np.float32, (B, Ho, Wo, Cc))


def interpret_gpu(preds, anchors_f64, K, classes, img_w, img_h, exp_thresh=1.0, device=0):
  lib = _lib.load()
  B, gh, gw, _ = preds.shape
  A = gh * gw * K
  dp = DeviceBuffer.from_numpy(preds.astype(np.float32), device)
  da = DeviceBuffer.from_numpy(np.asarray(anchors_f64, np.float64).astype(np.float32), device)
  db = DeviceBuffer(B * A * 16, device)
  dpr = DeviceBuffer(B * A * 4, device)
  dc = DeviceBuffer(B * A * 8, device)
  _lib.check(lib.sqdet_interpret(dp.ptr, da.ptr, db.ptr, dpr.ptr, dc.ptr, B, gh, gw, K, classes,
                                 img_w, img_h, C.c_float(exp_thresh), None))
  return (db.to_numpy(np.float32, (B, A, 4)), dpr.to_numpy(np.float32, (B, A)),
          dc.to_numpy(np.int64, (B, A)))


def topk_nms_gpu(boxes, probs, cls, classes, top_n, prob_thresh, nms_thresh, max_dets=None,
                 device=0):
  """boxes [B,A,4] probs [B,A] cls [B,A] -> (dets [B,max_dets], counts [B])."""
  lib = _lib.load()
  boxes = np.ascontiguousarray(boxes, np.float32)
  B, A = probs.shape
  if max_dets is None:
    max_dets = top_n if 0 < top_n < A else min(A, 1024)
  db = DeviceBuffer.from_numpy(boxes, device)
  dp = DeviceBuffer.from_numpy(np.ascontiguousarray(probs, np.float32), device)
  dc = DeviceBuffer.from_numpy(np.ascontiguousarray(cls, np.int64), device)
  dd = DeviceBuffer(B * max_dets * 28, device)
  dn = DeviceBuffer(B * 4, device)
  _lib.check(lib.sqdet_topk_nms(db.ptr, dp.ptr, dc.ptr, B, A, classes, top_n,
                                C.c_float(prob_thresh), C.c_float(nms_thresh), dd.ptr, dn.ptr,
                                max_dets, None))
  return dd.to_numpy(_lib.DET_DTYPE, (B, max_dets)), dn.to_numpy(np.int32, (B,))


def rel_err(got, want):
  """max |got-want| / max|want| — the per-tensor relative error used for activations."""
  want = np.asarray(want, np.float64)
  return float(np.abs(np.asarray(got, np.float64) - want).max() / max(np.abs(want).max(), 1e-30))


def preprocess_gpu(img_u8, width, height, bgr_means, order, device=0):
  """sqdet_preprocess_u8 on one uint8 [H0, W0, 3] image -> float32 [height, width, 3]."""
  lib = _lib.load()
  img = np.ascontiguousarray(img_u8, np.uint8)
  h0, w0 = img.shape[:2]
  src = DeviceBuffer.from_numpy(img, device)
  dst = DeviceBuffer(height * width * 3 * 4, device)
  means = np.ascontiguousarray(np.asarray(bgr_means, np.float64).reshape(3))
  code = {'demo': 0, 'eval': 1}[order]
  _lib.check(lib.sqdet_preprocess_u8(src.ptr, h0, w0, dst.ptr, height, width, means.ctypes.data,
                                     code, None))
  return dst.to_numpy(np.float32, (height, width, 3))


def class_margin(preds64, anchors_per_grid, classes):
  """Relative top-2 margin of the per-anchor class probabilities, from fp64 oracle preds
  [B,Hg,Wg,K*(C+5)]: (p_top1 - p_top2) / p_top1 (the sigmoid confidence is a common factor).
  An argmax may legitimately differ from the oracle's only where this is below fp noise."""
  p = np.asarray(preds64, np.float64)
  B = p.shape[0]
  K, C = anchors_per_grid, classes
  logits = p[..., :K * C].reshape(B, -1, C)
  z = logits - logits.max(axis=2, keepdims=True)
  e = np.exp(z)
  pr = e / e.sum(axis=2, keepdims=True)
  top = np.sort(pr, axis=2)
  if C == 1:
    return np.ones(pr.shape[:2])
  return (top[..., -1] - top[..., -2]) / top[..., -1]


def assert_classes_match(got_cls, want_cls, preds64, anchors_per_grid, classes, tol):
  """north_star: class ids bit-exact.  A mismatch is tolerated ONLY where the fp64 oracle's
  own top-2 class margin is below 10*tol (a near tie that fp32 rounding may order either way);
  returns the number of such near-tie mismatches."""
  mism = np.asarray(got_cls) != np.asarray(want_cls)
  if not mism.any():
    return 0
  margin = class_margin(preds64, anchors_per_grid, classes)
  bad = mism & (margin >= 10 * tol)
  assert not bad.any(), ('class id differs outside a near tie', int(bad.sum()),
                         float(margin[bad].max()))
  return int(mism.sum())


def fire_gpu(x, wsq, bsq, we1, be1, we3, be3, math_mode=1, device=0):
  """sqdet_fire on host arrays: x [B,H,W,Cin], HWIO kernels -> y [B,H,W,E1+E3]."""
  lib = _lib.load()
  B, H, W, Cin = x.shape
  S, E1, E3 = wsq.shape[3], we1.shape[3], we3.shape[3]
  bufs = [DeviceBuffer.from_numpy(np.ascontiguousarray(a, np.float32), device)
          for a in (x, wsq, bsq, we1, be1, we3, be3)]
  y0 = np.full((B, H, W, E1 + E3), np.nan, np.float32)
  dy = DeviceBuffer.from_numpy(y0, device)
  _lib.check(lib.sqdet_fire(*[b.ptr for b in bufs], dy.ptr, B, H, W, Cin, S, E1, E3,
                            int(math_mode), None))
  _lib.check(lib.sqdet_stream_sync(device, None))
  return dy.to_numpy(np.float32, y0.shape)
