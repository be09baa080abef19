"""ctypes binding of ``libsqdet_b200.so`` (the C ABI declared in
``include/sqdet_b200.h``).  There is no CPU fallback: if the library is missing
or no B200 is visible, calls fail loudly with :class:`SqdetError`."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libsqdet_b200.so')

OK = 0
PAD_SAME, PAD_VALID = 0, 1
MATH_FP32_SIMT, MATH_TF32X3_TC = 0, 1
IMG_F32, IMG_U8 = 0, 1
_PAD = {'SAME': PAD_SAME, 'VALID': PAD_VALID}


class SqdetError(RuntimeError):
  def __init__(self, code, msg):
    super().__init__('sqdet error %d: %s' % (code, msg))
    self.code = code


class Det(C.Structure):
  """struct sqdet_det — one filtered detection (28 bytes)."""
  _fields_ = [('anchor', C.c_int32), ('cls', C.c_int32), ('prob', C.c_float),
              ('cx', C.c_float), ('cy', C.c_float), ('w', C.c_float),
              ('h', C.c_float)]


DET_DTYPE = np.dtype([('anchor', '<i4'), ('cls', '<i4'), ('prob', '<f4'),
                      ('cx', '<f4'), ('cy', '<f4'), ('w', '<f4'), ('h', '<f4')])
assert DET_DTYPE.itemsize == C.sizeof(Det) == 28


class Config(C.Structure):
  """struct sqdet_config."""
  _fields_ = [('batch_size', C.c_int32), ('image_height', C.c_int32),
              ('image_width', C.c_int32), ('classes', C.c_int32),
              ('anchors_per_grid', C.c_int32), ('top_n_detection', C.c_int32),
              ('prob_thresh', C.c_float), ('nms_thresh', C.c_float),
              ('exp_thresh', C.c_float), ('batch_norm_epsilon', C.c_float),
              ('math_mode', C.c_int32), ('max_dets', C.c_int32)]


_vp, _i, _f, _i64 = C.c_void_p, C.c_int, C.c_float, C.c_int64
_ip = C.POINTER(C.c_int)
_i64p = C.POINTER(C.c_int64)
_fp = C.c_void_p      # float* passed as raw address (numpy .ctypes.data / device ptr)

# name -> (restype, argtypes): every symbol include/sqdet_b200.h declares.
SIGNATURES = {
    'sqdet_last_error': (C.c_char_p, []),
    'sqdet_version': (C.c_char_p, []),
    'sqdet_device_count': (_i, []),
    'sqdet_create': (_i, [C.POINTER(Config), _i, C.POINTER(_vp)]),
    'sqdet_destroy': (_i, [_vp]),
    'sqdet_add_conv': (_i, [_vp, C.c_char_p, _i, _i, _i, _i, _i, _i, _ip]),
    'sqdet_add_conv_bn': (_i, [_vp, C.c_char_p, _i, _i, _i, _i, _i, _i, _ip]),
    'sqdet_add_pool': (_i, [_vp, C.c_char_p, _i, _i, _i, _i, _ip]),
    'sqdet_add_fire': (_i, [_vp, C.c_char_p, _i, _i, _i, _i, _ip]),
    'sqdet_add_add_relu': (_i, [_vp, C.c_char_p, _i, _i, _ip]),
    'sqdet_set_preds': (_i, [_vp, _i, _vp, _i64]),
    'sqdet_finalize': (_i, [_vp]),
    'sqdet_num_params': (_i, [_vp]),
    'sqdet_param_info': (_i, [_vp, _i, C.c_char_p, _i, _i64p, _ip]),
    'sqdet_set_param': (_i, [_vp, C.c_char_p, _fp, _i64p, _i]),
    'sqdet_num_tensors': (_i, [_vp]),
    'sqdet_tensor_info': (_i, [_vp, _i, C.c_char_p, _i, _i64p]),
    'sqdet_read_tensor': (_i, [_vp, _i, _fp]),
    'sqdet_num_ops': (_i, [_vp]),
    'sqdet_op_info': (_i, [_vp, _i, C.c_char_p, _i, _i64p, _i64p, _i64p]),
    'sqdet_forward': (_i, [_vp, _fp, _vp]),
    'sqdet_forward_profiled': (_i, [_vp, _fp, _vp, _fp]),
    'sqdet_results_dev': (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                               C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int32)]),
    'sqdet_detect': (_i, [_vp, _fp, _fp, _fp, _fp, _fp, _fp, _vp]),
    'sqdet_set_bgr_means': (_i, [_vp, _vp]),
    'sqdet_submit': (_i, [_vp, _vp, _i, _vp, _vp]),
    'sqdet_wait': (_i, [_vp]),
    'sqdet_submit_frames': (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    'sqdet_set_box_scale': (_i, [_vp, _vp]),
    'sqdet_launches_per_forward': (_i, [_vp]),
    'sqdet_engine_stream': (_vp, [_vp]),
    'sqdet_comm_unique_id': (_i, [_vp]),
    'sqdet_comm_init': (_i, [_vp, _i, _i, _vp]),
    'sqdet_comm_attach': (_i, [_vp, _vp, _i, _i]),
    'sqdet_comm_destroy': (_i, [_vp]),
    'sqdet_set_gather_in_forward': (_i, [_vp, _i]),
    'sqdet_allgather': (_i, [_vp, _vp, _vp]),
    'sqdet_gathered_dev': (_i, [_vp, C.POINTER(_vp), C.POINTER(C.c_int64),
                                C.POINTER(C.c_int32)]),
    'sqdet_fire': (_i, [_fp] * 8 + [_i] * 8 + [_vp]),
    'sqdet_conv2d': (_i, [_fp, _fp, _fp, _fp, _fp, _fp] + [_i] * 12 + [_vp]),
    'sqdet_maxpool_nhwc': (_i, [_fp, _fp] + [_i] * 7 + [_vp]),
    'sqdet_preprocess_u8': (_i, [_vp, _i, _i, _fp, _i, _i, _vp, _i, _vp]),
    'sqdet_interpret': (_i, [_fp, _fp, _fp, _fp, _fp] + [_i] * 7 + [_f, _vp]),
    'sqdet_topk_nms': (_i, [_fp, _fp, _fp, _i, _i, _i, _i, _f, _f, _fp, _fp, _i, _vp]),
    'sqdet_malloc': (_i, [_i, _i64, C.POINTER(_vp)]),
    'sqdet_free': (_i, [_i, _vp]),
    'sqdet_malloc_host': (_i, [_i64, C.POINTER(_vp)]),
    'sqdet_free_host': (_i, [_vp]),
    'sqdet_memcpy_h2d': (_i, [_vp, _vp, _i64, _vp]),
    'sqdet_memcpy_d2h': (_i, [_vp, _vp, _i64, _vp]),
    'sqdet_stream_sync': (_i, [_i, _vp]),
}

_lib = None


def load():
  """Load the shared library (once) and type every entry point."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.isfile(LIB_PATH):
    raise SqdetError(-100, 'libsqdet_b200.so is not built (%s); run '
                     '`python -c "import __graft_entry__ as g; g.build()"` or '
                     '`make -C squeezedet_b200/csrc`' % LIB_PATH)
  lib = C.CDLL(LIB_PATH)
  for name, (res, args) in SIGNATURES.items():
    fn = getattr(lib, name)          # AttributeError if a declared symbol is missing
    fn.restype = res
    fn.argtypes = args
  _lib = lib
  return lib


def check(rc):
  if rc != OK:
    raise SqdetError(rc, load().sqdet_last_error().decode('utf-8', 'replace'))


def pad_code(padding):
  try:
    return _PAD[padding.upper()]
  except (KeyError, AttributeError):
    raise ValueError("padding must be 'SAME' or 'VALID', got %r" % (padding,))


def device_count():
  return load().sqdet_device_count()


def comm_unique_id():
  """128-byte ncclUniqueId (rank 0 calls this and shares the bytes with the other ranks)."""
  buf = (C.c_char * 128)()
  check(load().sqdet_comm_unique_id(buf))
  return bytes(buf)


# ---- small helpers for callers that keep buffers outside torch ---------------------------
class DeviceBuffer:
  """Device allocation owned through sqdet_malloc/sqdet_free."""

  def __init__(self, nbytes, device=0):
    self.device = device
    self.nbytes = int(nbytes)
    p = _vp()
    check(load().sqdet_malloc(device, self.nbytes, C.byref(p)))
    self.ptr = p.value

  @classmethod
  def from_numpy(cls, arr, device=0):
    arr = np.ascontiguousarray(arr)
    buf = cls(arr.nbytes, device)
    check(load().sqdet_memcpy_h2d(buf.ptr, arr.ctypes.data, arr.nbytes, None))
    check(load().sqdet_stream_sync(device, None))
    return buf

  def to_numpy(self, dtype, shape):
    out = np.empty(shape, dtype=dtype)
    assert out.nbytes <= self.nbytes
    check(load().sqdet_memcpy_d2h(out.ctypes.data, self.ptr, out.nbytes, None))
    check(load().sqdet_stream_sync(self.device, None))
    return out

  def free(self):
    if self.ptr:
      load().sqdet_free(self.device, self.ptr)
      self.ptr = None

  def __del__(self):
    try:
      self.free()
    except Exception:
      pass


class ScratchPool:
  """Grow-only device scratch, one ONE allocation, reused call after call: the reference-style
  two-step loop (`sess.run` then `model.filter_prediction`, demo.py:193-199) calls the stage-isolated
  entries thousands of times, and five cudaMalloc/cudaFree pairs per call dominated them."""

  def __init__(self, device=0):
    self.device = device
    self.buf = None

  def carve(self, *sizes):
    """-> device pointers of len(sizes) regions (256-byte aligned) inside the pooled allocation."""
    offs, total = [], 0
    for n in sizes:
      offs.append(total)
      total += (int(n) + 255) & ~255
    if self.buf is None or self.buf.nbytes < total:
      if self.buf is not None:
        self.buf.free()
      self.buf = DeviceBuffer(max(total, 1 << 16), self.device)
    return [self.buf.ptr + o for o in offs]

  def upload(self, ptr, arr):
    arr = np.ascontiguousarray(arr)
    check(load().sqdet_memcpy_h2d(ptr, arr.ctypes.data, arr.nbytes, None))

  def download(self, ptr, dtype, shape):
    out = np.empty(shape, dtype=dtype)
    check(load().sqdet_memcpy_d2h(out.ctypes.data, ptr, out.nbytes, None))
    check(load().sqdet_stream_sync(self.device, None))
    return out


_scratch_pools = {}


def scratch_pool(device=0):
  if device not in _scratch_pools:
    _scratch_pools[device] = ScratchPool(device)
  return _scratch_pools[device]


class PinnedArray:
  """numpy view over cudaMallocHost memory (for the end-to-end host path)."""

  def __init__(self, shape, dtype):
    self.dtype = np.dtype(dtype)
    self.shape = tuple(shape)
    nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
    p = _vp()
    check(load().sqdet_malloc_host(max(nbytes, 1), C.byref(p)))
    self.ptr = p.value
    buf = (C.c_char * nbytes).from_address(self.ptr)
    self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

  def free(self):
    if self.ptr:
      self.array = None
      load().sqdet_free_host(self.ptr)
      self.ptr = None

  def __del__(self):
    try:
      self.free()
    except Exception:
      pass
