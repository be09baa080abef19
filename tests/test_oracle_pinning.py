"""The oracle's numpy half against the committed fixtures produced by the reference's own
functions (tests/golden/make_golden.py)."""
import hashlib
import os

import numpy as np

import oracle
from oracle import postproc as P
from golden.make_golden import filter_trials, trial_sha256


def _run_oracle(c):
  return oracle.filter_prediction(c['boxes'], c['probs'], c['cls'], c['classes'],
                                  c['top_n'], c['prob_thresh'], c['nms_thresh'])


def test_filter_prediction_matches_reference_fixtures(postproc_kat):
  assert len(postproc_kat['cases']) >= 12
  for c in postproc_kat['cases']:
    fb, fp, fc, src = _run_oracle(c)
    assert fc == c['out_cls'].tolist(), c['name']
    assert np.array_equal(np.asarray(fb, np.float32).reshape(-1, 4), c['out_boxes']), c['name']
    assert np.array_equal(np.asarray(fp, np.float32), c['out_probs']), c['name']
    # kept-box indices point back at the same rows
    for s, b in zip(src, fb):
      assert np.array_equal(c['boxes'][s], b)


def test_nms_matches_reference_fixtures(postproc_kat):
  n_checked = 0
  for c in postproc_kat['cases']:
    if len(c['nms_keep']) == 0:
      continue
    keep = oracle.nms(c['boxes'], c['probs'], c['nms_thresh'])
    assert keep == c['nms_keep'].tolist(), c['name']
    n_checked += 1
  assert n_checked >= 10


def test_chain_case_is_not_greedy_nms(postproc_kat):
  c = [x for x in postproc_kat['cases'] if x['name'].startswith('chain')][0]
  assert c['nms_keep'].tolist() == [True, False, False]   # greedy NMS would keep C
  assert oracle.nms(c['boxes'], c['probs'], c['nms_thresh']) == [True, False, False]


def test_batch_iou_bit_exact(postproc_kat):
  b = postproc_kat['iou_boxes']
  for row, i in zip(postproc_kat['iou_out'], (0, 17, 256)):
    got = oracle.batch_iou(b, b[i])
    assert got.dtype == np.float32
    assert np.array_equal(got, row, equal_nan=True)


CONFIGS = {
    'kitti_squeezeDet_config': (1248, 384, 24, 78, P.ANCHOR_SHAPES_SQUEEZE),
    'kitti_squeezeDetPlus_config': (1242, 375, 22, 76, P.ANCHOR_SHAPES_SQUEEZE),
    'kitti_vgg16_config': (1242, 375, 24, 78, P.ANCHOR_SHAPES_SQUEEZE),
    'kitti_res50_config': (1242, 375, 24, 78, P.ANCHOR_SHAPES_RES50),
}


def test_set_anchors_matches_reference_fixtures(anchors_golden):
  for fn, (w, h, gh, gw, shapes) in CONFIGS.items():
    a = oracle.set_anchors(w, h, gh, gw, shapes)
    g = anchors_golden[fn]
    assert list(a.shape) == g['shape']
    assert hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest() == g['sha256'], fn
    assert a[0].tolist() == g['first'] and a[-1].tolist() == g['last']


def test_reference_filter_prediction_recorded_outputs():
  """60 seeded cases through the oracle, against what the reference's own filter_prediction
  returned for them (reference_filter.npz: the input rows it kept, in its output order)."""
  z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_filter.npz'))
  ends = np.cumsum(z['counts'])
  trials = list(filter_trials())
  assert len(trials) == len(ends) == 60
  for t, (boxes, probs, cls, top_n) in enumerate(trials):
    assert trial_sha256(boxes, probs, cls, top_n) == z['input_sha256'][t], t
    rows = z['rows'][ends[t] - z['counts'][t]:ends[t]].astype(np.int64)
    ob, op, oc, _ = oracle.filter_prediction(boxes, probs, cls, 3, top_n, 0.005, 0.4)
    assert oc == cls[rows].tolist(), t
    assert len(ob) == len(rows) and all(np.array_equal(x, boxes[r]) for x, r in zip(ob, rows)), t
    assert [float(x) for x in op] == [float(x) for x in probs[rows]], t


def test_interpret_output_hand_case():
  """A 1x1 grid, K=1, C=2 case worked by hand (SURVEY App. A.4/A.5)."""
  anchors = np.array([[50., 40., 20., 10.]])
  # logits (2), conf, dx dy dw dh ; dw = 2 > EXP_THRESH exercises the linear tail
  preds = np.array([[[[0.0, np.log(3.0), 0.0, 0.5, -1.0, 2.0, 0.0]]]], np.float32)
  boxes, probs, cls = oracle.interpret_output(preds, anchors, 2, 1, 100, 80, 1.0)
  assert cls.tolist() == [[1]]
  np.testing.assert_allclose(probs[0, 0], 0.75 * 0.5, rtol=1e-6)
  w = 20 * np.e * 2.0            # safe_exp(2) = e*(2-1+1)
  cx, cy, h = 50 + 0.5 * 20, 40 - 1.0 * 10, 10.0
  xmin, xmax = max(cx - w / 2, 0), min(cx + w / 2, 99)
  ymin, ymax = max(cy - h / 2, 0), min(cy + h / 2, 79)
  want = [xmin + 0.5 * (xmax - xmin + 1), ymin + 0.5 * (ymax - ymin + 1),
          xmax - xmin + 1, ymax - ymin + 1]
  np.testing.assert_allclose(boxes[0, 0], want, rtol=1e-6)
