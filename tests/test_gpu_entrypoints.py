"""The reference's two inference entry points executed end to end on the GPU with synthetic
weights (SURVEY config 1 = plumbing): `demo.image_demo` (src/demo.py:161-225) and
`eval.eval_once` (src/eval.py:48-134 + src/dataset/kitti.py:100-159), on generated PNGs, checked
against the oracle pipeline: oracle pre-processing (pinned to cv2) -> torch-CPU forward ->
interpret_output -> [eval: rescale ALL boxes, eval.py:83-84] -> filter_prediction."""
import os

import numpy as np
import pytest

import oracle
from oracle import preproc
from oracle.torch_port import TorchForward
from squeezedet_b200 import _lib, demo, eval as sq_eval
from squeezedet_b200 import config as cfg
from squeezedet_b200.utils import synth, viz
from squeezedet_b200.utils.util import bbox_transform

pytestmark = pytest.mark.gpu
TOL = 1e-4


def make_png(path, h, w, seed):
  """A frame with structure (rectangles on noise) so detections spread over the image."""
  import cv2
  rng = np.random.default_rng(seed)
  im = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
  for _ in range(12):
    y0, x0 = int(rng.integers(0, h - 40)), int(rng.integers(0, w - 80))
    im[y0:y0 + int(rng.integers(20, 120)), x0:x0 + int(rng.integers(40, 300))] = \
        rng.integers(0, 256, 3, dtype=np.uint8)
  assert cv2.imwrite(path, im)
  return im


def oracle_pipeline(net, mc, weights, frame_u8, order, rescale):
  fed = preproc.preprocess(frame_u8, mc.IMAGE_WIDTH, mc.IMAGE_HEIGHT, mc.BGR_MEANS, order)
  preds = TorchForward(net, weights)(fed[None])
  boxes, probs, cls = oracle.interpret_output(preds, mc.ANCHOR_BOX, mc.CLASSES,
                                              mc.ANCHOR_PER_GRID, mc.IMAGE_WIDTH,
                                              mc.IMAGE_HEIGHT, mc.EXP_THRESH)
  boxes, probs, cls = boxes[0].copy(), probs[0], cls[0]
  if rescale:
    # eval.py:72-74,83-84 (scales are Python floats; numpy divides the float32 array in float32)
    x_scale = mc.IMAGE_WIDTH / float(frame_u8.shape[1])
    y_scale = mc.IMAGE_HEIGHT / float(frame_u8.shape[0])
    boxes[:, 0::2] /= x_scale
    boxes[:, 1::2] /= y_scale
  fb, fp, fc, src = oracle.filter_prediction(boxes, probs, cls, mc.CLASSES, mc.TOP_N_DETECTION,
                                             mc.PROB_THRESH, mc.NMS_THRESH)
  order66 = np.argsort(-probs.astype(np.float64), kind='stable')[:66]
  top = probs[order66].astype(np.float64)
  gap = np.abs(top[:, None] - top[None, :]) <= 10 * TOL * top[:, None]
  np.fill_diagonal(gap, False)
  return fb, fp, fc, bool(gap.any())


def compare(got_boxes, got_probs, got_cls, want, what):
  fb, fp, fc, near_tie = want
  if near_tie:                       # an fp-level reordering of the top-64 is legitimate
    assert abs(len(got_cls) - len(fc)) <= 2, what
    return
  assert list(got_cls) == list(fc), what
  np.testing.assert_allclose(np.asarray(got_probs, np.float64), np.asarray(fp, np.float64),
                             rtol=2 * TOL, atol=1e-7, err_msg=what)
  for g, w in zip(got_boxes, fb):
    np.testing.assert_allclose(np.asarray(g, np.float64), np.asarray(w, np.float64),
                               rtol=2 * TOL, atol=2e-2, err_msg=what)


def test_image_demo_runs_and_matches_oracle(tmp_path, gpu_device):
  frames = {}
  for k, (h, w) in enumerate([(375, 1242), (370, 1224)]):
    frames['%06d.png' % k] = make_png(str(tmp_path / ('%06d.png' % k)), h, w, seed=10 + k)
  flags = demo.parse_flags(['--mode', 'image', '--checkpoint', 'synthetic',
                            '--input_path', str(tmp_path / '0*.png'),
                            '--out_dir', str(tmp_path / 'out'), '--gpu', str(gpu_device)])
  results = demo.image_demo(flags)
  assert len(results) == 2
  mc = cfg.kitti_squeezeDet_config()
  weights = synth.synthetic_weights(oracle.param_specs('squeezeDet'), seed=0)
  for path, boxes, probs, classes in results:
    name = os.path.basename(path)
    assert os.path.exists(tmp_path / 'out' / ('out_' + name))
    fb, fp, fc, near = oracle_pipeline('squeezeDet', mc, weights, frames[name], 'demo', False)
    keep = [i for i in range(len(fp)) if fp[i] > mc.PLOT_PROB_THRESH]       # demo.py:201-205
    want = ([fb[i] for i in keep], [fp[i] for i in keep], [fc[i] for i in keep], near)
    compare(boxes, probs, classes, want, name)


def test_eval_once_reference_order_files_and_scorer(tmp_path, gpu_device):
  data = tmp_path / 'KITTI'
  (data / 'training' / 'image_2').mkdir(parents=True)
  (data / 'training' / 'label_2').mkdir(parents=True)
  (data / 'ImageSets').mkdir()
  ids, frames = [], {}
  for k, (h, w) in enumerate([(375, 1242), (370, 1224), (376, 1241)]):
    idx = '%06d' % k
    ids.append(idx)
    frames[idx] = make_png(str(data / 'training' / 'image_2' / (idx + '.png')), h, w, seed=20 + k)
    (data / 'training' / 'label_2' / (idx + '.txt')).write_text(
        'Car 0.00 0 -1.57 100.00 120.00 300.00 250.00 1.5 1.6 3.9 1.0 1.7 10.0 -1.5\n')
  (data / 'ImageSets' / 'val.txt').write_text('\n'.join(ids) + '\n')
  flags = sq_eval.parse_flags(['--data_path', str(data), '--image_set', 'val',
                               '--eval_dir', str(tmp_path / 'eval'),
                               '--checkpoint_path', 'synthetic', '--net', 'squeezeDet',
                               '--gpu', str(gpu_device)])
  all_boxes, aps, names = sq_eval.eval_once(flags)
  mc = cfg.kitti_squeezeDet_config()
  weights = synth.synthetic_weights(oracle.param_specs('squeezeDet'), seed=0)
  det_dir = tmp_path / 'eval' / 'detection_files_0' / 'data'
  for i, idx in enumerate(ids):
    fb, fp, fc, near = oracle_pipeline('squeezeDet', mc, weights, frames[idx], 'eval', True)
    # the reference's all_boxes[c][i].append(bbox_transform(b) + [s])  (eval.py:89-91)
    want = [[] for _ in range(mc.CLASSES)]
    for c, b, s in zip(fc, fb, fp):
      want[c].append(bbox_transform(b) + [s])
    lines = (det_dir / (idx + '.txt')).read_text().splitlines()
    got_n = sum(len(all_boxes[c][i]) for c in range(mc.CLASSES))
    assert len(lines) == got_n
    if near:
      continue
    k = 0
    for c in range(mc.CLASSES):
      assert len(all_boxes[c][i]) == len(want[c]), (idx, c)
      for g, w in zip(all_boxes[c][i], want[c]):
        np.testing.assert_allclose(np.asarray(g, np.float64), np.asarray(w, np.float64),
                                   rtol=2 * TOL, atol=2e-2)
        # and the file holds exactly that record in the KITTI line format (kitti.py:116-127)
        assert lines[k] == viz.kitti_detection_line(mc.CLASS_NAMES[c], g[:4], g[4]).rstrip('\n')
        k += 1
  # the reference's unmodified scorer ran and its AP files were parsed (kitti.py:129-159)
  if not os.path.exists(sq_eval.EVAL_TOOL):
    pytest.skip('scorer binary absent: __graft_entry__.build() compiles it into oracle/_ref where '
                'the reference checkout exists')
  assert aps is not None and len(aps) == 3 * mc.CLASSES and names[0] == 'car_easy'
  # evaluate_object writes stats_<class>_ap.txt for exactly the classes that occur in the detection
  # files (its eval_car / eval_pedestrian / eval_cyclist flags, evaluate_object.cpp:695-776)
  res = tmp_path / 'eval' / 'detection_files_0'
  for c, name in enumerate(mc.CLASS_NAMES):
    has = any(len(all_boxes[c][i]) > 0 for i in range(len(ids)))
    assert os.path.exists(res / ('stats_%s_ap.txt' % name)) == has, name
  assert any(os.path.exists(res / ('stats_%s_ap.txt' % n)) for n in mc.CLASS_NAMES)


def test_rescale_before_filter_changes_nothing_but_coordinates(gpu_device):
  """sqdet_set_box_scale: det_boxes come back divided by the scales (float32 division, as numpy
  does in eval.py:83-84) and the records equal the oracle filter run on those rescaled boxes."""
  from squeezedet_b200.nets import SqueezeDet
  from test_gpu_e2e import make_mc
  mc = make_mc('squeezeDet', 416, 128, 2)
  m = SqueezeDet(mc, gpu_device)
  m.load_weights(synth.synthetic_weights(synth.model_param_specs(m), seed=5))
  imgs = synth.synthetic_images(2, 128, 416, seed=6)
  b0, p0, c0 = m.detect(imgs)
  scales = np.array([[1248 / 1242.0, 384 / 375.0], [0.75, 1.5]], np.float32)
  m.set_box_scale(scales)
  b1, p1, c1, dets, counts = m.detect(imgs, want_dets=True)
  want = b0.copy()
  for j in range(2):
    want[j, :, 0::2] /= float(scales[j, 0])
    want[j, :, 1::2] /= float(scales[j, 1])
  assert np.array_equal(b1, want) and np.array_equal(p1, p0) and np.array_equal(c1, c0)
  for j in range(2):
    fb, fp, fc, src = oracle.filter_prediction(b1[j], p1[j], c1[j], mc.CLASSES,
                                               mc.TOP_N_DETECTION, mc.PROB_THRESH, mc.NMS_THRESH)
    n = int(counts[j])
    assert dets[j]['anchor'][:n].tolist() == src and dets[j]['cls'][:n].tolist() == fc
  m.set_box_scale(None)
  b2, _, _ = m.detect(imgs)
  assert np.array_equal(b2, b0)
