#!/usr/bin/env python
"""Evaluation loop — drop-in for the detection part of reference ``src/eval.py``
(`eval_once`, lines 48-134), same flags: --dataset --data_path --image_set --eval_dir
--checkpoint_path --run_once --net --gpu.

Per image, in the reference's order (eval.py:69-92): the uint8 frame goes to the GPU, where it
is converted to float32, has the BGR means subtracted and is resized (src/dataset/imdb.py:85-97);
forward; ALL det boxes are rescaled to the original image (eval.py:83-84) and only then
filtered (filter_prediction + NMS on original-image coordinates, eval.py:86-87) - one
`sqdet_submit_frames(..., order=eval, rescale=1)` call; corner format + score go into
all_boxes[cls][image].  Then the KITTI detection files are written
(src/dataset/kitti.py:100-127) and the reference's unmodified `evaluate_object` binary
(built by oracle/build_kitti_eval.sh) is invoked and its stats_*_ap.txt parsed
(kitti.py:129-159).  The TensorBoard summaries and the checkpoint-polling loop
(eval.py:171-239) are not rebuilt.
"""
from __future__ import annotations

import argparse
import os
import subprocess

import numpy as np

from .utils.util import Timer, bbox_transform
from .utils.viz import parse_kitti_ap_files, write_kitti_detections


def parse_flags(argv=None):
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawTextHelpFormatter)
  ap.add_argument('--dataset', default='KITTI', help='Currently support KITTI dataset.')
  ap.add_argument('--data_path', default='', help='Root directory of data')
  ap.add_argument('--image_set', default='test', help='train, trainval, val, or test')
  ap.add_argument('--eval_dir', default='/tmp/bichen/logs/squeezeDet/eval')
  ap.add_argument('--checkpoint_path', default='/tmp/bichen/logs/squeezeDet/train',
                  help='TF checkpoint path, .npz keyed by reference variable names, or "synthetic".')
  ap.add_argument('--run_once', action='store_true', default=True)
  ap.add_argument('--net', default='squeezeDet', help='Neural net architecture.')
  ap.add_argument('--gpu', default='0', help='gpu id.')
  return ap.parse_args(argv)


NETS = {'vgg16': ('VGG16ConvDet', 'kitti_vgg16_config'),
        'resnet50': ('ResNet50ConvDet', 'kitti_res50_config'),
        'squeezeDet': ('SqueezeDet', 'kitti_squeezeDet_config'),
        'squeezeDet+': ('SqueezeDetPlus', 'kitti_squeezeDetPlus_config')}


def read_image(path, mc):
  """imdb.read_image_batch for one image (src/dataset/imdb.py:85-97): float32, subtract the
  BGR means in place, THEN resize; returns the image and (x_scale, y_scale)."""
  import cv2
  im = cv2.imread(path).astype(np.float32, copy=False)
  im -= mc.BGR_MEANS
  orig_h, orig_w = float(im.shape[0]), float(im.shape[1])
  im = cv2.resize(im, (mc.IMAGE_WIDTH, mc.IMAGE_HEIGHT))
  return im, (mc.IMAGE_WIDTH / orig_w, mc.IMAGE_HEIGHT / orig_h)


def detections_to_all_boxes(records, count, scale, num_classes):
  """One image's filtered records -> per-class lists of [xmin, ymin, xmax, ymax, score]
  (eval.py:89-91).  `scale` = (x_scale, y_scale) still to be divided out, or None when the
  engine already rescaled the boxes before the filter (the reference order, eval.py:83-87).
  count < 0 is the filter's overflow marker (PROB_THRESH branch above the record capacity)."""
  from ._lib import SqdetError
  if count < 0:
    raise SqdetError(-6, 'more boxes above PROB_THRESH than the record capacity')
  out = [[] for _ in range(num_classes)]
  x_scale, y_scale = scale if scale is not None else (1.0, 1.0)
  for r in records[:count]:
    if scale is None:
      box = np.array([r['cx'], r['cy'], r['w'], r['h']], dtype=np.float32)
    else:
      box = np.array([r['cx'] / x_scale, r['cy'] / y_scale, r['w'] / x_scale, r['h'] / y_scale],
                     dtype=np.float32)
    out[int(r['cls'])].append(bbox_transform(box) + [r['prob']])
  return out


# the reference's scorer as __graft_entry__.build() / oracle/build_kitti_eval.sh compile it
EVAL_TOOL = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle',
                         '_ref', 'evaluate_object')


def eval_once(flags):
  from . import config as cfg
  from . import nets
  from .utils import checkpoint as ckpt, synth
  assert flags.dataset == 'KITTI', 'Currently only supports KITTI dataset'
  assert flags.net in NETS, 'Selected neural net architecture not supported: {}'.format(flags.net)
  cls_name, cfg_name = NETS[flags.net]
  mc = getattr(cfg, cfg_name)()
  mc.BATCH_SIZE = 1                     # the reference evaluates image by image (eval.py:150)
  mc.LOAD_PRETRAINED_MODEL = False
  model = getattr(nets, cls_name)(mc, int(flags.gpu))
  if flags.checkpoint_path == 'synthetic':
    model.load_weights(synth.synthetic_weights(synth.model_param_specs(model), seed=0))
  else:
    model.load_weights(ckpt.load_weights_file(flags.checkpoint_path, names=model.param_names()))

  with open(os.path.join(flags.data_path, 'ImageSets', flags.image_set + '.txt')) as f:
    image_ids = [x.strip() for x in f.readlines()]
  image_dir = os.path.join(flags.data_path, 'training', 'image_2')
  num_images = len(image_ids)
  all_boxes = [[[] for _ in range(num_images)] for _ in range(mc.CLASSES)]
  _t = {'im_detect': Timer(), 'im_read': Timer(), 'misc': Timer()}
  for i, index in enumerate(image_ids):
    import cv2
    _t['im_read'].tic()
    frame = cv2.imread(os.path.join(image_dir, index + '.png'))     # uint8 BGR, original size
    _t['im_read'].toc()
    _t['im_detect'].tic()
    # imdb.py:85-97 pre-processing, forward, eval.py:83-84 rescale, filter: one GPU pass
    dets, counts = model.detect_frames([frame], order='eval', rescale=True)
    _t['im_detect'].toc()
    _t['misc'].tic()
    per_class = detections_to_all_boxes(dets[0], int(counts[0]), None, mc.CLASSES)
    for c in range(mc.CLASSES):
      all_boxes[c][i] = per_class[c]
    _t['misc'].toc()
    print('im_detect: {:d}/{:d} im_read: {:.3f}s detect: {:.3f}s misc: {:.3f}s'.format(
        i + 1, num_images, _t['im_read'].average_time, _t['im_detect'].average_time,
        _t['misc'].average_time))

  det_dir = os.path.join(flags.eval_dir, 'detection_files_{:s}'.format('0'), 'data')
  result_dir = write_kitti_detections(det_dir, image_ids, mc.CLASS_NAMES, all_boxes)
  tool = EVAL_TOOL
  aps = names = None
  if os.path.exists(tool):
    cmd = ' '.join([tool, os.path.join(flags.data_path, 'training'),
                    os.path.join(flags.data_path, 'ImageSets', flags.image_set + '.txt'),
                    result_dir, str(num_images)])
    print('Running: {}'.format(cmd))
    subprocess.call(cmd, shell=True)
    aps, names = parse_kitti_ap_files(result_dir, mc.CLASS_NAMES)
    for ap, name in zip(aps, names):
      print('    {}: {:.3f}'.format(name, ap))
    print('    Mean average precision: {:.3f}'.format(float(np.mean(aps))))
  else:
    print('KITTI scorer binary not found ({}; build it with oracle/build_kitti_eval.sh); '
          'detection files are in {}'.format(tool, det_dir))
  return all_boxes, aps, names


def main(argv=None):
  eval_once(parse_flags(argv))


if __name__ == '__main__':
  main()
