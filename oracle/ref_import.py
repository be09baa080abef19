"""Import the reference's OWN numpy half, unmodified, from /root/reference
(oracle — test infrastructure only; dev container only — the path does not
exist on the GPU box, so nothing in ``-m gpu`` tests / smoke / bench calls this).

What imports and runs as-is under Python 3.12 once ``tensorflow`` and
``easydict`` are stubbed in ``sys.modules`` (SURVEY.md §8c):
  * ``utils.util.nms / batch_iou / iou``                 (src/utils/util.py:9-76)
  * ``nn_skeleton.ModelSkeleton.filter_prediction``      (src/nn_skeleton.py:696-734)
  * ``config.kitti_*_config()`` incl. ``set_anchors``    (src/config/*.py)
Used by ``tests/golden/make_golden.py``, which records the reference's outputs as the fixtures
under ``tests/golden/`` that ``tests/test_oracle_pinning.py`` checks the oracle against.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_SRC = '/root/reference/src'


def available() -> bool:
  return os.path.isfile(os.path.join(REFERENCE_SRC, 'nn_skeleton.py'))


class _EasyDict(dict):
  """Minimal stand-in for easydict.EasyDict (attribute access on a dict)."""

  def __getattr__(self, k):
    try:
      return self[k]
    except KeyError as e:
      raise AttributeError(k) from e

  def __setattr__(self, k, v):
    self[k] = v


_loaded = None


def load():
  """Returns a namespace with .util, .ModelSkeleton, .configs{name: fn}."""
  global _loaded
  if _loaded is not None:
    return _loaded
  if not available():
    raise RuntimeError('reference tree not present at ' + REFERENCE_SRC)
  saved_path = list(sys.path)
  saved_mods = {k: sys.modules.get(k) for k in
                ('tensorflow', 'easydict', 'config', 'utils', 'utils.util',
                 'nn_skeleton', 'joblib_stub')}
  try:
    if 'tensorflow' not in sys.modules:
      sys.modules['tensorflow'] = types.ModuleType('tensorflow')
    ed = types.ModuleType('easydict')
    ed.EasyDict = _EasyDict
    sys.modules['easydict'] = ed
    # config dir first so the py2 implicit-relative `from config import ...`
    # inside src/config/*.py resolves to src/config/config.py
    sys.path[:0] = [os.path.join(REFERENCE_SRC, 'config'), REFERENCE_SRC]
    for m in ('config', 'utils', 'utils.util', 'nn_skeleton'):
      sys.modules.pop(m, None)
    import importlib
    cfgs = {}
    for mod, fn in (('kitti_squeezeDet_config', 'kitti_squeezeDet_config'),
                    ('kitti_squeezeDetPlus_config', 'kitti_squeezeDetPlus_config'),
                    ('kitti_vgg16_config', 'kitti_vgg16_config'),
                    ('kitti_res50_config', 'kitti_res50_config')):
      cfgs[fn] = getattr(importlib.import_module(mod), fn)
    # src/utils/util.py and src/nn_skeleton.py (needs `from utils import util`)
    sys.modules.pop('config', None)      # src/config/config.py shadowed `config`
    sys.path[:2] = [REFERENCE_SRC]
    util = importlib.import_module('utils.util')
    nn = importlib.import_module('nn_skeleton')
    ns = types.SimpleNamespace(util=util, ModelSkeleton=nn.ModelSkeleton,
                               configs=cfgs, EasyDict=_EasyDict)
    _loaded = ns
    return ns
  finally:
    sys.path[:] = saved_path
    for k, v in saved_mods.items():
      if v is None:
        sys.modules.pop(k, None)
      else:
        sys.modules[k] = v


def ref_filter_prediction(ns, boxes, probs, cls_idx, classes, top_n,
                          prob_thresh, nms_thresh):
  """Call the reference's unbound ``ModelSkeleton.filter_prediction`` with a
  fake ``self`` that only carries ``.mc``."""
  mc = _EasyDict(CLASSES=classes, TOP_N_DETECTION=top_n,
                 PROB_THRESH=prob_thresh, NMS_THRESH=nms_thresh)
  fake = types.SimpleNamespace(mc=mc)
  return ns.ModelSkeleton.filter_prediction(fake, boxes, probs, cls_idx)
