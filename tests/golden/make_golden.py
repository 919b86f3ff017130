"""Generates tests/golden/*.npz from the REAL reference modules that import without
TensorFlow in this container (SURVEY.md section 8c):

  /root/reference/efficientdet/nms_np.py          (numpy only)
  /root/reference/efficientdet/hparams_config.py  (with an empty `tensorflow` stub)
  /root/reference/efficientdet/tf2/fpn_configs.py (same stub)

Run from the repo root:  python tests/golden/make_golden.py
The GPU box has no /root/reference; tests there read the committed .npz / .json files.
"""
import json
import os
import sys
import types

import numpy as np

REF = '/root/reference/efficientdet'
OUT = os.path.dirname(os.path.abspath(__file__))
MAX_FILE_BYTES = 1000 * 1000


def _case_of(key):
  """Case index of a per-case array (`out_<case>_<method>`, `boxes_<case>`, ...), None otherwise."""
  parts = key.split('_')
  if parts[0] == 'out':
    return int(parts[1])
  return int(parts[-1]) if parts[-1].isdigit() else None


def save_split(name, arrays, groups):
  """Writes `arrays` as <name>.<i>.npz, part i holding the cases in groups[i] (arrays shared by
  all cases go with part 0), so that no file exceeds MAX_FILE_BYTES."""
  for i, cases in enumerate(groups):
    part = {k: v for k, v in arrays.items()
            if _case_of(k) in cases or (_case_of(k) is None and i == 0)}
    path = os.path.join(OUT, '%s.%d.npz' % (name, i))
    np.savez_compressed(path, **part)
    assert os.path.getsize(path) < MAX_FILE_BYTES, path


# cases per file of the per-class NMS fixtures (the 49 104-box cases fill a file of their own)
HARD_PARTS = [(0, 1, 2, 3, 4), (5, 6, 7, 8), (9,)]
SOFT_PARTS = [(0, 1, 2, 3, 4, 5), (6,)]


def write_nms_live(nms_np):
  """nms_np.nms on 3 / 64 / 400 boxes with evenly spread scores, every method
  (tests/test_oracle_pins.py::test_nms_np_live_against_reference)."""
  rng = np.random.default_rng(7)
  live = {}
  for k in (3, 64, 400):
    c = rng.uniform(0, 300, size=(k, 2))
    wh = rng.uniform(5, 120, size=(k, 2))
    dets = np.column_stack([c - wh / 2, c + wh / 2,
                            rng.permutation(np.linspace(0.01, 0.99, k))]).astype(np.float32)
    live['dets_%d' % k] = dets
    for method in ('hard', 'diou', 'gaussian', 'linear'):
      cfg = dict(method=method, iou_thresh=None, score_thresh=0.0, sigma=None)
      live['out_%d_%s' % (k, method)] = np.asarray(nms_np.nms(dets.copy(), cfg), np.float32)
  np.savez_compressed(os.path.join(OUT, 'nms_np_live.npz'), **live)


def import_reference():
  if 'tensorflow' not in sys.modules:
    sys.modules['tensorflow'] = types.ModuleType('tensorflow')  # only touched by yaml IO
  sys.path.insert(0, REF)
  import nms_np  # pylint: disable=g-import-not-at-top
  import hparams_config  # pylint: disable=g-import-not-at-top
  from tf2 import fpn_configs  # pylint: disable=g-import-not-at-top
  return nms_np, hparams_config, fpn_configs


def make_dets(rng, k, image=512.0, clusters=None):
  """COCO-shaped boxes [x1,y1,x2,y2,score] float32 with distinct scores."""
  if clusters:
    centres = rng.uniform(0, image, size=(clusters, 2))
    c = centres[rng.integers(0, clusters, size=k)] + rng.normal(0, 6.0, size=(k, 2))
  else:
    c = rng.uniform(0, image, size=(k, 2))
  wh = np.exp(rng.uniform(np.log(8), np.log(image / 2), size=(k, 2)))
  x1y1 = c - wh / 2
  x2y2 = c + wh / 2
  scores = 1.0 / (1.0 + np.exp(-rng.normal(-2.0, 2.0, size=k)))
  # make scores distinct in float32 (argsort tie order is implementation-defined)
  scores = np.unique(scores.astype(np.float32))
  while scores.size < k:
    extra = (1.0 / (1.0 + np.exp(-rng.normal(-2.0, 2.0, size=k)))).astype(np.float32)
    scores = np.unique(np.concatenate([scores, extra]))
  scores = rng.permutation(scores)[:k]
  return np.column_stack([x1y1, x2y2, scores]).astype(np.float32)


def make_dense_dets(rng, k, clusters, size=60.0, jitter=4.0, image=512.0):
  """Near-duplicate boxes around a few centres (heavy suppression), distinct float32 scores."""
  centres = rng.uniform(size, image - size, size=(clusters, 2))
  c = centres[rng.integers(0, clusters, size=k)] + rng.normal(0, jitter, size=(k, 2))
  wh = size + rng.normal(0, jitter, size=(k, 2))
  scores = np.unique(rng.uniform(0.01, 0.99, size=4 * k).astype(np.float32))
  scores = rng.permutation(scores)[:k]
  return np.column_stack([c - wh / 2, c + wh / 2, scores]).astype(np.float32)


def main():
  nms_np, hparams_config, fpn_configs = import_reference()
  rng = np.random.default_rng(20260922)

  # ---- nms_np goldens ---------------------------------------------------------------
  cases = {}
  methods = [
      dict(method='hard', iou_thresh=None, score_thresh=0.0, sigma=None),
      dict(method='hard', iou_thresh=0.3, score_thresh=0.0, sigma=None),
      dict(method='diou', iou_thresh=None, score_thresh=0.0, sigma=None),
      dict(method='gaussian', iou_thresh=None, score_thresh=0.0, sigma=None),
      dict(method='gaussian', iou_thresh=None, score_thresh=0.05, sigma=0.3),
      dict(method='linear', iou_thresh=None, score_thresh=0.0, sigma=None),
  ]
  for ci, (k, clusters) in enumerate([(1, None), (7, None), (100, 5), (1000, 40), (5000, 100)]):
    dets = make_dets(rng, k, clusters=clusters)
    for mi, cfg in enumerate(methods):
      out = nms_np.nms(dets.copy(), dict(cfg))
      cases['dets_%d' % ci] = dets
      cases['out_%d_%d' % (ci, mi)] = np.asarray(out, np.float32)
  cases['methods'] = np.asarray([json.dumps(m) for m in methods])
  np.savez_compressed(os.path.join(OUT, 'nms_np_nms.npz'), **cases)

  # per_class_nms goldens
  pc = {}
  for ci, k in enumerate([50, 600, 5000]):
    d = make_dets(rng, k, clusters=max(2, k // 40))
    boxes = d[:, [1, 0, 3, 2]].copy()  # [ymin,xmin,ymax,xmax] as produced by pre_nms
    scores = d[:, 4].copy()
    classes = rng.integers(0, 90, size=k).astype(np.int32)
    for mi, cfg in enumerate(methods[:1] + methods[3:4]):
      cfg = dict(cfg, max_output_size=100, pyfunc=True, max_nms_inputs=0)
      out = nms_np.per_class_nms(boxes, scores, classes, np.asarray([ci], np.float32),
                                 np.asarray([1.5], np.float32), 90, 100, cfg)
      pc['out_%d_%d' % (ci, mi)] = out
    pc['boxes_%d' % ci], pc['scores_%d' % ci], pc['classes_%d' % ci] = boxes, scores, classes
  np.savez_compressed(os.path.join(OUT, 'nms_np_per_class.npz'), **pc)

  # per_class_nms goldens for the CUDA replacement (hard / diou; tests/test_gpu_kernels.py):
  # many classes, few classes (long per-class lists), tight clusters (fewer than 100 survivors in
  # the top 2048 candidates -> several selection rounds on the device), fewer survivors than rows
  rng2 = np.random.default_rng(7051)
  hd = {}
  hd_cases = [(50, 90, None), (600, 90, 15), (5000, 90, 125), (20000, 90, 400), (6000, 3, 40),
              (12000, 2, 12), (3000, 1, 8)]
  hd_methods = [dict(method='hard', iou_thresh=None), dict(method='hard', iou_thresh=0.3),
                dict(method='diou', iou_thresh=None), dict(method='diou', iou_thresh=0.65)]
  hd_cases += [(8000, 1, -30), (20000, 2, -25), (49104, 90, -300)]   # negative: dense generator
  for ci, (k, ncls, clusters) in enumerate(hd_cases):
    d = make_dets(rng2, k, clusters=clusters) if clusters is None or clusters > 0 else \
        make_dense_dets(rng2, k, -clusters)
    boxes = d[:, [1, 0, 3, 2]].copy()
    scores = d[:, 4].copy()
    classes = rng2.integers(0, ncls, size=k).astype(np.int32)
    scale = np.asarray([0.75 + 0.25 * ci], np.float32)
    for mi, cfg in enumerate(hd_methods):
      cfg = dict(cfg, score_thresh=0.0, sigma=None, max_output_size=100, pyfunc=True, max_nms_inputs=0)
      hd['out_%d_%d' % (ci, mi)] = nms_np.per_class_nms(
          boxes, scores, classes, np.asarray([ci + 10], np.float32), scale, ncls, 100, cfg)
    hd['boxes_%d' % ci], hd['scores_%d' % ci], hd['classes_%d' % ci] = boxes, scores, classes
    hd['scale_%d' % ci], hd['ncls_%d' % ci] = scale, np.asarray(ncls)
  hd['methods'] = np.asarray([json.dumps(m) for m in hd_methods])
  save_split('nms_np_per_class_hard', hd, HARD_PARTS)

  # per_class_nms goldens for the soft methods (gaussian: NumPy's float32 exp is within 2 ulp of
  # the correctly rounded value and differs between CPUs, so the device is held to identical
  # indices / boxes / classes and scores within a few ulp; linear has no transcendental: bit-exact)
  rng3 = np.random.default_rng(9107)
  sf = {}
  sf_cases = [(50, 90, None), (600, 90, 15), (5000, 90, 125), (20000, 90, 400), (6000, 3, 40),
              (3000, 1, -8), (49104, 90, -300)]
  sf_methods = [dict(method='gaussian', iou_thresh=None, sigma=None, score_thresh=None),
                dict(method='gaussian', iou_thresh=None, sigma=0.3, score_thresh=0.05),
                dict(method='linear', iou_thresh=None, sigma=None, score_thresh=None),
                dict(method='linear', iou_thresh=0.5, sigma=None, score_thresh=0.01)]
  for ci, (k, ncls, clusters) in enumerate(sf_cases):
    d = make_dets(rng3, k, clusters=clusters) if clusters is None or clusters > 0 else \
        make_dense_dets(rng3, k, -clusters)
    boxes = d[:, [1, 0, 3, 2]].copy()
    scores = d[:, 4].copy()
    classes = rng3.integers(0, ncls, size=k).astype(np.int32)
    scale = np.asarray([0.5 + 0.25 * ci], np.float32)
    for mi, cfg in enumerate(sf_methods):
      cfg = dict(cfg, max_output_size=100, pyfunc=True, max_nms_inputs=0)
      sf['out_%d_%d' % (ci, mi)] = nms_np.per_class_nms(
          boxes, scores, classes, np.asarray([ci + 20], np.float32), scale, ncls, 100, cfg)
    sf['boxes_%d' % ci], sf['scores_%d' % ci], sf['classes_%d' % ci] = boxes, scores, classes
    sf['scale_%d' % ci], sf['ncls_%d' % ci] = scale, np.asarray(ncls)
  sf['methods'] = np.asarray([json.dumps(m) for m in sf_methods])
  save_split('nms_np_per_class_soft', sf, SOFT_PARTS)

  write_nms_live(nms_np)

  # ---- registry / fpn goldens ---------------------------------------------------------
  reg = {}
  names = (list(hparams_config.efficientdet_model_param_dict) +
           list(hparams_config.efficientdet_lite_param_dict))
  for n in names:
    reg[n] = hparams_config.get_efficientdet_config(n).as_dict()
  fpn = {}
  for lo, hi in [(3, 7), (2, 7), (3, 8)]:
    fpn['%d-%d' % (lo, hi)] = fpn_configs.bifpn_config(lo, hi, None).as_dict()
  with open(os.path.join(OUT, 'registry.json'), 'w') as f:
    json.dump({'configs': reg, 'bifpn': fpn}, f, indent=1, sort_keys=True)
  print('wrote goldens to', OUT)


if __name__ == '__main__':
  main()
