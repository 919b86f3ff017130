"""Structure pins: the oracle's own walk (oracle/structure_oracle.py) and the product's
DetArch against what the REAL reference constructors resolve (tests/golden/structure.json.gz,
made by tests/golden/make_structure_golden.py from /root/reference under a recording
TensorFlow stand-in).  Covers every registered detector: block args per MBConv block
(efficientnet_builder.BlockDecoder strings + width/depth rounding), every Keras layer the
reference constructs (filters / kernel / stride / bias / name), BiFPN node lists."""
import gzip
import json
import os

import pytest

from automl_b200 import arch
from automl_b200 import hparams_config
from oracle import structure_oracle as so

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'structure.json.gz')
with gzip.open(GOLDEN) as _f:
  STRUCT = json.load(_f)
MODELS = sorted(k for k in STRUCT if not k.startswith('__'))


@pytest.mark.parametrize('name', MODELS)
def test_oracle_structure_equals_real_reference(name):
  c = hparams_config.get_efficientdet_config(name)
  ref = STRUCT[name]
  assert so.raw_block_args(c.backbone_name) == ref['blocks']
  assert so.layer_log(c) == ref['layers']
  nodes = so.bifpn_nodes(c.min_level, c.max_level)
  for cell in ref['fnodes']:
    assert [[lvl - c.min_level, offs] for lvl, offs in nodes] == [[n[0], n[1]] for n in cell]
    assert all(n[2] == c.fpn_weight_method or (n[2] == 'fastattn' and not c.fpn_weight_method)
               for n in cell)
    assert all(n[3] == c.fpn_num_filters for n in cell)
  assert len(ref['fnodes']) == c.fpn_cell_repeats
  assert [s for s in ref['scopes'] if s.startswith('blocks_')] == \
      [b['name'] for b in so.backbone_blocks(c.backbone_name)[1]]


@pytest.mark.parametrize('name', MODELS)
def test_product_arch_equals_oracle_structure(name):
  """The product's DetArch (what the CUDA engine lowers) agrees with the oracle's independent
  walk block by block: channels, strides, SE widths, skip, layer names, endpoints."""
  c = hparams_config.get_efficientdet_config(name)
  a = arch.DetArch(c)
  stem, blocks = so.backbone_blocks(c.backbone_name)
  assert a.stem_filters == stem and len(a.blocks) == len(blocks)
  for pb, ob in zip(a.blocks, blocks):
    assert (pb.name, pb.kernel_size, pb.stride) == (ob['name'], ob['kernel_size'], ob['stride'])
    assert (pb.input_filters, pb.mid_filters, pb.output_filters) == \
        (ob['in_channels'], ob['mid_channels'], ob['output_filters'])
    assert pb.se_filters == ob['se_channels'] and pb.has_skip == ob['has_skip']
    assert (pb.expand_name, pb.expand_bn, pb.dw_bn, pb.project_name, pb.project_bn) == \
        (ob['expand_conv'], ob['expand_bn'], ob['dw_bn'], ob['project_conv'], ob['project_bn'])
    assert pb.reduction == ob['reduction']
  nodes = so.bifpn_nodes(c.min_level, c.max_level)
  for cell in a.cells:
    assert [(n.feat_level, [r.src for r in n.inputs]) for n in cell['nodes']] == nodes
  sizes = so.feature_sizes(c.image_size, c.max_level)
  assert [a.level_hw[l] for l in range(c.max_level + 1)] == sizes


def test_feature_sizes_odd_and_strings():
  # utils_test.py:108-127 style cases
  assert so.feature_sizes(640, 2) == [(640, 640), (320, 320), (160, 160)]
  assert so.feature_sizes('1280x640', 2) == [(640, 1280), (320, 640), (160, 320)]   # 'WxH'
  assert so.feature_sizes((511, 513), 3) == [(511, 513), (256, 257), (128, 129), (64, 65)]


def _anchor_case_args(case):
  lo, hi, ns, ar, sc, size = case
  if isinstance(size, list):
    size = tuple(size)
  return lo, hi, ns, ar, sc, size


@pytest.mark.parametrize('row', STRUCT['__anchors__'], ids=lambda r: str(r['case'][-1]))
def test_anchors_equal_real_reference(row):
  """Oracle anchors and product anchors are bit-identical to the REAL tf2/anchors.py output."""
  import hashlib
  import numpy as np
  from automl_b200 import anchors as product_anchors
  args = _anchor_case_args(row['case'])
  got = so.anchor_boxes(*args)
  assert list(got.shape) == row['shape']
  assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == row['sha256']
  np.testing.assert_array_equal(got[::997], np.asarray(row['sample'], np.float32))
  prod = product_anchors.Anchors(*args)
  np.testing.assert_array_equal(prod.boxes, got)
  assert prod.get_anchors_per_location() == row['per_location']


def test_feat_sizes_equal_real_reference():
  for row in STRUCT['__feat_sizes__']:
    size = tuple(row['image_size']) if isinstance(row['image_size'], list) else row['image_size']
    assert [list(s) for s in so.feature_sizes(so.image_hw(size), row['max_level'])] == row['sizes']
