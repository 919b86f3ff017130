"""GPU parity tests: every CUDA entry point (called through the C-ABI) against the CPU oracle on
the same seeded inputs.  Integer / index outputs must match exactly; floating point within the
tolerance written next to each assert (fp16 storage, fp32 accumulation)."""
import numpy as np
import pytest
import torch

from automl_b200 import anchors as anchors_lib
from automl_b200 import utils
from oracle import efficientdet_oracle as eo
from oracle import postprocess_oracle as po
from test_oracle_pins import load_split_golden   # same directory (pytest prepends tests/ to sys.path)

pytestmark = pytest.mark.gpu

DEV = 'cuda:0'


def _ops():
  from automl_b200 import ops  # deferred: loads the CUDA library
  return ops


def rel_l2(a, b):
  a, b = a.double().flatten(), b.double().flatten()
  return float((a - b).norm() / max(float(b.norm()), 1e-30))


def act_ref(x, act):
  return {utils.ACT_NONE: lambda t: t, utils.ACT_SWISH: lambda t: t * torch.sigmoid(t),
          utils.ACT_RELU6: lambda t: torch.clamp(t, 0, 6)}[act](x)


# ---------------------------------------------------------------------------------------------
PW_CASES = [
    # batch, rows, k, nout, act, residual, per-image weights
    (1, 128, 64, 64, utils.ACT_NONE, False, False),
    (1, 1000, 16, 96, utils.ACT_SWISH, False, False),       # K < 64 (TMA zero fill), ragged M
    (1, 777, 24, 144, utils.ACT_SWISH, False, False),       # K not a multiple of 16
    (1, 4096, 144, 24, utils.ACT_NONE, True, False),        # project + skip
    (2, 400, 1152, 192, utils.ACT_NONE, True, True),        # SE-scaled weights, rows % 128 != 0
    (3, 100, 672, 112, utils.ACT_NONE, False, True),
    (1, 2048, 192, 1152, utils.ACT_SWISH, False, False),    # nout > 256 -> several N tiles
    (1, 640, 64, 810, utils.ACT_NONE, False, False),        # class-predict, nout % 8 != 0
    (1, 25, 64, 36, utils.ACT_NONE, False, False),          # box-predict on a 5x5 level
    (2, 6400, 40, 64, utils.ACT_NONE, False, False),
    (1, 50000, 32, 16, utils.ACT_NONE, False, False),       # many tiles per CTA (pipeline wrap)
    (1, 3000, 320, 64, utils.ACT_RELU6, False, False),
    # wide single-tile N with deep K (D3-D7x BiFPN / head widths): the shared-memory plan has to
    # fall back to one store slab / 32-wide k-blocks
    (1, 1000, 160, 160, utils.ACT_SWISH, False, False),
    (2, 700, 224, 224, utils.ACT_NONE, False, False),
    (1, 513, 256, 256, utils.ACT_SWISH, True, False),
    (1, 900, 384, 384, utils.ACT_NONE, False, False),        # N > 256: tiles of 96 columns
    (1, 260, 1344, 224, utils.ACT_NONE, True, True),        # D4-sized project
]


@pytest.mark.parametrize('impl_name', ['tcgen05', 'simt'])
@pytest.mark.parametrize('case', PW_CASES)
def test_pointwise_conv(case, impl_name):
  ops = _ops()
  impl = ops.PW_TCGEN05 if impl_name == 'tcgen05' else ops.PW_SIMT
  batch, rows, k, nout, act, has_res, per_image = case
  g = torch.Generator().manual_seed(1234 + rows + k + nout)
  a = torch.randn(batch, rows, k, generator=g).half()
  wb = batch if per_image else 1
  w = (torch.randn(wb, nout, k, generator=g) / np.sqrt(k)).half()
  bias = torch.randn(nout, generator=g)
  ldo = (nout + 7) // 8 * 8
  res = torch.randn(batch, rows, ldo, generator=g).half() if has_res else None
  out = torch.full((batch, rows, ldo), 7.0).half().to(DEV)
  ops.pointwise_conv(a.to(DEV), w.to(DEV), bias.to(DEV), out, act,
                     residual=res.to(DEV) if has_res else None, rows=rows, batch=batch, nout=nout,
                     impl=impl)
  torch.cuda.synchronize()
  ref = torch.einsum('brk,bnk->brn', a.double(), w.double().expand(batch, nout, k)) + bias.double()
  ref = act_ref(ref, act)
  if has_res:
    ref = ref + res[..., :nout].double()
  got = out.cpu()[..., :nout].double()
  # fp16 output rounding (2^-11 relative) + fp32 accumulation
  assert torch.allclose(got, ref, rtol=2e-3, atol=2e-3), float((got - ref).abs().max())
  assert rel_l2(got, ref) < 5e-4
  if ldo > nout:
    # padding columns: untouched by the SIMT kernel; the TMA store works in 16-byte units, so
    # the tensor-core kernel may write zeros (never garbage) into the <8 trailing pad columns.
    pad = out.cpu()[..., nout:]
    assert bool(((pad == 7.0) | (pad == 0.0)).all())


@pytest.mark.parametrize('case', PW_CASES + [
    (1, 5000, 16, 96, utils.ACT_SWISH, False, False),      # expand widths: 3 / 5 / 8 units of 32
    (2, 3000, 24, 144, utils.ACT_SWISH, False, False),
    (1, 2500, 40, 240, utils.ACT_SWISH, False, False),
    (1, 1500, 80, 480, utils.ACT_SWISH, False, False),     # tiles of 96 columns with three teams
    (1, 900, 112, 672, utils.ACT_SWISH, False, False),
    (1, 300, 64, 88, utils.ACT_SWISH, True, False),        # 88 = 2 units + a 24-column tail (16 + 8)
])
def test_pointwise_epilogue_teams_agree(case):
  """The two epilogue organisations of pointwise_tc_kernel (two teams x 64-column chunks, three
  teams x 32-column units) read the same accumulators and do the same fp32 epilogue arithmetic:
  bit-identical outputs."""
  ops = _ops()
  batch, rows, k, nout, act, has_res, per_image = case
  g = torch.Generator().manual_seed(4321 + rows + k + nout)
  a = torch.randn(batch, rows, k, generator=g).half().to(DEV)
  wb = batch if per_image else 1
  w = (torch.randn(wb, nout, k, generator=g) / np.sqrt(k)).half().to(DEV)
  bias = torch.randn(nout, generator=g).to(DEV)
  ldo = -(-nout // 8) * 8
  res = torch.randn(batch, rows, ldo, generator=g).half().to(DEV) if has_res else None
  outs = []
  try:
    for teams in (2, 3):
      ops.set_option('pw_teams', teams)
      out = torch.full((batch, rows, ldo), 7.0, dtype=torch.float16, device=DEV)
      ops.pointwise_conv(a, w if per_image else w[0], bias, out, act, residual=res, rows=rows,
                         batch=batch, nout=nout)
      torch.cuda.synchronize()
      outs.append(out)
  finally:
    ops.set_option('pw_teams', 0)
  assert torch.equal(outs[0], outs[1])
  ref = torch.einsum('brk,bnk->brn', a.float().cpu().double(), w.float().cpu().double().expand(batch, -1, -1))
  ref = act_ref(ref + bias.cpu().double(), act)
  if has_res:
    ref = ref + res[..., :nout].cpu().double()
  assert torch.allclose(outs[1][..., :nout].cpu().double(), ref, rtol=2e-3, atol=2e-3)
  if ldo > nout:   # pad columns: untouched, or zeros from the 16-byte granular TMA store
    pad = outs[1][..., nout:]
    assert bool(((pad == 7.0) | (pad == 0.0)).all())


# ---------------------------------------------------------------------------------------------
DW_CASES = [
    # n, h, w, c, k, s, act, bias, se
    (2, 40, 40, 96, 3, 1, utils.ACT_SWISH, True, True),
    (1, 33, 47, 32, 3, 2, utils.ACT_SWISH, True, True),     # odd sizes, asymmetric SAME pad
    (2, 20, 20, 240, 5, 1, utils.ACT_SWISH, True, True),
    (1, 31, 29, 144, 5, 2, utils.ACT_SWISH, True, True),
    (2, 10, 10, 64, 3, 1, utils.ACT_NONE, False, False),    # head / BiFPN depthwise half
    (1, 5, 5, 64, 3, 1, utils.ACT_NONE, False, False),
    (1, 64, 64, 1152, 5, 1, utils.ACT_SWISH, True, True),
    (1, 12, 12, 672, 5, 2, utils.ACT_RELU6, True, False),
    # maps large enough for the TMA-tiled kernel (depthwise_tile.cu): ragged tiles in x and y,
    # channel counts that are not multiples of the 64-channel slice, every (k, stride)
    (2, 50, 70, 144, 3, 1, utils.ACT_SWISH, True, True),
    (1, 67, 45, 240, 5, 1, utils.ACT_SWISH, True, True),
    (2, 61, 83, 96, 3, 2, utils.ACT_SWISH, True, True),
    (1, 97, 59, 144, 5, 2, utils.ACT_SWISH, True, True),
    (3, 48, 48, 64, 3, 1, utils.ACT_NONE, False, False),    # head depthwise at level 3 size
    (1, 80, 80, 672, 5, 1, utils.ACT_RELU6, True, True),
    (1, 160, 160, 72, 5, 2, utils.ACT_RELU6, True, False),  # c % 16 != 0
    (2, 33, 200, 480, 3, 1, utils.ACT_NONE, True, False),   # many work units per CTA (ring wrap)
]


@pytest.mark.parametrize('case', DW_CASES)
def test_depthwise_conv(case):
  ops = _ops()
  n, h, w, c, k, s, act, has_bias, has_se = case
  g = torch.Generator().manual_seed(99 + h + c + k)
  x = torch.randn(n, h, w, c, generator=g).half()
  wk = (torch.randn(k, k, c, generator=g) / k).half()
  bias = torch.randn(c, generator=g) * 0.1 if has_bias else None
  ho, wo = -(-h // s), -(-w // s)
  out = torch.empty(n, ho, wo, c, dtype=torch.float16, device=DEV)
  partial = None
  if has_se:
    partial = torch.zeros(n, c, dtype=torch.int64, device=DEV)   # 2^-20 fixed-point sums
  ops.depthwise_conv(x.to(DEV), out, wk.reshape(k * k, c).float().to(DEV),
                     bias.to(DEV) if has_bias else None, act, k, s, partial)
  torch.cuda.synchronize()
  ref = eo.depthwise_conv2d_same(x.double().permute(0, 3, 1, 2), wk.double().unsqueeze(-1), s)
  if has_bias:
    ref = ref + bias.double().view(1, -1, 1, 1)
  ref = act_ref(ref, act).permute(0, 2, 3, 1)
  got = out.cpu().double()
  assert got.shape == ref.shape
  assert torch.allclose(got, ref, rtol=2e-3, atol=2e-3), float((got - ref).abs().max())
  if has_se:
    sums = partial.cpu().double() / 2.0**20
    np.testing.assert_allclose(sums.numpy(), ref.sum((1, 2)).numpy(), rtol=1e-4, atol=1e-3)
    # the squeeze is order independent: a second run gives the identical integers
    again = torch.zeros_like(partial)
    ops.depthwise_conv(x.to(DEV), out, wk.reshape(k * k, c).float().to(DEV),
                       bias.to(DEV) if has_bias else None, act, k, s, again)
    torch.cuda.synchronize()
    assert torch.equal(again, partial)


@pytest.mark.parametrize('case', [c for c in DW_CASES if c[1] >= 48 and c[3] >= 64])
def test_depthwise_tiled_equals_register_kernel(case):
  """The two depthwise implementations (TMA-tiled / register-tiled) do the same fp32 arithmetic in
  the same order: their fp16 outputs are bit-identical and the SE sums agree to the fixed-point
  rounding of the per-thread partial sums."""
  ops = _ops()
  n, h, w, c, k, s, act, has_bias, has_se = case
  g = torch.Generator().manual_seed(7 + h + c)
  x = torch.randn(n, h, w, c, generator=g).half().to(DEV)
  wk = (torch.randn(k * k, c, generator=g) / k).to(DEV)   # fp32 taps
  bias = (torch.randn(c, generator=g) * 0.1).to(DEV) if has_bias else None
  ho, wo = -(-h // s), -(-w // s)
  outs, sums = [], []
  try:
    for impl in (0, 1):
      ops.set_option('dw_impl', impl)
      assert ops.get_option('dw_impl') == impl
      out = torch.empty(n, ho, wo, c, dtype=torch.float16, device=DEV)
      part = torch.zeros(n, c, dtype=torch.int64, device=DEV) if has_se else None
      ops.depthwise_conv(x, out, wk, bias, act, k, s, part)
      torch.cuda.synchronize()
      outs.append(out)
      sums.append(part)
  finally:
    ops.set_option('dw_impl', 0)
  assert torch.equal(outs[0], outs[1])
  if has_se:
    # each partial sum is rounded to 2^-20 once: |difference| <= (number of partial sums) * 2^-20
    assert int((sums[0] - sums[1]).abs().max()) <= ho * wo
    np.testing.assert_allclose(sums[0].cpu().double().numpy(), sums[1].cpu().double().numpy(),
                               rtol=1e-5, atol=64)


# n, h, w, cin, cmid, k, stride, act, has_se   (D0 blocks 1-5 shapes at small sizes + edge cases)
MBF_CASES = [
    (2, 40, 40, 16, 96, 3, 2, utils.ACT_SWISH, True),     # block 1: one chunk, 32B swizzle
    (2, 33, 29, 24, 144, 3, 1, utils.ACT_SWISH, True),    # block 2: two chunks (80 + 64), K pad 24 -> 32
    (1, 37, 41, 24, 144, 5, 2, utils.ACT_SWISH, True),    # block 3
    (2, 20, 20, 40, 240, 5, 1, utils.ACT_SWISH, True),    # block 4: two k-blocks of 32
    (1, 23, 17, 40, 240, 3, 2, utils.ACT_RELU6, False),   # block 5 (lite flavour)
    (1, 16, 16, 80, 480, 3, 1, utils.ACT_SWISH, True),    # 4 chunks, 128B swizzle, two k-blocks
    (1, 5, 7, 16, 96, 5, 1, utils.ACT_SWISH, True),       # image smaller than one patch
    (3, 64, 64, 16, 96, 3, 2, utils.ACT_SWISH, True),     # several full tiles per image
]


@pytest.mark.parametrize('case', MBF_CASES)
def test_mbconv_expand_dw(case):
  ops = _ops()
  n, h, w, cin, cmid, k, s, act, has_se = case
  g = torch.Generator().manual_seed(7 + h + cmid + k)
  x = torch.randn(n, h, w, cin, generator=g).half()
  we = (torch.randn(cmid, cin, generator=g) / cin**0.5).half()
  be = torch.randn(cmid, generator=g) * 0.2
  wk = (torch.randn(k, k, cmid, generator=g) / k).half()
  bd = torch.randn(cmid, generator=g) * 0.1
  ho, wo = -(-h // s), -(-w // s)
  out = torch.full((n, ho, wo, cmid), 7.0, dtype=torch.float16, device=DEV)
  se = torch.zeros(n, cmid, dtype=torch.int64, device=DEV) if has_se else None
  args = (x.to(DEV), we.to(DEV), be.to(DEV), wk.reshape(k * k, cmid).float().to(DEV), bd.to(DEV))
  ops.mbconv_expand_dw(*args, out, act, k, s, se)
  torch.cuda.synchronize()
  # reference: the expanded map is an fp16 tensor (as in the unfused pipeline)
  e = act_ref(x.double() @ we.double().t() + be.double(), act).half().double()
  ref = eo.depthwise_conv2d_same(e.permute(0, 3, 1, 2), wk.double().unsqueeze(-1), s)
  ref = act_ref(ref + bd.double().view(1, -1, 1, 1), act).permute(0, 2, 3, 1)
  got = out.cpu().double()
  assert torch.allclose(got, ref, rtol=2e-3, atol=2e-3), float((got - ref).abs().max())
  if has_se:
    sums = se.cpu().double() / 2.0**20
    np.testing.assert_allclose(sums.numpy(), ref.sum((1, 2)).numpy(), rtol=1e-3, atol=0.05)
    again = torch.zeros_like(se)
    ops.mbconv_expand_dw(*args, out, act, k, s, again)
    torch.cuda.synchronize()
    assert torch.equal(again, se)


@pytest.mark.parametrize('shape', [(3, 96, 4, 24), (2, 144, 6, 24), (2, 1152, 48, 320),
                                   (2, 3840, 160, 640),    # D7x at batch 2: 8 warps share an output
                                   (2, 1000, 40, 64),      # ragged channel slices (4 warps)
                                   (32, 672, 28, 112)])    # D0 batch 32: one warp per output
def test_se_fc(shape):
  ops = _ops()
  n, c, se, nout = shape
  g = torch.Generator().manual_seed(5)
  sums = torch.randn(n, c, generator=g) * 20
  se_sum = torch.round(sums.double() * 2.0**20).to(torch.int64)
  nxt = torch.full((n, max(1160, c)), 123, dtype=torch.int64, device=DEV)
  w1, b1 = torch.randn(se, c, generator=g) * 2.0 / c**0.5, torch.randn(se, generator=g) * 0.1
  w2, b2 = torch.randn(c, se, generator=g) * 0.5, torch.randn(c, generator=g) * 0.1
  wt = torch.randn(nout, c, generator=g).half()
  gate = torch.empty(n, c, device=DEV)
  wt_scaled = torch.empty(n, nout, c, dtype=torch.float16, device=DEV)
  inv_hw = 1.0 / 50.0
  ops.se_fc(se_sum.to(DEV), inv_hw, w1.to(DEV), b1.to(DEV), w2.T.contiguous().to(DEV), b2.to(DEV), gate,
            utils.ACT_SWISH, wt.to(DEV), wt_scaled, nxt)
  torch.cuda.synchronize()
  assert int(nxt.abs().sum()) == 0          # the next block's accumulator was cleared
  mean = se_sum.double() / 2.0**20 * inv_hw
  r = mean @ w1.double().T + b1.double()
  r = r * torch.sigmoid(r)
  ref_gate = torch.sigmoid(r @ w2.double().T + b2.double())
  np.testing.assert_allclose(gate.cpu().double().numpy(), ref_gate.numpy(), rtol=1e-5, atol=1e-6)
  ref_w = wt.double()[None] * ref_gate[:, None, :]
  assert torch.allclose(wt_scaled.cpu().double(), ref_w, rtol=1e-3, atol=1e-4)


@pytest.mark.parametrize('impl', ['tensor_core', 'cuda_core'])
@pytest.mark.parametrize('hw,cout,n', [((64, 64), 32, 2), ((33, 47), 48, 2), ((8, 8), 64, 1),
                                      ((127, 129), 40, 1), ((200, 96), 56, 3), ((5, 3), 24, 1)])
def test_stem_conv(hw, cout, n, impl):
  """Both stem kernels (implicit GEMM on tcgen05 with the float32 input split into fp16 hi + lo;
  CUDA-core FFMA2) against the float64 oracle: even / odd sizes (asymmetric 'SAME' padding),
  widths that are not multiples of 16 (N padding), several tiles per CTA."""
  ops = _ops()
  h, w = hw
  g = torch.Generator().manual_seed(3 + h + cout)
  x = torch.randn(n, h, w, 3, generator=g) * 1.7
  k = (torch.randn(3, 3, 3, cout, generator=g) * 0.3).half()
  bias = torch.randn(cout, generator=g) * 0.1
  out = torch.empty(n, -(-h // 2), -(-w // 2), cout, dtype=torch.float16, device=DEV)
  try:
    ops.set_option('stem_impl', 0 if impl == 'tensor_core' else 1)
    ops.stem_conv(x.to(DEV), out, k.reshape(27, cout).to(DEV), bias.to(DEV), utils.ACT_SWISH)
    torch.cuda.synchronize()
  finally:
    ops.set_option('stem_impl', 0)
  ref = eo.conv2d_same(x.double().permute(0, 3, 1, 2), k.double(), stride=2) + bias.double().view(1, -1, 1, 1)
  ref = (ref * torch.sigmoid(ref)).permute(0, 2, 3, 1)
  got = out.cpu().double()
  assert torch.allclose(got, ref, rtol=2e-3, atol=2e-3), float((got - ref).abs().max())
  assert rel_l2(got, ref) < 4e-4          # one fp16 output rounding; the input keeps ~22 bits


# ---------------------------------------------------------------------------------------------
def test_fuse_dw_all_modes():
  """One node with an identity input, a nearest-upsampled input and a max-pooled input."""
  ops = _ops()
  n, c = 2, 88
  for (h, w) in [(20, 20), (13, 9)]:
    g = torch.Generator().manual_seed(h * 100 + w)
    uh, uw = (h - 1) // 2 + 1, (w - 1) // 2 + 1          # coarser level -> upsample
    dh, dw = h * 2 - (h % 2), w * 2 - (w % 2)            # finer level  -> max-pool 3x3 s2
    assert -(-dh // 2) == h and -(-dw // 2) == w
    same = torch.randn(n, h, w, c, generator=g).half()
    up = torch.randn(n, uh, uw, c, generator=g).half()
    down = torch.randn(n, dh, dw, c, generator=g).half()
    wts = [0.5, 0.3, 0.2]
    dwk = (torch.randn(3, 3, c, generator=g) / 3).half()
    out = torch.empty(n, h, w, c, dtype=torch.float16, device=DEV)
    specs = [(same.to(DEV), ops.RS_SAME, None, wts[0]), (up.to(DEV), ops.RS_UP, None, wts[1]),
             (down.to(DEV), ops.RS_DOWN, (3, 3, 2, 2), wts[2])]
    ops.fuse_dw(specs, dwk.reshape(9, c).float().to(DEV), out, utils.ACT_SWISH)
    torch.cuda.synchronize()
    nchw = lambda t: t.double().permute(0, 3, 1, 2)
    fused = (nchw(same) * np.float32(wts[0]) + eo.resize_nearest_tf1(nchw(up), h, w) * np.float32(wts[1]) +
             eo.max_pool_same(nchw(down), (3, 3), (2, 2)) * np.float32(wts[2]))
    fused = fused * torch.sigmoid(fused)
    ref = eo.depthwise_conv2d_same(fused, dwk.double().unsqueeze(-1)).permute(0, 2, 3, 1)
    assert torch.allclose(out.cpu().double(), ref, rtol=2e-3, atol=2e-3), (h, w)


@pytest.mark.parametrize('sig', ['same_up', 'same_same_down', 'same_down'])
@pytest.mark.parametrize('hw', [(20, 20), (13, 9), (40, 24), (5, 5)])
def test_fuse_dw_bifpn_signatures(sig, hw):
  """The three node shapes of a BiFPN cell run specialised instantiations (all input loads
  issued up front; padded max-pool cells replaced by a clamped in-window tap): same results as
  the oracle's resample / fuse / swish / depthwise on odd and even sizes."""
  ops = _ops()
  n, c = 2, 64
  h, w = hw
  g = torch.Generator().manual_seed(h * 31 + w + len(sig))
  uh, uw = (h - 1) // 2 + 1, (w - 1) // 2 + 1
  dh, dw = h * 2 - (h % 2), w * 2 - (w % 2)
  mk = lambda hh, ww: torch.randn(n, hh, ww, c, generator=g).half()
  nchw = lambda t: t.double().permute(0, 3, 1, 2)
  if sig == 'same_up':
    tens = [mk(h, w), mk(uh, uw)]
    modes = [(ops.RS_SAME, None), (ops.RS_UP, None)]
    res = [nchw(tens[0]), eo.resize_nearest_tf1(nchw(tens[1]), h, w)]
  elif sig == 'same_same_down':
    tens = [mk(h, w), mk(h, w), mk(dh, dw)]
    modes = [(ops.RS_SAME, None), (ops.RS_SAME, None), (ops.RS_DOWN, (3, 3, 2, 2))]
    res = [nchw(tens[0]), nchw(tens[1]), eo.max_pool_same(nchw(tens[2]), (3, 3), (2, 2))]
  else:
    tens = [mk(h, w), mk(dh, dw)]
    modes = [(ops.RS_SAME, None), (ops.RS_DOWN, (3, 3, 2, 2))]
    res = [nchw(tens[0]), eo.max_pool_same(nchw(tens[1]), (3, 3), (2, 2))]
  wts = [0.45, 0.35, 0.2][:len(tens)]
  dwk = (torch.randn(3, 3, c, generator=g) / 3).half()
  out = torch.empty(n, h, w, c, dtype=torch.float16, device=DEV)
  specs = [(t.to(DEV), m, pool, wt) for t, (m, pool), wt in zip(tens, modes, wts)]
  ops.fuse_dw(specs, dwk.reshape(9, c).float().to(DEV), out, utils.ACT_SWISH)
  torch.cuda.synchronize()
  fused = sum(r * np.float32(wt) for r, wt in zip(res, wts))
  fused = fused * torch.sigmoid(fused)
  ref = eo.depthwise_conv2d_same(fused, dwk.double().unsqueeze(-1)).permute(0, 2, 3, 1)
  assert torch.allclose(out.cpu().double(), ref, rtol=2e-3, atol=2e-3), (sig, hw)


CONV_CASES = [
    # n, h, w, cin, cout, k, stride, act, residual      (EfficientNetV2-S fused stages + edges)
    (2, 24, 24, 24, 24, 3, 1, utils.ACT_SWISH, True),      # stage 0: single 3x3 conv + act + skip
    (2, 24, 24, 24, 96, 3, 2, utils.ACT_SWISH, False),     # stage 1 first block: 3x3 s2 expand
    (1, 17, 23, 48, 192, 3, 1, utils.ACT_SWISH, False),    # stage 1 repeat: odd sizes, N = 192
    (1, 19, 13, 48, 192, 3, 2, utils.ACT_SWISH, False),    # stride 2 on odd sizes
    (2, 12, 12, 64, 256, 3, 1, utils.ACT_SWISH, False),    # stage 2: N = 256 (one accum stage)
    (1, 40, 56, 32, 32, 3, 1, utils.ACT_NONE, True),       # several tiles, 64B swizzle K
    (1, 9, 9, 160, 320, 3, 1, utils.ACT_RELU6, False),     # 3 k-blocks x 9 taps, 3 N tiles
    (1, 10, 14, 16, 40, 5, 2, utils.ACT_NONE, False),      # 5x5 stride 2
    (3, 64, 64, 24, 24, 3, 1, utils.ACT_SWISH, True),      # persistent loop over many tiles
]


@pytest.mark.parametrize('case', CONV_CASES)
def test_conv2d_tc(case):
  ops = _ops()
  n, h, w, cin, cout, k, s, act, has_res = case
  g = torch.Generator().manual_seed(17 + h + cin + cout)
  x = torch.randn(n, h, w, cin, generator=g).half()
  wk = (torch.randn(k, k, cin, cout, generator=g) / (k * cin**0.5)).half()     # HWIO like Keras
  bias = torch.randn(cout, generator=g) * 0.1
  ho, wo = -(-h // s), -(-w // s)
  res = torch.randn(n, ho, wo, cout, generator=g).half() if has_res else None
  out = torch.full((n, ho, wo, cout), 7.0, dtype=torch.float16, device=DEV)
  wt = wk.permute(0, 1, 3, 2).reshape(k * k, cout, cin).contiguous()            # [tap][cout][cin]
  ops.conv2d(x.to(DEV), wt.to(DEV), bias.to(DEV), out, act, k, s,
             residual=res.to(DEV) if has_res else None)
  torch.cuda.synchronize()
  ref = eo.conv2d_same(x.double().permute(0, 3, 1, 2), wk.double(), s) + bias.double().view(1, -1, 1, 1)
  ref = act_ref(ref, act).permute(0, 2, 3, 1)
  if has_res:
    ref = ref + res.double()
  got = out.cpu().double()
  assert got.shape == ref.shape
  assert rel_l2(got, ref) < 6e-4, rel_l2(got, ref)
  assert torch.allclose(got, ref, rtol=4e-3, atol=4e-3), float((got - ref).abs().max())


SEP_CASES = [
    # n, (h, w), c, nout, pre, post, inputs [(mode, (h, w))]
    (1, (13, 21), 88, 88, utils.ACT_NONE, utils.ACT_SWISH, ['same']),              # D1 width, 2 atoms
    (2, (5, 5), 64, 64, utils.ACT_NONE, utils.ACT_SWISH, ['same']),                # tower layer, tiny level
    (1, (40, 40), 64, 64, utils.ACT_NONE, utils.ACT_SWISH, ['same']),              # several tiles per CTA
    (1, (9, 17), 112, 112, utils.ACT_NONE, utils.ACT_RELU6, ['same']),             # D2 width
    (3, (80, 80), 64, 64, utils.ACT_NONE, utils.ACT_SWISH, ['same']),              # persistent loop
    (2, (33, 47), 64, 64, utils.ACT_NONE, utils.ACT_SWISH, ['same']),              # ragged tiles (TMA zero fill)
    (1, (17, 9), 48, 48, utils.ACT_NONE, utils.ACT_RELU6, ['same']),               # c < 64: box wider than the tensor
    (2, (24, 24), 64, 40, utils.ACT_NONE, utils.ACT_NONE, ['same']),               # nout != c
]


@pytest.mark.parametrize('impl', [0, 1, 2])
@pytest.mark.parametrize('case', SEP_CASES)
def test_sepconv(case, impl):
  """edet_sepconv (a head tower layer: depthwise 3x3 + pointwise in one kernel) == edet_fuse_dw +
  edet_pointwise_conv bit for bit (same fp16 rounding of the depthwise result), and both match
  the float64 restatement.  impl 0 / 1: input tile staged by TMA / loaded straight from global
  memory / staged by TMA in a single buffer (four CTAs per SM)."""
  ops = _ops()
  n, (h, w), c, nout, pre, post, modes = case
  ops.set_option('sepconv_impl', impl)
  g = torch.Generator().manual_seed(31 + h + c)
  specs, ref_in = [], []
  wsum = float(len(modes))
  for i, m in enumerate(modes):
    if m == 'same':
      hh, ww, pool = h, w, None
    elif m == 'up':
      hh, ww, pool = -(-h // 2), -(-w // 2), None
    else:
      hh, ww, pool = h * 2 - (h % 2), w * 2 - (w % 2), (3, 3, 2, 2)
    t = torch.randn(n, hh, ww, c, generator=g).half()
    wgt = (i + 1.0) / (wsum * (wsum + 1) / 2)
    specs.append((t.to(DEV), {'same': ops.RS_SAME, 'up': ops.RS_UP, 'down': ops.RS_DOWN}[m], pool, wgt))
    ref_in.append((t, m, wgt))
  dw_w = (torch.randn(9, c, generator=g) / 3).half()
  pw = (torch.randn(nout, c, generator=g) / c**0.5).half()
  bias = torch.randn(nout, generator=g) * 0.1
  ldo = nout + 8
  out = torch.full((n, h, w, ldo), 7.0, dtype=torch.float16, device=DEV)
  ops.sepconv(specs, pre, dw_w.float().to(DEV), pw.to(DEV), bias.to(DEV), out, post, nout=nout)
  tmp = torch.empty(n, h, w, c, dtype=torch.float16, device=DEV)
  two = torch.full((n, h, w, ldo), 7.0, dtype=torch.float16, device=DEV)
  ops.fuse_dw(specs, dw_w.float().to(DEV), tmp, pre)
  ops.pointwise_conv(tmp, pw.to(DEV), bias.to(DEV), two, post, rows=n * h * w, nout=nout)
  torch.cuda.synchronize()
  ops.set_option('sepconv_impl', 0)
  assert torch.equal(out[..., :nout], two[..., :nout])
  assert bool((out[..., nout:] == 7.0).all())       # the padding columns are not touched
  # float64 restatement
  fused = 0
  for t, m, wgt in ref_in:
    x = t.double().permute(0, 3, 1, 2)
    if m == 'up':
      x = eo.resize_nearest_tf1(x, h, w)
    elif m == 'down':
      x = eo.max_pool_same(x, (3, 3), (2, 2))
    fused = fused + x * float(np.float32(wgt))
  fused = act_ref(fused, pre)
  d = eo.depthwise_conv2d_same(fused, dw_w.double().view(3, 3, c, 1), 1).permute(0, 2, 3, 1)
  ref = act_ref(d.half().double() @ pw.double().t() + bias.double(), post)
  got = out[..., :nout].cpu().double()
  assert torch.allclose(got, ref, rtol=3e-3, atol=3e-3), float((got - ref).abs().max())


def test_max_pool():
  ops = _ops()
  for (h, w) in [(20, 20), (5, 5), (13, 9)]:
    x = torch.randn(2, h, w, 64, generator=torch.Generator().manual_seed(h)).half()
    out = torch.empty(2, -(-h // 2), -(-w // 2), 64, dtype=torch.float16, device=DEV)
    ops.max_pool(x.to(DEV), out, (3, 3), (2, 2))
    torch.cuda.synchronize()
    ref = eo.max_pool_same(x.permute(0, 3, 1, 2).float(), (3, 3), (2, 2)).permute(0, 2, 3, 1)
    assert torch.equal(out.cpu().float(), ref)      # max of fp16 values is exact


# ---------------------------------------------------------------------------------------------
def _synthetic_head_outputs(rng, n, image_size, min_level=3, max_level=7, a=9, c=90):
  fs = utils.get_feat_sizes(image_size, max_level)
  cls, box = [], []
  for l in range(min_level, max_level + 1):
    h, w = fs[l]['height'], fs[l]['width']
    cls.append(rng.normal(-4.0, 2.0, size=(n, h, w, a * c)).astype(np.float16))
    box.append(rng.normal(0.0, 0.5, size=(n, h, w, a * 4)).astype(np.float16))
  return cls, box


def _params(image_size, method='gaussian', **nms_over):
  nms = {'method': method, 'iou_thresh': None, 'score_thresh': 0., 'sigma': None,
         'pyfunc': False, 'max_nms_inputs': 0, 'max_output_size': 100}
  nms.update(nms_over)
  return {'min_level': 3, 'max_level': 7, 'num_scales': 3, 'aspect_ratios': [1.0, 2.0, 0.5],
          'anchor_scale': 4.0, 'image_size': image_size, 'num_classes': 90,
          'data_format': 'channels_last', 'nms_configs': nms}


def _pad_ld(arr, ld):
  out = np.zeros(arr.shape[:-1] + (ld,), arr.dtype)
  out[..., :arr.shape[-1]] = arr
  return out


@pytest.mark.parametrize('image_size', [128, (96, 160)])
def test_pre_nms(image_size):
  ops = _ops()
  rng = np.random.default_rng(11)
  n = 2
  cls, box = _synthetic_head_outputs(rng, n, image_size)
  params = _params(image_size)
  ref_boxes, ref_scores, ref_classes = po.pre_nms(params, cls, box)
  anc = anchors_lib.Anchors(3, 7, 3, [1.0, 2.0, 0.5], 4.0, image_size).boxes
  k = anc.shape[0]
  cls_d = [torch.from_numpy(_pad_ld(t, 816)).to(DEV) for t in cls]
  box_d = [torch.from_numpy(_pad_ld(t, 40)).to(DEV) for t in box]
  boxes = torch.empty(n, k, 4, device=DEV)
  scores = torch.empty(n, k, device=DEV)
  classes = torch.empty(n, k, dtype=torch.int32, device=DEV)
  hw = [(t.shape[1], t.shape[2]) for t in cls]
  ops.pre_nms(cls_d, box_d, hw, 9, 90, torch.from_numpy(anc).to(DEV), boxes, scores, classes)
  torch.cuda.synchronize()
  np.testing.assert_array_equal(classes.cpu().numpy(), ref_classes)          # bit-exact indices
  np.testing.assert_allclose(scores.cpu().numpy(), ref_scores, rtol=1e-6, atol=1e-7)
  np.testing.assert_allclose(boxes.cpu().numpy(), ref_boxes, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize('image_size,topk', [(128, 1000), ((96, 160), 5000), (64, 8192)])
def test_pre_nms_topk(image_size, topk):
  """max_nms_inputs > 0 (postprocess.py:88-102): the top-k (anchor, class) pairs.  fp16 logits
  tie massively at the threshold, so this also checks the lower-flat-index tie rule."""
  ops = _ops()
  rng = np.random.default_rng(13)
  n = 2
  cls, box = _synthetic_head_outputs(rng, n, image_size)
  params = _params(image_size, max_nms_inputs=topk)
  ref_boxes, ref_scores, ref_classes = po.pre_nms(params, cls, box)
  anc = anchors_lib.Anchors(3, 7, 3, [1.0, 2.0, 0.5], 4.0, image_size).boxes
  cls_d = [torch.from_numpy(_pad_ld(t, 816)).to(DEV) for t in cls]
  box_d = [torch.from_numpy(_pad_ld(t, 40)).to(DEV) for t in box]
  boxes = torch.empty(n, topk, 4, device=DEV)
  scores = torch.empty(n, topk, device=DEV)
  classes = torch.empty(n, topk, dtype=torch.int32, device=DEV)
  indices = torch.empty(n, topk, dtype=torch.int32, device=DEV)
  hw = [(t.shape[1], t.shape[2]) for t in cls]
  ops.pre_nms_topk(cls_d, box_d, hw, 9, 90, torch.from_numpy(anc).to(DEV), boxes, scores, classes, indices)
  torch.cuda.synchronize()
  np.testing.assert_array_equal(classes.cpu().numpy(), ref_classes)
  np.testing.assert_allclose(scores.cpu().numpy(), ref_scores, rtol=1e-6, atol=1e-7)
  np.testing.assert_allclose(boxes.cpu().numpy(), ref_boxes, rtol=1e-5, atol=1e-4)
  # the anchor index of every row (the oracle's `indices`)
  flat = np.concatenate([c.reshape(n, -1, 90) for c in cls], axis=1).astype(np.float32).reshape(n, -1)
  order = np.lexsort((np.arange(flat.shape[1])[None].repeat(n, 0), -flat), axis=-1)[:, :topk]
  np.testing.assert_array_equal(indices.cpu().numpy(), order // 90)


def _nms_inputs(rng, n, k, image=512.0, clustered=True):
  if clustered:
    centres = rng.uniform(0, image, size=(n, 40, 2))
    pick = rng.integers(0, 40, size=(n, k))
    c = np.take_along_axis(centres, pick[..., None].repeat(2, -1), 1) + rng.normal(0, 8, size=(n, k, 2))
  else:
    c = rng.uniform(0, image, size=(n, k, 2))
  wh = np.exp(rng.uniform(np.log(8), np.log(image / 2), size=(n, k, 2)))
  boxes = np.concatenate([c - wh / 2, c + wh / 2], -1).astype(np.float32)   # [ymin,xmin,ymax,xmax]
  scores = (1 / (1 + np.exp(-rng.normal(-3, 2, size=(n, k))))).astype(np.float32)
  classes = rng.integers(0, 90, size=(n, k)).astype(np.int32)
  return boxes, scores, classes


@pytest.mark.parametrize('method,k', [('gaussian', 3000), ('hard', 3000), ('gaussian', 20000),
                                      ('hard', 49104), ('gaussian', 64)])
def test_nms_v5_bit_exact(method, k):
  ops = _ops()
  rng = np.random.default_rng(k + len(method))
  n = 3
  boxes, scores, classes = _nms_inputs(rng, n, k)
  if method == 'hard':   # exercise exact ties: duplicate scores and boxes
    scores[:, 1::7] = scores[:, 0:1]
    boxes[:, 5] = boxes[:, 4]
  params = _params(512, method=method, score_thresh=0.0 if method == 'gaussian' else None)
  iou_t, score_t, tf_sigma = po.nms_v5_params(params['nms_configs'])
  scales = np.asarray([1.0, 1.5, 0.75], np.float32)
  det = torch.empty(n, 100, 7, device=DEV)
  sel = torch.empty(n, 100, dtype=torch.int32, device=DEV)
  valid = torch.empty(n, dtype=torch.int32, device=DEV)
  work = torch.empty(ops.nms_work_bytes(n, k), dtype=torch.uint8, device=DEV)
  ops.nms_v5(torch.from_numpy(boxes).to(DEV), torch.from_numpy(scores).to(DEV),
             torch.from_numpy(classes).to(DEV), torch.from_numpy(scales).to(DEV), 0, 100, iou_t,
             score_t, tf_sigma, (512.0, 512.0), det, sel, valid, work)
  torch.cuda.synchronize()
  det, sel, valid = det.cpu().numpy(), sel.cpu().numpy(), valid.cpu().numpy()
  flags = work[-4 * n:].view(torch.int32).cpu().numpy()
  if method == 'gaussian':
    assert (flags == 0).all(), flags      # the batched shared-memory path proved itself exact
  for i in range(n):
    idx, sc, v = po.non_max_suppression_v5(boxes[i], scores[i], 100, iou_t, score_t, tf_sigma, True)
    assert valid[i] == v
    np.testing.assert_array_equal(sel[i], idx)                      # bit-exact keep indices
    np.testing.assert_array_equal(det[i, :, 5], sc)                 # bit-exact (soft) scores
    ref_boxes = po.clip_boxes(boxes[i][idx], 512) * scales[i]
    np.testing.assert_array_equal(det[i, :, 1:5], ref_boxes)
    np.testing.assert_array_equal(det[i, :, 6], (classes[i][idx] + 1).astype(np.float32))
    np.testing.assert_array_equal(det[i, :, 0], np.full(100, i, np.float32))


def test_nms_v5_full_queue_fallback():
  """Massive exact ties overflow the shared-memory fast path (one histogram bin holds every
  candidate), so the full-queue kernel must take over and still match bit for bit."""
  ops = _ops()
  rng = np.random.default_rng(3)
  n, k = 2, 9000
  boxes, scores, classes = _nms_inputs(rng, n, k, clustered=False)
  scores[0, :] = np.float32(0.25)            # image 0: all tied -> index order decides
  scores[1, :8000] = np.float32(0.5)         # image 1: 8000-way tie above a few distinct ones
  det = torch.empty(n, 100, 7, device=DEV)
  sel = torch.empty(n, 100, dtype=torch.int32, device=DEV)
  valid = torch.empty(n, dtype=torch.int32, device=DEV)
  work = torch.empty(ops.nms_work_bytes(n, k), dtype=torch.uint8, device=DEV)
  ops.nms_v5(torch.from_numpy(boxes).to(DEV), torch.from_numpy(scores).to(DEV),
             torch.from_numpy(classes).to(DEV), None, 0, 100, 0.5, 0.001, 0.25, (512.0, 512.0),
             det, sel, valid, work)
  torch.cuda.synchronize()
  for i in range(n):
    idx, sc, v = po.non_max_suppression_v5(boxes[i], scores[i], 100, 0.5, 0.001, 0.25, True)
    assert int(valid[i]) == v
    np.testing.assert_array_equal(sel[i].cpu().numpy(), idx)
    np.testing.assert_array_equal(det[i, :, 5].cpu().numpy(), sc)


def test_nms_v5_fewer_than_max_and_empty():
  ops = _ops()
  rng = np.random.default_rng(0)
  boxes, scores, classes = _nms_inputs(rng, 2, 50)
  scores[1] = 0.0005          # nothing passes score_thresh 0.001 in image 1
  det = torch.empty(2, 100, 7, device=DEV)
  sel = torch.empty(2, 100, dtype=torch.int32, device=DEV)
  valid = torch.empty(2, dtype=torch.int32, device=DEV)
  work = torch.empty(ops.nms_work_bytes(2, 50), dtype=torch.uint8, device=DEV)
  ops.nms_v5(torch.from_numpy(boxes).to(DEV), torch.from_numpy(scores).to(DEV),
             torch.from_numpy(classes).to(DEV), None, 0, 100, 0.5, 0.001, 0.25, (512.0, 512.0),
             det, sel, valid, work)
  torch.cuda.synchronize()
  idx, sc, v = po.non_max_suppression_v5(boxes[0], scores[0], 100, 0.5, 0.001, 0.25, True)
  assert int(valid[0]) == v and int(valid[1]) == 0
  np.testing.assert_array_equal(sel[0].cpu().numpy(), idx)
  np.testing.assert_array_equal(det[0, :, 5].cpu().numpy(), sc)
  assert float(det[1, :, 5].abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------
# nms_np.per_class_nms replacement: rows bit-identical to the REAL reference module's output
# (tests/golden/nms_np_per_class_hard.*.npz, written by tests/golden/make_golden.py from
# the reference's efficientdet/nms_np.py)
@pytest.mark.parametrize('ci', range(10))
def test_per_class_nms_matches_reference_module(ci):
  import json
  ops = _ops()
  g = load_split_golden('nms_np_per_class_hard')
  methods = [json.loads(m) for m in g['methods']]
  boxes, scores, classes = g['boxes_%d' % ci], g['scores_%d' % ci], g['classes_%d' % ci]
  k = scores.shape[0]
  n = 2   # image 1 = the same candidates in reversed anchor order (same rows, mirrored indices)
  b = torch.from_numpy(np.stack([boxes, boxes[::-1]])).to(DEV).contiguous()
  s_ = torch.from_numpy(np.stack([scores, scores[::-1]])).to(DEV).contiguous()
  c = torch.from_numpy(np.stack([classes, classes[::-1]])).to(DEV).contiguous()
  ids = torch.full((n,), float(ci + 10), device=DEV)
  scl = torch.full((n,), float(g['scale_%d' % ci][0]), device=DEV)
  for mi, cfg in enumerate(methods):
    det = torch.empty(n, 100, 7, device=DEV)
    keep = torch.empty(n, 100, dtype=torch.int32, device=DEV)
    valid = torch.empty(n, dtype=torch.int32, device=DEV)
    ops.per_class_nms(b, s_, c, ids, scl, int(g['ncls_%d' % ci]), 100, cfg['method'],
                      cfg['iou_thresh'], det, keep, valid)
    torch.cuda.synchronize()
    ref = g['out_%d_%d' % (ci, mi)]
    got = det.cpu().numpy()
    np.testing.assert_array_equal(got[0], ref, err_msg='case %d method %d' % (ci, mi))
    np.testing.assert_array_equal(got[1], ref, err_msg='case %d method %d (reversed)' % (ci, mi))
    nv = int((ref[:, 5] > -1e4).sum())
    assert valid.cpu().tolist() == [nv, nv]
    kp = keep.cpu().numpy()
    # keep indices: the anchor each row came from (scores are distinct -> unique match)
    np.testing.assert_array_equal(scores[kp[0, :nv]], ref[:nv, 5])
    np.testing.assert_array_equal(kp[1, :nv], k - 1 - kp[0, :nv])
    assert (kp[:, nv:] == -1).all()


@pytest.mark.parametrize('ci', range(7))
def test_per_class_soft_nms_matches_reference_module(ci):
  """gaussian / linear soft NMS of nms_np.per_class_nms (tests/golden/nms_np_per_class_soft.*.npz,
  written by the real module): `linear` rows are bit-identical; `gaussian` selects the same
  anchors in the same order with the same boxes and classes, and its scores agree to 1e-6
  relative (NumPy's float32 exp is not correctly rounded, the device's is)."""
  import json
  ops = _ops()
  g = load_split_golden('nms_np_per_class_soft')
  methods = [json.loads(m) for m in g['methods']]
  boxes, scores, classes = g['boxes_%d' % ci], g['scores_%d' % ci], g['classes_%d' % ci]
  b = torch.from_numpy(boxes[None]).to(DEV).contiguous()
  s_ = torch.from_numpy(scores[None]).to(DEV).contiguous()
  c = torch.from_numpy(classes[None]).to(DEV).contiguous()
  ids = torch.full((1,), float(ci + 20), device=DEV)
  scl = torch.full((1,), float(g['scale_%d' % ci][0]), device=DEV)
  for mi, cfg in enumerate(methods):
    det = torch.empty(1, 100, 7, device=DEV)
    keep = torch.empty(1, 100, dtype=torch.int32, device=DEV)
    valid = torch.empty(1, dtype=torch.int32, device=DEV)
    ops.per_class_nms(b, s_, c, ids, scl, int(g['ncls_%d' % ci]), 100, cfg['method'],
                      cfg['iou_thresh'], det, keep, valid, sigma=cfg['sigma'],
                      score_thresh=cfg['score_thresh'])
    torch.cuda.synchronize()
    ref = g['out_%d_%d' % (ci, mi)]
    got = det.cpu().numpy()[0]
    nv = int((ref[:, 5] > -1e4).sum())
    assert int(valid.item()) == nv, (ci, mi)
    if cfg['method'] == 'linear':
      np.testing.assert_array_equal(got, ref, err_msg='case %d method %d' % (ci, mi))
    else:
      np.testing.assert_array_equal(got[:, [0, 1, 2, 3, 4, 6]], ref[:, [0, 1, 2, 3, 4, 6]])
      np.testing.assert_allclose(got[:, 5], ref[:, 5], rtol=1e-6, atol=0)
    kp = keep.cpu().numpy()[0]
    np.testing.assert_array_equal(boxes[kp[:nv]][:, [1, 0, 3, 2]] * g['scale_%d' % ci][0], ref[:nv, 1:5])
    assert (kp[nv:] == -1).all()


def test_per_class_nms_bad_method():
  ops = _ops()
  z = torch.zeros(1, 8, 4, device=DEV)
  with pytest.raises(ValueError):
    ops.per_class_nms(z, torch.zeros(1, 8, device=DEV), torch.zeros(1, 8, dtype=torch.int32, device=DEV),
                      None, None, 90, 100, 'median', None, torch.empty(1, 100, 7, device=DEV),
                      torch.empty(1, 100, dtype=torch.int32, device=DEV),
                      torch.empty(1, dtype=torch.int32, device=DEV))


def test_sepconv_rejects_the_removed_node_form():
  """The whole-BiFPN-node form (several inputs / pre-activation) was removed: loud error, no fallback."""
  ops = _ops()
  from automl_b200 import _lib
  a = torch.zeros(1, 8, 8, 64, dtype=torch.float16, device=DEV)
  out = torch.empty(1, 8, 8, 64, dtype=torch.float16, device=DEV)
  dw = torch.zeros(9, 64, device=DEV)
  pw = torch.zeros(64, 64, dtype=torch.float16, device=DEV)
  b = torch.zeros(64, device=DEV)
  with pytest.raises(_lib.EdetError):
    ops.sepconv([(a, ops.RS_SAME, None, 0.5), (a, ops.RS_SAME, None, 0.5)], utils.ACT_SWISH, dw, pw, b,
                out, utils.ACT_NONE)
