"""Masked conv / linear fprop, dgrad and dense wgrad vs the float64 CPU oracle.

Tolerance (floating point, north_star: 1e-5 rel on fp32 accumulators): inputs are
rounded to bf16 ONCE on the host and fed identically to both sides, so the only
differences are fp32 accumulation order (checked at rtol 2e-5 of the output scale
on the fp32 outputs) and the single final rounding to bf16 (<= 1 bf16 ulp =
2^-8 relative, checked on the bf16 outputs).
"""
import numpy as np
import pytest
import torch

from oracle import rigl_oracle as orc
from rigl_b200 import _cabi
from rigl_b200.layers import SparseConv2d, SparseLinear
from rigl_b200 import pruning

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _bf16(a):
  return torch.from_numpy(np.asarray(a, np.float32)).to(torch.bfloat16)


def _check_bf16(got, want, what):
  got = got.detach().float().cpu().numpy().astype(np.float64)
  scale = np.abs(want).max() + 1e-30
  err = np.abs(got - want)
  tol = np.maximum(np.abs(want) * 2.0 ** -8, scale * 2.0 ** -16) * 1.01 + scale * 2e-5
  assert (err <= tol).all(), '%s: max err %g (scale %g) at %d positions' % (
      what, err.max(), scale, int((err > tol).sum()))


def _check_f32(got, want, what, rtol=2e-5):
  got = got.detach().float().cpu().numpy().astype(np.float64)
  scale = np.abs(want).max() + 1e-30
  assert np.abs(got - want).max() <= rtol * scale, '%s: max err %g scale %g' % (
      what, np.abs(got - want).max(), scale)


CONV_CASES = [
    # n, h, w, cin, cout, k, stride, sparsity
    (2, 8, 8, 16, 32, 3, 1, 0.5),
    (2, 9, 7, 8, 16, 3, 2, 0.8),
    (3, 8, 8, 64, 64, 1, 1, 0.0),
    (2, 14, 14, 64, 128, 1, 2, 0.4),
    (2, 12, 12, 3, 8, 7, 2, 0.14),      # stem-like: cin=3 (patch matrix / SIMT)
    (3, 32, 32, 3, 64, 7, 2, 0.14),
    (2, 17, 17, 3, 16, 3, 1, 0.3),
    (4, 16, 16, 64, 64, 3, 1, 0.64),
    (8, 14, 14, 128, 128, 3, 1, 0.82),
    (4, 28, 28, 128, 128, 3, 2, 0.82),
    (16, 7, 7, 256, 256, 3, 1, 0.95),
    (32, 7, 7, 512, 128, 1, 1, 0.7),
    # TensorFlow 'SAME' incl. the asymmetric stride-2 case (WRN, cifar_resnet/resnet_model.py:158-181)
    (4, 32, 32, 16, 32, 3, 2, 0.8, 'SAME'),
    (2, 16, 16, 64, 128, 3, 2, 0.9, 'SAME'),
    (2, 15, 15, 32, 64, 3, 2, 0.5, 'SAME'),
    (2, 16, 16, 32, 64, 1, 2, 0.2, 'VALID'),
    (2, 9, 9, 16, 16, 3, 1, 0.3, 'VALID'),
]


def _conv_case(case, force_simt):
  n, h, w, cin, cout, k, stride, sparsity = case[:8]
  padding = case[8] if len(case) > 8 else 'FIXED'
  rng = np.random.RandomState(abs(hash(case[:8])) % (2 ** 31))
  pruning.reset_default_registry()
  _cabi.lib().rigl_set_force_simt(1 if force_simt else 0)
  try:
    layer = SparseConv2d(cin, cout, k, strides=stride, padding=padding, name='t', device=DEV)
    w_np = _bf16(rng.standard_normal((k, k, cin, cout)) / np.sqrt(k * k * cin)).float().numpy()
    m_np = orc.get_mask_random_numpy((k, k, cin, cout), sparsity, rng).astype(np.float32)
    with torch.no_grad():
      layer.weight.copy_(torch.from_numpy(w_np))
    layer.mask.assign(m_np)
    x_np = _bf16(rng.standard_normal((n, h, w, cin))).float().numpy()
    x = torch.from_numpy(x_np).permute(0, 3, 1, 2).to(DEV).to(torch.bfloat16) \
        .contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = layer(x)
    wm = (w_np * m_np).astype(np.float64)
    (ho, pad), (wo, _) = layer.out_size(h), layer.out_size(w)
    if padding == 'SAME':
      assert (ho, pad) == orc.tf_same_padding(h, k, stride)[:2]
    y_want = orc.conv2d_nhwc_general(x_np.astype(np.float64), wm, stride, pad, (ho, wo))
    assert tuple(y.shape) == (n, cout, y_want.shape[1], y_want.shape[2])
    _check_bf16(y.permute(0, 2, 3, 1), y_want, 'fprop %s' % (case,))
    dy_np = _bf16(rng.standard_normal(y_want.shape)).float().numpy()
    dy = torch.from_numpy(dy_np).permute(0, 3, 1, 2).to(DEV).to(torch.bfloat16) \
        .contiguous(memory_format=torch.channels_last)
    y.backward(dy)
    dx_want, dw_want = orc.conv2d_nhwc_general_bwd(x_np.astype(np.float64), wm, dy_np.astype(np.float64), stride, pad)
    _check_bf16(x.grad.permute(0, 2, 3, 1), dx_want, 'dgrad %s' % (case,))
    # dense wgrad: every position, including masked-out ones (RigL grow scores)
    _check_f32(layer.masked_weights.dense_grad.view(k, k, cin, cout), dw_want, 'wgrad %s' % (case,))
    # dL/dweights = mask * dense
    _check_f32(layer.weight.grad, dw_want * m_np, 'masked wgrad %s' % (case,))
    assert (layer.weight.grad.detach().cpu().numpy()[m_np == 0] == 0).all()
  finally:
    _cabi.lib().rigl_set_force_simt(0)


@pytest.mark.parametrize('case', CONV_CASES[:6])
def test_conv_simt_path(case):
  _conv_case(case, force_simt=True)


@pytest.mark.parametrize('case', CONV_CASES)
def test_conv_default_path(case):
  _conv_case(case, force_simt=False)


LINEAR_CASES = [(1, 3, 5, 0.5), (100, 784, 300, 0.9), (100, 300, 100, 0.81), (100, 100, 10, 0.0),
                (256, 2048, 1000, 0.85), (37, 64, 64, 0.3)]


@pytest.mark.parametrize('case', LINEAR_CASES)
@pytest.mark.parametrize('force_simt', [True, False])
def test_linear(case, force_simt):
  m_rows, n_in, n_out, sparsity = case
  rng = np.random.RandomState(m_rows + n_in)
  pruning.reset_default_registry()
  _cabi.lib().rigl_set_force_simt(1 if force_simt else 0)
  try:
    layer = SparseLinear(n_in, n_out, name='fc', device=DEV, out_dtype=torch.float32)
    w_np = _bf16(rng.standard_normal((n_in, n_out)) / np.sqrt(n_in)).float().numpy()
    m_np = orc.get_mask_random_numpy((n_in, n_out), sparsity, rng).astype(np.float32)
    b_np = rng.standard_normal(n_out).astype(np.float32)
    with torch.no_grad():
      layer.weight.copy_(torch.from_numpy(w_np))
      layer.bias.copy_(torch.from_numpy(b_np))
    layer.mask.assign(m_np)
    x_np = _bf16(rng.standard_normal((m_rows, n_in))).float().numpy()
    x = torch.from_numpy(x_np).to(DEV).to(torch.bfloat16).requires_grad_(True)
    y = layer(x)
    assert y.dtype == torch.float32
    y_want = orc.masked_linear_fwd(x_np, w_np, m_np, b_np)
    _check_f32(y, y_want, 'linear fprop')
    dy_np = _bf16(rng.standard_normal(y_want.shape)).float().numpy()
    y.backward(torch.from_numpy(dy_np).to(DEV))
    dx_want, dw_dense, dw_masked = orc.masked_linear_bwd(x_np, w_np, m_np, dy_np)
    _check_bf16(x.grad, dx_want, 'linear dgrad')
    _check_f32(layer.masked_weights.dense_grad.view(n_in, n_out), dw_dense, 'linear dense wgrad')
    _check_f32(layer.weight.grad, dw_masked, 'linear masked wgrad')
    _check_f32(layer.bias.grad, dy_np.astype(np.float64).sum(0), 'bias grad')
  finally:
    _cabi.lib().rigl_set_force_simt(0)


def test_rank_and_channel_errors():
  pruning.reset_default_registry()
  layer = SparseConv2d(8, 8, 3, name='e', device=DEV)
  with pytest.raises(ValueError):
    layer(torch.zeros(2, 8, 4, device=DEV))
  with pytest.raises(ValueError):
    layer(torch.zeros(2, 4, 4, 4, device=DEV))


@pytest.mark.parametrize('case', [(2, 16, 16, 3, 64, 7, 2, 0.14), (3, 32, 32, 3, 64, 7, 2, 0.14),
                                  (2, 64, 48, 3, 16, 7, 2, 0.5), (2, 224, 224, 3, 64, 7, 2, 0.14)])
def test_conv_stem_s2d_path(case):
  """The space-to-depth stem (layers.STEM_S2D_PATH, the default): same oracle, same tolerances."""
  from rigl_b200 import layers
  old, layers.STEM_S2D_PATH = layers.STEM_S2D_PATH, True
  try:
    _conv_case(case, force_simt=False)
  finally:
    layers.STEM_S2D_PATH = old


@pytest.mark.parametrize('case', [(3, 32, 32, 3, 64, 7, 2, 0.14), (2, 64, 48, 3, 16, 7, 2, 0.5),
                                  (2, 12, 12, 3, 8, 7, 2, 0.14), (2, 17, 17, 3, 16, 3, 1, 0.3)])
def test_conv_stem_patch_matrix_path(case):
  """RIGL_STEM_S2D=0 fallback: the im2col patch-matrix stem."""
  from rigl_b200 import layers
  old, layers.STEM_S2D_PATH = layers.STEM_S2D_PATH, False
  try:
    _conv_case(case, force_simt=False)
  finally:
    layers.STEM_S2D_PATH = old


# 3x3 / stride 1 / pad 1 layers with <= 64 reduction channels run on the halo kernels (one halo tile in
# shared memory feeds all nine taps): full and partial channel blocks, H not a multiple of the strip,
# H smaller than a strip, several N tiles, every halo pitch (16 / 32 / 64).
HALO_CASES = [
    (2, 14, 14, 64, 64, 3, 1, 0.6),
    (3, 56, 56, 64, 64, 3, 1, 0.64),
    (2, 28, 28, 32, 128, 3, 1, 0.8),
    (2, 13, 27, 64, 24, 3, 1, 0.5),
    (5, 6, 14, 16, 64, 3, 1, 0.3),
    (2, 28, 28, 64, 64, 3, 1, 0.9, 'SAME'),
]


@pytest.mark.parametrize('case', HALO_CASES)
def test_conv_halo_path(case):
  _conv_case(case, force_simt=False)


@pytest.mark.parametrize('case', [HALO_CASES[1], HALO_CASES[3]])
def test_conv_halo_disabled_matches(case):
  """RIGL_HALO3X3=0 routes the same layers through the generic per-tap kernels."""
  import os, subprocess, sys
  code = ('import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_conv_gpu as t; '
          't._conv_case(%r, False); print("GEN_OK")' % (os.path.dirname(os.path.dirname(__file__)),
                                                        os.path.dirname(__file__), case))
  env = dict(os.environ, RIGL_HALO3X3='0')
  out = subprocess.run([sys.executable, '-c', code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  assert 'GEN_OK' in out.stdout, out.stdout[-1500:]


@pytest.mark.parametrize('case', [CONV_CASES[0], CONV_CASES[5], CONV_CASES[7], CONV_CASES[8], CONV_CASES[9], CONV_CASES[10],
                                  CONV_CASES[11], CONV_CASES[12]])
def test_conv_single_cta_mma_path(case):
  """The default K-major kernel is the CTA-pair one (cta_group::2); this keeps the single-CTA
  (M = 128) kernel covered."""
  import os, subprocess, sys
  code = ('import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_conv_gpu as t; '
          't._conv_case(%r, False); print("ONE_OK")' % (os.path.dirname(os.path.dirname(__file__)),
                                                        os.path.dirname(__file__), case))
  env = dict(os.environ, RIGL_CTA_PAIR='0')
  out = subprocess.run([sys.executable, '-c', code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  assert 'ONE_OK' in out.stdout, out.stdout[-1500:]


# ---- BASELINE-size problems (C2: ResNet-50, batch 256, 224x224): many more tiles than CTAs, so the persistent
# loops' TMEM double buffering, smem-ring wrap and split-K schedules run for many tiles per CTA.
def _r50_erk80_sparsity():
  layers = orc.resnet50_masked_layers()
  sp = orc.get_sparsities([orc.FakeMask(n + '/mask:0', sh) for n, sh, _, _ in layers], 'erdos_renyi_kernel', 0.8, {})
  return layers, sp


def _r50_b256_shapes():
  """Distinct (n,h,w,cin,cout,k,stride,sparsity) of the 53 ResNet-50 convs at batch 256."""
  layers, sp = _r50_erk80_sparsity()
  seen, out = set(), []
  for name, sh, stride, out_hw in layers:
    if len(sh) != 4:
      continue
    k, _, cin, cout = sh
    key = (out_hw * stride, cin, cout, k, stride)
    if key in seen:
      continue
    seen.add(key)
    out.append((256, out_hw * stride, out_hw * stride, cin, cout, k, stride, round(float(sp[name + '/mask:0']), 3)))
  return out


# the four shapes VERDICT r1 asked for: 56^2 64->256 1x1, 56^2->28^2 128 3x3 s2, 14^2 256 3x3, 7^2 512 3x3
_B256_ORACLE = [c for c in _r50_b256_shapes() if (c[1], c[3], c[4], c[5], c[6]) in
                ((56, 64, 256, 1, 1), (56, 128, 128, 3, 2), (14, 256, 256, 3, 1), (7, 512, 512, 3, 1))]


@pytest.mark.parametrize('case', _B256_ORACLE, ids=lambda c: 'h%d_c%d_%d_k%d_s%d' % (c[1], c[3], c[4], c[5], c[6]))
def test_conv_b256_baseline_shapes_vs_fp64_oracle(case):
  assert len(_B256_ORACLE) == 4
  _conv_case(case, force_simt=False)


def _run_both(layer, x, dy, force_simt):
  _cabi.lib().rigl_set_force_simt(1 if force_simt else 0)
  try:
    xx = x.detach().clone().requires_grad_(True)
    layer.masked_weights.fresh = False
    layer.weight.grad = None
    y = layer(xx)
    y.backward(dy)
    torch.cuda.synchronize()
    return y.detach().float(), xx.grad.detach().float() if xx.grad is not None else None, \
        layer.masked_weights.dense_grad.clone()
  finally:
    _cabi.lib().rigl_set_force_simt(0)


@pytest.mark.parametrize('case', _r50_b256_shapes(), ids=lambda c: 'h%d_c%d_%d_k%d_s%d' % (c[1], c[3], c[4], c[5], c[6]))
def test_conv_b256_every_r50_shape_tensor_core_vs_cuda_core(case):
  """Every distinct ResNet-50 conv shape at batch 256: the tcgen05 kernels against the shape-agnostic CUDA-core
  kernels on the SAME device inputs and packed operands (fp32 accumulation on both sides; bf16 outputs may differ
  by one rounding)."""
  n, h, w, cin, cout, k, stride, sparsity = case
  rng = np.random.RandomState(cin * 7 + cout + k)
  pruning.reset_default_registry()
  layer = SparseConv2d(cin, cout, k, strides=stride, padding='FIXED', name='t', device=DEV)
  layer.mask.assign(orc.get_mask_random_numpy((k, k, cin, cout), sparsity, rng).astype(np.float32))
  g = torch.Generator(device=DEV).manual_seed(cin + cout)
  x = torch.randn((n, cin, h, w), device=DEV, generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
  ho = layer.out_size(h)[0]
  dy = torch.randn((n, cout, ho, ho), device=DEV, generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
  y1, dx1, dw1 = _run_both(layer, x, dy, force_simt=False)
  y0, dx0, dw0 = _run_both(layer, x, dy, force_simt=True)
  for got, want, what in ((y1, y0, 'fprop'), (dx1, dx0, 'dgrad')):
    scale = float(want.abs().max())
    bad = (got - want).abs() > want.abs() * 2.0 ** -7 + scale * 2e-5
    assert not bool(bad.any()), '%s %s: %d elements off, max err %g (scale %g)' % (
        what, case, int(bad.sum()), float((got - want).abs().max()), scale)
  scale = float(dw0.abs().max())
  assert float((dw1 - dw0).abs().max()) <= 5e-5 * scale, 'wgrad %s: %g vs scale %g' % (
      case, float((dw1 - dw0).abs().max()), scale)


def test_batched_pack_equals_per_layer_pack():
  """layers.pack_all (ONE launch over a tile table) writes byte-identical operand blobs -- both K-major layouts and
  the 64x64 survivor counts -- to the per-layer rigl_pack_masked_weights calls, incl. ragged channel counts, the
  stem's patch-matrix form and a linear layer."""
  from rigl_b200 import layers
  pruning.reset_default_registry()
  rng = np.random.RandomState(5)
  ls = [SparseConv2d(3, 64, 7, strides=2, padding='FIXED', name='stem', device=DEV),
        SparseConv2d(64, 256, 1, name='a', device=DEV), SparseConv2d(72, 40, 3, name='ragged', device=DEV),
        SparseConv2d(128, 128, 3, strides=2, name='b', device=DEV), SparseLinear(300, 100, name='fc', device=DEV),
        SparseConv2d(5, 3, 3, name='tiny', device=DEV)]
  for l in ls:
    l.mask.assign(orc.get_mask_random_numpy(tuple(l.weight.shape), 0.8, rng).astype(np.float32))
  blobs = lambda l: [b for b in (getattr(l, 'packed_patch', None), l.packed, getattr(l, 'packed_s2d', None)) if b is not None]
  want = []
  for l in ls:
    for b in blobs(l):
      b.fill_(0x5a)          # (alignment padding between the blob's sections is never written: same filler twice)
    l.pack()
    want.append([b.clone() for b in blobs(l)])
  for l in ls:
    for b in blobs(l):
      b.fill_(0x5a)
  layers.pack_all(ls)
  torch.cuda.synchronize()
  for l, ws in zip(ls, want):
    got = blobs(l)
    if getattr(l, 'patch_mode', False):       # patch-mode layers only pack their patch / special forms
      got, ws = [got[0]] + got[2:], [ws[0]] + ws[2:]
    for g, w in zip(got, ws):
      assert torch.equal(g, w), l.scope
  layers._PACKED_AHEAD.clear()


def test_conv_wgrad_accumulates_over_backward_passes():
  """beta = 1: a second backward before the gradients are consumed ADDS to the dense gradient (k_splitk_reduce
  reads dw back and adds the split-K partials to it in split order)."""
  pruning.reset_default_registry()
  torch.manual_seed(3)
  layer = SparseConv2d(128, 256, 3, padding='FIXED', name='acc', device=DEV)
  x = torch.randn(8, 128, 14, 14, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
  dy = torch.randn(8, 256, 14, 14, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
  layer.masked_weights.fresh = False
  layer(x).backward(dy)
  once = layer.masked_weights.dense_grad.clone()
  layer(x).backward(dy)                       # fresh is still True: accumulates
  assert torch.allclose(layer.masked_weights.dense_grad, once + once, rtol=1e-5, atol=1e-5 * float(once.abs().max()))


@pytest.mark.parametrize('case', [(2, 16, 16, 32, 1), (2, 17, 13, 64, 2), (3, 14, 14, 256, 1), (2, 8, 8, 1024, 2),
                                  (4, 112, 112, 32, 1), (2, 56, 56, 128, 2), (1, 5, 7, 24, 1)])
def test_depthwise3x3_vs_fp64(case):
  """Native depthwise 3x3 (csrc/depthwise.cu; MobileNet-v1's depthwise_conv2d_fixed_padding, mobilenetv1_model.py:
  120-153) forward, input gradient and weight gradient against a float64 grouped convolution on the same
  bf16-rounded operands."""
  from rigl_b200.workloads import DepthwiseConv2d
  n, h, w, c, stride = case
  torch.manual_seed(c + h)
  dw = DepthwiseConv2d(c, stride=stride, device=DEV)
  dw.native = True                       # the csrc/depthwise.cu kernels (the default path is cuDNN)
  with torch.no_grad():
    dw.weight.copy_(dw.weight.to(torch.bfloat16).float() * 3)
    dw.weight.copy_(dw.weight.to(torch.bfloat16).float())
  x = torch.randn(n, c, h, w, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
  y = dw(x)
  x64 = x.detach().double().cpu().requires_grad_(True)
  w64 = dw.weight.detach().double().cpu().requires_grad_(True)
  y64 = torch.nn.functional.conv2d(x64, w64, None, stride, 1, 1, c)
  assert tuple(y.shape) == tuple(y64.shape)
  dy = torch.randn_like(y64).to(torch.bfloat16)
  y.backward(dy.to(DEV).contiguous(memory_format=torch.channels_last))
  y64.backward(dy.double())
  _check_bf16(y.permute(0, 2, 3, 1), y64.detach().permute(0, 2, 3, 1).numpy(), 'depthwise fprop %s' % (case,))
  _check_bf16(x.grad.permute(0, 2, 3, 1), x64.grad.permute(0, 2, 3, 1).numpy(), 'depthwise dgrad %s' % (case,))
  _check_f32(dw.weight.grad, w64.grad.numpy(), 'depthwise wgrad %s' % (case,))
