"""Frozen inference (rigl_b200.inference, rigl_masked_conv2d_fprop_affine) on the GPU.

Per-op: the fused epilogue y = [relu](conv(x, mask*W) * scale + shift (+ residual)) against an fp64 numpy
restatement on the same bf16-rounded inputs; tolerance 1 bf16 ulp of the element + 2e-5 of the tensor's max
(the single final rounding + fp32 accumulation order), as in test_conv_gpu.py.
Whole model: frozen logits against `model.eval()` logits.  The two differ by rounding only: eval rounds every
conv output to bf16 before the BN, the frozen path rounds once after it.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import rigl_oracle as orc
from rigl_b200 import _cabi
from rigl_b200 import pruning
from rigl_b200 import workloads as wl
from rigl_b200.inference import freeze
from rigl_b200.layers import SparseConv2d

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNSUPPORTED = -4

# Relative L2 of frozen vs model.eval() logits measured on B200 (profiles/r03_inference.md); the bound is 3x that.
# ResNet-50 0.0806, MobileNet-v1 0.0849 (a one-ulp perturbation of the input moves model.eval()'s own logits by 0.115
# and 0.143); WRN-22-2 and MnistFC 0: on those every op of the frozen path is the eval path's kernel.
REL_L2_BOUND = {'resnet50': 0.242, 'mobilenet_v1': 0.255, 'wrn': 0.0, 'mnist_fc': 0.0}


def policy_declines(n, ho, wo, cin, cout, k, residual):
  """Restatement of affine_profitable() in igemm_tc.cu (tensor-core shapes only)."""
  K = k * k * cin
  return residual or (K <= 512 and cout >= 2 * K and n * ho * wo <= 12544)


def _bf16_np(a):
  return torch.from_numpy(np.asarray(a, np.float32)).to(torch.bfloat16).float().numpy()


def _check_bf16(got, want, what):
  got = got.detach().float().cpu().numpy().astype(np.float64)
  scale = np.abs(want).max() + 1e-30
  err = np.abs(got - want)
  tol = np.maximum(np.abs(want) * 2.0 ** -8, scale * 2.0 ** -16) * 1.01 + scale * 2e-5
  assert (err <= tol).all(), '%s: max err %g (scale %g) at %d positions' % (
      what, err.max(), scale, int((err > tol).sum()))


def _nhwc(t_np):
  return torch.from_numpy(t_np).permute(0, 3, 1, 2).to(DEV).to(torch.bfloat16).contiguous(
      memory_format=torch.channels_last)


def _make_layer(n, h, w, cin, cout, k, stride, sparsity=0.7, seed=0):
  rng = np.random.RandomState(seed)
  pruning.reset_default_registry()
  layer = SparseConv2d(cin, cout, k, strides=stride, padding='FIXED', name='inf', device=DEV)
  w_np = _bf16_np(rng.standard_normal((k, k, cin, cout)) / np.sqrt(k * k * cin))
  m_np = orc.get_mask_random_numpy((k, k, cin, cout), sparsity, rng).astype(np.float32)
  with torch.no_grad():
    layer.weight.copy_(torch.from_numpy(w_np))
  layer.mask.assign(m_np)
  layer.pack()
  x_np = _bf16_np(rng.standard_normal((n, h, w, cin)))
  return layer, (w_np * m_np).astype(np.float64), x_np, rng


def _affine(layer, x, scale, shift, res, relu):
  n, c, h, w = x.shape
  d = layer._desc(n, h, w)
  y = torch.empty((n, layer._cout, d.out_h, d.out_w), dtype=torch.bfloat16, device=DEV,
                  memory_format=torch.channels_last)
  p = lambda t: None if t is None else t.data_ptr()
  rc = _cabi.lib().rigl_masked_conv2d_fprop_affine(d, x.data_ptr(), layer.packed.data_ptr(), p(scale), p(shift),
                                                   p(res), int(relu), y.data_ptr(), None, 0, _cabi.stream_ptr())
  return rc, y


def _plain(layer, x):
  n, c, h, w = x.shape
  d = layer._desc(n, h, w)
  y = torch.empty((n, layer._cout, d.out_h, d.out_w), dtype=torch.bfloat16, device=DEV,
                  memory_format=torch.channels_last)
  _cabi.check(_cabi.lib().rigl_masked_conv2d_fprop(d, x.data_ptr(), layer.packed.data_ptr(), y.data_ptr(), None, None,
                                                   None, 0, _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
  return y


# n, h, w, cin, cout, k, stride
SHAPES = [
    (4, 14, 14, 64, 24, 1, 1),        # cout 24: one partial 64-channel slab
    (2, 9, 9, 128, 200, 3, 1),        # 3x3 s1 (cin > 64: not a halo layer), cout 200
    (4, 14, 14, 128, 1024, 1, 2),     # 1x1 s2, cout 1024
    (2, 15, 15, 72, 64, 3, 2),        # 3x3 s2
    (1, 8, 8, 64, 64, 1, 1),          # one M tile: k_igemm_kmajor
    (1, 4, 4, 128, 200, 3, 1),        # one M tile, 3x3, cout 200
]
# scale, shift, residual, relu (0/1 = NULL/given)
EPILOGUES = [(1, 1, 1, 1), (1, 1, 0, 1), (1, 1, 1, 0), (1, 1, 0, 0), (0, 1, 1, 1), (1, 0, 1, 1), (0, 0, 1, 0),
             (0, 0, 0, 1)]
BASELINE_SHAPES = [(256, 28, 28, 128, 512, 1, 1), (256, 14, 14, 256, 1024, 1, 1)]


def run_case(shape, ep, force_simt=False, expect_declined=False):
  n, h, w, cin, cout, k, stride = shape
  layer, wm, x_np, rng = _make_layer(*shape, seed=abs(hash((shape, ep))) % (2 ** 31))
  pad = layer.pad
  (ho, _), (wo, _) = layer.out_size(h), layer.out_size(w)
  conv = orc.conv2d_nhwc_general(x_np.astype(np.float64), wm, stride, pad, (ho, wo))
  sc = rng.uniform(-1.5, 1.5, cout).astype(np.float32) if ep[0] else None
  sh = rng.standard_normal(cout).astype(np.float32) if ep[1] else None
  rs = _bf16_np(rng.standard_normal((n, ho, wo, cout))) if ep[2] else None
  want = conv * (sc.astype(np.float64) if sc is not None else 1.0)
  if sh is not None:
    want = want + sh
  if rs is not None:
    want = want + rs
  if ep[3]:
    want = np.maximum(want, 0.0)
  t = lambda a: None if a is None else torch.from_numpy(a).to(DEV)
  _cabi.lib().rigl_set_force_simt(1 if force_simt else 0)
  try:
    rc, y = _affine(layer, _nhwc(x_np), t(sc), t(sh), None if rs is None else _nhwc(rs), ep[3])
  finally:
    _cabi.lib().rigl_set_force_simt(0)
  if expect_declined:
    assert rc == UNSUPPORTED and b'not profitable' in _cabi.lib().rigl_last_error()
    return
  _cabi.check(rc, 'rigl_masked_conv2d_fprop_affine')
  _check_bf16(y.permute(0, 2, 3, 1), want, 'affine %s %s simt=%d' % (shape, ep, force_simt))


def _declined(shape, ep):
  n, h, w, cin, cout, k, stride = shape
  ho, wo = (h + stride - 1) // stride, (w + stride - 1) // stride     # FIXED padding, k in {1, 3}
  return policy_declines(n, ho, wo, cin, cout, k, bool(ep[2]))


@pytest.mark.parametrize('ep', EPILOGUES)
@pytest.mark.parametrize('shape', SHAPES)
def test_affine_epilogue_vs_fp64(shape, ep):
  """Default policy: fused where profitable, RIGL_ERR_UNSUPPORTED where the measured rule declines."""
  run_case(shape, ep, expect_declined=_declined(shape, ep))


@pytest.mark.parametrize('ep', EPILOGUES)
@pytest.mark.parametrize('shape', SHAPES)
def test_affine_epilogue_simt_vs_fp64(shape, ep):
  run_case(shape, ep, force_simt=True)


def _in_fresh_process(calls, **env):
  """Runs `calls` (python source over this module as `t`) in a new process: the RIGL_* switches are read once,
  when the library initialises."""
  code = ('import sys, importlib.util; sys.path.insert(0, %r); '
          'spec = importlib.util.spec_from_file_location("t", %r); t = importlib.util.module_from_spec(spec); '
          'spec.loader.exec_module(t); %s; print("subprocess ok")' % (ROOT, os.path.abspath(__file__), calls))
  r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, **env), cwd=ROOT, stdout=subprocess.PIPE,
                     stderr=subprocess.STDOUT, text=True, timeout=900)
  assert r.returncode == 0 and 'subprocess ok' in r.stdout, r.stdout[-4000:]


def test_affine_epilogue_every_case_fused():
  """RIGL_AFFINE_ALWAYS=1 lifts the profitability rule: the fused kernels on every case, including the residual
  epilogue and two BASELINE-size residual shapes at b256 (28x28 128->512, 14x14 256->1024)."""
  _in_fresh_process('[t.run_case(s, e) for s in t.SHAPES for e in t.EPILOGUES]; '
                    '[t.run_case(s, (1, 1, 1, 1)) for s in t.BASELINE_SHAPES]', RIGL_AFFINE_ALWAYS='1')


def test_affine_epilogue_direct_store_path():
  """RIGL_TMA_STORE=0: per-thread global stores instead of the staged slab + TMA store."""
  _in_fresh_process('[t.run_case(s, e) for s in t.SHAPES for e in [(1, 1, 1, 1), (0, 1, 0, 0)]]',
                    RIGL_AFFINE_ALWAYS='1', RIGL_TMA_STORE='0')


@pytest.mark.parametrize('shape', [SHAPES[0], (4, 14, 14, 256, 256, 1, 2), SHAPES[4], (8, 28, 28, 256, 128, 3, 2)])
def test_affine_identity_equals_plain_fprop(shape):
  layer, _, x_np, _ = _make_layer(*shape)
  x = _nhwc(x_np)
  rc, y = _affine(layer, x, None, None, None, 0)
  _cabi.check(rc, 'rigl_masked_conv2d_fprop_affine')
  assert torch.equal(y, _plain(layer, x))


def test_halo_shape_is_declined():
  layer, _, x_np, _ = _make_layer(2, 56, 56, 64, 64, 3, 1)
  one = torch.ones(64, device=DEV)
  rc, _ = _affine(layer, _nhwc(x_np), one, one, None, 1)
  assert rc == UNSUPPORTED
  assert b'halo' in _cabi.lib().rigl_last_error()


@pytest.mark.parametrize('shape', [(2, 112, 112, 64), (3, 9, 7, 24)])
def test_maxpool_without_argmax_is_bit_identical(shape):
  n, h, w, c = shape
  x = torch.randn(n, c, h, w, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
  oh, ow = (h + 1) // 2, (w + 1) // 2
  ys = [torch.empty((n, c, oh, ow), dtype=torch.bfloat16, device=DEV, memory_format=torch.channels_last)
        for _ in range(2)]
  arg = torch.empty((n, oh, ow, c), dtype=torch.uint8, device=DEV)
  for y, a in zip(ys, (arg.data_ptr(), None)):
    _cabi.check(_cabi.lib().rigl_maxpool_same_forward(x.data_ptr(), n, h, w, c, 3, 2, y.data_ptr(), a,
                                                      _cabi.stream_ptr()), 'rigl_maxpool_same_forward')
  assert torch.equal(ys[0], ys[1])


# ---- whole models ----
def _randomise_bn_and_fill_running_stats(model, x):
  g = torch.Generator(device=DEV).manual_seed(5)
  bns = [m for m in model.modules() if isinstance(m, wl.FusedBatchNormReLU)]
  with torch.no_grad():
    for bn in bns:
      sign = torch.randint(0, 2, (bn.channels,), device=DEV, generator=g) * 2 - 1
      bn.weight.copy_(sign * (0.5 + torch.rand(bn.channels, device=DEV, generator=g)))
      bn.bias.copy_(0.2 * torch.randn(bn.channels, device=DEV, generator=g))
    momenta = [bn.momentum for bn in bns]
    for bn in bns:
      bn.momentum = 1.0                 # running statistics <- this batch's statistics
    model.train()
    model(x)
    for bn, mo in zip(bns, momenta):
      bn.momentum = mo
  model.eval()


MODELS = {
    'resnet50': (lambda: wl.ResNet50(device=DEV), (16, 3, 224, 224), 'erdos_renyi_kernel', 0.8),
    'mobilenet_v1': (lambda: wl.MobileNetV1(device=DEV), (16, 3, 224, 224), 'random', 0.9),
    'wrn': (lambda: wl.WideResNet(depth=22, width=2, device=DEV), (32, 3, 32, 32), 'erdos_renyi_kernel', 0.95),
    'mnist_fc': (lambda: wl.MnistFC(device=DEV), (64, 784), 'random', 0.9),
}


def _input(shape, seed=1):
  g = torch.Generator(device=DEV).manual_seed(seed)
  x = torch.randn(*shape, device=DEV, generator=g).to(torch.bfloat16)
  return x.contiguous(memory_format=torch.channels_last) if len(shape) == 4 else x


@pytest.fixture(scope='module')
def models():
  out = {}
  for name, (ctor, shape, method, sparsity) in MODELS.items():
    torch.manual_seed(0)
    m = ctor()
    wl.init_masks(m, method, sparsity, seed=0)
    x = _input(shape)
    if name == 'mnist_fc':
      m.eval()
    else:
      _randomise_bn_and_fill_running_stats(m, x)
    out[name] = (m, x)
  return out


def _one_ulp_perturbed(x, seed=3):
  """x with each nonzero element moved by -1, 0 or +1 bf16 ulp at random."""
  g = torch.Generator(device=DEV).manual_seed(seed)
  bits = x.view(torch.int16)
  step = torch.randint(-1, 2, x.shape, device=DEV, generator=g).to(torch.int16)
  return (bits + step * (x != 0).to(torch.int16)).view(torch.bfloat16)


@pytest.mark.parametrize('name', sorted(MODELS))
def test_whole_model_frozen_vs_eval(models, name):
  m, x = models[name]
  with torch.no_grad():
    want = m(x)
    noisy = m(_one_ulp_perturbed(x))
  fz = freeze(m)
  got = fz(x)
  assert got.dtype == want.dtype and got.shape == want.shape
  g, w = got.double(), want.double()
  rel = float((g - w).norm() / w.norm())
  floor = float((noisy.double() - w).norm() / w.norm())
  # Rows whose top-2 gap exceeds 1e-2 of the logit scale, and that a one-ulp perturbation of the input does not
  # already reorder (the randomly initialised networks amplify rounding: see the printed `floor`).
  top2 = w.topk(2, dim=1).values
  gap = top2[:, 0] - top2[:, 1]
  clear = (gap > 1e-2 * float(w.abs().max())) & (gap > 2 * float((noisy.double() - w).abs().max()))
  print('WHOLE_MODEL %s rel_l2 %.6g one_ulp_input_rel_l2 %.6g clear_rows %d/%d' % (
      name, rel, floor, int(clear.sum()), w.shape[0]))
  assert rel <= REL_L2_BOUND[name], rel
  assert bool((g.argmax(1) == w.argmax(1))[clear].all())
  assert fz.bn_apply_calls == len(fz.fallback)
  if name == 'resnet50':
    bns = [n for n, mod in m.named_modules() if isinstance(mod, wl.FusedBatchNormReLU)]
    assert len(bns) == 53 and sorted(fz.folded + list(fz.fallback)) == sorted(bns)
    want_fb, h = {'initial_bn'}, 56
    for i, blk in enumerate(m.blocks):
      s = blk.conv2.stride
      if blk.conv2._cin <= 64 and s == 1:                             # the halo 3x3 layers
        want_fb.add('blocks.%d.bn2' % i)
      for conv, bn, hout, res in ((blk.proj, 'proj_bn', h // s, False), (blk.conv1, 'bn1', h, False),
                                  (blk.conv2, 'bn2', h // s, False), (blk.conv3, 'bn3', h // s, True)):
        if conv is not None and policy_declines(16, hout, hout, conv._cin, conv._cout, conv.ksize, res):
          want_fb.add('blocks.%d.%s' % (i, bn))
      h //= s
    assert set(fz.fallback) == want_fb, (sorted(fz.fallback), sorted(want_fb))


def test_fallback_is_plain_fprop_plus_bn_apply(models):
  m, _ = models['resnet50']
  fz = freeze(m)
  blk = m.blocks[0]
  x = _input((16, 64, 56, 56), seed=7)
  fz._folded, fz._fallback, fz._calls = [], {}, 0
  got = fz._conv(blk.conv2, x, blk.bn2)
  assert 'blocks.0.bn2' in fz._fallback and fz._calls == 1
  with torch.no_grad():
    want = blk.bn2(blk.conv2(x))        # eval mode: plain fprop, then rigl_bn_apply
  assert torch.equal(got, want)


def test_cuda_graph_replay_equals_eager(models):
  m, x = models['resnet50']
  fz = freeze(m)
  eager = fz(x).clone()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    fz(x)
  torch.cuda.current_stream().wait_stream(side)
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g):
    out = fz(x)
  g.replay()
  torch.cuda.synchronize()
  assert torch.equal(out, eager)


def _wrn_with_harness(seed=0):
  torch.manual_seed(seed)
  m = wl.WideResNet(depth=22, width=2, device=DEV)
  wl.init_masks(m, 'erdos_renyi_kernel', 0.9, seed=0)
  return m, wl.TrainHarness(m)


def _batch(seed):
  g = torch.Generator(device=DEV).manual_seed(seed)
  x = torch.randn(16, 3, 32, 32, device=DEV, generator=g).to(torch.bfloat16).contiguous(
      memory_format=torch.channels_last)
  return x, torch.randint(0, 10, (16,), device=DEV, generator=g)


def test_snapshot_and_refresh():
  torch.backends.cudnn.deterministic = True
  m, h = _wrn_with_harness()
  x, y = _batch(11)
  h.step(x, y)                                   # non-trivial running statistics
  m.eval()
  fz = freeze(m)
  before = fz(x).clone()
  m.train()
  h.step(*_batch(12))                            # the first step of the schedule also updates the masks
  m.eval()
  assert torch.equal(fz(x), before)
  fz.refresh()
  assert torch.equal(fz(x), freeze(m)(x))
  assert not torch.equal(fz(x), before)


def test_frozen_forward_does_not_disturb_training():
  torch.backends.cudnn.deterministic = True
  states = []
  for with_eval in (False, True):
    m, h = _wrn_with_harness()
    fz = freeze(m) if with_eval else None
    h.step(*_batch(21))
    if with_eval:
      fz.refresh()
      fz(_batch(23)[0])
    h.step(*_batch(22))
    torch.cuda.synchronize()
    st = {'param.' + n: p.detach().clone() for n, p in m.named_parameters()}
    st.update({'buf.' + n: b.clone() for n, b in m.named_buffers()})
    st.update({'mask.%d' % i: l.mask.bits.clone() for i, l in enumerate(m.registry.layers())})
    st.update({'mom.' + n: h.inner.state[p]['momentum_buffer'].clone() for n, p in m.named_parameters()
               if 'momentum_buffer' in h.inner.state[p]})
    states.append(st)
  assert states[0].keys() == states[1].keys()
  for k in states[0]:
    assert torch.equal(states[0][k], states[1][k]), k
