"""Masked conv2d / fully-connected layers on the CUDA hot path.

Mirror of the reference's masked-layer shim rigl/imagenet_resnet/pruning_layers.py
(sparse_conv2d :72-172, sparse_fully_connected :175-248), which delegates to
tf.contrib.model_pruning's masked_conv2d / masked_fully_connected:
  y = conv(x, mask * W) (+ bias)     weights HWIO [kh,kw,Cin,Cout] / [in,out] float32
Each layer owns
  .weight           float32 Parameter in the reference layout, `.name` '<scope>/weights:0'
  .mask             MaskVariable (1-bit bitmap), `.name` '<scope>/mask:0'
  .masked_weights   handle whose `.dense_grad` receives dL/d(mask*W) -- the DENSE
                    gradient RigL ranks for regrowth (sparse_optimizers_base.py:481-484)
and registers itself in `rigl_b200.pruning` (the graph-collection analogue).
Activations are bf16 NHWC: conv inputs are torch tensors of logical shape
[N,C,H,W] in `torch.channels_last` memory format.
"""
import math

import numpy as np
import torch
from torch import nn

from . import _cabi
from . import pruning
from .masks import MaskVariable

import ctypes as C

_WS = {}
import os as _os
# The conv epilogue emits the following BN's batch statistics (column sums / sums of squares of the bf16 output
# slab it has just staged for the TMA store), so the BN forward needs no stats pass over the activation.
# RIGL_FUSE_BN_STATS=0: separate stats pass.
FUSE_BN_STATS = _os.environ.get('RIGL_FUSE_BN_STATS', '1') != '0'
_BN_ROWS = []


def _bn_partial_rows():
  if not _BN_ROWS:
    _BN_ROWS.append(int(_cabi.lib().rigl_bn_partial_rows()))
  return _BN_ROWS[0]


# space-to-depth halo kernels for the 7x7/2 3-channel stem (csrc/stem_s2d.cuh, DESIGN.md 3.7): validated on
# B200 at the start of round 2 (tools/umma_sw32_probe.cu + tests/test_conv_gpu.py::test_conv_stem_s2d_path);
# RIGL_STEM_S2D=0 falls back to the patch-matrix (im2col) stem
STEM_S2D_PATH = _os.environ.get('RIGL_STEM_S2D', '1') != '0'


class Profiler(object):
  """Optional per-call CUDA-event timing of the hot-path kernels (bench.py's roofline leg)."""
  enabled = False
  records = []

  @classmethod
  def start(cls):
    cls.enabled, cls.records = True, []

  @classmethod
  def stop(cls):
    """-> list of (kind, scope, milliseconds); synchronises."""
    cls.enabled = False
    torch.cuda.synchronize()
    out = [(k, sc, s.elapsed_time(e)) for k, sc, s, e in cls.records]
    cls.records = []
    return out


def _timed(kind, layer, fn):
  if not Profiler.enabled:
    return fn()
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  r = fn()
  e.record()
  Profiler.records.append((kind, layer.scope, s, e))
  return r


def _workspace(device, nbytes):
  key = (device, _WS_SLOT[0])          # one scratch buffer per (device, stream role)
  ws = _WS.get(key)
  if ws is None or ws.numel() < nbytes:
    ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
    _WS[key] = ws
  return ws


# ---- dense wgrad on a second stream ---------------------------------------------------------------
# The dense weight gradient of a layer (and mask * grad) is needed only by the optimizer / the mask
# update, not by the rest of the backward pass, while the chain dgrad -> BN backward -> dgrad ... is
# serial and half of it (BN) leaves the tensor cores idle.  With WGRAD_SIDE_STREAM the wgrad kernels
# of layer k run on a forked stream concurrently with the BN backward of layer k-1 (they fit on
# the same SM: 198 KB + <= 16 KB shared memory).  Opt-in (TrainHarness enables it in CUDA-graph mode):
# the weight gradient is then written straight into `weight.grad` on the side stream instead of
# being returned to autograd, and the caller must `join_side_streams()` after `backward()`.
WGRAD_SIDE_STREAM = False
# Set by TrainHarness around backward() when the inner optimizer is optim.FusedMomentumSGD: it forms
# mask * dense_grad while loading the dense gradient, so the layers neither compute nor return the masked
# weight gradient (`weight.grad` stays untouched).
MASKED_GRAD_IN_OPTIMIZER = False
# data_parallel.DataParallel while a backward pass should launch its bucketed all-reduces (set by TrainHarness):
# `layer_done(layer, stream)` is called right after a layer's dense wgrad has been issued on `stream`.
DP_HOOK = None
_WS_SLOT = ['main']
_SIDE = {}
_SIDE_KEEP = []        # tensors the side stream may still be reading (released at the join)


def side_stream(device):
  st = _SIDE.get(device)
  if st is None:
    st = torch.cuda.Stream(device=device)
    _SIDE[device] = st
  return st


_PACKED_AHEAD = set()     # id(layer): operands already packed on the side stream for this step
_PACK_JOIN = {}           # device -> True while the main stream has not yet waited for those packs


def pack_ahead(layers):
  """Packs the operands of `layers` on the side stream (they depend only on weights and masks, not on
  activations), concurrently with whatever the caller's stream does next (the stem of the forward
  pass); the first of these layers to run makes the main stream wait for all of them."""
  layers = [l for l in layers if l.weight.is_cuda]
  if not layers:
    return
  dev = layers[0].weight.device
  main, side = torch.cuda.current_stream(dev), side_stream(dev)
  side.wait_stream(main)                     # weights / masks were last written on the main stream
  with torch.cuda.stream(side):
    for l in layers:
      l.pack()
      _PACKED_AHEAD.add(id(l))
  _PACK_JOIN[dev] = True


class PackPlan(object):
  """ONE launch packing the operands of a fixed list of layers (rigl_pack_plan_*): `mask * W` -> bf16 GEMM
  operands + tile survivor counts for every layer.  Raw pointers are captured, so the plan is rebuilt whenever a
  weight / bitmap / blob is reallocated."""

  def __init__(self):
    self._plan, self._key = C.c_void_p(None), None

  def __del__(self):
    try:
      self._destroy()
    except Exception:
      pass

  def _destroy(self):
    if self._plan and self._plan.value:
      _cabi.lib().rigl_pack_plan_destroy(self._plan)
      self._plan = C.c_void_p(None)

  @staticmethod
  def _entries(layer):
    """(weights ptr, bitmap ptr, blob ptr, taps, cin, cout) of every generic blob `layer.pack()` would write."""
    if getattr(layer, 'patch_mode', False):
      return [(layer.weight.data_ptr(), layer.mask.bits.data_ptr(), layer.packed_patch.data_ptr(), 1, layer._kdim,
               layer._cout)]
    return [(layer.weight.data_ptr(), layer.mask.bits.data_ptr(), layer.packed.data_ptr(), layer._taps, layer._cin,
             layer._cout)]

  def run(self, layers):
    ents = [e for l in layers for e in self._entries(l)]
    key = tuple(ents)
    if key != self._key:
      self._destroy()
      descs = (_cabi.PackDesc * len(ents))()
      for d, (w, b, pk, taps, cin, cout) in zip(descs, ents):
        d.weights, d.mask_bits, d.packed, d.taps, d.cin, d.cout = w, b, pk, taps, cin, cout
      plan = C.c_void_p(None)
      _cabi.check(_cabi.lib().rigl_pack_plan_create(descs, len(ents), C.byref(plan)), 'rigl_pack_plan_create')
      self._plan, self._key = plan, key
    _cabi.check(_cabi.lib().rigl_pack_plan_run(self._plan, _cabi.stream_ptr()), 'rigl_pack_plan_run')
    for l in layers:          # the small special-format stem operands are not part of the batch
      if getattr(l, 's2d_mode', False):
        l.pack_special()


_PACK_PLANS = {}


class _AllLayers(object):
  scope = 'all_layers'


_ALL_LAYERS = _AllLayers()


def pack_all(layers):
  """Packs the operands of all `layers` with one launch on the current stream; their forward passes then skip
  the per-layer pack for this step."""
  layers = [l for l in layers if l.weight.is_cuda]
  if not layers:
    return
  key = tuple(id(l) for l in layers)
  plan = _PACK_PLANS.get(key)
  if plan is None:
    plan = _PACK_PLANS[key] = PackPlan()
  _timed('pack', _ALL_LAYERS, lambda: plan.run(layers))
  for l in layers:
    _PACKED_AHEAD.add(id(l))


def _pack_for_forward(layer):
  if id(layer) in _PACKED_AHEAD:
    _PACKED_AHEAD.discard(id(layer))
    dev = layer.weight.device
    if _PACK_JOIN.get(dev):
      torch.cuda.current_stream(dev).wait_stream(side_stream(dev))
      _PACK_JOIN[dev] = False
    return
  _timed('pack', layer, layer.pack)


def join_side_streams():
  """The current stream of every device waits for the forked wgrad work; releases the kept tensors."""
  for dev, st in _SIDE.items():
    torch.cuda.current_stream(dev).wait_stream(st)
  del _SIDE_KEEP[:]


class NamedParameter(nn.Parameter):
  """Parameter that can carry the TF-style variable name ('<scope>/weights:0') and the
  `initial_value` tensor some grow-init modes read (sparse_optimizers_base.py:374-380)."""
  name = None
  initial_value = None


class MaskedWeights(object):
  """Handle for `mask * weights`; carries the dense gradient buffer."""

  def __init__(self, scope, numel, device):
    self.name = scope + '/masked_weights:0'
    self.dense_grad = torch.zeros(numel, dtype=torch.float32, device=device)
    self.fresh = False        # True once a backward has written dense_grad this step


def variance_scaling_(tensor_hwio, scale=2.0):
  """fan_in variance scaling on an HWIO / [in,out] tensor (resnet_model.py:283 uses
  tf.variance_scaling_initializer; a plain normal is used here -- only the
  synthetic weight distribution depends on it, not parity)."""
  fan_in = int(np.prod(tensor_hwio.shape[:-1]))
  with torch.no_grad():
    tensor_hwio.normal_(0., math.sqrt(scale / max(fan_in, 1)))
  return tensor_hwio


class _MaskedConvFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, weight, bias, layer, out_f32):
    _pack_for_forward(layer)
    y = _timed('fprop', layer, lambda: layer._fprop(x, bias, out_f32))
    ctx.layer = layer
    ctx.save_for_backward(x)
    ctx.has_bias = bias is not None
    return y

  @staticmethod
  def backward(ctx, dy):
    layer = ctx.layer
    x, = ctx.saved_tensors
    dy16 = layer._as_activation(dy, layer.out_channels)
    dx = _timed('dgrad', layer, lambda: layer._dgrad(dy16, x)) if ctx.needs_input_grad[0] else None
    mw = layer.masked_weights
    gw = None
    if WGRAD_SIDE_STREAM and x.is_cuda and not Profiler.enabled:
      want_gw = ctx.needs_input_grad[1] and not MASKED_GRAD_IN_OPTIMIZER
      if want_gw and layer.weight.grad is None:
        layer.weight.grad = torch.zeros_like(layer.weight)
      patch_keep = getattr(layer, '_patch_cache', None)     # (the stem's patch matrix is dropped inside _wgrad)
      main, side = torch.cuda.current_stream(x.device), side_stream(x.device)
      side.wait_stream(main)                       # x and dy16 were produced on the main stream
      _WS_SLOT[0] = 'side'
      try:
        with torch.cuda.stream(side):
          layer._wgrad(x, dy16, mw.dense_grad, accumulate=mw.fresh)
          if want_gw:
            layer.mask.apply_to(mw.dense_grad, out=layer.weight.grad.view(-1))
      finally:
        _WS_SLOT[0] = 'main'
      _SIDE_KEEP.append((x, dy16, patch_keep))     # no reuse of these blocks before the join
      mw.fresh = True
      mw.dense_grad.rigl_reduced = False           # rewritten: not yet summed over the replicas
      if DP_HOOK is not None:
        DP_HOOK.layer_done(layer, side)
    else:
      _timed('wgrad', layer, lambda: layer._wgrad(x, dy16, mw.dense_grad, accumulate=mw.fresh))
      mw.fresh = True
      mw.dense_grad.rigl_reduced = False
      if DP_HOOK is not None:
        DP_HOOK.layer_done(layer, None)
      if ctx.needs_input_grad[1] and not MASKED_GRAD_IN_OPTIMIZER:
        gw = layer.mask.apply_to(mw.dense_grad).view(layer.weight.shape)
    gb = None
    if ctx.has_bias and ctx.needs_input_grad[2]:
      gb = dy.float().reshape(-1, layer.out_channels).sum(0) if dy.dim() == 2 else \
          dy.float().sum(dim=(0, 2, 3))
    return dx, gw, gb, None, None


class _MaskedLayer(nn.Module):
  is_rigl_masked_layer = True

  def _setup(self, scope, shape_hwio, device, registry, kernel_initializer):
    self.scope = scope
    w = torch.empty(shape_hwio, dtype=torch.float32, device=device)
    (kernel_initializer or variance_scaling_)(w)
    self.weight = NamedParameter(w)
    self.weight.name = scope + '/weights:0'
    self.mask = MaskVariable(scope, shape_hwio, device)
    self.masked_weights = MaskedWeights(scope, w.numel(), device)
    taps = int(np.prod(shape_hwio[:-2])) if len(shape_hwio) > 2 else 1
    self._taps, self._cin, self._cout = taps, int(shape_hwio[-2]), int(shape_hwio[-1])
    nbytes = int(_cabi.lib().rigl_packed_weights_bytes(taps, self._cin, self._cout))
    self.packed = torch.zeros(nbytes, dtype=torch.uint8, device=device)
    (registry if registry is not None else pruning.default_registry()).register(self)

  @property
  def in_channels(self):
    return self._cin

  @property
  def out_channels(self):
    return self._cout

  def pack(self):
    """mask * W -> bf16 GEMM operands (both K-major layouts) + tile survivor counts."""
    _cabi.check(_cabi.lib().rigl_pack_masked_weights(
        self.weight.data_ptr(), self.mask.bits.data_ptr(), self._taps, self._cin, self._cout,
        self.packed.data_ptr(), _cabi.stream_ptr()), 'rigl_pack_masked_weights')

  def extra_repr(self):
    return '%s, hwio=%s' % (self.scope, tuple(self.weight.shape))


class SparseConv2d(_MaskedLayer):
  """Masked 2-D convolution, square kernel/stride, no bias (resnet_model.py:296).

  Layers whose input-channel count is not a multiple of 8 (the 7x7x3 stem) run in
  "patch-matrix" mode: `rigl_im2col_nhwc` builds the [pixels, k*k*Cin] matrix once per
  forward and the conv becomes a masked dense layer over it with the SAME HWIO weights
  and mask (HWIO flattened over (kh,kw,ci) is exactly the [in,out] matrix)."""

  def __init__(self, in_channels, units, kernel_size, strides=1, padding='SAME', name=None,
               kernel_initializer=None, device='cuda', registry=None):
    super(SparseConv2d, self).__init__()
    k = int(kernel_size[0] if isinstance(kernel_size, (tuple, list)) else kernel_size)
    s = int(strides[0] if isinstance(strides, (tuple, list)) else strides)
    if padding not in ('SAME', 'VALID', 'FIXED'):
      raise ValueError('padding must be SAME, VALID or FIXED')
    self.ksize, self.stride = k, s
    # 'FIXED' = conv2d_fixed_padding (resnet_model.py:234-303): explicit (k-1)//2 pad, then VALID.
    # 'SAME'  = TensorFlow SAME: out = ceil(in/s), pad_before = pad_total // 2 (asymmetric for
    #           stride 2 on even inputs -- what cifar_resnet/resnet_model.py:158-181 uses).
    self.padding = padding
    self._setup(name or 'Conv', (k, k, int(in_channels), int(units)), device, registry,
                kernel_initializer)
    self.patch_mode = (int(in_channels) % 8 != 0) and k > 1
    if self.patch_mode:
      self._kdim = k * k * int(in_channels)
      self._kpitch = (self._kdim + 7) // 8 * 8
      nbytes = int(_cabi.lib().rigl_packed_weights_bytes(1, self._kdim, self._cout))
      self.packed_patch = torch.zeros(nbytes, dtype=torch.uint8, device=device)
    self.s2d_mode = bool(STEM_S2D_PATH and self.patch_mode and k == 7 and s == 2 and int(in_channels) <= 3 and
                         int(units) <= 64 and int(units) % 8 == 0 and padding == 'FIXED')
    if self.s2d_mode:
      self.packed_s2d = torch.zeros(16 * int(units) * 32, dtype=torch.uint8, device=device)
    self._use_s2d = False
    self.collect_bn_stats = False   # set by the model when a FusedBatchNormReLU consumes this output
    self.bn_partial = None

  def pack(self):
    if self.patch_mode:      # both stem operand forms are tiny; which one runs is decided per call
      _cabi.check(_cabi.lib().rigl_pack_masked_weights(
          self.weight.data_ptr(), self.mask.bits.data_ptr(), 1, self._kdim, self._cout,
          self.packed_patch.data_ptr(), _cabi.stream_ptr()), 'rigl_pack_masked_weights')
      self.pack_special()
    else:
      super(SparseConv2d, self).pack()

  def pack_special(self):
    """The stem's own operand format (space-to-depth kernels)."""
    if self.s2d_mode:
      d = self._desc(1, 16, 16)
      _cabi.check(_cabi.lib().rigl_stem_s2d_pack_weights(
          d, self.weight.data_ptr(), self.mask.bits.data_ptr(), self.packed_s2d.data_ptr(),
          _cabi.stream_ptr()), 'rigl_stem_s2d_pack_weights')

  @property
  def pad(self):
    """pad_before when it does not depend on the input size (FIXED / VALID / stride-1 SAME)."""
    return 0 if self.padding == 'VALID' else (self.ksize - 1) // 2

  def out_size(self, size):
    """(output extent, pad_before) along one spatial dimension."""
    k, s = self.ksize, self.stride
    if self.padding == 'SAME':
      out = (size + s - 1) // s
      return out, max((out - 1) * s + k - size, 0) // 2
    if self.padding == 'FIXED':
      return (size + 2 * ((k - 1) // 2) - k) // s + 1, (k - 1) // 2
    return (size - k) // s + 1, 0

  def _desc(self, n, h, w):
    d = _cabi.ConvDesc()
    d.batch, d.in_h, d.in_w, d.cin = n, h, w, self._cin
    d.out_h, pad_h = self.out_size(h)
    d.out_w, pad_w = self.out_size(w)
    if pad_h != pad_w:
      raise ValueError('unequal vertical/horizontal padding is not supported (%d vs %d)' % (pad_h, pad_w))
    d.cout, d.ksize, d.stride, d.pad = self._cout, self.ksize, self.stride, pad_h
    d.x_pitch = 0
    return d

  def _patch_desc(self, rows):
    d = _cabi.ConvDesc()
    d.batch, d.in_h, d.in_w, d.cin = rows, 1, 1, self._kdim
    d.out_h, d.out_w, d.cout, d.ksize, d.stride, d.pad = 1, 1, self._cout, 1, 1, 0
    d.x_pitch = self._kpitch
    return d

  @staticmethod
  def _as_activation(t, channels):
    if t.dtype != torch.bfloat16:
      t = t.to(torch.bfloat16)
    return t.contiguous(memory_format=torch.channels_last)

  def _patches(self, x):
    n, c, h, w = x.shape
    d = self._desc(n, h, w)
    rows = n * d.out_h * d.out_w
    a = torch.empty((rows, self._kpitch), dtype=torch.bfloat16, device=x.device)
    _cabi.check(_cabi.lib().rigl_im2col_nhwc(d, x.data_ptr(), a.data_ptr(), self._kpitch,
                                             _cabi.stream_ptr()), 'rigl_im2col_nhwc')
    return a

  def _fprop(self, x, bias, out_f32):
    n, c, h, w = x.shape
    d = self._desc(n, h, w)
    y = torch.empty((n, self._cout, d.out_h, d.out_w), dtype=torch.bfloat16, device=x.device,
                    memory_format=torch.channels_last)
    packed, src = self.packed, x
    self._use_s2d = bool(self.s2d_mode and _cabi.lib().rigl_stem_s2d_supported(d))
    if self._use_s2d:
      xs = torch.empty(int(_cabi.lib().rigl_stem_s2d_folded_bytes(d)), dtype=torch.uint8, device=x.device)
      _cabi.check(_cabi.lib().rigl_stem_s2d_fold_input(d, x.data_ptr(), xs.data_ptr(), _cabi.stream_ptr()),
                  'rigl_stem_s2d_fold_input')
      _cabi.check(_cabi.lib().rigl_stem_s2d_fprop(d, xs.data_ptr(), self.packed_s2d.data_ptr(), y.data_ptr(),
                                                  _cabi.stream_ptr()), 'rigl_stem_s2d_fprop')
      self._patch_cache = xs
      return y
    if self.patch_mode:
      self._patch_cache = src = self._patches(x)
      d, packed = self._patch_desc(src.shape[0]), self.packed_patch
    ws = _workspace(x.device, _cabi.lib().rigl_conv_workspace_bytes(d))
    self.bn_partial = None
    if self.collect_bn_stats and self.training and FUSE_BN_STATS:
      # the epilogue also emits per-CTA column sums / sums of squares of the output (BN statistics)
      rows = C.c_int(0)
      part = torch.empty(_bn_partial_rows() * 2 * self._cout, dtype=torch.float32, device=x.device)
      rc = _cabi.lib().rigl_masked_conv2d_fprop_bnstats(
          d, src.data_ptr(), packed.data_ptr(), y.data_ptr(), part.data_ptr(), C.byref(rows), ws.data_ptr(),
          ws.numel(), _cabi.stream_ptr())
      if rc == 0:
        self.bn_partial = (part, rows.value, y.data_ptr())
        return y
      if rc != -4:        # RIGL_ERR_UNSUPPORTED: fall through to the plain call
        _cabi.check(rc, 'rigl_masked_conv2d_fprop_bnstats')
    _cabi.check(_cabi.lib().rigl_masked_conv2d_fprop(
        d, src.data_ptr(), packed.data_ptr(), y.data_ptr(), None, None, ws.data_ptr(),
        ws.numel(), _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
    return y

  def _dgrad(self, dy, x):
    n, c, h, w = x.shape
    d = self._desc(n, h, w)
    if self.patch_mode:                 # rare (image gradients): CUDA-core kernels on the conv form
      super(SparseConv2d, self).pack()
    dx = torch.empty_like(x, memory_format=torch.channels_last)
    ws = _workspace(x.device, _cabi.lib().rigl_conv_workspace_bytes(d))
    _cabi.check(_cabi.lib().rigl_masked_conv2d_dgrad(
        d, dy.data_ptr(), self.packed.data_ptr(), dx.data_ptr(), ws.data_ptr(), ws.numel(),
        _cabi.stream_ptr()), 'rigl_masked_conv2d_dgrad')
    return dx

  def _wgrad(self, x, dy, out, accumulate):
    n, c, h, w = x.shape
    d, src = self._desc(n, h, w), x
    if self._use_s2d and getattr(self, '_patch_cache', None) is not None:
      xs, self._patch_cache = self._patch_cache, None
      ws = _workspace(x.device, _cabi.lib().rigl_stem_s2d_workspace_bytes(d))
      _cabi.check(_cabi.lib().rigl_stem_s2d_wgrad(
          d, xs.data_ptr(), dy.data_ptr(), out.data_ptr(), 1.0 if accumulate else 0.0, ws.data_ptr(),
          ws.numel(), _cabi.stream_ptr()), 'rigl_stem_s2d_wgrad')
      return
    if self.patch_mode:
      src = self._patch_cache if getattr(self, '_patch_cache', None) is not None else self._patches(x)
      self._patch_cache = None
      d = self._patch_desc(src.shape[0])
    ws = _workspace(x.device, _cabi.lib().rigl_conv_workspace_bytes(d))
    _cabi.check(_cabi.lib().rigl_conv2d_wgrad_dense(
        d, src.data_ptr(), dy.data_ptr(), out.data_ptr(), 1.0 if accumulate else 0.0, ws.data_ptr(),
        ws.numel(), _cabi.stream_ptr()), 'rigl_conv2d_wgrad_dense')

  def forward(self, x):
    if x.dim() != 4:
      raise ValueError('Rank not supported {}'.format(x.dim()))
    if x.shape[1] != self._cin:
      raise ValueError('expected %d input channels, got %d' % (self._cin, x.shape[1]))
    x = self._as_activation(x, self._cin)
    return _MaskedConvFn.apply(x, self.weight, None, self, False)


class SparseLinear(_MaskedLayer):
  """Masked fully-connected layer, weights [in,out], dense zero-init bias."""

  def __init__(self, in_features, units, use_bias=True, name=None, kernel_initializer=None,
               device='cuda', registry=None, out_dtype=torch.bfloat16):
    super(SparseLinear, self).__init__()
    self.ksize, self.stride, self.pad = 1, 1, 0
    self.out_dtype = out_dtype
    self._setup(name or 'Dense', (int(in_features), int(units)), device, registry,
                kernel_initializer)
    if use_bias:
      self.bias = NamedParameter(torch.zeros(int(units), dtype=torch.float32, device=device))
      self.bias.name = self.scope + '/biases:0'
    else:
      self.register_parameter('bias', None)

  def _desc(self, m):
    d = _cabi.ConvDesc()
    d.batch, d.in_h, d.in_w, d.cin = m, 1, 1, self._cin
    d.out_h, d.out_w, d.cout, d.ksize, d.stride, d.pad = 1, 1, self._cout, 1, 1, 0
    d.x_pitch = 0
    return d

  @staticmethod
  def _as_activation(t, channels):
    t = t.reshape(-1, channels)
    if t.dtype != torch.bfloat16:
      t = t.to(torch.bfloat16)
    return t.contiguous()

  def _fprop(self, x, bias, out_f32):
    d = self._desc(x.shape[0])
    ws = _workspace(x.device, _cabi.lib().rigl_conv_workspace_bytes(d))
    y16 = None if out_f32 else torch.empty((x.shape[0], self._cout), dtype=torch.bfloat16, device=x.device)
    y32 = torch.empty((x.shape[0], self._cout), dtype=torch.float32, device=x.device) if out_f32 else None
    _cabi.check(_cabi.lib().rigl_masked_conv2d_fprop(
        d, x.data_ptr(), self.packed.data_ptr(), None if y16 is None else y16.data_ptr(),
        None if y32 is None else y32.data_ptr(), None if bias is None else bias.data_ptr(),
        ws.data_ptr(), ws.numel(), _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
    return y32 if out_f32 else y16

  def _dgrad(self, dy, x):
    d = self._desc(x.shape[0])
    dx = torch.empty_like(x)
    ws = _workspace(x.device, _cabi.lib().rigl_conv_workspace_bytes(d))
    _cabi.check(_cabi.lib().rigl_masked_conv2d_dgrad(
        d, dy.data_ptr(), self.packed.data_ptr(), dx.data_ptr(), ws.data_ptr(), ws.numel(),
        _cabi.stream_ptr()), 'rigl_masked_conv2d_dgrad')
    return dx

  def _wgrad(self, x, dy, out, accumulate):
    d = self._desc(x.shape[0])
    ws = _workspace(x.device, _cabi.lib().rigl_conv_workspace_bytes(d))
    _cabi.check(_cabi.lib().rigl_conv2d_wgrad_dense(
        d, x.data_ptr(), dy.data_ptr(), out.data_ptr(), 1.0 if accumulate else 0.0, ws.data_ptr(),
        ws.numel(), _cabi.stream_ptr()), 'rigl_conv2d_wgrad_dense')

  def forward(self, x):
    lead = x.shape[:-1]
    x2 = self._as_activation(x, self._cin)
    y = _MaskedConvFn.apply(x2, self.weight, self.bias, self, self.out_dtype == torch.float32)
    return y.reshape(*lead, self._cout)


# ---- functional, reference-signature entry points (variable-scope style reuse) ----
_SCOPED = {}


def reset_scopes():
  _SCOPED.clear()


def sparse_conv2d(x, units, kernel_size, activation=None, use_bias=False, kernel_initializer=None,
                  kernel_regularizer=None, bias_initializer=None, biases_regularizer=None,
                  sparsity_technique='baseline', normalizer_fn=None, strides=(1, 1), padding='SAME',
                  data_format='channels_last', name=None):
  """Reference-signature conv (pruning_layers.py:72-86).  `x` is a 4-D bf16 tensor of
  logical shape [N,C,H,W] (channels_last memory = NHWC).  The layer object is created
  on first use of `name` and reused afterwards (variable_scope reuse semantics)."""
  if data_format not in ('channels_last', 'channels_first'):
    raise ValueError('Not a valid channel string:', data_format)
  if x.dim() != 4:
    raise ValueError('Rank not supported {}'.format(x.dim()))
  key = ('conv', name)
  layer = _SCOPED.get(key) if name else None
  if layer is None:
    if sparsity_technique == 'threshold':
      layer = SparseConv2d(x.shape[1], units, kernel_size, strides=strides, padding=padding,
                           name=name, kernel_initializer=kernel_initializer, device=x.device)
    elif sparsity_technique == 'baseline':
      k = kernel_size[0] if isinstance(kernel_size, (tuple, list)) else kernel_size
      s = strides[0] if isinstance(strides, (tuple, list)) else strides
      layer = nn.Conv2d(x.shape[1], units, k, stride=s, padding=(k - 1) // 2 if padding != 'VALID' else 0,
                        bias=use_bias, device=x.device, dtype=x.dtype)
    else:
      raise ValueError('Unsupported sparsity technique {}'.format(sparsity_technique))
    if name:
      _SCOPED[key] = layer
  y = layer(x)
  if normalizer_fn is not None:
    y = normalizer_fn(y)
  return activation(y) if activation is not None else y


def sparse_fully_connected(x, units, activation=None, use_bias=True, kernel_initializer=None,
                           kernel_regularizer=None, bias_initializer=None, biases_regularizer=None,
                           sparsity_technique='baseline', name=None):
  """Reference-signature dense layer (pruning_layers.py:175-184)."""
  key = ('dense', name)
  layer = _SCOPED.get(key) if name else None
  if layer is None:
    if sparsity_technique == 'threshold':
      layer = SparseLinear(x.shape[-1], units, use_bias=use_bias, name=name,
                           kernel_initializer=kernel_initializer, device=x.device)
    elif sparsity_technique == 'baseline':
      layer = nn.Linear(x.shape[-1], units, bias=use_bias, device=x.device, dtype=x.dtype)
    else:
      raise ValueError('Unsupported sparsity technique {}'.format(sparsity_technique))
    if name:
      _SCOPED[key] = layer
  y = layer(x)
  return activation(y) if activation is not None else y
