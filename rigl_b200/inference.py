"""Frozen sparse inference: the EVAL / PREDICT forward of a trained model.

The reference evaluates with batch norm on its moving averages (`is_training = (mode == TRAIN)`,
imagenet_resnet/imagenet_train_eval.py:544-566, resnet_model.py:41-80).  With running statistics a BN is a
per-channel affine transform known before the conv runs, so `freeze(model)` folds it -- together with the
residual add and the ReLU that follow -- into the epilogue of the masked conv that produces the tensor
(rigl_masked_conv2d_fprop_affine): one bf16 store per conv instead of a store, a BN read and a second store.

`InferenceModel` owns its operands: one pack-plan launch writes `mask * W` for every masked layer into buffers
of its own; the folded scale / shift, the dense convs' weights and the linear biases are its own copies too.  It never writes a layer's `packed`,
`bn_partial` or the training-side pack bookkeeping, so evaluation can be interleaved with training.  `refresh()`
re-packs and re-folds in place (same buffers), so a captured CUDA graph of `forward` stays valid.

Wiring per model (what is folded into a conv epilogue; everything else runs as in `model.eval()`):
  ResNet50     every conv -> BN pair; conv3 also takes the shortcut and the ReLU.  The stem's BN and layers the
               kernel declines (the halo 3x3 layers, unprofitable shapes) run plain fprop + rigl_bn_apply.
  MobileNetV1  the 13 pointwise convs + bn_pw; initial conv, depthwise convs and their BNs as today.
  WideResNet   conv_b + skip as a residual-only epilogue; every BN is pre-activation (rigl_bn_apply).
  MnistFC      hidden layers: bias as `shift`, plus the ReLU; the last layer keeps its fp32 logits.
"""
import ctypes as C

import torch
import torch.nn.functional as F

from . import _cabi
from .norm import FusedBatchNormReLU
from .workloads import DenseConv2d, DepthwiseConv2d

_UNSUPPORTED = -4


def _p(t):
  return None if t is None else t.data_ptr()


def _cl(t):
  return t.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)


class InferenceModel(object):
  """Snapshot of a model for evaluation.  Attributes after each `forward`:
    folded    names of the BNs (or residual adds) applied inside a conv epilogue
    fallback  {name: reason} of those run by rigl_bn_apply
    bn_apply_calls  number of rigl_bn_apply launches (== len(fallback))"""

  def __init__(self, model):
    from . import workloads as wl
    kinds = ((wl.ResNet50, 'resnet50'), (wl.MobileNetV1, 'mobilenet_v1'), (wl.WideResNet, 'wrn'),
             (wl.MnistFC, 'mnist_fc'))
    self.kind = next((k for cls, k in kinds if isinstance(model, cls)), None)
    if self.kind is None:
      raise TypeError('freeze: unsupported model %s' % type(model).__name__)
    self.model = model
    self._names = {id(m): n for n, m in model.named_modules()}
    self._layers = [l for l in model.registry.layers()]
    dev = self._layers[0].weight.device
    self._packed, ents = {}, []
    for l in self._layers:
      if getattr(l, 'patch_mode', False):        # the stem: patch-matrix blob (+ its space-to-depth operand)
        blob = torch.zeros_like(l.packed_patch)
        ents.append((l.weight, l.mask.bits, blob, 1, l._kdim, l._cout))
        if l.s2d_mode:
          self._s2d = torch.zeros_like(l.packed_s2d)
      else:
        blob = torch.zeros_like(l.packed)
        ents.append((l.weight, l.mask.bits, blob, l._taps, l._cin, l._cout))
      self._packed[id(l)] = blob
    descs = (_cabi.PackDesc * len(ents))()
    for d, (w, b, pk, taps, cin, cout) in zip(descs, ents):
      d.weights, d.mask_bits, d.packed, d.taps, d.cin, d.cout = w.data_ptr(), b.data_ptr(), pk.data_ptr(), taps, cin, cout
    self._plan = C.c_void_p(None)
    _cabi.check(_cabi.lib().rigl_pack_plan_create(descs, len(ents), C.byref(self._plan)), 'rigl_pack_plan_create')
    self._plan_keep = ents                       # the plan holds raw pointers into these tensors
    self._bns = [m for m in model.modules() if isinstance(m, FusedBatchNormReLU)]
    self._fold = {id(bn): (torch.empty(bn.channels, device=dev), torch.empty(bn.channels, device=dev))
                  for bn in self._bns}
    self._unit = {}                              # channels -> (ones, zeros): rigl_bn_apply of a plain residual add
    # the un-masked parameters the forward reads (dense convs, linear biases): snapshotted like the masked operands
    self._dense = {id(mod): torch.empty_like(mod.weight) for mod in model.modules()
                   if isinstance(mod, (DenseConv2d, DepthwiseConv2d))}
    self._bias = {id(l): torch.empty_like(l.bias) for l in self._layers if getattr(l, 'bias', None) is not None}
    self.folded, self.fallback, self.bn_apply_calls = [], {}, 0
    self.refresh()

  def __del__(self):
    try:
      if self._plan and self._plan.value:
        _cabi.lib().rigl_pack_plan_destroy(self._plan)
    except Exception:
      pass

  @torch.no_grad()
  def refresh(self):
    """Re-packs every masked operand and re-folds every BN from the model's current state (same buffers)."""
    _cabi.check(_cabi.lib().rigl_pack_plan_run(self._plan, _cabi.stream_ptr()), 'rigl_pack_plan_run')
    for l in self._layers:
      if getattr(l, 's2d_mode', False):
        _cabi.check(_cabi.lib().rigl_stem_s2d_pack_weights(
            l._desc(1, 16, 16), l.weight.data_ptr(), l.mask.bits.data_ptr(), self._s2d.data_ptr(),
            _cabi.stream_ptr()), 'rigl_stem_s2d_pack_weights')
    mods = {id(mod): mod for mod in self.model.modules()}
    for k, w in self._dense.items():
      w.copy_(mods[k].weight)
    for l in self._layers:
      if id(l) in self._bias:
        self._bias[id(l)].copy_(l.bias)
    for bn in self._bns:                          # the formula of FusedBatchNormReLU in eval mode
      scale, shift = self._fold[id(bn)]
      s = bn.weight.detach() * torch.rsqrt(bn.running_var + bn.eps)
      scale.copy_(s)
      shift.copy_(bn.bias.detach() - bn.running_mean * s)
    return self

  # ---- building blocks ----
  def _name(self, m):
    return self._names.get(id(m), type(m).__name__)

  def _apply(self, y, scale, shift, residual, relu, name, reason):
    out = torch.empty_like(y, memory_format=torch.channels_last)
    n, c, h, w = y.shape
    _cabi.check(_cabi.lib().rigl_bn_apply(y.data_ptr(), _p(residual), scale.data_ptr(), shift.data_ptr(), n * h * w,
                                          c, int(relu), out.data_ptr(), _cabi.stream_ptr()), 'rigl_bn_apply')
    self._fallback[name] = reason
    self._calls += 1
    return out

  def _bn(self, bn, y, reason='no masked producer'):
    """A BN that is not folded into a conv: rigl_bn_apply on the folded coefficients."""
    scale, shift = self._fold[id(bn)]
    return self._apply(_cl(y), scale, shift, None, bn.relu, self._name(bn), reason)

  def _conv(self, layer, x, bn=None, residual=None, name=None):
    """layer(x), with the epilogue [relu](acc * scale + shift (+ residual)) when there is a `bn` (scale, shift,
    its ReLU) or a `residual` (plain add) to fold."""
    n, c, h, w = x.shape
    d = layer._desc(n, h, w)
    y = torch.empty((n, layer._cout, d.out_h, d.out_w), dtype=torch.bfloat16, device=x.device,
                    memory_format=torch.channels_last)
    packed = self._packed[id(layer)]
    lib = _cabi.lib()
    if bn is None and residual is None:
      _cabi.check(lib.rigl_masked_conv2d_fprop(d, x.data_ptr(), packed.data_ptr(), y.data_ptr(), None, None, None, 0,
                                               _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
      return y
    scale, shift, relu = None, None, False
    if bn is not None:
      (scale, shift), relu, name = self._fold[id(bn)], bn.relu, self._name(bn)
    rc = lib.rigl_masked_conv2d_fprop_affine(d, x.data_ptr(), packed.data_ptr(), _p(scale), _p(shift), _p(residual),
                                             int(relu), y.data_ptr(), None, 0, _cabi.stream_ptr())
    if rc == 0:
      self._folded.append(name)
      return y
    if rc != _UNSUPPORTED:
      _cabi.check(rc, 'rigl_masked_conv2d_fprop_affine')
    reason = lib.rigl_last_error().decode('utf-8', 'replace')
    _cabi.check(lib.rigl_masked_conv2d_fprop(d, x.data_ptr(), packed.data_ptr(), y.data_ptr(), None, None, None, 0,
                                             _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
    if scale is None:
      scale, shift = self._unit_coeffs(layer._cout, x.device)
    return self._apply(y, scale, shift, residual, relu, name, reason)

  def _unit_coeffs(self, c, dev):
    if c not in self._unit:                      # (allocated on first use; warm up before capturing a graph)
      self._unit[c] = (torch.ones(c, device=dev), torch.zeros(c, device=dev))
    return self._unit[c]

  def _stem(self, layer, x):
    n, c, h, w = x.shape
    d = layer._desc(n, h, w)
    y = torch.empty((n, layer._cout, d.out_h, d.out_w), dtype=torch.bfloat16, device=x.device,
                    memory_format=torch.channels_last)
    lib = _cabi.lib()
    if layer.s2d_mode and lib.rigl_stem_s2d_supported(d):
      xs = torch.empty(int(lib.rigl_stem_s2d_folded_bytes(d)), dtype=torch.uint8, device=x.device)
      _cabi.check(lib.rigl_stem_s2d_fold_input(d, x.data_ptr(), xs.data_ptr(), _cabi.stream_ptr()),
                  'rigl_stem_s2d_fold_input')
      _cabi.check(lib.rigl_stem_s2d_fprop(d, xs.data_ptr(), self._s2d.data_ptr(), y.data_ptr(), _cabi.stream_ptr()),
                  'rigl_stem_s2d_fprop')
      return y
    a = layer._patches(x)
    _cabi.check(lib.rigl_masked_conv2d_fprop(layer._patch_desc(a.shape[0]), a.data_ptr(),
                                             self._packed[id(layer)].data_ptr(), y.data_ptr(), None, None, None, 0,
                                             _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
    return y

  def _linear(self, layer, x, shift=None, relu=False, out_f32=False):
    d = layer._desc(x.shape[0])
    x = layer._as_activation(x, layer._cin)
    packed = self._packed[id(layer)].data_ptr()
    if out_f32:                                   # the logits: fp32 + bias, exactly as the training layer
      y = torch.empty((x.shape[0], layer._cout), dtype=torch.float32, device=x.device)
      _cabi.check(_cabi.lib().rigl_masked_conv2d_fprop(d, x.data_ptr(), packed, None, y.data_ptr(),
                                                       _p(self._bias.get(id(layer))),
                                                       None, 0, _cabi.stream_ptr()), 'rigl_masked_conv2d_fprop')
      return y
    y = torch.empty((x.shape[0], layer._cout), dtype=torch.bfloat16, device=x.device)
    _cabi.check(_cabi.lib().rigl_masked_conv2d_fprop_affine(d, x.data_ptr(), packed, None, _p(shift), None, int(relu),
                                                            y.data_ptr(), None, 0, _cabi.stream_ptr()),
                'rigl_masked_conv2d_fprop_affine')
    self._folded.append(self._name(layer))
    return y

  def _dense_conv(self, m, x):
    """The un-masked convs, as their modules run them, on the snapshot weights."""
    w = self._dense[id(m)]
    if isinstance(m, DepthwiseConv2d):
      if m.native and m.channels % 8 == 0:
        x = _cl(x)
        n, c, h, wd = x.shape
        y = torch.empty((n, c, (h - 1) // m.stride + 1, (wd - 1) // m.stride + 1), dtype=torch.bfloat16,
                        device=x.device, memory_format=torch.channels_last)
        _cabi.check(_cabi.lib().rigl_depthwise3x3_fprop(x.data_ptr(), w.data_ptr(), n, h, wd, c, m.stride, y.data_ptr(),
                                                        _cabi.stream_ptr()), 'rigl_depthwise3x3_fprop')
        return y
      return F.conv2d(x, w.to(torch.bfloat16), None, m.stride, 1, 1, m.channels)
    return F.conv2d(x, w.to(torch.bfloat16), None, m.stride, m.padding, m.dilation, m.groups)

  def _max_pool(self, x, ksize=3, stride=2):
    n, c, h, w = x.shape
    y = torch.empty((n, c, (h + stride - 1) // stride, (w + stride - 1) // stride), dtype=torch.bfloat16,
                    device=x.device, memory_format=torch.channels_last)
    _cabi.check(_cabi.lib().rigl_maxpool_same_forward(x.data_ptr(), n, h, w, c, ksize, stride, y.data_ptr(), None,
                                                      _cabi.stream_ptr()), 'rigl_maxpool_same_forward')
    return y

  # ---- model forwards ----
  def _resnet50(self, m, x):
    x = self._bn(m.initial_bn, self._stem(m.initial_conv, _cl(x)), 'stem: its kernels have no inference epilogue')
    x = self._max_pool(x, 3, 2)
    for blk in m.blocks:
      shortcut = x if blk.proj is None else self._conv(blk.proj, x, blk.proj_bn)
      y = self._conv(blk.conv1, x, blk.bn1)
      y = self._conv(blk.conv2, y, blk.bn2)
      x = self._conv(blk.conv3, y, blk.bn3, residual=shortcut)
    return self._linear(m.final_dense, x.mean(dim=(2, 3)), out_f32=True)

  def _mobilenet(self, m, x):
    x = self._bn(m.initial_bn, self._dense_conv(m.initial_conv, _cl(x)))
    for blk in m.blocks:
      x = self._bn(blk.bn_dw, self._dense_conv(blk.depthwise, x))
      x = self._conv(blk.pointwise, x, blk.bn_pw)
    return self._linear(m.final_dense, x.mean(dim=(2, 3)), out_f32=True)

  def _wrn(self, m, x):
    net = self._dense_conv(m.conv_1, _cl(x))
    for blk in m.blocks:
      skip = net
      net = self._bn(blk.bn_a, net)
      if blk.skip is not None:
        skip = self._conv(blk.skip, net)
      net = self._conv(blk.conv_a, net)
      net = self._bn(blk.bn_b, net)                # dropout is the identity in evaluation
      net = self._conv(blk.conv_b, net, residual=_cl(skip), name=self._name(blk.conv_b) + '+skip')
    net = self._bn(m.final_bn, net)
    return self._linear(m.logits, net.mean(dim=(2, 3)), out_f32=True)

  def _mnist(self, m, x):
    last = len(m.layers) - 1
    for i, l in enumerate(m.layers):
      x = self._linear(l, x, out_f32=True) if i == last else self._linear(l, x, shift=self._bias[id(l)], relu=True)
    return x

  @torch.no_grad()
  def forward(self, images):
    """Logits of the frozen model: same dtype and shape as `model(images)` in eval mode.  No host
    synchronisation and no allocation outside torch's caching allocator: capturable in a CUDA graph for a
    fixed input shape (after one eager call)."""
    self._folded, self._fallback, self._calls = [], {}, 0
    fwd = {'resnet50': self._resnet50, 'mobilenet_v1': self._mobilenet, 'wrn': self._wrn,
           'mnist_fc': self._mnist}[self.kind]
    out = fwd(self.model, images)
    self.folded, self.fallback, self.bn_apply_calls = self._folded, self._fallback, self._calls
    return out

  __call__ = forward


def freeze(model):
  """Snapshot of `model` for EVAL / PREDICT (see the module docstring)."""
  return InferenceModel(model)


def evaluate(logits, labels, label_smoothing):
  """The reference's EVAL metrics (imagenet_train_eval.py:594-606) over one batch:
    eval_accuracy        mean(argmax(logits) == labels)
    top_5_eval_accuracy  mean(in_top_k(logits, labels, 5)): the label's logit has fewer than 5 strictly larger
                         logits (tf.nn.in_top_k counts ties at the boundary as inside); non-finite -> outside
    cross_loss           softmax cross-entropy against label-smoothed one-hot targets, mean over the batch
                         (tf.losses.softmax_cross_entropy(label_smoothing=...), :577-580)
  Returns python floats."""
  z = logits.detach().double()
  labels = labels.to(z.device).long()
  k = z.shape[1]
  target = z.gather(1, labels[:, None])
  top1 = (z.argmax(dim=1) == labels).double().mean()
  top5 = (((z > target).sum(dim=1) < min(5, k)) & torch.isfinite(target[:, 0])).double().mean()
  onehot = F.one_hot(labels, k).double()
  soft = onehot * (1.0 - label_smoothing) + label_smoothing / k
  cross = -(soft * torch.log_softmax(z, dim=1)).sum(dim=1).mean()
  return {'eval_accuracy': float(top1), 'top_5_eval_accuracy': float(top5), 'cross_loss': float(cross)}
