"""Inference forward of the sparse models: today's eval path vs the frozen, epilogue-fused path (rigl_b200.inference).

  python tools/bench_inference.py [--configs c2,c4] [--batches 256,1000] [--seconds 1.0] [--json OUT]
  python tools/bench_inference.py --shapes [--shape-batch 256] [--shape-seconds 0.3] [--json OUT]

Models and masks as bench.py builds them: C2 = ResNet-50 ERK 80 %, C4 = MobileNet-v1 uniform 90 % on the pointwise
convs + classifier.  BN running statistics are filled by one train-mode forward at momentum 1 after randomising gamma
and beta (the default zero gamma of the last BN of a ResNet block would make the residual branch vanish).

Per config and batch, timed with CUDA events over a window of at least --seconds after warm-up:
  (a) eval      model.eval() + torch.no_grad() forward (what evaluation runs today)
  (b) frozen    InferenceModel.forward, eager
  (c) graph     InferenceModel.forward captured once in a CUDA graph and replayed
plus images/s, per-kind kernel time of (a) and (b) from a separate torch.profiler pass, and the largest logit
difference between (a) and (b).

--shapes: for every distinct ResNet-50 and MobileNet-v1 conv that has a BN to fold, the fused call
(rigl_masked_conv2d_fprop_affine, forced on with RIGL_AFFINE_ALWAYS=1) against the plain fprop + rigl_bn_apply,
each timed over a rotation of input / output buffers larger than the 126 MB L2 (so both read HBM as in a forward
pass).  This is the table the profitability rule in tc_fprop rests on (DESIGN.md 3.8).
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {'c2': ('resnet50', 'erdos_renyi_kernel', 0.8), 'c4': ('mobilenet_v1', 'random', 0.9)}


def gpu_info():
  out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  return out.stdout.strip().splitlines()[0] if out.returncode == 0 else 'nvidia-smi failed: ' + out.stdout.strip()


def build(cfg, dev):
  import torch
  from rigl_b200 import workloads as wl
  kind, method, sparsity = CONFIGS[cfg]
  torch.manual_seed(0)
  m = wl.ResNet50(device=dev) if kind == 'resnet50' else wl.MobileNetV1(device=dev)
  wl.init_masks(m, method, sparsity, seed=0)
  g = torch.Generator(device=dev).manual_seed(5)
  bns = [b for b in m.modules() if isinstance(b, wl.FusedBatchNormReLU)]
  with torch.no_grad():
    for bn in bns:
      sign = torch.randint(0, 2, (bn.channels,), device=dev, generator=g) * 2 - 1
      bn.weight.copy_(sign * (0.5 + torch.rand(bn.channels, device=dev, generator=g)))
      bn.bias.copy_(0.2 * torch.randn(bn.channels, device=dev, generator=g))
      bn.momentum = 1.0
    m.train()
    m(images(64, dev, seed=9))
    for bn in bns:
      bn.momentum = 0.1
  m.eval()
  return m


def images(n, dev, seed=1):
  import torch
  g = torch.Generator(device=dev).manual_seed(seed)
  return torch.randn(n, 3, 224, 224, device=dev, generator=g).to(torch.bfloat16).contiguous(
      memory_format=torch.channels_last)


def timed(fn, seconds):
  """ms per call: warm-up, then one CUDA-event window of at least `seconds`."""
  import time
  import torch
  for _ in range(3):
    fn()
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  for _ in range(3):
    fn()
  torch.cuda.synchronize()
  per = (time.perf_counter() - t0) / 3
  reps = max(5, int(math.ceil(seconds / max(per, 1e-6))))
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(reps):
    fn()
  e.record()
  torch.cuda.synchronize()
  ms = s.elapsed_time(e)
  return ms / reps, reps, ms / 1e3


def kind_of(name):
  if any(k in name for k in ('k_igemm', 'k_halo3x3', 'k_stem_s2d', 'k_simt_fprop', 'k_im2col')):
    return 'fprop'
  if 'k_bn_' in name:
    return 'bn'
  if 'maxpool' in name or 'k_depthwise' in name or 'conv' in name.lower():
    return 'pool' if 'maxpool' in name else 'other_conv'
  return 'other'


def per_kind(fn):
  """ms per call by kernel kind, from torch.profiler over 3 calls (separate from the timed window)."""
  import torch
  from torch.profiler import ProfilerActivity, profile
  fn()
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
      fn()
    torch.cuda.synchronize()
  out = {}
  for ev in prof.key_averages():
    t = getattr(ev, 'self_device_time_total', None)
    if t is None:
      t = getattr(ev, 'self_cuda_time_total', 0)
    if t <= 0:
      continue
    k = kind_of(ev.key)
    out[k] = out.get(k, 0.0) + t / 1e3 / 3
  return {k: round(v, 4) for k, v in sorted(out.items())}


def run_forward(args, dev):
  import torch
  from rigl_b200.inference import freeze
  res = []
  for cfg in args.configs.split(','):
    model = build(cfg, dev)
    fz = freeze(model)
    for b in [int(v) for v in args.batches.split(',')]:
      x = images(b, dev)
      with torch.no_grad():
        eval_fwd = lambda: model(x)
        a = eval_fwd().float()
      bl = fz(x).float()
      diff = float((a - bl).abs().max())
      rel = float((a.double() - bl.double()).norm() / a.double().norm())
      t_a = timed(eval_fwd, args.seconds)
      t_b = timed(lambda: fz(x), args.seconds)
      side = torch.cuda.Stream()
      side.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(side):
        fz(x)
      torch.cuda.current_stream().wait_stream(side)
      graph = torch.cuda.CUDAGraph()
      with torch.cuda.graph(graph):
        gout = fz(x)
      t_c = timed(graph.replay, args.seconds)
      torch.cuda.synchronize()
      row = {'config': cfg, 'batch': b,
             'eval_ms': round(t_a[0], 4), 'frozen_ms': round(t_b[0], 4), 'graph_ms': round(t_c[0], 4),
             'eval_img_s': round(b / t_a[0] * 1e3, 1), 'frozen_img_s': round(b / t_b[0] * 1e3, 1),
             'graph_img_s': round(b / t_c[0] * 1e3, 1),
             'window_s': {'eval': round(t_a[2], 3), 'frozen': round(t_b[2], 3), 'graph': round(t_c[2], 3)},
             'max_abs_logit_diff_eval_vs_frozen': diff, 'rel_l2_eval_vs_frozen': rel,
             'graph_equals_eager': bool(torch.equal(gout.float(), bl)),
             'kernel_ms_by_kind': {'eval': per_kind(eval_fwd), 'frozen': per_kind(lambda: fz(x))},
             'folded': len(fz.folded), 'fallback': sorted(fz.fallback)}
      del graph
      print(json.dumps(row), flush=True)
      res.append(row)
    del fz, model
    torch.cuda.empty_cache()
  return res


def run_shapes(args, dev):
  import torch
  from rigl_b200 import _cabi
  from rigl_b200.inference import InferenceModel, freeze
  lib = _cabi.lib()
  rows = []
  for cfg in ('c2', 'c4'):
    model = build(cfg, dev)
    fz = freeze(model)
    seen = []
    orig = InferenceModel._conv

    def record(self, layer, x, bn=None, residual=None, name=None):
      if bn is not None:
        seen.append((layer, tuple(x.shape), bn, residual is not None))
      return orig(self, layer, x, bn, residual, name)
    InferenceModel._conv = record
    try:
      fz(images(args.shape_batch, dev))
    finally:
      InferenceModel._conv = orig
    done = set()
    for layer, xs, bn, has_res in seen:
      n, c, h, w = xs
      key = (n, h, w, c, layer._cout, layer.ksize, layer.stride, has_res)
      if key in done:
        continue
      done.add(key)
      d = layer._desc(n, h, w)
      ybytes = n * d.out_h * d.out_w * layer._cout * 2
      per_call = n * h * w * c * 2 + ybytes * (3 if has_res else 2)
      copies = max(2, int(math.ceil(300e6 / per_call)))
      xs_ = [torch.randn(n, c, h, w, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
             for _ in range(copies)]
      mk = lambda: torch.randn(n, layer._cout, d.out_h, d.out_w, device=dev).to(torch.bfloat16).contiguous(
          memory_format=torch.channels_last)
      ys, tmp = [mk() for _ in range(copies)], [mk() for _ in range(copies)]
      rs = [mk() for _ in range(copies)] if has_res else [None] * copies
      scale, shift = fz._fold[id(bn)]
      packed = fz._packed[id(layer)].data_ptr()
      st = _cabi.stream_ptr()
      it = [0]
      p = lambda t: None if t is None else t.data_ptr()

      def fused():
        i = it[0] = (it[0] + 1) % copies
        _cabi.check(lib.rigl_masked_conv2d_fprop_affine(d, xs_[i].data_ptr(), packed, scale.data_ptr(),
                                                        shift.data_ptr(), p(rs[i]), int(bn.relu), ys[i].data_ptr(),
                                                        None, 0, st), 'affine')

      def plain_apply():
        i = it[0] = (it[0] + 1) % copies
        _cabi.check(lib.rigl_masked_conv2d_fprop(d, xs_[i].data_ptr(), packed, tmp[i].data_ptr(), None, None, None, 0,
                                                 st), 'fprop')
        _cabi.check(lib.rigl_bn_apply(tmp[i].data_ptr(), p(rs[i]), scale.data_ptr(), shift.data_ptr(),
                                      n * d.out_h * d.out_w, layer._cout, int(bn.relu), ys[i].data_ptr(), st),
                    'bn_apply')
      rc = lib.rigl_masked_conv2d_fprop_affine(d, xs_[0].data_ptr(), packed, scale.data_ptr(), shift.data_ptr(),
                                               p(rs[0]), int(bn.relu), ys[0].data_ptr(), None, 0, st)
      if rc != 0:                                 # the halo layers: no fused form exists
        row = {'config': cfg, 'layer': layer.scope, 'n': n, 'h': h, 'w': w, 'cin': c, 'cout': layer._cout,
               'k': layer.ksize, 'stride': layer.stride, 'residual': has_res, 'K': layer.ksize ** 2 * c,
               'fused_ms': None, 'plain_apply_ms': round(timed(plain_apply, args.shape_seconds)[0], 4),
               'declined': lib.rigl_last_error().decode()}
        print(json.dumps(row), flush=True)
        rows.append(row)
        continue
      # alternate the two forms twice so that drift in clocks hits both
      tf, tp = [], []
      for _ in range(2):
        tf.append(timed(fused, args.shape_seconds)[0])
        tp.append(timed(plain_apply, args.shape_seconds)[0])
      f, pa = min(tf), min(tp)
      row = {'config': cfg, 'layer': layer.scope, 'n': n, 'h': h, 'w': w, 'cin': c, 'cout': layer._cout,
             'k': layer.ksize, 'stride': layer.stride, 'residual': has_res, 'K': layer.ksize ** 2 * c,
             'fused_ms': round(f, 4), 'plain_apply_ms': round(pa, 4), 'fused_over_plain': round(f / pa, 3),
             'fused_ms_runs': [round(v, 4) for v in tf], 'plain_apply_ms_runs': [round(v, 4) for v in tp]}
      print(json.dumps(row), flush=True)
      rows.append(row)
      del xs_, ys, tmp, rs
    del fz, model
    torch.cuda.empty_cache()
  return rows


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--configs', default='c2,c4')
  ap.add_argument('--batches', default='256,1000')
  ap.add_argument('--seconds', type=float, default=1.0)
  ap.add_argument('--shapes', action='store_true')
  ap.add_argument('--shape-batch', type=int, default=256)
  ap.add_argument('--shape-seconds', type=float, default=0.3)
  ap.add_argument('--json', default=None)
  args = ap.parse_args()
  if args.shapes:
    os.environ['RIGL_AFFINE_ALWAYS'] = '1'     # read when the library initialises: time every shape fused
  import torch
  if not torch.cuda.is_available():
    raise SystemExit('bench_inference: no CUDA device')
  dev = 'cuda:0'
  info = gpu_info()
  print('gpu:', info, flush=True)
  out = {'gpu': info, 'torch': torch.__version__}
  if args.shapes:
    out['shapes'] = run_shapes(args, dev)
  else:
    out['forward'] = run_forward(args, dev)
  if args.json:
    os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
    with open(args.json, 'w') as f:
      json.dump(out, f, indent=1)


if __name__ == '__main__':
  main()
