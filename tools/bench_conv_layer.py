"""Per-layer micro-benchmark of the masked conv kernels (fprop / dgrad / dense wgrad) through the
same host calls the training step makes.  One JSON line per (shape, op): microseconds (CUDA
events, median of --iters, inputs rotated through buffers larger than L2), dense-executed TFLOP/s
and algorithmic GB/s.  Kernel-selection switches (RIGL_HALO3X3, RIGL_CTA_PAIR, RIGL_TMA_STORE ...)
are read once per process: run one process per configuration.

  python tools/bench_conv_layer.py [--shapes r50s1] [--iters 20] [--tag name]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rigl_b200 import pruning  # noqa: E402
from rigl_b200.layers import SparseConv2d  # noqa: E402

DEV = 'cuda:0'
SHAPES = {
    # n, h, w, cin, cout, k, stride
    'r50s1': [(256, 56, 56, 64, 64, 3, 1)],
    'r50s2': [(256, 28, 28, 128, 128, 3, 1)],
    'r50_c3': [(256, 14, 14, 1024, 256, 1, 1)],
    'r50_33c3': [(256, 14, 14, 256, 256, 3, 1)],
    'r50_3x3': [(256, 56, 56, 64, 64, 3, 1), (256, 28, 28, 128, 128, 3, 1), (256, 14, 14, 256, 256, 3, 1),
                (256, 7, 7, 512, 512, 3, 1)],
    'stats': [(256, 56, 56, 64, 256, 1, 1), (256, 28, 28, 128, 512, 1, 1), (256, 56, 56, 256, 64, 1, 1),
              (256, 28, 28, 512, 128, 1, 1)],
    'r50_1x1': [(256, 56, 56, 64, 256, 1, 1), (256, 56, 56, 256, 64, 1, 1), (256, 28, 28, 512, 128, 1, 1),
                (256, 14, 14, 1024, 256, 1, 1), (256, 7, 7, 2048, 512, 1, 1)],
}


REPS = 5


def timed(fn, iters):
  """Median GPU time of one call.  A spin kernel ahead of the start event lets the host enqueue
  the REPS calls before the GPU reaches them, so host launch latency is not in the interval."""
  ts = []
  for i in range(iters + 3):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(1000000)
    a.record()
    for r in range(REPS):
      fn(i * REPS + r)
    b.record()
    b.synchronize()
    if i >= 3:
      ts.append(a.elapsed_time(b) * 1e3 / REPS)
  ts.sort()
  return ts[len(ts) // 2]


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--shapes', default='r50s1')
  ap.add_argument('--iters', type=int, default=20)
  ap.add_argument('--tag', default='')
  args = ap.parse_args()
  for (n, h, w, cin, cout, k, stride) in SHAPES[args.shapes]:
    pruning.reset_default_registry()
    layer = SparseConv2d(cin, cout, k, strides=stride, padding='FIXED', name='t', device=DEV)
    layer.mask.assign((torch.rand(k, k, cin, cout, device=DEV) >= 0.8).float())
    layer.pack()
    ho, wo = layer.out_size(h)[0], layer.out_size(w)[0]
    in_bytes, out_bytes = n * h * w * cin * 2, n * ho * wo * cout * 2
    copies = max(2, int(300e6 // max(in_bytes + out_bytes, 1)) + 1)          # rotate through > 2x L2
    xs = [torch.randn(n, cin, h, w, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
          for _ in range(copies)]
    dys = [torch.randn(n, cout, ho, wo, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
           for _ in range(copies)]
    dw = torch.empty(k * k * cin * cout, dtype=torch.float32, device=DEV)
    flops = 2.0 * n * ho * wo * k * k * cin * cout
    from rigl_b200 import layers as L, _cabi
    def fprop_stats(i):
      L.FUSE_BN_STATS, layer.collect_bn_stats = True, True
      layer.train()
      try:
        return layer._fprop(xs[i % copies], None, False)
      finally:
        L.FUSE_BN_STATS, layer.collect_bn_stats = False, False
    _cabi.lib().rigl_set_bn_stats_always(1)
    L.FUSE_BN_STATS = False
    ops = (('fprop', lambda i: layer._fprop(xs[i % copies], None, False)), ('fprop_stats', fprop_stats),
           ('dgrad', lambda i: layer._dgrad(dys[i % copies], xs[i % copies])),
           ('wgrad', lambda i: layer._wgrad(xs[i % copies], dys[i % copies], dw, False)))
    for name, fn in ops:
      us = timed(fn, args.iters)
      print(json.dumps({'tag': args.tag, 'shape': [n, h, w, cin, cout, k, stride], 'op': name, 'us': round(us, 2),
                        'tflops_dense': round(flops / us * 1e-6, 1),
                        'gbps_algorithmic': round((in_bytes + out_bytes) / us * 1e-3, 1)}), flush=True)


if __name__ == '__main__':
  main()
