"""Benchmark of the RigL hot path: sparse train step (+ the periodic mask update) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5] [--impl ours|reference]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Configs (BASELINE.json `configs`; the metric is quoted on c2, the default):
  c2  ResNet-50, ImageNet-shaped synthetic, 80 % ERK, bf16, batch 256 per GPU
  c3  ResNet-50, 90 % ERK, batch 256 per GPU (global 2048 at 8 GPUs)
  c4  MobileNet-v1, 90 % uniform on the 13 pointwise convs + classifier (~89 % overall), batch 256 per GPU
  c5  WideResNet-22-2, CIFAR-shaped synthetic, 95 % ERK, batch 128 per GPU, mask update every 100 steps
All: RigL, drop fraction 0.3 cosine, update every 100 steps, Nesterov momentum, weak scaling (fixed per-GPU
batch).  The timed region always contains ceil(steps/100) mask updates (the schedule is aligned so that the
first one falls in the middle of the region), so `value` includes their cost at the reference's own cadence
or denser.  One JSON line on rank 0: the driver contract plus `roofline`, `cpu_baseline`, `mask_update_ms`.
"""
import argparse
import functools
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    'c2': dict(model='resnet50', sparsity=0.8, method='erdos_renyi_kernel', batch=256, image=224, classes=1000,
               metric='sparse_train_step_images_per_sec_resnet50_erk80',
               workload='ResNet-50 ImageNet-shaped, 80% ERK (54 masked tensors, 25.5M weights), batch 256/GPU'),
    'c3': dict(model='resnet50', sparsity=0.9, method='erdos_renyi_kernel', batch=256, image=224, classes=1000,
               metric='sparse_train_step_images_per_sec_resnet50_erk90',
               workload='ResNet-50 ImageNet-shaped, 90% ERK (54 masked tensors, 25.5M weights), batch 256/GPU'),
    'c4': dict(model='mobilenet_v1', sparsity=0.9, method='random', batch=256, image=224, classes=1000,
               metric='sparse_train_step_images_per_sec_mobilenetv1_uniform90',
               workload='MobileNet-v1 ImageNet-shaped, 90% uniform on 13 pointwise convs + classifier '
                        '(~89% overall), depthwise convs dense (cuDNN), batch 256/GPU'),
    'c5': dict(model='wrn22_2', sparsity=0.95, method='erdos_renyi_kernel', batch=128, image=32, classes=10,
               metric='sparse_train_step_images_per_sec_wrn22_2_erk95',
               workload='WideResNet-22-2 CIFAR-shaped, 95% ERK (22 masked tensors), batch 128/GPU'),
}
UPDATE_EVERY = 100


def _peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      d = json.load(f)
    return d.get('hbm_gbs', 6650.0), d.get('bf16_tflops_sustained', 1400.0), 'measured'
  return 6650.0, 1400.0, 'fallback'


def _recorded_traffic(cfg_name):
  """DRAM bytes per step of the conv kernel family from the committed ncu pass of the SAME workload
  (profiles/*_dram_traffic_step.json: dram__bytes_read.sum + dram__bytes_write.sum, c2 at batch 256).  ncu
  cannot run inside a timed bench, so this is the recorded capture, not a live measurement; null for the
  configs that have no capture."""
  if cfg_name != 'c2':
    return None
  for name in ('r02_dram_traffic_step.json', 'r01_dram_traffic_step.json'):
    path = os.path.join(ROOT, 'profiles', name)
    try:
      with open(path) as f:
        d = json.load(f)
      return {'dram_bytes_per_step': d['conv_family_dram_bytes_per_step'], 'launches': d['conv_family_launches'],
              'source': 'profiles/' + name + ' (recorded ncu capture, not measured by this run)'}
    except Exception:
      continue
  return None


class ClockSampler(object):
  """Samples nvidia-smi clocks / throttle reasons during the timed region."""

  def __init__(self, gpu_index=0):
    self.rows, self.proc, self.thread, self.idx = [], None, None, gpu_index

  def start(self):
    q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + q,
                                    '--format=csv,noheader,nounits', '-lms', '200'],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
      return
    self.thread = threading.Thread(target=self._pump, daemon=True)
    self.thread.start()

  def _pump(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(',')])

  def mark(self):
    """Samples taken so far (while nvidia-smi was starting up, before the timed region) are dropped."""
    self.skip = len(self.rows)

  def stop(self):
    self.rows = self.rows[getattr(self, 'skip', 0):]
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      self.proc.kill()
    sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
    mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == 'Active' for r in self.rows)]
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': reasons, 'samples': len(sm)}


def _dist_setup(n_gpus):
  import torch.distributed as dist
  world = int(os.environ.get('WORLD_SIZE', '1'))
  if world > 1:
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    return dist, dist.get_rank(), world, local
  torch.cuda.set_device(0)
  return None, 0, 1, 0


def build_model(cfg, dev):
  from rigl_b200 import workloads
  if cfg['model'] == 'resnet50':
    model = workloads.ResNet50(num_classes=cfg['classes'], device=dev)
  elif cfg['model'] == 'mobilenet_v1':
    model = workloads.MobileNetV1(num_classes=cfg['classes'], device=dev)
  else:
    model = workloads.WideResNet(depth=22, width=2, num_classes=cfg['classes'], device=dev)
  workloads.init_masks(model, cfg['method'], cfg['sparsity'], seed=0)
  return model


def masked_flops_per_image(model, image, dev):
  """SURVEY 8(d) accounting from the model's own masked layers: per image, 2*MAC, maskable layers only.
  f_D = dense-executed fprop FLOPs, f_S = the same scaled by each layer's density.  This build computes the DENSE
  wgrad every step (as the TF1 reference effectively does), so a step costs
    algorithmic = 2*f_S + f_D - f_S(first masked conv: no input gradient);  dense-executed = 3*f_D - f_D(first)."""
  from rigl_b200.layers import SparseConv2d
  shapes = {}
  hooks = []
  for l in model.registry.layers():
    hooks.append(l.register_forward_hook(lambda mod, inp, out, l=l: shapes.__setitem__(l.scope, tuple(out.shape))))
  was = model.training
  model.eval()
  with torch.no_grad():
    model(torch.zeros(1, 3, image, image, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
  model.train(was)
  for h in hooks:
    h.remove()
  f_d = f_s = 0.0
  first_d = first_s = None
  for l in model.registry.layers():
    sh = shapes[l.scope]
    pixels = sh[2] * sh[3] if len(sh) == 4 else 1
    macs = pixels * l.weight.numel()
    dens = l.mask.count_ones() / float(l.mask.size)
    f_d += 2.0 * macs
    f_s += 2.0 * macs * dens
    if first_d is None and isinstance(l, SparseConv2d) and l.in_channels == 3:
      first_d, first_s = 2.0 * macs, 2.0 * macs * dens
  first_d, first_s = first_d or 0.0, first_s or 0.0
  return {'f_dense_gflop': f_d / 1e9, 'f_sparse_gflop': f_s / 1e9,
          'algorithmic_gflop': (2 * f_s + f_d - first_s) / 1e9, 'dense_executed_gflop': (3 * f_d - first_d) / 1e9}


DUMP_SAMPLE = 1 << 21       # elements per dumped array (8 MB in float32): a whole dump stays under 41 MB


@functools.lru_cache(maxsize=None)
def _dump_index(n):
  """A fixed, seeded sample of DUMP_SAMPLE of the positions 0..n-1, ascending."""
  return torch.from_numpy(np.sort(np.random.RandomState(0).choice(n, DUMP_SAMPLE, replace=False)))


def _dump_sample(t):
  return t if t.numel() <= DUMP_SAMPLE else t[_dump_index(t.numel()).to(t.device)]


def dump_outputs(out_dir, model, harness, loss):
  """Writes what the last timed step computed as DIR/<name>.npy (float32): its loss and the model it leaves behind.
  The per-layer arrays are concatenated in registry order (each layer flat, C order) and sampled at the same
  positions: masked weights, masks, momentum slots and the step's dense gradients; other_params holds every
  parameter that carries no mask (batch-norm scales and offsets, biases, dense depthwise weights)."""
  os.makedirs(out_dir, exist_ok=True)
  layers = model.registry.layers()
  masked = set(id(l.weight) for l in layers)
  parts = {
      'masked_weights': [l.weight.reshape(-1) for l in layers],
      'masks': [l.mask.to_dense().reshape(-1) for l in layers],
      'momentum': [harness.inner.state[l.weight]['momentum_buffer'].reshape(-1) for l in layers],
      'dense_grads': [l.masked_weights.dense_grad.reshape(-1) for l in layers],
      'other_params': [p.reshape(-1) for p in model.parameters() if id(p) not in masked],
  }
  arrays = {'loss': loss.float().reshape(())}
  for name, ts in parts.items():
    arrays[name] = _dump_sample(torch.cat([t.detach().float() for t in ts]))
  for name, t in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy())


def run_ours(args):
  from rigl_b200 import _cabi
  from rigl_b200 import workloads
  from rigl_b200.layers import Profiler

  cfg = CONFIGS[args.config]
  batch, image = cfg['batch'], cfg['image']
  dist, rank, world, local = _dist_setup(args.gpus)
  if args.scaling == 'strong':               # fixed GLOBAL batch (the config's), split over the ranks
    if batch % world:
      raise SystemExit('--scaling strong: batch %d is not divisible by %d ranks' % (batch, world))
    batch //= world
  dev = torch.device('cuda', local)
  torch.manual_seed(0)
  model = build_model(cfg, dev)
  flops = masked_flops_per_image(model, image, dev)
  dp = None
  if world > 1:
    from rigl_b200.data_parallel import DataParallel
    dp = DataParallel()
  wd = 5e-4 if cfg['model'] == 'wrn22_2' else 1e-4
  smooth = 0.0 if cfg['model'] == 'wrn22_2' else 0.1
  harness = workloads.TrainHarness(model, lr=0.1, weight_decay=wd, label_smoothing=smooth, frequency=UPDATE_EVERY,
                                   data_parallel=dp)
  g = torch.Generator(device=dev).manual_seed(1 + rank)
  images = torch.randn(batch, 3, image, image, device=dev, generator=g).to(torch.bfloat16) \
      .contiguous(memory_format=torch.channels_last)
  labels = torch.randint(0, cfg['classes'], (batch,), device=dev, generator=g)

  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize()

  harness.step(images, labels)               # eager: first step is the initial mask update
  harness.step(images, labels)
  graphed = False
  if not args.no_graph:
    graphed = harness.enable_cuda_graph(images, labels)
  # nvidia-smi is started BEFORE the warm-up: its start-up initialises NVML on every GPU of the box, which stalls
  # them for tens of milliseconds (measured at N = 8) -- that belongs to no step; it then samples every 200 ms
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  # warm-up of the UPDATE path too: the first update after the momentum slots exist rebuilds the launch plan
  # (device allocations), like a first step does; the timed updates then run the steady-state path
  harness.opt.collect_masked_grads()
  harness.opt.drop_fraction = np.float32(0.3)
  harness.opt.mask_update_op()
  for _ in range(args.warmup):
    harness.step(images, labels)
  # align the schedule: the next update is due in the middle of the timed region (then every 100 steps)
  harness.opt._last_update_step = harness.global_step.value + min(args.steps, UPDATE_EVERY) // 2 - UPDATE_EVERY
  barrier()
  sampler.mark()
  launches0 = _cabi.launch_count() + getattr(harness, 'replayed_kernel_launches', 0)
  start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
  start.record()
  marks[0].record()
  n_updates, update_steps = 0, []
  for i in range(args.steps):
    loss = harness.step(images, labels).detach()      # (keeps no autograd graph alive into the next step)
    marks[i + 1].record()
    if harness.opt.last_update_was_mask_update:
      n_updates += 1
      update_steps.append(i)
  stop.record()
  barrier()
  if args.dump_outputs and rank == 0:
    # before the legs below train on and change the model
    dump_outputs(args.dump_outputs, model, harness, loss)
  per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]
  clocks = sampler.stop() if rank == 0 else None
  launches = _cabi.launch_count() + getattr(harness, 'replayed_kernel_launches', 0) - launches0
  ms = torch.tensor([start.elapsed_time(stop)], device=dev, dtype=torch.float64)
  if dist is not None:
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
  total_ms = float(ms.item())
  value = world * batch * args.steps / (total_ms / 1e3)
  masks_identical = None
  if dp is not None:
    masks_identical = bool(dp.masks_identical(model))     # replicas must still agree after the updates
    if not masks_identical:
      raise RuntimeError('masks diverged across replicas')

  # ---- end-to-end leg: host (pinned) -> device copy of every batch, loss read back ----
  e2e_steps = max(3, min(args.steps, 20))
  host_images = torch.empty((batch, image, image, 3), dtype=torch.bfloat16).pin_memory()
  host_images.copy_(images.permute(0, 2, 3, 1).cpu())
  host_labels = labels.cpu().pin_memory()
  barrier()
  e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  copy_stream = torch.cuda.Stream(device=dev)

  # two device staging buffers, allocated once: the prefetch never goes through the caching allocator (a fresh
  # `.to(device)` per step made the leg bimodal, 22.8 vs 29.9 ms per step on the same box: an allocation that
  # cannot reuse the block still held for the running step falls back to cudaMalloc and serialises the copy)
  stage_x = [torch.empty((batch, image, image, 3), dtype=torch.bfloat16, device=dev) for _ in range(2)]
  stage_y = [torch.empty_like(labels) for _ in range(2)]

  def fetch(i):           # host -> device copy of batch i on the copy stream (input prefetch)
    with torch.cuda.stream(copy_stream):
      stage_x[i % 2].copy_(host_images, non_blocking=True)
      stage_y[i % 2].copy_(host_labels, non_blocking=True)
      ev = torch.cuda.Event()
      ev.record(copy_stream)
    return stage_x[i % 2], stage_y[i % 2], ev

  copy_stream.wait_stream(torch.cuda.current_stream())
  e_start.record()
  nxt = fetch(0)
  for i in range(e2e_steps):
    xb, yb, ev = nxt
    torch.cuda.current_stream().wait_event(ev)
    if i + 1 < e2e_steps:
      nxt = fetch(i + 1)  # overlaps the next batch's H2D with this step's compute; buffer (i+1)%2 was last read by
                          # step i-1, which has completed (its loss was read back)
    loss = harness.step(xb.permute(0, 3, 1, 2), yb)
    _ = float(loss.item())
  e_stop.record()
  barrier()
  e_ms = torch.tensor([e_start.elapsed_time(e_stop)], device=dev, dtype=torch.float64)
  if dist is not None:
    dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
  e2e_value = world * batch * e2e_steps / (float(e_ms.item()) / 1e3)

  # ---- roofline leg: per-call CUDA-event times of the conv kernels (all ranks step: the
  # data-parallel all-reduce is collective; only rank 0 records) ----
  prof_steps = 3
  harness.graphed = False                    # the per-call event timing needs the eager path
  for _ in range(2):                         # re-warm the eager allocator state after graph replay
    harness.step(images, labels)
  barrier()
  if rank == 0:
    Profiler.start()
  for _ in range(prof_steps):
    harness.step(images, labels)
  barrier()
  if rank != 0:
    _teardown(dist, harness)
    return
  rec = Profiler.stop()
  per_kind = {}
  for kind, _, t in rec:
    per_kind[kind] = per_kind.get(kind, 0.0) + t / prof_steps
  if args.layer_report:
    agg = {}
    for kind, scope, t in rec:
      agg[(kind, scope)] = agg.get((kind, scope), 0.0) + t / prof_steps
    with open(args.layer_report, 'w') as f:
      json.dump([{'kind': k, 'scope': sc, 'ms': v} for (k, sc), v in agg.items()], f, indent=0)
  conv_ms = sum(per_kind.get(k, 0.0) for k in ('fprop', 'dgrad', 'wgrad'))
  n_conv_launch = sum(1 for k, _, _ in rec if k in ('fprop', 'dgrad', 'wgrad')) / prof_steps
  hbm_peak, tf_peak, peak_src = _peaks()
  alg = flops['algorithmic_gflop']
  achieved_tf = alg * batch / conv_ms                             # GFLOP/ms == TFLOP/s
  step_ms = total_ms / args.steps
  step_tf = alg * batch * world / step_ms                         # whole job, all ranks
  # ---- mask update alone (all masked layers, one update), through the public optimizer call ----
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
  mu = []
  harness.opt.drop_fraction = np.float32(0.3)
  for i in range(8):
    flush.zero_()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    harness.opt.mask_update_op()
    e.record()
    torch.cuda.synchronize()
    if i >= 3:
      mu.append(s.elapsed_time(e))
  mask_ms = float(np.median(mu))
  total_w = sum(m.size for m in model.registry.get_masks())

  out = {
      'metric': cfg['metric'], 'value': value, 'unit': 'images/sec', 'n_gpus': world, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': step_ms, 'higher_is_better': True,
      'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
      'config': {'workload': cfg['workload'] + ', RigL drop 0.3 cosine every 100 steps, Nesterov momentum',
                 'name': args.config, 'global_batch': batch * world, 'per_gpu_batch': batch,
                 'parallelism': 'dp%d' % world,
                 'l2_policy': 'inputs larger than L2 (activations per step >> 126 MB)',
                 'mask_updates_in_timed_region': n_updates, 'mask_update_steps': update_steps,
                 'step_ms': {'p50': float(np.median(per_step)), 'p90': float(np.percentile(per_step, 90)),
                             'max': float(max(per_step)), 'argmax': int(np.argmax(per_step)),
                             'note': 'rank 0, per step, device events'},
                 'masks_identical_across_replicas': masks_identical,
                 'cuda_graph': bool(graphed)},
      'clocks': clocks,
      'e2e': {'value': e2e_value, 'unit': 'images/sec', 'steps': e2e_steps,
              'h2d_bytes_per_step': int(host_images.numel() * 2 + host_labels.numel() * 8),
              'd2h_bytes_per_step': 4},
      'gpu_launches': int(launches),
      'mask_update_ms': mask_ms,
      'mask_update_algorithmic_GBps': 8.25 * total_w / mask_ms / 1e6,
      'roofline': {'bound': 'tensor',
                   'kernel': 'k_igemm_kmajor2 / k_igemm_wgrad / k_halo3x3_* / k_stem_s2d_* (all masked conv+linear launches)',
                   'achieved': achieved_tf, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': achieved_tf / tf_peak,
                   # the metric's own fraction: masked FLOPs of the whole job over the whole step (all kernels)
                   'achieved_step': step_tf, 'frac_step': step_tf / (tf_peak * world),
                   'peak_source': peak_src + ' bf16_tflops_sustained',
                   'algorithmic_gflop_per_image': alg,
                   'dense_executed_gflop_per_image': flops['dense_executed_gflop'],
                   'dense_executed_tflops': flops['dense_executed_gflop'] * batch / conv_ms,
                   'conv_ms_per_step': conv_ms, 'conv_launches_per_step': n_conv_launch,
                   'ms_per_step_by_kind': per_kind, 'traffic': _recorded_traffic(args.config)},
  }
  if world == 1 and not args.no_cpu_baseline:
    out['cpu_baseline'] = cpu_baseline_leg(args.config, sample_batch=args.cpu_batch)
  _emit(out)
  _teardown(dist, harness)


def _teardown(dist, harness):
  """NCCL refuses to finalise a communicator while CUDA graphs that captured its collectives are alive
  (ncclCommDestroy waits for them): release the graphs first, then destroy the process group -- and never let a
  stuck teardown turn a finished measurement into a hang."""
  if dist is None:
    return
  import gc

  def bail():
    os._exit(0)
  t = threading.Timer(45.0, bail)
  t.daemon = True
  t.start()
  harness.release_cuda_graph()
  gc.collect()
  torch.cuda.synchronize()
  try:
    dist.barrier()
    dist.destroy_process_group()
  finally:
    t.cancel()


def _cpu_port_timing(cfg_name, batch, steps, warmup):
  """Times the CPU port in a FRESH interpreter whose OpenMP environment is not the one
  torchrun exports (OMP_NUM_THREADS=1): torch then sizes its intra-op pool to the host's
  cores.  Returns {'times' (s per step, every timed step), 'mask_update_sec', 'threads'}."""
  cfg = CONFIGS[cfg_name]
  env = dict(os.environ)
  for k in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS', 'OMP_PROC_BIND', 'OMP_PLACES', 'GOMP_CPU_AFFINITY',
            'KMP_AFFINITY', 'CUDA_VISIBLE_DEVICES'):
    env.pop(k, None)
  env['CUDA_VISIBLE_DEVICES'] = ''
  code = ('import json,sys,torch; sys.path.insert(0, %r); '
          'from oracle import cpu_train_step as c; '
          'times, net, dense = c.time_train_steps_model(%r, %d, %d, warmup=%d, image_hw=%d, sparsity=%r); '
          'mu = c.time_mask_update(net, dense); '
          'print("CPUPORT " + json.dumps({"times": times, "mask_update_sec": mu, '
          '"threads": torch.get_num_threads()}))' % (ROOT, cfg['model'], batch, steps, warmup, cfg['image'],
                                                     cfg['sparsity']))
  out = subprocess.run([sys.executable, '-c', code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=1500)
  for line in out.stdout.splitlines():
    if line.startswith('CPUPORT '):
      return json.loads(line[len('CPUPORT '):])
  raise RuntimeError('CPU port failed: ' + out.stderr[-2000:])


def _spread(times, batch):
  t = np.asarray(times, np.float64)
  return {'median_images_per_sec': batch / float(np.median(t)),
          'p10_images_per_sec': batch / float(np.percentile(t, 90)),     # slow steps -> low throughput
          'p90_images_per_sec': batch / float(np.percentile(t, 10)),
          'timed_steps': int(t.size)}


def cpu_baseline_leg(cfg_name, sample_batch=16, steps=5):
  """Times the CPU port of the reference path on the host cores (bounded sample)."""
  t = _cpu_port_timing(cfg_name, sample_batch, steps, 1)
  sp = _spread(t['times'], sample_batch)
  return {'value': sp['median_images_per_sec'], 'unit': 'images/sec', 'cores': t['threads'], 'kind': 'port',
          'sample': '%s fp32 train step (fwd + dense&masked bwd + momentum), batch %d, %d timed steps after 1 '
                    'warm-up (median), torch-CPU port of the TF1 graph' % (CONFIGS[cfg_name]['workload'], sample_batch,
                                                                        steps),
          'spread': sp,
          'mask_update_ms': t['mask_update_sec'] * 1e3,
          'mask_update_sample': 'one drop/grow update of all masked layers (numpy stable argsort x2 per layer)'}


def run_reference(args):
  """The reference's own CPU implementation of the path (torch-CPU / numpy port of the
  TF1 graph -- TensorFlow is not installable in this image), all host threads."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  cfg = CONFIGS[args.config]
  batch = args.cpu_batch
  steps = max(5, min(args.steps, 8))         # >= 5 timed steps: a 3-step sample was too noisy (VERDICT r1)
  warm = max(1, min(args.warmup, 2))
  t0 = time.perf_counter()
  t = _cpu_port_timing(args.config, batch, steps, warm)
  sp = _spread(t['times'], batch)
  value = sp['median_images_per_sec']
  _emit({
      'impl': 'reference', 'metric': cfg['metric'], 'value': value, 'unit': 'images/sec',
      'n_gpus': args.gpus, 'steps': steps, 'warmup': warm, 'ms_per_step': batch / value * 1e3,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': '%s, CPU port of the reference TF1 train step, bounded sample of batch %d per step'
                             % (cfg['workload'], batch), 'name': args.config},
      'cpu_baseline': {'value': value, 'unit': 'images/sec', 'cores': t['threads'], 'kind': 'port',
                       'sample': 'batch %d, %d timed steps (median), wall %.1fs' % (batch, steps, time.perf_counter() - t0),
                       'spread': sp},
      'mask_update_ms': t['mask_update_sec'] * 1e3,
      'e2e': {'value': value, 'unit': 'images/sec', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'gpu_launches': 0})


_JSON_FD = None


def _emit(obj):
  """The ONE JSON line of the contract, on the process's original stdout."""
  line = (json.dumps(obj) + '\n').encode()
  if _JSON_FD is None:
    sys.stdout.write(line.decode())
    sys.stdout.flush()
  else:
    os.write(_JSON_FD, line)


def main():
  # stdout carries exactly one JSON line: everything else that writes to fd 1 (NCCL prints its
  # version banner there when NCCL_DEBUG is set, library warnings) is sent to stderr.
  global _JSON_FD
  sys.stdout.flush()
  _JSON_FD = os.dup(1)
  os.dup2(2, 1)
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=100)
  ap.add_argument('--warmup', type=int, default=5)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--config', default='c2', choices=sorted(CONFIGS))
  ap.add_argument('--cpu-batch', type=int, default=16)
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--layer-report', default=None)
  ap.add_argument('--no-graph', action='store_true', help='run the step eagerly (no CUDA-graph replay)')
  ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                  help='weak (default, the driver contract): the per-GPU batch is fixed; strong: the GLOBAL batch of '
                       'the config is fixed and split over the ranks')
  ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                  help='write what the last timed step computed (loss, sampled weights / masks / momentum / dense '
                       'gradients, other parameters) as DIR/<name>.npy, to compare two builds on the same inputs')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs writes the outputs of --impl ours')
  if args.warmup < 3 and args.impl == 'ours':
    args.warmup = 3
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
