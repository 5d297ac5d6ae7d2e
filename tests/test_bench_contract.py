"""bench.py's JSON contract, checked on the CPU: the reference arm (the CPU port of the reference's train step) runs
without a GPU, so its line can be produced here; the product arm must refuse to run without one (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
  env = dict(os.environ, OMP_NUM_THREADS=os.environ.get('OMP_NUM_THREADS', '8'))
  return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, cwd=ROOT, env=env,
                        stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)


def test_reference_arm_line_has_every_contract_key():
  # the smallest BASELINE config (WideResNet-22-2, CIFAR-shaped): a bounded sample of batch 16 per step
  r = _run(['--impl', 'reference', '--config', 'c5', '--steps', '2', '--warmup', '1'])
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, 'exactly ONE JSON line on stdout'
  d = json.loads(lines[0])
  assert d['impl'] == 'reference'
  for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e', 'gpu_launches'):
    assert key in d, key
  assert d['unit'] == 'images/sec' and d['higher_is_better'] is True and d['n_gpus'] == 1
  assert d['metric'].startswith('sparse_train_step_images_per_sec')
  assert d['value'] > 0 and d['ms_per_step'] > 0
  assert d['steps'] >= 5, 'the CPU arm times at least five steps (VERDICT r1: 3 steps were too noisy)'
  assert d['gpu_launches'] == 0 and d['dtype'] == 'f32' and d['data'] == 'synthetic'
  assert 'workload' in d['config'] and 'model' not in d['config']
  cb = d['cpu_baseline']
  assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['unit'] == d['unit'] and cb['value'] == d['value']
  assert 'sample' in cb and {'p10_images_per_sec', 'p90_images_per_sec'} <= set(cb['spread'])
  assert cb['spread']['p10_images_per_sec'] <= cb['value'] <= cb['spread']['p90_images_per_sec'] * 1.0001
  e = d['e2e']
  assert e['value'] == d['value'] and e['unit'] == d['unit']
  assert e['h2d_bytes_per_step'] == 0 and e['d2h_bytes_per_step'] == 0
  # images / second and milliseconds / step describe the same run (a step = one bounded sample of 16 images)
  assert abs(d['value'] * d['ms_per_step'] / 1e3 - 16.0) <= 0.05 * 16.0


def test_product_arm_refuses_to_run_without_a_gpu():
  if torch.cuda.is_available():
    return            # on a GPU box the product arm is what `python bench.py` measures
  r = _run(['--steps', '1', '--warmup', '0', '--no-cpu-baseline'], timeout=300)
  assert r.returncode != 0, 'bench.py must not fall back to a CPU path'
  assert r.stdout.strip() == '', 'and must not print a bench line'


@pytest.mark.gpu
def test_product_arm_dumps_what_the_last_timed_step_computed(tmp_path):
  r = _run(['--config', 'c5', '--steps', '3', '--warmup', '3', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)])
  assert r.returncode == 0, r.stderr[-2000:]
  d = json.loads(r.stdout)
  assert d['steps'] == 3
  names = {'loss', 'masked_weights', 'masks', 'momentum', 'dense_grads', 'other_params'}
  assert {f for f in os.listdir(tmp_path)} == {n + '.npy' for n in names}
  assert sum(os.path.getsize(os.path.join(tmp_path, n + '.npy')) for n in names) <= 64 << 20
  a = {n: np.load(os.path.join(tmp_path, n + '.npy')) for n in names}
  assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
  assert a['loss'].shape == () and a['loss'] > 0
  n = a['masked_weights'].size
  assert n > 0 and all(a[k].size == n for k in ('masks', 'momentum', 'dense_grads'))
  assert set(np.unique(a['masks'])) == {0.0, 1.0} and abs(a['masks'].mean() - 0.05) < 0.01     # 95 % ERK
  assert np.count_nonzero(a['dense_grads']) > 0.5 * n                                          # dense, not masked


def test_reference_arm_under_torchrun_prints_one_line_from_rank_0():
  # the driver launches the reference arm like the product arm (torchrun, N ranks): rank 0 alone measures and prints
  env = dict(os.environ)
  r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
                      '--master-addr', '127.0.0.1', '--master-port', '29541', os.path.join(ROOT, 'bench.py'),
                      '--impl', 'reference', '--config', 'c5', '--gpus', '2', '--steps', '2', '--warmup', '1'],
                     cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip().startswith('{')]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d['impl'] == 'reference' and d['n_gpus'] == 2 and d['value'] > 0
  assert d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
