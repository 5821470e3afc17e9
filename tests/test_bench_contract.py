"""bench.py's reference arm (`--impl reference`: the oracle port on the host cores) runs without a GPU, so its side of the
JSON contract is checked here on a tiny shape: one line on stdout, the base keys, `"impl": "reference"`, a
`cpu_baseline` describing the run, an `e2e` object without copies, the evaluation record nested under `"eval"`; under
torchrun only rank 0 prints, the other ranks exit 0 without work.  The GPU arm's line and its --dump-outputs files are
checked by the last test, on the B200; profiles/r2_bench_default_final.json holds a full line of that arm."""

import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
             'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'cpu_baseline', 'impl'}


def _run(extra_env=None, extra_args=()):
  env = dict(os.environ)
  env.update(extra_env or {})
  cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
         '--height', '64', '--width', '96', '--batch', '2', *extra_args]
  return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)


def _check_record(rec, metric, unit):
  assert BASE_KEYS <= set(rec), sorted(BASE_KEYS - set(rec))
  assert rec['impl'] == 'reference' and rec['metric'] == metric and rec['unit'] == unit
  assert rec['value'] > 0 and rec['higher_is_better'] is True and rec['vs_baseline'] is None and rec['gpu_launches'] == 0
  assert rec['data'] == 'synthetic' and rec['dtype'] == 'f32' and 'workload' in rec['config'] and 'model' not in rec['config']
  cpu = rec['cpu_baseline']
  assert set(cpu) >= {'value', 'unit', 'cores', 'kind', 'sample'} and cpu['kind'] == 'port' and cpu['value'] == rec['value']
  assert cpu['cores'] >= 1 and cpu['unit'] == unit
  e2e = rec['e2e']
  assert e2e == {'value': rec['value'], 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_reference_arm_prints_one_contract_line():
  r = _run()
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, r.stdout
  rec = json.loads(lines[0])
  _check_record(rec, 'train_images_per_s', 'images/s')
  assert rec['steps'] == 1 and rec['warmup'] == 0 and rec['n_gpus'] == 1
  assert '2 strong + 0 bbox + 0 image-level images/GPU' in rec['config']['workload'] and '64x96' in rec['config']['workload']
  _check_record(rec['eval'], 'eval_mpix_per_s', 'Mpix/s')


def test_reference_arm_other_ranks_exit_without_work():
  r = _run({'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2'}, ('--gpus', '2'))
  assert r.returncode == 0 and r.stdout.strip() == '', (r.stdout, r.stderr[-500:])


def test_reference_arm_times_exactly_the_requested_steps():
  r = _run(extra_args=('--steps', '5', '--warmup', '2'))
  assert r.returncode == 0, r.stderr[-2000:]
  rec = json.loads(r.stdout)
  for half in (rec, rec['eval']):
    assert half['steps'] == 5 and half['warmup'] == 2
    assert half['cpu_baseline']['sample'].startswith('5 ') and '2 warm-up' in half['cpu_baseline']['sample']


def test_bench_refuses_zero_steps_and_dumps_of_the_reference_arm(tmp_path):
  r = _run(extra_args=('--dump-outputs', str(tmp_path)))
  assert r.returncode == 2 and '--dump-outputs' in r.stderr and not os.listdir(tmp_path)
  r = _run(extra_args=('--steps', '0'))
  assert r.returncode == 2 and '--steps' in r.stderr


def test_dump_outputs_writes_float_arrays(tmp_path):
  import numpy as np
  import torch
  sys.path.insert(0, ROOT)
  import bench
  bench.dump_outputs(str(tmp_path / 'out'), {'counts': torch.tensor([[3, 2 ** 40]]),
                                             'x': torch.randn(7, 3).to(torch.bfloat16),
                                             'y': torch.ones(2, dtype=torch.float64)})
  assert sorted(os.listdir(tmp_path / 'out')) == ['counts.npy', 'x.npy', 'y.npy']
  counts = np.load(tmp_path / 'out' / 'counts.npy')
  assert counts.dtype == np.float64 and counts.tolist() == [[3.0, 2.0 ** 40]]
  assert np.load(tmp_path / 'out' / 'x.npy').dtype == np.float32
  assert np.load(tmp_path / 'out' / 'y.npy').dtype == np.float64


@pytest.mark.gpu
def test_wlseg_arm_dumps_the_outputs_of_its_last_timed_step(cuda, tmp_path):
  """Both halves at a small evaluation size: one JSON line, and the arrays of the last timed step under DIR as float
  .npy files, 64 MB at most."""
  import numpy as np
  out = tmp_path / 'dump'
  cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '3', '--warmup', '1', '--height', '128', '--width',
         '256', '--batch', '2', '--no-cpu-baseline', '--no-e2e', '--sustained-seconds', '0', '--dump-outputs', str(out)]
  r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
  assert r.returncode == 0, r.stderr[-3000:]
  rec = json.loads(r.stdout)
  assert rec['steps'] == 3 and rec['eval']['steps'] == 3
  arrays = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
  assert set(arrays) == {'eval_confusion_matrix', 'eval_invalid_labels', 'train_losses'}
  assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in arrays.values())
  assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 << 20
  cm = arrays['eval_confusion_matrix']
  assert cm.shape == (20, 20) and cm.sum() == 3 * 2 * 128 * 256 and arrays['eval_invalid_labels'].tolist() == [0.0]
  losses = arrays['train_losses']
  assert losses.shape == (6,) and losses.tolist() == rec['config']['last_loss']
