"""Throughput of training on a split read from disk (wlseg/train_input.py + wlseg_train_inputs), one JSON line.

    python tools/train_dataset_bench.py [--images 64] [--steps 50] [--repeats 4] [--e2e-steps 100] [--workdir DIR]

Writes a seeded Cityscapes-layout training split of 1024 x 2048 PNG image / label pairs into --workdir (a temporary
directory, removed at the end, when not given), then measures on cuda:0:
  fill_images_per_s          decode (PIL in DataLoader workers) + copy into the device arena, wall clock
  train_inputs_us_per_batch  wlseg_train_inputs alone, 4 examples -> 4 x 512 x 1024, CUDA events over --launches
                             launches whose indices rotate over the whole arena (8 MB per example: 512 MB at the
                             default 64 images, more than the 126 MB L2); its algorithmic GB/s counts 16 B written +
                             13 B gathered (4 RGB taps + 1 label id) per output pixel
  train_images_per_s_arena / _synthetic
                             Estimator.train at 4 x 512 x 1024 (bf16) fed from the arena vs fed from the on-device
                             synthetic generator (per-pixel part only), CUDA events, the two arms alternated --repeats
                             times; reported as the median of each arm
  step_footprint_bytes       drop of free device memory across the first Estimator.train call after the network
                             exists, at Cityscapes 4 x 512 x 1024 and Vistas 4 x 621 x 855 (what
                             wlseg.train_input.STEP_RESERVE_BYTES must leave free next to the arena)
  e2e_s                      cli.train_main --per_pixel_split_path for --e2e-steps steps, wall clock, fill included
The card's name and power limit are read in the same run.  Needs a GPU: there is no CPU fallback.
"""

import argparse
import contextlib
import gc
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'iv2019-boosting-semantic-segmentation-with-weak-labels_b200')
for _p in (ROOT, os.path.join(ROOT, 'tools'), PKG):
  if _p not in sys.path:
    sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from eval_dataset_bench import card, write_split  # noqa: E402


def _train_settings(log_dir, dataset, dev, extra=()):
  from wlseg import settings as wsettings, system_factory
  argv = [log_dir, dataset, '--learning_rate_values', '0.01'] + list(extra)   # Estimator.train without the facade's schedule
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(argv))
  st.device, st.rank, st.world_size, st.save_checkpoints = str(dev), 0, 1, False
  system_factory.attach_problem_definitions(st)
  return st


def _estimator(st, dev):
  from wlseg import estimator as est, hierarchy
  e = est.Estimator(st, hierarchy.Hierarchy(st.per_pixel_dataset_name, st.training_problem_def['cids2labels']), device=dev)
  e.initialize(for_training=True)
  return e


def step_footprint(dataset, dev, tmp):
  """Free device memory before minus after the first 3 training steps on synthetic per-pixel batches."""
  from wlseg import synthetic
  st = _train_settings(os.path.join(tmp, f'fp_{dataset}'), dataset, dev)
  st.Nb_per_bbox = st.Nb_per_image = 0
  e = _estimator(st, dev)
  st.output_Nclasses = e.hier.num_classes
  torch.cuda.synchronize()
  free0, _ = torch.cuda.mem_get_info(dev)
  e.train(synthetic.train_input_fn(None, st), 3)
  torch.cuda.synchronize()
  free1, _ = torch.cuda.mem_get_info(dev)
  del e
  gc.collect()
  torch.cuda.empty_cache()
  return free0 - free1


def main():
  ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
  ap.add_argument('--images', type=int, default=64)
  ap.add_argument('--steps', type=int, default=50, help='training steps per timed repeat')
  ap.add_argument('--repeats', type=int, default=4)
  ap.add_argument('--launches', type=int, default=200, help='wlseg_train_inputs launches timed')
  ap.add_argument('--e2e-steps', type=int, default=100)
  ap.add_argument('--workdir', default=None)
  args = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('train_dataset_bench.py measures on a GPU; none is available')
  from wlseg import cli, dataset_input, estimator as est, ops, problem_defs, synthetic, train_input
  dev = torch.device('cuda:0')
  torch.cuda.set_device(dev)
  problem_defs.write_all()
  tmp = args.workdir or tempfile.mkdtemp(prefix='wlseg_train_bench_')
  os.makedirs(tmp, exist_ok=True)
  quiet = open(os.devnull, 'w')
  Nb, hw = 4, (512, 1024)
  try:
    # 0. the step's own device memory at train.py's two per-pixel sizes, before anything else is resident
    with contextlib.redirect_stdout(quiet):
      footprint = {'cityscapes_4x512x1024': step_footprint('cityscapes', dev, tmp),
                   'vistas_4x621x855': step_footprint('vistas', dev, tmp)}

    t0 = time.perf_counter()
    root = os.path.join(tmp, 'data')
    val = write_split(root, args.images, 1024, 2048, seed=0)
    split = os.path.join(root, 'leftImg8bit', 'train')
    os.rename(val, split)
    os.rename(os.path.join(root, 'gtFine', 'val'), os.path.join(root, 'gtFine', 'train'))
    write_s = time.perf_counter() - t0

    # 1. fill: decode + copy into the arena
    pairs = train_input.split_pairs(split, 'cityscapes')
    sizes, _, _ = dataset_input.check_pairs(pairs)
    table = est._replacevoids(problem_defs.cityscapes()['lids2cids'])
    shard = train_input.Shard(pairs, sizes, len(table), dev, budget=train_input.device_budget(dev))
    fill_s = shard.seconds

    # 2. wlseg_train_inputs alone, indices rotating over the whole arena
    lut = torch.tensor(table, dtype=torch.int32, device=dev)
    order = torch.from_numpy(np.concatenate([np.random.default_rng(r).permutation(len(pairs)) for r in range(8)])
                             .astype(np.int32)).to(dev)
    per_pass = order.numel() // Nb
    outs = [(torch.empty((Nb,) + hw + (3,), dtype=torch.float32, device=dev),
             torch.empty((Nb,) + hw, dtype=torch.int32, device=dev)) for _ in range(2)]
    invalid = torch.zeros(1, dtype=torch.int64, device=dev)

    def launch(i):
      k = i % per_pass
      ops.train_inputs(shard.arena, shard.offsets, shard.sizes, order[k * Nb:(k + 1) * Nb], lut, max(table), hw,
                       *outs[i % 2], invalid)
    for i in range(8):
      launch(i)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.launches):
      launch(i)
    ev1.record()
    torch.cuda.synchronize()
    assert int(invalid.item()) == 0
    us_per_batch = ev0.elapsed_time(ev1) * 1e3 / args.launches
    del shard
    gc.collect()

    # 3. device-side training, arena-fed vs synthetic-fed, alternated
    st = _train_settings(os.path.join(tmp, 'log_dev'), 'cityscapes', dev, ['--per_pixel_split_path', split])
    st.Nb_per_bbox = st.Nb_per_image = 0
    e = _estimator(st, dev)
    st.output_Nclasses = e.hier.num_classes
    with contextlib.redirect_stdout(quiet):
      arms = {'arena': train_input.train_input_fn(None, st), 'synthetic': synthetic.train_input_fn(None, st)}
    for it in arms.values():
      e.train(it, 4)                       # warm-up: eager steps, graph capture (one graph: the shapes are equal)
    times = {k: [] for k in arms}
    for _ in range(args.repeats):
      for k, it in arms.items():
        torch.cuda.synchronize()
        ev0.record()
        losses = e.train(it, args.steps)
        ev1.record()
        torch.cuda.synchronize()
        assert np.isfinite(losses).all()
        times[k].append(ev0.elapsed_time(ev1) / 1e3)
    del arms, e
    gc.collect()
    torch.cuda.empty_cache()
    rate = {k: args.steps * Nb / float(np.median(v)) for k, v in times.items()}

    # 4. end to end: train.py on the directory, fill included
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(quiet):
      losses = cli.train_main([os.path.join(tmp, 'log_e2e'), 'cityscapes', '--per_pixel_split_path', split,
                               '--steps', str(args.e2e_steps)])
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert losses.shape == (args.e2e_steps, 6) and np.isfinite(losses).all()

    name, limit = card()
    print(json.dumps({
        'tool': 'train_dataset_bench', 'gpu': name, 'power_limit': limit, 'images': len(pairs), 'Nb': Nb,
        'source_size': [1024, 2048], 'network_size': list(hw), 'decode_workers': dataset_input._workers_per_rank(),
        'host_cpus': os.cpu_count(), 'split_write_s': round(write_s, 2),
        'arena_bytes': sum(h * w * 4 for h, w in sizes),
        'fill_images_per_s': round(len(pairs) / fill_s, 2),
        'train_inputs_us_per_batch': round(us_per_batch, 2),
        'train_inputs_algorithmic_GBps': round(Nb * hw[0] * hw[1] * (16 + 13) / (us_per_batch * 1e-6) / 1e9, 1),
        'train_images_per_s_arena': round(rate['arena'], 2),
        'train_images_per_s_synthetic': round(rate['synthetic'], 2),
        'arena_vs_synthetic': round(rate['arena'] / rate['synthetic'], 4),
        'repeat_s': {k: [round(t, 4) for t in v] for k, v in times.items()},
        'step_footprint_bytes': footprint,
        'e2e_steps': args.e2e_steps, 'e2e_s': round(e2e_s, 2),
        'e2e_includes': 'discovery, header checks, fill, estimator construction, warm-up and graph capture',
    }), flush=True)
  finally:
    quiet.close()
    if not args.workdir:
      shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
  main()
