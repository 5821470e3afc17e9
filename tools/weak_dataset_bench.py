"""Throughput of training on a Cityscapes split plus Open Images weak labels read from disk (wlseg/weak_input.py +
wlseg_weak_train_inputs), one JSON line.

    python tools/weak_dataset_bench.py [--images 96] [--pairs 32] [--steps 30] [--repeats 4] [--e2e-steps 60]
                                       [--workdir DIR]

Writes a seeded Open Images-layout split (JPEGs of mixed sizes and aspect ratios up to 1024 on the long side, the
descriptions file, one bbox CSV and one image-level CSV) and a seeded Cityscapes-layout training split of 1024 x 2048
PNG pairs into --workdir (a temporary directory, removed at the end, when not given), then measures on cuda:0:
  mixed_step_footprint_bytes  drop of free device memory across the first 3 steps of Estimator.train on synthetic
                              4 + 8 + 4 batches with dense weak labels, at Cityscapes 512 x 1024 and Vistas 621 x 855
                              (what wlseg.train_input.MIXED_STEP_RESERVE_BYTES must leave free next to the arenas)
  fill_images_per_s           decode (PIL in DataLoader workers) + copy of the Open Images split into one weak arena
  weak_inputs_us_per_step     wlseg_weak_train_inputs alone: one 8-example bbox launch + one 4-example image-level
                              launch -> 512 x 1024, CUDA events over --launches launch pairs whose indices rotate over
                              an arena larger than the 126 MB L2; its algorithmic GB/s counts 12 B image + 60 B label
                              written and 12 B gathered (4 RGB taps) per output pixel
  train_images_per_s_arenas / _synthetic
                              Estimator.train at 4 + 8 + 4 x 512 x 1024 (bf16) fed from the three arenas vs fed from
                              the on-device synthetic generator with dense weak labels, CUDA events, the two arms
                              alternated --repeats times; the median of each arm
  e2e_s                       cli.train_main with all three split flags for --e2e-steps steps, wall clock, fills included
The card's name and power limit are read in the same run.  Needs a GPU: there is no CPU fallback.
"""

import argparse
import contextlib
import csv
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
from train_dataset_bench import _estimator, _train_settings  # noqa: E402

# (H, W) of the generated Open Images JPEGs: landscape, portrait, square and panorama, long side <= 1024 as in the release
SIZES = ((768, 1024), (1024, 768), (683, 1024), (1024, 1024), (576, 1024), (1024, 681), (400, 1024))


def write_open_images(root, n, seed=0):
  """n seeded JPEGs (smooth colour fields + noise, so JPEG sizes are realistic) with 1..12 boxes and 1..4 positive tags
  of the 14 weak classes each, plus boxes / tags of another class."""
  from PIL import Image
  from wlseg import hierarchy
  rng = np.random.default_rng(seed)
  os.makedirs(os.path.join(root, 'images'), exist_ok=True)
  mids = [f'/m/bench{c:02d}' for c in range(14)]
  with open(os.path.join(root, 'class-descriptions-boxable.csv'), 'w', newline='') as f:
    w = csv.writer(f)
    w.writerows([(m, hierarchy.weak_display_name(c)) for c, m in enumerate(mids)] + [('/m/benchtree', 'Tree')])
  boxes, tags = [], []
  for i in range(n):
    h, w = SIZES[i % len(SIZES)]
    base = rng.integers(0, 256, (h // 32 + 1, w // 32 + 1, 3)).astype(np.uint8)
    img = np.repeat(np.repeat(base, 32, 0), 32, 1)[:h, :w]
    img = (img.astype(np.int16) + rng.integers(-12, 13, img.shape)).clip(0, 255).astype(np.uint8)
    image_id = f'{i:016x}'
    Image.fromarray(img).save(os.path.join(root, 'images', image_id + '.jpg'), quality=90)
    for _ in range(int(rng.integers(1, 13))):
      x, y = np.sort(rng.random(2)), np.sort(rng.random(2))
      boxes.append((image_id, 'xclick', mids[int(rng.integers(0, 14))], 1, f'{x[0]:.6f}', f'{x[1]:.6f}', f'{y[0]:.6f}',
                    f'{y[1]:.6f}', 0, 0, 0, 0, 0))
    boxes.append((image_id, 'xclick', '/m/benchtree', 1, '0.1', '0.9', '0.1', '0.9', 0, 0, 0, 0, 0))
    for c in rng.choice(14, int(rng.integers(1, 5)), replace=False):
      tags.append((image_id, 'verification', mids[int(c)], 1))
    tags.append((image_id, 'verification', '/m/benchtree', 1))
  with open(os.path.join(root, 'train-annotations-bbox.csv'), 'w', newline='') as f:
    w = csv.writer(f)
    w.writerow(['ImageID', 'Source', 'LabelName', 'Confidence', 'XMin', 'XMax', 'YMin', 'YMax', 'IsOccluded',
                'IsTruncated', 'IsGroupOf', 'IsDepiction', 'IsInside'])
    w.writerows(boxes)
  with open(os.path.join(root, 'train-annotations-human-imagelabels-boxable.csv'), 'w', newline='') as f:
    w = csv.writer(f)
    w.writerow(['ImageID', 'Source', 'LabelName', 'Confidence'])
    w.writerows(tags)
  return root


def mixed_step_footprint(dataset, dev, tmp):
  """Free device memory before minus after the first 3 training steps on synthetic 4 + 8 + 4 batches."""
  from wlseg import synthetic
  st = _train_settings(os.path.join(tmp, f'fp_{dataset}'), dataset, dev)
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
  ap.add_argument('--images', type=int, default=96, help='Open Images JPEGs generated')
  ap.add_argument('--pairs', type=int, default=32, help='Cityscapes image / label pairs generated')
  ap.add_argument('--steps', type=int, default=30, help='training steps per timed repeat')
  ap.add_argument('--repeats', type=int, default=4)
  ap.add_argument('--launches', type=int, default=200, help='launch pairs (bbox + image-level) timed')
  ap.add_argument('--e2e-steps', type=int, default=60)
  ap.add_argument('--workdir', default=None)
  args = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('weak_dataset_bench.py measures on a GPU; none is available')
  from wlseg import cli, problem_defs, synthetic, train_input, weak_input
  dev = torch.device('cuda:0')
  torch.cuda.set_device(dev)
  problem_defs.write_all()
  tmp = args.workdir or tempfile.mkdtemp(prefix='wlseg_weak_bench_')
  os.makedirs(tmp, exist_ok=True)
  quiet = open(os.devnull, 'w')
  hw = (512, 1024)
  try:
    # 0. the mixed step's own device memory at train.py's two sizes, before anything else is resident
    with contextlib.redirect_stdout(quiet):
      footprint = {'cityscapes_4+8+4x512x1024': mixed_step_footprint('cityscapes', dev, tmp),
                   'vistas_4+8+4x621x855': mixed_step_footprint('vistas', dev, tmp)}

    t0 = time.perf_counter()
    oi = write_open_images(os.path.join(tmp, 'oi'), args.images)
    root = os.path.join(tmp, 'cs')
    val = write_split(root, args.pairs, 1024, 2048, seed=0)
    split = os.path.join(root, 'leftImg8bit', 'train')
    os.rename(val, split)
    os.rename(os.path.join(root, 'gtFine', 'val'), os.path.join(root, 'gtFine', 'train'))
    write_s = time.perf_counter() - t0

    # 1. fill of one weak arena; the image-level part holds the same images
    parts = {p: weak_input.WeakPart(p, oi, nb, hw, 0, 1, 0) for p, nb in (('bbox', 8), ('image', 4))}
    with contextlib.redirect_stdout(quiet):
      for part in parts.values():
        part.fill(dev)
    fill_s = parts['bbox'].shard.seconds
    arena_bytes = parts['bbox'].shard.bytes

    # 2. wlseg_weak_train_inputs alone: one bbox + one image-level launch per step, orders rotating over the arena
    outs = [(torch.empty((8,) + hw + (3,), device=dev), torch.empty((8,) + hw + (15,), device=dev),
             torch.empty((4,) + hw + (3,), device=dev), torch.empty((4,) + hw + (15,), device=dev)) for _ in range(2)]
    # steps of epoch 0 only, so that no order is uploaded inside the timed window; one bbox epoch covers every image
    spe = min(p.steps_per_epoch for p in parts.values())

    def launch(i):
      o = outs[i % 2]
      parts['bbox'].gather(i % spe, o[0], o[1])
      parts['image'].gather(i % spe, o[2], o[3])
    for i in range(spe):
      launch(i)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for i in range(args.launches):
      launch(i)
    ev1.record()
    torch.cuda.synchronize()
    assert all(int(p.invalid.item()) == 0 for p in parts.values())
    us_per_step = ev0.elapsed_time(ev1) * 1e3 / args.launches
    del parts, outs
    gc.collect()
    torch.cuda.empty_cache()

    # 3. device-side training, arena-fed vs synthetic-fed (dense weak labels), alternated
    st = _train_settings(os.path.join(tmp, 'log_dev'), 'cityscapes', dev,
                         ['--per_pixel_split_path', split, '--per_bbox_split_path', oi, '--per_image_split_path', oi])
    e = _estimator(st, dev)
    st.output_Nclasses = e.hier.num_classes
    with contextlib.redirect_stdout(quiet):
      arms = {'arenas': train_input.train_input_fn(None, st), 'synthetic': synthetic.train_input_fn(None, st)}
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
    rate = {k: args.steps * 16 / float(np.median(v)) for k, v in times.items()}

    # 4. end to end: train.py on the two directories, fills included
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(quiet):
      losses = cli.train_main([os.path.join(tmp, 'log_e2e'), 'cityscapes', '--per_pixel_split_path', split,
                               '--per_bbox_split_path', oi, '--per_image_split_path', oi, '--steps', str(args.e2e_steps)])
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert losses.shape == (args.e2e_steps, 6) and np.isfinite(losses).all()

    name, limit = card()
    npix = 12 * hw[0] * hw[1]
    print(json.dumps({
        'tool': 'weak_dataset_bench', 'gpu': name, 'power_limit': limit, 'open_images': args.images,
        'cityscapes_pairs': args.pairs, 'batch': '4 + 8 + 4', 'network_size': list(hw), 'host_cpus': os.cpu_count(),
        'split_write_s': round(write_s, 2), 'weak_arena_bytes': arena_bytes,
        'fill_images_per_s': round(args.images / fill_s, 2),
        'weak_inputs_us_per_step': round(us_per_step, 2),
        'weak_inputs_algorithmic_GBps': round(npix * (12 + 60 + 12) / (us_per_step * 1e-6) / 1e9, 1),
        'train_images_per_s_arenas': round(rate['arenas'], 2),
        'train_images_per_s_synthetic': round(rate['synthetic'], 2),
        'arenas_vs_synthetic': round(rate['arenas'] / rate['synthetic'], 4),
        'repeat_s': {k: [round(t, 4) for t in v] for k, v in times.items()},
        'mixed_step_footprint_bytes': footprint,
        'e2e_steps': args.e2e_steps, 'e2e_s': round(e2e_s, 2),
        'e2e_includes': 'discovery, CSV and header checks, fills, estimator construction, warm-up and graph capture',
    }), flush=True)
  finally:
    quiet.close()
    if not args.workdir:
      shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
  main()
