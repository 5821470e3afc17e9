"""Throughput of evaluation on a split read from disk (wlseg/dataset_input.py + wlseg_eval_inputs), one JSON line.

    python tools/eval_dataset_bench.py [--images 64] [--Nb 4]

Writes a seeded Cityscapes-layout split of 1024 x 2048 PNG image / label pairs into a temporary directory (removed at
the end), then measures on cuda:0:
  decode_images_per_s       the DataLoader alone (PIL decoding in worker processes), no GPU work
  device_images_per_s       packed raw batches already on the device through Estimator.evaluate: wlseg_eval_inputs +
                            the evaluation step, CUDA events
  e2e_images_per_s          cli.evaluate_main on the directory, wall clock around the call (it ends in a synchronise)
  eval_inputs_us_per_image  wlseg_eval_inputs alone, CUDA events over many launches rotating through 4 batches of
                            inputs and outputs (~280 MB at the defaults, more than the 126 MB L2); its algorithmic GB/s
                            counts 16 B written + 13 B gathered (4 RGB taps + 1 label id) per output pixel
  h2d_bytes_per_image       bytes of a packed batch per image (what the staging ring copies)
The card's name and power limit are read in the same run.  Needs a GPU: there is no CPU fallback.
"""

import argparse
import contextlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'iv2019-boosting-semantic-segmentation-with-weak-labels_b200')
for _p in (ROOT, PKG):
  if _p not in sys.path:
    sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def write_split(root, n, h, w, seed):
  """Smooth colour fields with noise (compress like photographs more than white noise does) and blocky label ids."""
  from PIL import Image
  rng = np.random.default_rng(seed)
  split = os.path.join(root, 'leftImg8bit', 'val')
  for i in range(n):
    city = ('aachen', 'bochum', 'zurich')[i % 3]
    for d in ('leftImg8bit', 'gtFine'):
      os.makedirs(os.path.join(root, d, 'val', city), exist_ok=True)
    coarse = rng.integers(0, 256, (h // 64, w // 64, 3), dtype=np.uint8)
    img = np.repeat(np.repeat(coarse, 64, 0), 64, 1).astype(np.int16) + rng.integers(-12, 13, (h, w, 3), dtype=np.int16)
    Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)).save(
        os.path.join(split, city, f'b_{i:04d}_leftImg8bit.png'), compress_level=1)
    ids = np.repeat(np.repeat(rng.integers(0, 34, (h // 32, w // 32), dtype=np.uint8), 32, 0), 32, 1)
    Image.fromarray(ids, mode='L').save(os.path.join(root, 'gtFine', 'val', city, f'b_{i:04d}_gtFine_labelIds.png'),
                                        compress_level=1)
  return split


def card():
  name = torch.cuda.get_device_name(0)
  try:
    limit = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
  except (OSError, subprocess.SubprocessError):
    limit = 'not measured'
  return name, limit or 'not measured'


def main():
  ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
  ap.add_argument('--images', type=int, default=64)
  ap.add_argument('--Nb', type=int, default=4)
  ap.add_argument('--height', type=int, default=512, help='height_feature_extractor')
  ap.add_argument('--width', type=int, default=1024, help='width_feature_extractor')
  ap.add_argument('--launches', type=int, default=200, help='wlseg_eval_inputs launches timed')
  args = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('eval_dataset_bench.py measures on a GPU; none is available')
  from oracle import network as onet
  from wlseg import checkpoints, cli, dataset_input, estimator as est, ops, problem_defs, settings as wsettings
  from wlseg.system_factory import SemanticSegmentation
  dev = torch.device('cuda:0')
  torch.cuda.set_device(dev)
  steps = args.images // args.Nb
  n = steps * args.Nb
  hw = (args.height, args.width)
  tmp = tempfile.mkdtemp(prefix='wlseg_eval_bench_')
  quiet = open(os.devnull, 'w')
  try:
    t0 = time.perf_counter()
    split = write_split(tmp, n, 1024, 2048, seed=0)
    write_s = time.perf_counter() - t0
    problem_defs.write_all()
    log_dir = os.path.join(tmp, 'log')
    os.makedirs(log_dir)
    ckpt = checkpoints.save_file(os.path.join(log_dir, 'model.ckpt-1.pt'),
                                 onet.init_params('cityscapes', seed=0, randomize_bn=True, tame=True), 1)
    argv = [log_dir, str(n), problem_defs.default_path('cityscapes'), split, 'cityscapes', '--Nb', str(args.Nb),
            '--height_feature_extractor', str(hw[0]), '--width_feature_extractor', str(hw[1]), '--ckpt_path', ckpt]

    # 1. decoding alone
    params = argparse.Namespace(tfrecords_path=split, Nb=args.Nb, num_eval_steps=steps, rank=0, world_size=1)
    t0 = time.perf_counter()
    staged, h2d = [], 0
    for features, labels in dataset_input.eval_input_fn(None, params):
      h2d += sum(t.numel() * t.element_size() for t in list(features.values()) + list(labels.values()))
      if len(staged) < 4:
        staged.append(({k: v.to(dev) for k, v in features.items()}, {k: v.to(dev) for k, v in labels.items()}))
    decode_s = time.perf_counter() - t0

    # 2. device side: pre-staged packed batches through Estimator.evaluate (eval_inputs + evaluation step)
    st = wsettings.eval_extra_args(wsettings.build_parser(wsettings.EVAL).parse_args(argv))
    st.device, st.rank, st.world_size = str(dev), 0, 1
    with contextlib.redirect_stdout(quiet):
      system = SemanticSegmentation({'eval': None}, None, st)
      e = system._create_estimator(ckpt_path=ckpt)
    lut = est._replacevoids(system.settings.training_cids2evaluation_cids)
    num_classes = max(lut) + 1
    lut = None if lut == list(range(len(lut))) else lut
    rounds = max(1, steps // len(staged))
    e.evaluate(staged * 2, num_classes, lut=lut)          # warm-up: first step eager, graph capture
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    e.evaluate(staged * rounds, num_classes, lut=lut)
    ev1.record()
    torch.cuda.synchronize()
    device_s = ev0.elapsed_time(ev1) / 1e3
    device_images = rounds * len(staged) * args.Nb

    # 3. wlseg_eval_inputs alone
    lut_ids = torch.tensor(est._replacevoids(system.settings.evaluation_problem_def['lids2cids']), dtype=torch.int32,
                           device=dev)
    void_id = int(lut_ids.max())
    outs = [(torch.empty((args.Nb,) + hw + (3,), dtype=torch.float32, device=dev),
             torch.empty((args.Nb,) + hw, dtype=torch.int32, device=dev)) for _ in staged]
    invalid = torch.zeros(1, dtype=torch.int64, device=dev)

    def launch(i):
      f, l = staged[i % len(staged)]
      ops.eval_inputs(f[dataset_input.PACKED_IMAGES], l[dataset_input.PACKED_LIDS], f[dataset_input.PACKED_SIZES], lut_ids,
                      void_id, hw, *outs[i % len(staged)], invalid)
    for i in range(8):
      launch(i)
    ev0.record()
    for i in range(args.launches):
      launch(i)
    ev1.record()
    torch.cuda.synchronize()
    assert int(invalid.item()) == 0
    us_per_image = ev0.elapsed_time(ev1) * 1e3 / (args.launches * args.Nb)
    bytes_per_image = hw[0] * hw[1] * (16 + 13)

    # 4. end to end (after 2 and 3: the library's modules are loaded): evaluate.py on the directory
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(quiet):
      m = cli.evaluate_main(argv)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert m[0]['steps'] == steps

    name, limit = card()
    print(json.dumps({
        'tool': 'eval_dataset_bench', 'gpu': name, 'power_limit': limit, 'images': n, 'Nb': args.Nb,
        'source_size': [1024, 2048], 'network_size': list(hw), 'decode_workers': dataset_input._workers_per_rank(),
        'host_cpus': os.cpu_count(), 'split_write_s': round(write_s, 2),
        'decode_images_per_s': round(n / decode_s, 2),
        'device_images_per_s': round(device_images / device_s, 2),
        'e2e_images_per_s': round(n / e2e_s, 2),
        'e2e_includes': 'estimator construction, checkpoint restore, first-step warm-up and graph capture',
        'eval_inputs_us_per_image': round(us_per_image, 2),
        'eval_inputs_algorithmic_GBps': round(bytes_per_image / (us_per_image * 1e-6) / 1e9, 1),
        'h2d_bytes_per_image': h2d // n,
    }), flush=True)
  finally:
    quiet.close()
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
  main()
