#!/usr/bin/env python
"""bench.py -- headline benchmark of the wlseg hot path.

BASELINE.json's metric has two halves; the default run measures BOTH in one process and prints ONE line:

  headline  (BASELINE configs[2]) Cityscapes strong-label TRAINING step, 768x768 crops, batch 4 per GPU, bf16,
            data parallel over the ranks with the NCCL gradient all-reduce inside the timed region
            -> metric train_images_per_s (value, e2e, roofline, cpu_baseline, sustained, clocks)
  "eval"    (BASELINE configs[1]) Cityscapes-shaped EVALUATION: ResNet-50 OS8 forward + hierarchical heads +
            argmax + confusion matrix at 1024x2048, batch 4 per step, image-sharded over the ranks
            -> nested object with the same keys, metric eval_mpix_per_s

  python bench.py --gpus N --steps K --warmup W          # this implementation, both halves
  python bench.py --workload train|eval ...              # one half only (the line is that half's record)
  python bench.py --impl reference --steps K --warmup W  # the reference algorithm on the host CPU (oracle port;
                                                         # TF 1.12 is uninstallable): the training step, same
                                                         # config as the headline, eval nested
  python bench.py --dump-outputs DIR ...                 # also write what the last timed step computed, as
                                                         # DIR/<name>.npy, so that two builds can be compared

One JSON line is printed by rank 0.  The inputs and the initial parameters are seeded: the same arguments give the same
inputs on every run.
"""

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'iv2019-boosting-semantic-segmentation-with-weak-labels_b200')
for _p in (ROOT, PKG):
  if _p not in sys.path:
    sys.path.insert(0, _p)

EVAL_H, EVAL_W, EVAL_NB = 1024, 2048, 4
TRAIN_H, TRAIN_W, TRAIN_NB = 768, 768, 4


def parse_args():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', type=str, default='wlseg', choices=['wlseg', 'reference'])
  ap.add_argument('--workload', type=str, default='both', choices=['both', 'eval', 'train'])
  ap.add_argument('--dataset', type=str, default='cityscapes', choices=['cityscapes', 'vistas'])
  ap.add_argument('--height', type=int, default=None)
  ap.add_argument('--width', type=int, default=None)
  ap.add_argument('--batch', type=int, default=None)
  ap.add_argument('--mixed', action='store_true', help='train workload: add 8 bbox + 4 image-level images per GPU')
  ap.add_argument('--boxes', action='store_true', help='--mixed: weak labels generated inside the loss kernel from box / class lists')
  ap.add_argument('--sustained-seconds', type=float, default=3.0, help='length of the extra sustained-clock loop (0 = skip)')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-e2e', action='store_true')
  ap.add_argument('--detail', type=str, default=None, help='write the per-kernel-class roofline table here')
  ap.add_argument('--dump-outputs', type=str, default=None, metavar='DIR',
                  help='write the outputs of the last timed step as DIR/<name>.npy (float32 / float64)')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'wlseg':
    ap.error('--dump-outputs records the wlseg arm only')
  return args


def load_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as fp:
      p = json.load(fp)
    return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
            'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
  return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


def load_traffic(workload, kernel_prefix):
  """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, averaged over the launches of
  one step) of the dominant kernel, from the committed ncu capture of this same command
  (profiles/rNN_traffic.json, written by tools/make_profiles.py).  None when no capture is committed."""
  pdir = os.path.join(ROOT, 'profiles')
  if not os.path.isdir(pdir):
    return None, None
  files = sorted(f for f in os.listdir(pdir) if f.endswith('_traffic.json'))
  if not files:
    return None, None
  with open(os.path.join(pdir, files[-1])) as fp:
    t = json.load(fp).get(workload, {})
  # the kernel class spans several template instantiations (single CTA / CTA pair / BN-backward epilogue):
  # launch-weighted mean over all of them
  hits = [v for k, v in t.items() if k.startswith(kernel_prefix)]
  n = sum(v['launches'] for v in hits)
  if not n:
    return None, None
  return sum(v['dram_bytes_per_launch'] * v['launches'] for v in hits) / n, files[-1]


def dump_outputs(out_dir, arrays):
  """--dump-outputs: every array as out_dir/<name>.npy, integer and float64 arrays as float64 (exact for counts below
  2**53), the others as float32."""
  import numpy as np
  import torch
  os.makedirs(out_dir, exist_ok=True)
  for name, t in arrays.items():
    t = t.detach().double() if t.dtype in (torch.int32, torch.int64, torch.float64) else t.detach().float()
    np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy())


class ClockSampler:
  """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, index=0):
    self.file = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
    self.proc = None
    try:
      self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                    '-i', str(index), '-lms', '100'], stdout=self.file, stderr=subprocess.DEVNULL)
    except OSError:
      self.proc = None

  def stop(self):
    out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
    if self.proc is None:
      return out
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except subprocess.TimeoutExpired:
      self.proc.kill()
    self.file.flush()
    self.file.seek(0)
    sm, mx, reasons = [], [], set()
    names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
    for line in self.file.read().splitlines():
      f = [x.strip() for x in line.split(',')]
      if len(f) < 9:
        continue
      try:
        sm.append(float(f[1]))
        mx.append(float(f[2]))
      except ValueError:
        continue
      for name, val in zip(names, f[5:9]):
        if val.lower().startswith('active'):
          reasons.add(name)
    self.file.close()
    os.unlink(self.file.name)
    if sm:
      out['sm_mhz'] = statistics.median(sm)
      out['sm_max_mhz'] = max(mx)
      out['samples'] = len(sm)
    out['reasons'] = sorted(reasons)
    return out


def cpu_reference_eval(dataset, h, w, steps, warmup, images_per_step=1):
  """The reference algorithm (oracle port: PyTorch-CPU fp32 restatement of the TF-1.12 graph)
  timed on the host cores: forward + argmax + confusion matrix, `images_per_step` images per step."""
  import numpy as np
  import torch
  from oracle import metrics as ometrics
  from oracle import network as onet
  from oracle.tables import TABLES
  torch.set_num_threads(os.cpu_count() or 1)
  ncls = TABLES[dataset]['num_classes']
  params = onet.init_params(dataset, seed=0)
  net = onet.Net(params, dataset)
  g = torch.Generator().manual_seed(1234)
  images = torch.rand(images_per_step, h, w, 3, generator=g) * 2 - 1
  labels = torch.randint(0, ncls, (images_per_step, h, w), generator=g, dtype=torch.int32).numpy()
  cm = np.zeros((ncls, ncls), dtype=np.int64)
  times = []
  with torch.no_grad():
    for i in range(warmup + steps):
      t0 = time.perf_counter()
      pred = net.forward(images)
      cm += ometrics.confusion_matrix(labels, pred['decisions'].numpy(), ncls)
      dt = time.perf_counter() - t0
      if i >= warmup:
        times.append(dt)
  total = sum(times)
  mpix = images_per_step * h * w * len(times) / 1e6
  return {'value': mpix / total, 'unit': 'Mpix/s', 'cores': torch.get_num_threads(), 'kind': 'port',
          'sample': f'{len(times)} step(s) of {images_per_step} image(s) {h}x{w}, oracle fp32 on CPU, '
                    f'{warmup} warm-up', 'ms_per_step': 1e3 * total / len(times)}


def cpu_reference_train(dataset, h, w, steps=1, warmup=0, images_per_step=1, mixed=False):
  """The reference algorithm's training step (oracle: fp32 PyTorch-CPU restatement, autograd
  backward, momentum update) on `images_per_step` images per step, all host cores."""
  import torch
  from oracle import losses as olosses
  from oracle import network as onet
  from oracle import optimizer as oopt
  from oracle.tables import TABLES
  torch.set_num_threads(os.cpu_count() or 1)
  ncls = TABLES[dataset]['num_classes']
  params = {k: v.clone().requires_grad_(not k.endswith(('moving_mean', 'moving_variance')))
            for k, v in onet.init_params(dataset, seed=0).items()}
  g = torch.Generator().manual_seed(1234)
  nb = images_per_step
  npb, npi = (2 * nb, nb) if mixed else (0, 0)
  images = torch.rand(nb + npb + npi, h, w, 3, generator=g) * 2 - 1
  labels = {'prolabels_per_pixel': torch.randint(0, ncls, (nb, h, w), generator=g, dtype=torch.int32)}
  if mixed:
    from oracle import weak_labels as oweak
    labels['prolabels_per_bbox'] = torch.stack([torch.from_numpy(oweak.bbox_labels(
        [(int(torch.randint(0, 14, (1,), generator=g)), 0.1, 0.6, 0.2, 0.9)], h, w)) for _ in range(npb)])
    labels['prolabels_per_image'] = torch.stack([torch.from_numpy(oweak.image_labels(
        [int(torch.randint(0, 14, (1,), generator=g))], h, w)) for _ in range(npi)])
  acc = {k: torch.zeros_like(v) for k, v in params.items() if v.requires_grad}
  times = []
  for i in range(warmup + steps):
    t0 = time.perf_counter()
    for v in params.values():
      v.grad = None
    net = onet.Net(params, dataset, training=True)
    pred = net.forward(images)
    loss = olosses.define_losses(pred, labels, dataset)['total']
    loss.backward()
    with torch.no_grad():
      for k, v in params.items():
        if v.requires_grad:
          wn, an = oopt.momentum_step(v, v.grad + (0.00017 * v if k.endswith('weights') else 0.0), acc[k], 0.01)
          v.copy_(wn)
          acc[k] = an
      for k, v in net.new_moving.items():   # UPDATE_OPS: the moving statistics follow the batch
        params[k].copy_(v.detach())
    dt = time.perf_counter() - t0
    if i >= warmup:
      times.append(dt)
  total = sum(times)
  nimg = nb + npb + npi
  return {'value': nimg * len(times) / total, 'unit': 'images/s', 'cores': torch.get_num_threads(), 'kind': 'port',
          'sample': f'{len(times)} training step(s) on {nimg} image(s) {h}x{w}, oracle fp32 autograd on CPU, '
                    f'{warmup} warm-up', 'ms_per_step': 1e3 * total / len(times)}


def train_workload_name(dataset, H, W, NB, npb, npi, mixed):
  """config.workload of the training half - the SAME string in both arms (the driver compares them)."""
  return (f'{dataset} training step (BASELINE configs[{3 if mixed else 2}]): ResNet-50 OS8 + hierarchical heads, '
          f'fwd (batch-stat BN) + masked strong{"+weak" if mixed else ""} loss + bwd + SGD-momentum, {H}x{W} crops, '
          f'{NB} strong + {npb} bbox + {npi} image-level images/GPU, random init')


def eval_workload_name(dataset, H, W, NB):
  return (f'{dataset} eval (BASELINE configs[1]): ResNet-50 OS8 forward + hierarchical heads + argmax + confusion '
          f'matrix, {H}x{W}, batch {NB}/GPU/step, random init')


def reference_eval_record(args, steps, warm):
  h, w, nb = args.height or EVAL_H, args.width or EVAL_W, args.batch or EVAL_NB
  r = cpu_reference_eval(args.dataset, h, w, steps, warm, images_per_step=nb)
  return {'impl': 'reference', 'metric': 'eval_mpix_per_s', 'value': r['value'], 'unit': 'Mpix/s', 'n_gpus': args.gpus,
          'steps': steps, 'warmup': warm, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
          'config': {'workload': eval_workload_name(args.dataset, h, w, nb),
                     'sample': 'reference arm = the oracle port of the TF-1.12 graph (TensorFlow cannot be installed) on '
                               f'the host cores; {steps} timed step(s) of the same batch of {nb}'},
          'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
          'e2e': {'value': r['value'], 'unit': 'Mpix/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
          'gpu_launches': 0}


def reference_train_record(args, steps, warm):
  h, w, nb = args.height or TRAIN_H, args.width or TRAIN_W, args.batch or TRAIN_NB
  mixed = bool(getattr(args, 'mixed', False))
  npb, npi = (2 * nb, nb) if mixed else (0, 0)
  r = cpu_reference_train(args.dataset, h, w, steps, warm, images_per_step=nb, mixed=mixed)
  return {'impl': 'reference', 'metric': 'train_images_per_s', 'value': r['value'], 'unit': 'images/s',
          'n_gpus': args.gpus, 'steps': steps, 'warmup': warm, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True,
          'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
          'config': {'workload': train_workload_name(args.dataset, h, w, nb, npb, npi, mixed),
                     'sample': 'reference arm = the oracle port of the TF-1.12 graph (TensorFlow cannot be installed) on '
                               f'the host cores, fp32 autograd; {steps} timed step(s) of the same per-GPU batch'},
          'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
          'e2e': {'value': r['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
          'gpu_launches': 0}


def run_reference(args):
  """Reference arm: the reference's own algorithm (oracle port) on the host cores, rank 0 only.  Same config as the
  GPU arm (a full per-GPU batch per step) and the same step counts: a 4 x 768 x 768 fp32 training step takes ~10 s on
  16 cores, a 4 x 1024 x 2048 evaluation step ~10 s, so pass a small --steps / --warmup here."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  if args.workload == 'eval':
    line = reference_eval_record(args, args.steps, args.warmup)
  else:
    line = reference_train_record(args, args.steps, args.warmup)
    if args.workload == 'both':
      line['eval'] = reference_eval_record(args, args.steps, args.warmup)
  print(json.dumps(line), flush=True)


def tensor_roofline(name, dom, peaks, region_seconds, traffic, tsrc, share, timed_over):
  """Roofline object of a tensor-core kernel class.  `frac` is against the peak the region EARNS: the burst figure
  for a timed region shorter than 1 s (boost clocks, before the power cap settles; also what a kernel timed alone
  between event pairs sees), the sustained one for a long region; both fractions are always reported."""
  ach = dom['flops'] / (dom['ms'] / 1e3) / 1e12
  burst, sust = peaks['bf16_tflops'], peaks['bf16_tflops_sustained']
  kind = 'burst' if region_seconds < 1.0 else 'sustained'
  peak = burst if kind == 'burst' else sust
  return {'bound': 'tensor', 'kernel': name, 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak,
          'peak_kind': kind, 'frac_burst': ach / burst, 'frac_sustained': ach / sust, 'peak_burst': burst,
          'peak_sustained': sust, 'traffic': traffic,
          'traffic_unit': 'DRAM bytes per launch (ncu, mean over the launches of a step)',
          'traffic_source': None if tsrc is None else 'profiles/' + tsrc,
          'algorithmic_bytes_per_launch': dom['bytes'] / dom['launches'],
          'flops_per_launch': dom['flops'] / dom['launches'],
          'peak_source': peaks['source'] + f' (cuBLAS bf16, {kind}; timed region {region_seconds:.2f} s)',
          'launches': dom['launches'], 'share_of_step': share, 'timed_over': timed_over}


def sustained_loop(step, seconds, ms_per_step_hint, units_per_step, unit, dev, world, rank, local_rank):
  """The same graph replays for >= `seconds` (the power cap settles after ~1 s of dense tensor work): the regime
  a long job runs in, next to the short K-step region the contract times."""
  import torch
  import torch.distributed as dist
  if seconds <= 0:
    return None
  n = max(8, int(seconds * 1e3 / max(ms_per_step_hint, 1e-3)) + 1)
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  sampler = ClockSampler(local_rank) if rank == 0 else None
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(n):
    step(i)
  e1.record()
  torch.cuda.synchronize()
  clocks = sampler.stop() if sampler else None
  t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms = float(t.item())
  return {'steps': n, 'seconds': ms / 1e3, 'ms_per_step': ms / n, 'value': world * n * units_per_step / (ms / 1e3),
          'unit': unit, 'clocks': clocks}


class Ctx:
  """Process-wide set-up shared by the two halves: device, ranks, one NCCL communicator."""

  def __init__(self):
    import torch
    self.world = int(os.environ.get('WORLD_SIZE', '1'))
    self.rank = int(os.environ.get('RANK', '0'))
    self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
      raise SystemExit('bench.py: no CUDA device; wlseg has no CPU fallback')
    torch.cuda.set_device(self.local_rank)
    self.dev = torch.device('cuda', self.local_rank)
    if self.world > 1:
      import torch.distributed as dist
      with StdoutToStderr():   # the NCCL banner must not land on stdout (one JSON line only)
        dist.init_process_group('nccl', device_id=self.dev)
        dist.all_reduce(torch.zeros(1, device=self.dev))  # communicator set-up outside every timed region
        torch.cuda.synchronize()


def run_wlseg_eval(args, ctx):
  import torch
  import torch.distributed as dist
  from wlseg import arch, hierarchy, network, ops, problem_defs, synthetic

  world, rank, local_rank, dev = ctx.world, ctx.rank, ctx.local_rank, ctx.dev
  quiet = StdoutToStderr()
  quiet.__enter__()

  H, W, NB = args.height or EVAL_H, args.width or EVAL_W, args.batch or EVAL_NB
  pd = problem_defs.GENERATORS[args.dataset]()
  hier = hierarchy.Hierarchy(args.dataset, pd['cids2labels'])
  ncls = hier.num_classes
  params = network.Params(hier, dev)
  params.init_random(0)
  net = network.Network(params, dtype=torch.bfloat16)
  src = synthetic.SyntheticInputs(ncls, dev, rank=rank)
  batches = [src.eval_batch(NB, H, W) for _ in range(2)]  # 2 x 133 MB + GBs of activations >> 126 MB L2
  # the product's evaluation step: forward + decisions + confusion-matrix update replayed as one CUDA graph per
  # resident input batch (network.EvalStep, what Estimator.evaluate runs)
  evstep = network.EvalStep(net, ncls)
  cm = evstep.cm

  def step(i):
    f, l = batches[i % 2]
    evstep(f['proimages'], l['prolabels'])

  for i in range(max(args.warmup, 3)):   # one eager step, then the two graph captures happen here
    step(i)
  evstep.reset()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  quiet.__exit__()

  sampler = ClockSampler(local_rank) if rank == 0 else None
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(args.steps):
    step(i)
  if world > 1:
    dist.all_reduce(cm, op=dist.ReduceOp.SUM)  # evaluation sharded by image: one exact integer reduction
  e1.record()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  clocks = sampler.stop() if sampler else None
  ms = e0.elapsed_time(e1)
  assert int(cm.sum()) == world * args.steps * NB * H * W, 'confusion matrix does not cover the timed pixels'
  if args.dump_outputs and rank == 0:
    # what a caller of the evaluation step receives: the confusion matrix over the timed steps (it was reset before
    # them) and the count of labels outside the class range
    dump_outputs(args.dump_outputs, {'eval_confusion_matrix': cm, 'eval_invalid_labels': evstep.invalid})
  t = torch.tensor([ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_max = float(t.item())
  sustained = sustained_loop(step, args.sustained_seconds, ms_max / args.steps, NB * H * W / 1e6, 'Mpix/s', dev, world,
                             rank, local_rank)
  # roofline pass, live, right after the timed region: the same steps launched eagerly with a CUDA event pair
  # around every convolution launch (events cannot sit inside a replayed graph)
  prof_steps = min(3, args.steps)
  net.profile = []
  launches0 = ops.launches
  for i in range(prof_steps):
    step(i)
  torch.cuda.synchronize()
  launches = (ops.launches - launches0) // prof_steps * args.steps
  prof = net.profile
  net.profile = None
  total_pix = world * args.steps * NB * H * W
  value = total_pix / 1e6 / (ms_max / 1e3)

  # ---- roofline of the dominant kernel: conv_igemm_kernel<BN=256> (bulk of the FLOPs) ----------
  peaks = load_peaks()
  classes = {}
  for rec in prof:
    rec['ms'] = rec['e0'].elapsed_time(rec['e1'])
    c = classes.setdefault(rec['cls'], {'flops': 0.0, 'ms': 0.0, 'launches': 0, 'bytes': 0.0})
    c['flops'] += rec['flops']
    c['ms'] += rec['ms']
    c['bytes'] += rec['bytes']
    c['launches'] += 1
  dom = classes.get('igemm_bn256')
  roofline = None
  if dom and dom['ms'] > 0:
    traffic, tsrc = load_traffic('eval', 'conv_igemm_kernel<256')
    roofline = tensor_roofline('conv_igemm_kernel<256, bf16>', dom, peaks, ms_max / 1e3, traffic, tsrc,
                               (dom['ms'] / prof_steps) / (ms / args.steps),
                               f'{prof_steps} eagerly launched steps after the timed region (graph replays)')
    roofline['whole_step_tflops'] = world * args.steps * NB * arch.conv_flops(params.specs, H, W) / (ms_max / 1e3) / 1e12
    roofline['whole_step_frac_burst'] = roofline['whole_step_tflops'] / world / peaks['bf16_tflops']
  if args.detail and rank == 0:
    table = {k: {'launches': v['launches'], 'ms_per_step': v['ms'] / prof_steps,
                 'tflops': v['flops'] / (v['ms'] / 1e3) / 1e12 if v['ms'] else None,
                 'gbs_algorithmic': v['bytes'] / (v['ms'] / 1e3) / 1e9 if v['ms'] else None}
             for k, v in sorted(classes.items())}
    with open(args.detail + ('.eval' if args.workload == 'both' else ''), 'w') as fp:
      json.dump({'ms_per_step': ms / args.steps, 'classes': table}, fp, indent=1)

  # ---- end to end through the public API with host buffers -------------------------------------
  e2e = None
  if not args.no_e2e:
    e2e = measure_e2e(args, dev, rank, world, H, W, NB)

  cpu = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    cpu = cpu_reference_eval(args.dataset, H, W, steps=2, warmup=1, images_per_step=1)
    cpu = {k: cpu[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
  fwd_gflop = arch.conv_flops(params.specs, H, W) / 1e9
  del evstep, net, params, batches, src
  torch.cuda.empty_cache()

  return {'metric': 'eval_mpix_per_s', 'value': value, 'unit': 'Mpix/s', 'n_gpus': world, 'steps': args.steps,
          'warmup': args.warmup, 'ms_per_step': ms_max / args.steps, 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
          'config': {'workload': eval_workload_name(args.dataset, H, W, NB),
                     'l2': 'inputs (2 rotating 133 MB batches) and multi-GB activations exceed the 126 MB L2',
                     'launch': 'whole step replayed as one CUDA graph per resident batch',
                     'parallelism': f'image-sharded x{world}, int64 confusion-matrix all-reduce' if world > 1 else 'single GPU',
                     'fwd_gflop_per_image': fwd_gflop},
          'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches * world, 'roofline': roofline,
          'sustained': sustained, 'cpu_baseline': cpu}


def host_link_probe(dev, world):
  """What the end-to-end number rides on besides the step: pinned host -> device copy bandwidth of this rank's
  PCIe path (128 MB, best of 3, CUDA events) and the CPUs this process may run on; the slowest rank is reported
  (the job runs at its pace).  Explains an e2e value that falls below the device-resident one."""
  import torch
  import torch.distributed as dist
  src = torch.empty(128 << 20, dtype=torch.uint8).pin_memory()
  dst = torch.empty(128 << 20, dtype=torch.uint8, device=dev)
  best = 0.0
  for _ in range(4):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    dst.copy_(src, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    best = max(best, src.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9)
  cpus = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 0)
  t = torch.tensor([-best, -float(cpus)], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  return {'h2d_gbs_slowest_rank': round(-float(t[0]), 2), 'cpus_per_rank_min': int(-float(t[1]))}


def measure_e2e(args, dev, rank, world, H, W, NB):
  """Same metric through the reference-facing API (`SemanticSegmentation.evaluate` machinery) with
  HOST buffers: every step copies its fp32 images + int32 labels from pinned host memory and reads
  the running confusion matrix back."""
  import types

  import torch
  import torch.distributed as dist
  from wlseg import problem_defs, settings as wsettings
  from wlseg.system_factory import SemanticSegmentation

  tmp = tempfile.mkdtemp(prefix='wlseg_bench_')
  ss = wsettings.build_parser(wsettings.EVAL)
  argv = [tmp, str(NB * (args.warmup + args.steps) * world), problem_defs.default_path(args.dataset), 'synthetic',
          args.dataset, '--Nb', str(NB), '--height_feature_extractor', str(H), '--width_feature_extractor', str(W),
          '--synthetic']
  st = wsettings.eval_extra_args(ss.parse_args(argv))
  st.device, st.rank, st.world_size = str(dev), rank, world
  nsteps = {'n': args.warmup}
  # two pinned host batches reused round-robin (what a host input pipeline would hand over)
  g = torch.Generator().manual_seed(1234 + rank)
  host = []
  for _ in range(2):
    img = (torch.rand((NB, H, W, 3), generator=g) * 2 - 1).pin_memory()
    lab = torch.randint(0, 20 if args.dataset == 'cityscapes' else 66, (NB, H, W), generator=g,
                        dtype=torch.int32).pin_memory()
    host.append(({'proimages': img}, {'prolabels': lab}))

  def input_fn(config, params):
    for i in range(nsteps['n']):
      yield host[i % 2]

  system = SemanticSegmentation({'eval': input_fn}, None, st)
  import contextlib
  import io
  with contextlib.redirect_stdout(io.StringIO()):
    system.evaluate()  # builds the estimator, warm-up steps
  est = system.estimator
  nsteps['n'] = args.steps
  ncls = system.settings.output_Nclasses
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  # wall clock around the public call, max over ranks; the K-step region is short (tens of ms), so it
  # is repeated three times and the MEDIAN is reported (a single host hiccup would otherwise halve it)
  dts = []
  for _ in range(3):
    if world > 1:
      dist.barrier()
    t0 = time.perf_counter()
    m = est.evaluate(input_fn(None, st), ncls)
    if world > 1:
      system._reduce_across_ranks(m)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dts.append(float(t.item()))
    assert int(m['confusion_matrix_int64'].sum()) == world * args.steps * NB * H * W
  dt = statistics.median(dts)
  import shutil
  shutil.rmtree(tmp, ignore_errors=True)
  del types
  return {'value': world * args.steps * NB * H * W / 1e6 / dt, 'unit': 'Mpix/s',
          'h2d_bytes_per_step': est.last_h2d_bytes // args.steps, 'd2h_bytes_per_step': est.last_d2h_bytes // args.steps,
          'ms_per_step': 1e3 * dt / args.steps, 'repeats': 3, 'stat': 'median of 3 repeats of the K-step region',
          'repeat_ms_per_step': [round(1e3 * d / args.steps, 3) for d in dts], 'host_link': host_link_probe(dev, world)}


class StdoutToStderr:
  """NCCL prints its version banner on stdout when the first communicator comes up; the contract is
  ONE JSON line on stdout, so file descriptor 1 points at stderr until the warm-up is over."""

  def __enter__(self):
    sys.stdout.flush()
    self.saved = os.dup(1)
    os.dup2(2, 1)
    return self

  def __exit__(self, *exc):
    sys.stdout.flush()
    os.dup2(self.saved, 1)
    os.close(self.saved)


def main():
  args = parse_args()
  if args.impl == 'reference':
    return run_reference(args)
  ctx = Ctx()
  line = None
  if args.workload in ('both', 'eval'):
    line = run_wlseg_eval(args, ctx)
  if args.workload in ('both', 'train'):
    from wlseg import train_bench
    ev = line
    line = train_bench.run(args, ctx, cpu_train_sample=cpu_reference_train)
    if ev is not None and line is not None:
      line['eval'] = ev
  if ctx.rank == 0:
    print(json.dumps(line), flush=True)
  if ctx.world > 1:
    # captured NCCL collectives keep the communicator busy: the graphs were dropped by the training half; drain
    # and leave without running the process-group destructor (it can wait forever on a communicator a graph held)
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == '__main__':
  main()
