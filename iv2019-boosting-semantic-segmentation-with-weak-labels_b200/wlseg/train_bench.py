"""`bench.py --workload train`: training images/s at 768x768 crops (BASELINE.json configs[2] / [3]).

One step = forward with batch statistics + fused hierarchical loss fwd/bwd + backward through the
whole network + gradient all-reduce (N > 1) + fused SGD-momentum update, on synthetic
Cityscapes-shaped batches of 4 images per GPU (strong labels; `--mixed` adds 8 bbox + 4 image-level
images per GPU, the reference's 4:8:4 ratio, train.py:52-55).
"""

import json
import time

import torch


def run(args, ctx, cpu_train_sample=None):
  """-> the JSON line (dict) of the training half; `ctx` is bench.Ctx (device, ranks, NCCL already up)."""
  import torch.distributed as dist
  import bench  # noqa: E402 (bench.py is the caller)
  from bench import ClockSampler, StdoutToStderr, load_peaks
  from wlseg import arch, hierarchy, network, ops, problem_defs, synthetic, trainer as wtrainer

  world, rank, local_rank, dev = ctx.world, ctx.rank, ctx.local_rank, ctx.dev
  quiet = StdoutToStderr()
  quiet.__enter__()  # nothing but the one JSON line may land on stdout
  H, W, NB = args.height or 768, args.width or 768, args.batch or 4
  if args.workload == 'both':   # the nested evaluation half owns --height / --width / --batch overrides
    H, W, NB = 768, 768, 4
  mixed = getattr(args, 'mixed', False)
  npb, npi = (2 * NB, NB) if mixed else (0, 0)
  boxes = bool(mixed and getattr(args, 'boxes', False))
  hier = hierarchy.Hierarchy(args.dataset, problem_defs.GENERATORS[args.dataset]()['cids2labels'])
  params = network.Params(hier, dev)
  params.init_random(0)

  class S:
    pass
  st = S()
  st.momentum, st.use_nesterov, st.optimizer, st.regularization_weight = 0.9, False, 'SGDM', 0.00017
  st.batch_norm_decay, st.distribute, st.ema_decay = 0.9, world > 1, 0.0
  tr = wtrainer.Trainer(params, st, dtype=torch.bfloat16, rank=rank, world_size=world)
  src = synthetic.SyntheticInputs(hier.num_classes, dev, rank=rank)
  batches = [src.train_batch(NB, npb, npi, H, W, compact=boxes) for _ in range(2)]

  def step(i):
    f, l = batches[i % 2]
    return tr.step(f, {k: v for k, v in l.items() if v is not None}, 0.01)

  for i in range(max(args.warmup, 3)):  # two eager steps + the graph capture happen here
    step(i)
  torch.cuda.synchronize()
  quiet.__exit__()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  # timed region: the step as the product runs it (one CUDA-graph replay per step after the warm-up)
  sampler = ClockSampler(local_rank) if rank == 0 else None
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(args.steps):
    out = step(i)
  e1.record()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  clocks = sampler.stop() if sampler else None
  ms = e0.elapsed_time(e1)
  if args.dump_outputs and rank == 0:
    # what a caller of the training step receives: the loss vector of the last timed step.  The updated parameters are
    # left out: from random init this network amplifies rounding-order differences ~10^2 per step (DESIGN.md), and
    # after the default 3 + 20 steps two runs of one build hold momentum slots with cosine ~0 (measured on a B200 at
    # 1000 W), while their losses agree to 1e-2 relative
    bench.dump_outputs(args.dump_outputs, {'train_losses': out})
  # roofline pass, live, right after the timed region: the same steps launched eagerly with a CUDA
  # event pair around every convolution launch (events cannot sit inside a replayed graph)
  prof_steps = min(3, args.steps)
  tr.net.profile = []
  l0 = ops.launches
  pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  pe0.record()
  for i in range(prof_steps):
    step(i)
  pe1.record()
  torch.cuda.synchronize()
  launches = (ops.launches - l0) // prof_steps * args.steps
  prof, tr.net.profile = tr.net.profile, None
  prof_ms = pe0.elapsed_time(pe1)
  t = torch.tensor([ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_max = float(t.item())
  nimg = NB + npb + npi
  value = world * args.steps * nimg / (ms_max / 1e3)
  sustained = bench.sustained_loop(step, args.sustained_seconds, ms_max / args.steps, nimg, 'images/s', dev, world,
                                   rank, local_rank)

  peaks = load_peaks()
  classes = {}
  for rec in prof:
    rec['ms'] = rec['e0'].elapsed_time(rec['e1'])
    c = classes.setdefault(rec['cls'], {'flops': 0.0, 'ms': 0.0, 'launches': 0, 'bytes': 0.0})
    c['flops'] += rec['flops']
    c['ms'] += rec['ms']
    c['bytes'] += rec['bytes']
    c['launches'] += 1
  roofline = None
  tc = {k: v for k, v in classes.items() if k.startswith(('igemm', 'wgrad_tc'))}
  if tc:
    name, dom = max(tc.items(), key=lambda kv: kv[1]['ms'])
    from bench import load_traffic, tensor_roofline
    kname = 'conv_igemm_kernel<256' if name == 'igemm_bn256' else 'conv_wgrad_kernel<256'
    traffic, tsrc = load_traffic('train', kname)
    # kernel time per step (event pairs of the eager pass) over the step time of the timed region (graph replay):
    # the eager pass's own wall time is inflated by Python launch gaps and is not the step
    roofline = tensor_roofline(kname + ('' if name.endswith('256') else f' [{name}]') + ', bf16>', dom, peaks, ms_max / 1e3,
                               traffic, tsrc, (dom['ms'] / prof_steps) / (ms_max / args.steps),
                               f'{prof_steps} eagerly launched steps after the timed region')
    # every tensor-core launch of the step (fprop + dgrad + wgrad) against the same peak, and the whole step
    all_flops = sum(v['flops'] for v in tc.values())
    all_ms = sum(v['ms'] for v in tc.values())
    roofline['all_conv_tflops'] = all_flops / (all_ms / 1e3) / 1e12
    roofline['all_conv_share_of_step'] = (all_ms / prof_steps) / (ms_max / args.steps)
    roofline['whole_step_tflops'] = (all_flops / prof_steps) / (ms_max / args.steps / 1e3) / 1e12
    roofline['whole_step_frac_burst'] = roofline['whole_step_tflops'] / peaks['bf16_tflops']
  if args.detail and rank == 0:
    table = {k: {'launches': v['launches'], 'ms_per_step': v['ms'] / prof_steps,
                 'tflops': v['flops'] / (v['ms'] / 1e3) / 1e12 if v['ms'] else None,
                 'gbs_algorithmic': v['bytes'] / (v['ms'] / 1e3) / 1e9 if v['ms'] else None}
             for k, v in sorted(classes.items())}
    with open(args.detail, 'w') as fp:
      json.dump({'ms_per_step': ms / args.steps, 'ms_per_step_eager_profiled': prof_ms / prof_steps, 'classes': table}, fp, indent=1)

  # ---- end to end: host batches (pinned fp32 images + int32 labels) -> step -> loss back to the host
  e2e = None
  if not args.no_e2e:
    from wlseg import estimator as west
    g = torch.Generator().manual_seed(1234 + rank)
    host = []
    for _ in range(2):
      img = (torch.rand((nimg, H, W, 3), generator=g) * 2 - 1).pin_memory()
      lab = {'prolabels_per_pixel': torch.randint(0, hier.num_classes, (NB, H, W), generator=g, dtype=torch.int32).pin_memory()}
      if mixed:
        f, l = batches[0]
        for k in ('prolabels_per_bbox', 'prolabels_per_image', 'bbox_coords', 'bbox_cids', 'image_vectors'):
          if l.get(k) is not None:
            lab[k] = l[k].cpu().pin_memory()
      host.append(({'proimages': img}, lab))
    est = west.Estimator.__new__(west.Estimator)
    st.rank, st.world_size = rank, world
    st.learning_rate_schedule, st.learning_rate_boundaries, st.learning_rate_values = 'piecewise_constant', [10 ** 9], [0.01, 0.01]
    est.settings, est.hier, est.device, est.dtype, est.params = st, hier, dev, torch.bfloat16, params
    est.global_step, est.trainer = tr.global_step, tr

    stamps = []

    def gen(n):
      for i in range(n):
        stamps.append(time.perf_counter())
        yield host[i % 2]
    est.train(gen(args.steps), args.steps)  # same step count: same pinned result buffer size
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    # wall clock around the public call, max over ranks, median of three repeats of the K-step region
    dts = []
    for _ in range(3):
      if world > 1:
        dist.barrier()
      t0 = time.perf_counter()
      est.train(gen(args.steps), args.steps)
      torch.cuda.synchronize()
      dt = time.perf_counter() - t0
      tt = torch.tensor([dt], dtype=torch.float64, device=dev)
      if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
      dts.append(float(tt.item()))
    raw_dts = list(dts)
    dts.sort()
    dt = dts[1]
    e2e = {'value': world * args.steps * nimg / dt, 'unit': 'images/s', 'h2d_bytes_per_step': est.last_h2d_bytes // args.steps,
           'd2h_bytes_per_step': est.last_d2h_bytes // args.steps, 'ms_per_step': 1e3 * dt / args.steps,
           'repeats': 3, 'stat': 'median of 3 repeats of the K-step region',
           'repeat_ms_per_step': [round(1e3 * d / args.steps, 3) for d in raw_dts]}
    from bench import host_link_probe
    e2e['host_link'] = host_link_probe(dev, world)

  cpu = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline and cpu_train_sample is not None:
    # one step over the arm's own batch (about 10 s of host work at 4 x 768 x 768)
    cpu = cpu_train_sample(args.dataset, H, W, images_per_step=NB if not mixed else 1, mixed=mixed)

  fwd = arch.conv_flops(params.specs, H, W) / 1e9
  line = {'metric': 'train_images_per_s', 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
          'warmup': args.warmup, 'ms_per_step': ms_max / args.steps, 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
          'config': {'workload': bench.train_workload_name(args.dataset, H, W, NB, npb, npi, mixed),
                     'l2': 'two rotating input batches; activations + gradients (GBs) exceed the 126 MB L2',
                     'launch': 'whole step replayed as one CUDA graph',
                     'parallelism': (f'data parallel x{world}, NCCL gradient all-reduce ({tr.grad_payload}) bucketed behind '
                                     f'backward, inside the timed region') if world > 1 else 'single GPU',
                     'weak_labels': ('generated in the loss kernel from box / class lists' if boxes else 'dense 60 B/pixel maps') if mixed else None,
                     'fwd_gflop_per_image': fwd, 'last_loss': [float(x) for x in out.tolist()]},
          'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches * world, 'roofline': roofline, 'sustained': sustained,
          'cpu_baseline': cpu}
  # captured NCCL collectives keep the communicator busy: drop the graphs before the caller drains and exits
  tr._graphs.clear()
  torch.cuda.synchronize()
  return line
