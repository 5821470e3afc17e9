"""Cityscapes / Mapillary Vistas training splits read from disk for train.py, decoded once into device memory.

train.py does not preserve the aspect ratio of per-pixel examples (code/train.py:42-68) and the augmentation library is
dead code upstream, so a per-pixel training example is the evaluation contract's arithmetic: legacy resizes of the image
and label-id map to the feature-extractor size, [-1, 1) scaling and the _replacevoids(lids2cids) lookup.  Decoding a
1024 x 2048 PNG pair costs far more host time than the device spends on it in a training step, so the rank's whole shard
is decoded once (PIL in DataLoader worker processes) into one uint8 arena in device memory, and every step is one gather
launch (ops.train_inputs) over a device-resident permutation.

Files are found and checked by wlseg.dataset_input (the layouts its docstring lists).  Rank r of R owns the files i with
i % R == r.  Each epoch is a fresh permutation of the rank's shard, a pure function of (seed, rank, world, epoch); every
rank takes the same number of batches per epoch and drops the rest, so a run resumed at global step k feeds exactly the
batches an uninterrupted run feeds from step k on.  The bounding-box and image-level parts of the batch come from Open
Images splits (wlseg.weak_input) when train.py names them, and are empty otherwise.
"""

import time

import numpy as np
import torch

from wlseg import dataset_input
from wlseg.dataset_input import DatasetError

# Device memory left free next to the arena for the training step itself (activations, gradients, the CUDA graph's
# pool).  The step's own footprint at train.py's two per-pixel sizes, measured by tools/train_dataset_bench.py on one
# B200 at a 1000 W power limit (DESIGN.md 8.2) as the drop of free device memory across the first 3 steps of
# Estimator.train after the network exists: 10.37 GB at Cityscapes 4 x 512 x 1024, 10.94 GB at Vistas 4 x 621 x 855.
# The reserve is the larger of the two plus a quarter, rounded up to whole GiB.
STEP_RESERVE_BYTES = 13 << 30
# The same for the mixed 4 + 8 + 4 step (per-pixel + bounding-box + image-level examples), which holds four times the
# images of a per-pixel-only step and its 15-way dense weak labels.  NOT MEASURED yet: an estimate, the Vistas
# per-pixel footprint above scaled to 16 images (4 x 10.94 GB = 43.76 GB) plus a quarter (54.7 GB), rounded up to 51
# GiB.  tools/weak_dataset_bench.py measures it (mixed_step_footprint_bytes, DESIGN.md 8.3).
MIXED_STEP_RESERVE_BYTES = 51 << 30


def split_pairs(path, dataset_name):
  """[(image path, label path)] of the training split at `path`, which must be in the layout of `dataset_name`."""
  layout = dataset_input.detect_layout(path)
  if layout != dataset_name:
    found = f'a {layout} split' if layout else 'neither a Cityscapes leftImg8bit/<split> nor a Vistas split (images/ + labels/)'
    raise DatasetError(f'--per_pixel_split_path {path} is {found}, but per_pixel_dataset_name is {dataset_name}')
  return dataset_input.list_pairs(path)


def steps_per_epoch(n_files, world, Nb):
  """Batches every rank takes per epoch: the smallest shard holds n_files // world files."""
  return (n_files // world) // Nb


def epoch_order(seed, rank, world, n_files, Nb, epoch, rng=None):
  """Shard positions rank `rank` feeds in epoch `epoch`, in order: a permutation of its shard cut to whole batches.
  `rng` replaces the per-pixel generator of (seed, rank, world, epoch) (the weak parts draw from their own)."""
  n_shard = len(range(rank, n_files, world))
  if rng is None:
    rng = np.random.default_rng([seed % (1 << 64), rank, world, epoch])
  return rng.permutation(n_shard)[:steps_per_epoch(n_files, world, Nb) * Nb].astype(np.int32)


def batch_at(seed, rank, world, n_files, Nb, global_step):
  """Shard positions of the batch rank `rank` feeds at `global_step` (0-based)."""
  epoch, k = divmod(global_step, steps_per_epoch(n_files, world, Nb))
  return epoch_order(seed, rank, world, n_files, Nb, epoch)[k * Nb:(k + 1) * Nb]


def arena_layout(sizes, bytes_per_pixel=4):
  """-> (int64 byte offsets of the examples, total bytes): each holds H * W * 3 image bytes, then (4 bytes per pixel,
  per-pixel examples) H * W label ids."""
  nbytes = np.asarray([h * w * bytes_per_pixel for h, w in sizes], dtype=np.int64)
  offsets = np.zeros(len(sizes), dtype=np.int64)
  np.cumsum(nbytes[:-1], out=offsets[1:])
  return offsets, int(nbytes.sum())


def device_budget(device, reserve=STEP_RESERVE_BYTES):
  """Arena bytes the device can hold next to a training step that needs `reserve` bytes (None on the CPU: no limit)."""
  device = torch.device(device)
  if device.type != 'cuda':
    return None
  free, _ = torch.cuda.mem_get_info(device)
  return free - reserve


def check_budget(what, need, budget):
  """Refuses `need` bytes of decoded examples over `budget` (None: no limit), naming `what`."""
  if budget is not None and need > budget:
    raise DatasetError(f'{what} needs {need} bytes of device memory but {max(budget, 0)} are available next to a '
                       'training step; more ranks (--distribute) shrink each shard')


class _Examples(torch.utils.data.Dataset):
  """Item i = (i, uint8 [H * W * 4]): file pair i decoded, its RGB image (HWC) followed by its label ids."""

  def __init__(self, pairs, sizes, n_lids):
    self.pairs, self.sizes, self.n_lids = pairs, sizes, n_lids

  def __len__(self):
    return len(self.pairs)

  def __getitem__(self, i):
    img_path, lab_path = self.pairs[i]
    img, lab = dataset_input._decode_image(img_path), dataset_input._decode_label(lab_path)
    h, w = self.sizes[i]
    if img.shape[:2] != (h, w) or lab.shape != (h, w):
      raise DatasetError(f'{img_path}: decoded size {img.shape[:2]} / label {lab.shape} differ from the header size '
                         f'{(h, w)}')
    top = int(lab.max())
    if top >= self.n_lids:
      raise DatasetError(f'{lab_path}: label id {top} is outside the {self.n_lids} label ids (lids2cids) of the '
                         'training problem definition')
    out = torch.empty(h * w * 4, dtype=torch.uint8)
    out[:h * w * 3].numpy()[:] = img.reshape(-1)     # PIL's arrays are read-only: copy
    out[h * w * 3:].numpy()[:] = lab.reshape(-1)
    return i, out


class Shard:
  """One rank's examples in one uint8 arena on `device`: .arena, .offsets (int64 [E]), .sizes (int32 [E, 2])."""

  def __init__(self, pairs, sizes, n_lids, device, budget=None, workers=None, examples=None, bytes_per_pixel=4):
    """Checks the arena against `budget` bytes (None: no limit) before anything is decoded, then fills it.  `examples`
    (default: the per-pixel image / label pairs) is a dataset of (i, uint8 [H * W * bytes_per_pixel]) items."""
    device = torch.device(device)
    offsets, total = arena_layout(sizes, bytes_per_pixel)
    check_budget(f'the decoded shard of {len(pairs)} files', total, budget)
    t0 = time.perf_counter()
    self.arena = torch.empty(total, dtype=torch.uint8, device=device)
    workers = min(workers or dataset_input._workers_per_rank(), len(pairs))
    if examples is None:
      examples = _Examples(pairs, sizes, n_lids)
    loader = torch.utils.data.DataLoader(examples, batch_size=None, shuffle=False,
                                         num_workers=workers, pin_memory=device.type == 'cuda')
    for i, chunk in loader:
      off = int(offsets[i])
      self.arena[off:off + chunk.numel()].copy_(chunk, non_blocking=device.type == 'cuda')
    if device.type == 'cuda':
      torch.cuda.synchronize(device)
    self.seconds = time.perf_counter() - t0
    self.offsets = torch.from_numpy(offsets).to(device)
    self.sizes = torch.tensor(sizes, dtype=torch.int32).reshape(len(sizes), 2).to(device)
    self.files, self.bytes = len(pairs), total


def train_input_fn(config, params):
  """Drop-in `input_fn(config, params)` for SemanticSegmentation({'train': ...}) over the training split at
  params.per_pixel_split_path.  Discovery, the header checks, the device-memory check and the fill run here, before any
  step; the returned iterator yields this rank's batches ({'proimages'}, {'prolabels_per_pixel'}) from step
  params.initial_global_step on, as device tensors from a ring of two: a batch is overwritten when the iterator is
  advanced twice more, by a launch on the stream of the step that reads it."""
  del config
  from wlseg import ops
  from wlseg.estimator import _replacevoids, get_temp_Nb
  rank, world = getattr(params, 'rank', 0), getattr(params, 'world_size', 1)
  device = torch.device(getattr(params, 'device', 'cuda'))
  Nb = get_temp_Nb(params, params.Nb_per_pixel)
  pairs = split_pairs(params.per_pixel_split_path, params.per_pixel_dataset_name)
  if len(pairs) // world < Nb:
    raise DatasetError(f'{params.per_pixel_split_path} holds {len(pairs)} image / label pairs: the smallest shard of '
                       f'{world} rank(s) has {len(pairs) // world}, fewer than one batch of {Nb}')
  if len(pairs) != params.Ntrain and rank == 0:
    print(f'The split holds {len(pairs)} image / label pairs, the learning-rate schedule assumes Ntrain = {params.Ntrain}: '
          'training on the files found.', flush=True)
  mine = pairs[rank::world]
  sizes, _, _ = dataset_input.check_pairs(mine)
  hw = (params.height_feature_extractor, params.width_feature_extractor)
  from wlseg import weak_input
  weak = weak_input.parts(params, hw, rank, world)   # CSVs and headers only: nothing is decoded yet
  for part in weak:
    print(f'{"" if world == 1 else f"rank {rank}: "}{part.summary()}', flush=True)
  budget = None
  if weak:
    check_budget('the decoded per-pixel, bounding-box and image-level shards', arena_layout(sizes)[1] +
                 sum(part.bytes for part in weak), device_budget(device, MIXED_STEP_RESERVE_BYTES))
  else:
    budget = device_budget(device)
  table = _replacevoids(params.training_problem_def['lids2cids'])
  shard = Shard(mine, sizes, len(table), device, budget=budget)
  print(f'{"" if world == 1 else f"rank {rank}: "}decoded {shard.files} files into {shard.bytes} bytes of '
        f'{device.type} memory in {shard.seconds:.1f} s', flush=True)
  for part in weak:
    part.fill(device)
  lut = torch.tensor(table, dtype=torch.int32, device=device)
  n, spe, step = len(pairs), steps_per_epoch(len(pairs), world, Nb), int(getattr(params, 'initial_global_step', 0))
  rows = Nb + sum(part.Nb for part in weak)
  # two output sets: the estimator's prefetcher enqueues batch i + 1 before step i copies batch i into its inputs.
  # proimages holds the per-pixel rows, then the bounding-box rows, then the image-level rows.
  ring = [(torch.empty((rows,) + hw + (3,), dtype=torch.float32, device=device),
           torch.empty((Nb,) + hw, dtype=torch.int32, device=device),
           [torch.empty((part.Nb,) + hw + (15,), dtype=torch.float32, device=device) for part in weak])
          for _ in range(2)]
  invalid = torch.zeros(1, dtype=torch.int64, device=device)

  def batches(step):
    order = None
    while True:
      epoch, k = divmod(step, spe)
      if order is None or k == 0:
        if int(invalid.item()):
          raise ops.WlsegError(f'{int(invalid.item())} label ids or indices outside the training arena\'s tables')
        order = torch.from_numpy(epoch_order(params.seed, rank, world, n, Nb, epoch)).to(device)
      pro, lab, weak_labels = ring[step % 2]
      ops.train_inputs(shard.arena, shard.offsets, shard.sizes, order[k * Nb:(k + 1) * Nb], lut, max(table), hw, pro[:Nb],
                       lab, invalid)
      labels = {'prolabels_per_pixel': lab}
      row = Nb
      for part, out in zip(weak, weak_labels):
        part.gather(step, pro[row:row + part.Nb], out)
        labels[part.label_key] = out
        row += part.Nb
      yield {'proimages': pro}, labels
      step += 1
  return batches(step)
