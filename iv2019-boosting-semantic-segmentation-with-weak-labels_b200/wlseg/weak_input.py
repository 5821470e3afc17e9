"""Open Images weak labels read from disk for train.py: the bounding-box and image-level parts of the training batch,
decoded once into device memory.

Layout (the CSV release of Open Images), in the directory --per_bbox_split_path / --per_image_split_path names (both
may name the same one):
  class-descriptions-boxable.csv            MID,DisplayName rows, with or without a header row
  *annotations-bbox.csv                     exactly one; bounding-box part.  Columns found by header name:
                                            ImageID, LabelName (the MID), XMin, XMax, YMin, YMax (normalised)
  *annotations-human-imagelabels*.csv       exactly one; image-level part.  ImageID, LabelName, Confidence: a row counts
                                            when Confidence == 1
  images/<ImageID>.jpg

MIDs map onto the 14 weak classes of wlseg.hierarchy.WEAK_CLASSES by display name (case-insensitive,
hierarchy.WEAK_DISPLAY_NAMES); boxes and tags of any other MID are skipped, as the reference skips MIDs that are not in
its mid2cid.  An example is an image under images/ with at least one box (bbox part) or positive tag (image part) of
those classes; annotation rows of absent images and images without a weak class are counted, not refused, since a user
holds a subset of CSVs that cover the whole release.

Restated here, because the reference's pickles and the bodies of its input_subset_* pipelines are not in this checkout:
  * the host form of the labels: per bbox example its boxes (float32 xmin, xmax, ymin, ymax + int32 weak class id) in
    one CSR table, which the device rasterises with _generate_rla (csrc/weak_boxes.cuh); per image-level example one
    float32 15-vector uniform over its distinct classes, built as input_subset_image_labels._generate_rla;
  * every box is used (no IsGroupOf / IsDepiction filtering), and the EXIF orientation is ignored, as
    tf.image.decode_jpeg ignores it.
train.py preserves the aspect ratio of weak examples: each is resized to preprocess.resized_size(H, W, target, True) and
cut at a random offset, both in one gather launch per part per step (ops.weak_train_inputs).  Rank r of R owns the
examples i with i % R == r of each part; a part's order and crop offsets in an epoch are a pure function of (seed, part,
rank, world, epoch), so a run resumed at global step k feeds exactly the batches, crops included, an uninterrupted run
feeds from step k on.
"""

import csv
import glob
import os

import numpy as np
import torch

from wlseg import dataset_input, hierarchy, preprocess, train_input
from wlseg.dataset_input import DatasetError

DESCRIPTIONS = 'class-descriptions-boxable.csv'
MAX_BOXES_PER_IMAGE = 1024   # boxes of one image the gather kernel holds in shared memory (kMaxBoxesSmem)
NUM_WEAK = len(hierarchy.WEAK_CLASSES)
_PARTS = {   # part -> (generator key, train.py flag, CSV pattern, batch-size setting, label key)
    'bbox': (1, '--per_bbox_split_path', '*annotations-bbox.csv', 'Nb_per_bbox', 'prolabels_per_bbox'),
    'image': (2, '--per_image_split_path', '*annotations-human-imagelabels*.csv', 'Nb_per_image', 'prolabels_per_image'),
}


def weak_class_ids(path):
  """{MID: weak class id} of the descriptions file in directory `path`; refuses a file that lacks one of the 14."""
  fname = os.path.join(path, DESCRIPTIONS)
  if not os.path.isfile(fname):
    raise DatasetError(f'{path} has no {DESCRIPTIONS}')
  wanted = {hierarchy.weak_display_name(c).lower(): c for c in range(NUM_WEAK - 1)}
  mids = {}
  with open(fname, newline='', encoding='utf-8') as f:
    for row in csv.reader(f):
      if len(row) >= 2 and row[1].strip().lower() in wanted:
        mids[row[0].strip()] = wanted[row[1].strip().lower()]
  missing = sorted(set(wanted.values()) - set(mids.values()))
  if missing:
    raise DatasetError(f'{fname} lacks the display name(s) {", ".join(hierarchy.weak_display_name(c) for c in missing)} '
                       'of the weak classes')
  return mids


def _one_csv(path, pattern):
  found = sorted(glob.glob(os.path.join(path, pattern)))
  if len(found) != 1:
    raise DatasetError(f'{path} must hold exactly one {pattern} file, found {len(found)}'
                       + (f': {", ".join(os.path.basename(f) for f in found)}' if found else ''))
  return found[0]


def _rows(fname, columns):
  """Yields (line number, [the named columns]) of a CSV whose header row names them."""
  with open(fname, newline='', encoding='utf-8') as f:
    reader = csv.reader(f)
    header = [h.strip() for h in next(reader, [])]
    missing = [c for c in columns if c not in header]
    if missing:
      raise DatasetError(f'{fname}: the header row lacks the column(s) {", ".join(missing)}')
    idx = [header.index(c) for c in columns]
    for line, row in enumerate(reader, start=2):
      if row:
        yield line, [row[i] for i in idx]


def image_vector(cids):
  """input_subset_image_labels._generate_rla: float32 15-vector uniform over the distinct classes `cids`."""
  v = np.zeros(NUM_WEAK, dtype=np.float32)
  v[sorted(set(cids))] = 1.0
  return v / v.sum()


def read_part(part, path):
  """-> (csv path, {ImageID: labels}, absent rows, no-weak-class images) for the examples of one part: labels are
  [(cid, xmin, xmax, ymin, ymax)] (bbox) or [cid] (image); ImageIDs in sorted order."""
  mids = weak_class_ids(path)
  fname = _one_csv(path, _PARTS[part][2])
  present = {os.path.splitext(f)[0] for f in os.listdir(os.path.join(path, 'images')) if f.endswith('.jpg')} \
      if os.path.isdir(os.path.join(path, 'images')) else set()
  labels, absent = {}, 0
  if part == 'bbox':
    for line, (image, mid, *xy) in _rows(fname, ('ImageID', 'LabelName', 'XMin', 'XMax', 'YMin', 'YMax')):
      if image not in present:
        absent += 1
        continue
      if mid not in mids:
        continue
      try:
        xmin, xmax, ymin, ymax = (np.float32(v) for v in xy)
      except ValueError:
        raise DatasetError(f'{fname}:{line}: coordinates {xy} are not numbers') from None
      if not (0 <= xmin <= xmax <= 1 and 0 <= ymin <= ymax <= 1):
        raise DatasetError(f'{fname}:{line}: box (XMin, XMax, YMin, YMax) = ({", ".join(xy)}) of {image} is outside '
                           '[0, 1] or has min > max')
      labels.setdefault(image, []).append((mids[mid], xmin, xmax, ymin, ymax))
    for image, boxes in labels.items():
      if len(boxes) > MAX_BOXES_PER_IMAGE:
        raise DatasetError(f'{fname}: image {image} has {len(boxes)} boxes of the weak classes, more than the '
                           f'{MAX_BOXES_PER_IMAGE} the gather kernel holds per image')
  else:
    for line, (image, mid, confidence) in _rows(fname, ('ImageID', 'LabelName', 'Confidence')):
      if image not in present:
        absent += 1
        continue
      try:
        confidence = float(confidence)
      except ValueError:
        raise DatasetError(f'{fname}:{line}: Confidence {confidence!r} of {image} is not a number') from None
      if mid in mids and confidence == 1:
        labels.setdefault(image, []).append(mids[mid])
  return fname, {k: labels[k] for k in sorted(labels)}, absent, len(present - set(labels))


class _Images(torch.utils.data.Dataset):
  """Item i = (i, uint8 [H * W * 3]): image i decoded to RGB (HWC)."""

  def __init__(self, paths, sizes):
    self.paths, self.sizes = paths, sizes

  def __len__(self):
    return len(self.paths)

  def __getitem__(self, i):
    img = dataset_input._decode_image(self.paths[i])
    if img.shape[:2] != tuple(self.sizes[i]):
      raise DatasetError(f'{self.paths[i]}: decoded size {img.shape[:2]} differs from the header size {self.sizes[i]}')
    return i, torch.from_numpy(img.reshape(-1).copy())


class WeakPart:
  """One weak part of this rank's batch: the examples found at `path`, checked from the CSVs and headers.  .fill()
  decodes them into device memory; .gather(step, proimages, labels) writes the part's batch of global step `step`."""

  def __init__(self, part, path, Nb, hw, rank, world, seed):
    self.part, self.path, self.Nb, self.hw, self.rank, self.world, self.seed = part, path, Nb, hw, rank, world, seed
    self.key, flag, _, _, self.label_key = _PARTS[part]
    self.csv, labels, self.absent_rows, self.no_weak_class = read_part(part, path)
    ids = list(labels)
    self.n_examples = len(ids)
    if len(ids) // world < Nb:
      raise DatasetError(f'{flag} {path} holds {len(ids)} {part} examples: the smallest shard of {world} rank(s) has '
                         f'{len(ids) // world}, fewer than one batch of {Nb}')
    self.ids = ids[rank::world]
    self.paths = [os.path.join(path, 'images', i + '.jpg') for i in self.ids]
    self.sizes = _check_images(self.paths)
    self.resized = [preprocess.resized_size(h, w, hw, True) for h, w in self.sizes]
    if part == 'bbox':
      boxes = [labels[i] for i in self.ids]
      self.box_start = np.zeros(len(boxes) + 1, dtype=np.int32)
      np.cumsum([len(b) for b in boxes], out=self.box_start[1:])
      flat = [b for bs in boxes for b in bs]
      self.box_cids = np.asarray([b[0] for b in flat], dtype=np.int32)
      self.box_coords = np.asarray([b[1:] for b in flat], dtype=np.float32).reshape(-1, 4)
      tables = self.box_start.nbytes + self.box_cids.nbytes + self.box_coords.nbytes
    else:
      self.vectors = np.stack([image_vector(labels[i]) for i in self.ids])
      tables = self.vectors.nbytes
    self.n_boxes = int(self.box_start[-1]) if part == 'bbox' else 0
    self.n_tags = 0 if part == 'bbox' else sum(len(set(labels[i])) for i in self.ids)   # distinct, on this rank
    self.bytes = train_input.arena_layout(self.sizes, 3)[1] + tables + 24 * len(self.ids)   # + offsets, sizes, resized
    self.steps_per_epoch = train_input.steps_per_epoch(len(ids), world, Nb)

  def summary(self):
    what = f'{self.n_boxes} boxes' if self.part == 'bbox' else f'{self.n_tags} positive tags'
    return (f'{self.part} part: {self.csv}: {self.n_examples} examples, {len(self.ids)} on this rank ({what}); '
            f'{self.absent_rows} annotation rows of images absent from {os.path.join(self.path, "images")}, '
            f'{self.no_weak_class} images without a weak class')

  def epoch(self, epoch):
    """-> (shard positions int32 [steps_per_epoch * Nb], crop offsets int32 [.., 2]) of epoch `epoch`: a pure function
    of (seed, part, rank, world, epoch); offsets ~ U{0..RH - TH} x U{0..RW - TW} per position."""
    rng = np.random.default_rng([self.seed % (1 << 64), self.key, self.rank, self.world, epoch])
    order = train_input.epoch_order(self.seed, self.rank, self.world, self.n_examples, self.Nb, epoch, rng=rng)
    extra = np.asarray(self.resized, dtype=np.int64).reshape(-1, 2)[order] - np.asarray(self.hw, dtype=np.int64)
    crops = np.stack([rng.integers(0, extra[:, 0] + 1), rng.integers(0, extra[:, 1] + 1)], axis=1)
    return order, crops.astype(np.int32)

  def batch_at(self, global_step):
    """(shard positions, crop offsets) of the batch this part feeds at `global_step` (0-based)."""
    epoch, k = divmod(global_step, self.steps_per_epoch)
    order, crops = self.epoch(epoch)
    return order[k * self.Nb:(k + 1) * self.Nb], crops[k * self.Nb:(k + 1) * self.Nb]

  def fill(self, device, workers=None):
    device = torch.device(device)
    self.shard = train_input.Shard(self.paths, self.sizes, None, device, workers=workers,
                                   examples=_Images(self.paths, self.sizes), bytes_per_pixel=3)
    print(f'{"" if self.world == 1 else f"rank {self.rank}: "}decoded {self.shard.files} {self.part} images into '
          f'{self.shard.bytes} bytes of {device.type} memory in {self.shard.seconds:.1f} s', flush=True)
    self.resized_dev = torch.tensor(self.resized, dtype=torch.int32).reshape(-1, 2).to(device)
    if self.part == 'bbox':
      self.tables = dict(boxes=tuple(torch.from_numpy(a).to(device) for a in
                                     (self.box_start, self.box_coords, self.box_cids)))
    else:
      self.tables = dict(vectors=torch.from_numpy(self.vectors).to(device))
    self.invalid = torch.zeros(1, dtype=torch.int64, device=device)
    self._epoch = None

  def gather(self, step, proimages, labels):
    from wlseg import ops
    epoch, k = divmod(step, self.steps_per_epoch)
    if self._epoch != epoch:
      if int(self.invalid.item()):
        raise ops.WlsegError(f'{int(self.invalid.item())} indices or crop offsets outside the {self.part} arena')
      order, crops = self.epoch(epoch)
      device = self.shard.arena.device
      self._order, self._crops, self._epoch = (torch.from_numpy(order).to(device), torch.from_numpy(crops).to(device),
                                               epoch)
    s = slice(k * self.Nb, (k + 1) * self.Nb)
    ops.weak_train_inputs(self.shard.arena, self.shard.offsets, self.shard.sizes, self.resized_dev, self._order[s],
                          self._crops[s], self.hw, proimages, labels, self.invalid, **self.tables)


def _check_images(paths):
  """Headers only: every image exists and has a supported mode.  -> [(H, W)]."""
  from PIL import Image
  sizes = []
  for p in paths:
    with Image.open(p) as im:
      if im.mode not in dataset_input._IMAGE_MODES:
        raise DatasetError(f'{p}: image mode {im.mode} is not supported (one of {", ".join(dataset_input._IMAGE_MODES)})')
      w, h = im.size
    sizes.append((h, w))
  return sizes


def parts(params, hw, rank, world):
  """The weak parts train.py names (--per_bbox_split_path, --per_image_split_path), checked but not decoded: [] when
  neither is given."""
  from wlseg.estimator import get_temp_Nb
  out = []
  for part, (_, _, _, nb_key, _) in _PARTS.items():
    path = getattr(params, f'per_{part}_split_path', None)
    if path:
      out.append(WeakPart(part, path, get_temp_Nb(params, getattr(params, nb_key)), hw, rank, world, params.seed))
  return out
