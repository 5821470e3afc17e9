"""Cityscapes / Mapillary Vistas validation splits read from disk for evaluate.py.

The host only decodes: PIL in DataLoader worker processes turns each batch into packed raw bytes, and the resize, the
dtype conversion and the label-id lookup of the evaluation contract (SURVEY.md 3.5) run on the device in one launch
(ops.eval_inputs, called by Estimator.evaluate).

Layouts, recognised from the directory `tfrecords_path` names:
  Cityscapes  .../leftImg8bit/<split>/<city>/<stem>_leftImg8bit.png, labels
              .../gtFine/<split>/<city>/<stem>_gtFine_labelIds.png
  Vistas      <split>/images/<stem>.jpg, labels <split>/labels/<stem>.png (palette-indexed: the index is the label id)

Files are taken in the order of their relative paths; the first num_eval_steps * Nb are evaluated and batch b goes to
rank b % world_size (as wlseg.synthetic.eval_input_fn shards).  Every batch carries rows of one width - the largest
image and label map of the evaluated files - so the device staging ring keeps its addresses.
"""

import glob
import os

import numpy as np
import torch

# keys of a batch in packed raw form (Estimator.evaluate turns them into proimages / prolabels on the device)
PACKED_IMAGES, PACKED_SIZES, PACKED_LIDS = 'packed_images', 'packed_sizes', 'packed_lids'

_IMAGE_MODES = ('RGB', 'L', 'P', 'RGBA')   # L, P, RGBA are converted to RGB, as wlseg/image_input.py does
_LABEL_MODES = ('L', 'P')                  # read as indices, never converted


class DatasetError(ValueError):
  pass


def detect_layout(path):
  """'cityscapes', 'vistas' or None for a directory in neither layout (or no directory)."""
  if not path or not os.path.isdir(path):
    return None
  path = os.path.abspath(path)
  if os.path.basename(os.path.dirname(path)) == 'leftImg8bit' and glob.glob(os.path.join(path, '*', '*_leftImg8bit.png')):
    return 'cityscapes'
  if os.path.isdir(os.path.join(path, 'images')) and os.path.isdir(os.path.join(path, 'labels')):
    return 'vistas'
  return None


def list_pairs(path):
  """[(image path, label path)] of a split, sorted by the image's path relative to the split directory."""
  layout = detect_layout(path)
  path = os.path.abspath(path)
  if layout == 'cityscapes':
    split = os.path.basename(path)
    gt = os.path.join(os.path.dirname(os.path.dirname(path)), 'gtFine', split)
    rels = sorted(os.path.relpath(f, path) for f in glob.glob(os.path.join(path, '*', '*_leftImg8bit.png')))
    return [(os.path.join(path, r), os.path.join(gt, r[:-len('_leftImg8bit.png')] + '_gtFine_labelIds.png')) for r in rels]
  if layout == 'vistas':
    rels = sorted(os.path.relpath(f, path) for f in glob.glob(os.path.join(path, 'images', '*.jpg')))
    return [(os.path.join(path, r), os.path.join(path, 'labels', os.path.splitext(os.path.basename(r))[0] + '.png'))
            for r in rels]
  raise DatasetError(f'{path} is neither a Cityscapes leftImg8bit/<split> directory nor a Vistas split directory '
                     '(images/ + labels/)')


def check_pairs(pairs):
  """Headers only (nothing is decoded): every label exists, modes are supported, image and label agree in size.
  -> (sizes [(H, W)], cap_img = max H*W*3, cap_lab = max H*W)."""
  from PIL import Image
  sizes = []
  for img_path, lab_path in pairs:
    if not os.path.isfile(lab_path):
      raise DatasetError(f'{img_path} has no label file {lab_path}')
    with Image.open(img_path) as im:
      if im.mode not in _IMAGE_MODES:
        raise DatasetError(f'{img_path}: image mode {im.mode} is not supported (one of {", ".join(_IMAGE_MODES)})')
      w, h = im.size
    with Image.open(lab_path) as lb:
      if lb.mode not in _LABEL_MODES:
        raise DatasetError(f'{lab_path}: label mode {lb.mode} is not supported: label ids are 8-bit single-channel '
                           '(mode L, or P whose palette index is the id)')
      if lb.size != (w, h):
        raise DatasetError(f'{lab_path}: label size {lb.size[0]}x{lb.size[1]} differs from the image size {w}x{h} of '
                           f'{img_path}')
    sizes.append((h, w))
  return sizes, max(h * w * 3 for h, w in sizes), max(h * w for h, w in sizes)


def _decode_image(path):
  from PIL import Image
  with Image.open(path) as im:
    if im.mode != 'RGB':
      im = im.convert(mode='RGB')
    return np.asarray(im, dtype=np.uint8)


def _decode_label(path):
  from PIL import Image
  with Image.open(path) as lb:
    return np.asarray(lb, dtype=np.uint8)   # mode P: the palette indices


class PackedBatches(torch.utils.data.Dataset):
  """Item i = batch `batches[i]` decoded into rows of fixed width: (features, labels) with
  features = {PACKED_IMAGES: uint8 [Nb, cap_img], PACKED_SIZES: int32 [Nb, 2]}, labels = {PACKED_LIDS: uint8 [Nb, cap_lab]}."""

  def __init__(self, pairs, sizes, batches, Nb, cap_img, cap_lab):
    self.pairs, self.sizes, self.batches, self.Nb = pairs, sizes, batches, Nb
    self.cap_img, self.cap_lab = cap_img, cap_lab

  def __len__(self):
    return len(self.batches)

  def __getitem__(self, i):
    first = self.batches[i] * self.Nb
    images = torch.zeros((self.Nb, self.cap_img), dtype=torch.uint8)
    lids = torch.zeros((self.Nb, self.cap_lab), dtype=torch.uint8)
    sizes = torch.zeros((self.Nb, 2), dtype=torch.int32)
    for j in range(self.Nb):
      img_path, lab_path = self.pairs[first + j]
      img, lab = _decode_image(img_path), _decode_label(lab_path)
      if img.shape[:2] != tuple(self.sizes[first + j]) or lab.shape != img.shape[:2]:
        raise DatasetError(f'{img_path}: decoded size {img.shape[:2]} / label {lab.shape} differ from the header size '
                           f'{tuple(self.sizes[first + j])}')
      images[j, :img.size].numpy()[:] = img.reshape(-1)     # PIL's arrays are read-only: copy into the row
      lids[j, :lab.size].numpy()[:] = lab.reshape(-1)
      sizes[j, 0], sizes[j, 1] = img.shape[0], img.shape[1]
    return {PACKED_IMAGES: images, PACKED_SIZES: sizes}, {PACKED_LIDS: lids}


def _workers_per_rank():
  """Host cores shared evenly by the processes of this node (torchrun's LOCAL_WORLD_SIZE)."""
  try:
    cores = len(os.sched_getaffinity(0))
  except AttributeError:
    cores = os.cpu_count() or 1
  return max(1, cores // max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1'))))


def eval_input_fn(config, params):
  """Drop-in `input_fn(config, params)` for SemanticSegmentation({'eval': ...}) over the split at params.tfrecords_path.
  Discovery and the header checks run here, before any step; the returned iterator yields this rank's batches."""
  del config
  Nb, steps = params.Nb, params.num_eval_steps
  rank, world = getattr(params, 'rank', 0), getattr(params, 'world_size', 1)
  pairs = list_pairs(params.tfrecords_path)
  need = steps * Nb
  if len(pairs) < need:
    raise DatasetError(f'{params.tfrecords_path} holds {len(pairs)} image / label pairs but {steps} evaluation steps of '
                       f'{Nb} need {need}')
  pairs = pairs[:need]
  sizes, cap_img, cap_lab = check_pairs(pairs)
  mine = [b for b in range(steps) if b % world == rank]
  ds = PackedBatches(pairs, sizes, mine, Nb, cap_img, cap_lab)
  workers = min(_workers_per_rank(), len(mine))
  return iter(torch.utils.data.DataLoader(ds, batch_size=None, shuffle=False, num_workers=workers,
                                          pin_memory=torch.cuda.is_available()))
