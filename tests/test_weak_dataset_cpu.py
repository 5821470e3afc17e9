"""Open Images weak labels read from disk for training (wlseg/weak_input.py, its use by wlseg/train_input.py and
cli.train_main's flags), on CPU.  ops.weak_train_inputs is replaced by its contract restated with the oracle's legacy
resizes and `_generate_rla`; the kernel's own bit equality is tests/test_gpu_weak_dataset.py."""

import contextlib
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

from tests.test_eval_dataset_cpu import _rgb
from tests.test_train_dataset_cpu import cityscapes_train, emulated_train_inputs, train_settings

HERE = os.path.dirname(os.path.abspath(__file__))
# the three MIDs tests/golden/reference_run.npz pins (rla/cids), the others made up
MIDS = {'Car': '/m/0k4j', 'Bus': '/m/01bjv', 'Person': '/m/01g317'}


def mid(name):
  return MIDS.get(name, '/m/x_' + name.lower().replace(' ', '_'))


def write_descriptions(root, header=True, names=None, case=str):
  from wlseg import hierarchy
  names = names if names is not None else [hierarchy.weak_display_name(c) for c in range(14)] + ['Tree', 'Dog']
  os.makedirs(root, exist_ok=True)
  with open(os.path.join(root, 'class-descriptions-boxable.csv'), 'w') as f:
    if header:
      f.write('LabelName,DisplayName\n')
    for n in names:
      f.write(f'{mid(n)},{case(n)}\n')


def write_open_images(root, images, boxes=(), tags=(), bbox_csv='train-annotations-bbox.csv',
                      tags_csv='train-annotations-human-imagelabels-boxable.csv', header=True):
  """images: [(ImageID, PIL image)]; boxes: [(ImageID, display name, xmin, xmax, ymin, ymax)]; tags: [(ImageID, display
  name, confidence)] -> root in the Open Images CSV layout; returns root."""
  write_descriptions(root, header=header)
  os.makedirs(os.path.join(root, 'images'), exist_ok=True)
  for image_id, im in images:
    im.save(os.path.join(root, 'images', f'{image_id}.jpg'), quality=90)
  if bbox_csv:
    with open(os.path.join(root, bbox_csv), 'w') as f:
      f.write('ImageID,Source,LabelName,Confidence,XMin,XMax,YMin,YMax,IsOccluded,IsTruncated,IsGroupOf,IsDepiction,'
              'IsInside\n')
      for image_id, name, *xy in boxes:
        f.write(f'{image_id},xclick,{mid(name)},1,{",".join(str(v) for v in xy)},0,0,0,0,0\n')
  if tags_csv:
    with open(os.path.join(root, tags_csv), 'w') as f:
      f.write('ImageID,Source,LabelName,Confidence\n')
      for image_id, name, conf in tags:
        f.write(f'{image_id},verification,{mid(name)},{conf}\n')
  return root


def random_open_images(root, n, seed=0, sizes=((40, 60), (70, 45), (33, 90), (50, 50)), absent=3, no_weak=2,
                       max_boxes=5):
  """n images with boxes and tags of random weak classes, `absent` annotated ImageIDs without a file and `no_weak`
  images whose only annotations are of other classes."""
  from wlseg import hierarchy
  rng = np.random.default_rng(seed)
  names = [hierarchy.weak_display_name(c) for c in range(14)]
  images, boxes, tags = [], [], []
  for i in range(n + no_weak):
    h, w = sizes[i % len(sizes)]
    images.append((f'img{i:04d}', Image.fromarray(_rgb(rng, h, w))))
  for i in range(n + no_weak + absent):
    image_id = f'img{i:04d}'
    weak = i < n or i >= n + no_weak
    for _ in range(int(rng.integers(1, max_boxes + 1))):
      x = np.sort(rng.random(2)).round(4)
      y = np.sort(rng.random(2)).round(4)
      boxes.append((image_id, names[int(rng.integers(0, 14))] if weak else 'Tree', x[0], x[1], y[0], y[1]))
    for _ in range(int(rng.integers(1, 4))):
      tags.append((image_id, names[int(rng.integers(0, 14))] if weak else 'Dog', 1))
    tags.append((image_id, names[int(rng.integers(0, 14))], 0))          # negative tags never count
  return write_open_images(root, images, boxes, tags)


def weak_settings(split, bbox=None, image=None, **kw):
  return train_settings(split, per_bbox_split_path=bbox, per_image_split_path=image, Nb_per_bbox=2, Nb_per_image=1,
                        **kw)


def oracle_weak_example(img, boxes, vector, hw, offset):
  """One weak example through the oracle: u8 * (float)(1/255), resize_images_and_labels(preserve_aspect_ratio=True) at
  `offset` on the image and on its dense label (_generate_rla at H x W, or the vector tiled), then [-1, 1)."""
  from oracle import preprocess as opre
  from oracle import weak_labels as oweak
  h, w = img.shape[:2]
  if boxes is not None:
    dense = oweak.bbox_labels([(int(c),) + tuple(float(v) for v in xy) for c, xy in boxes], h, w)
  else:
    dense = np.broadcast_to(vector, (h, w, 15)).copy()
  x = torch.as_tensor(img)[None].to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
  pro, lab = opre.resize_images_and_labels(x, torch.from_numpy(dense)[None], hw, preserve_aspect_ratio=True,
                                           offset=offset)
  return (pro[0] - 0.5) / 0.5, lab[0]


def emulated_weak_train_inputs(monkeypatch):
  """ops.weak_train_inputs restated per output example: the oracle's bilinear resize of the image, and the label of the
  source pixel min(floor((Y + oy) * (H / RH)), H - 1) (x alike) rasterised by the oracle's `_generate_rla`."""
  from oracle import preprocess as opre
  from oracle import weak_labels as oweak
  from wlseg import ops

  def weak_train_inputs(arena, offsets, sizes, resized, index, crops, target_hw, proimages, labels, invalid, boxes=None,
                        vectors=None):
    th, tw = target_hw
    for n, e in enumerate(index.tolist()):
      oy, ox = (int(v) for v in crops[n])
      if not 0 <= e < offsets.numel():
        invalid += 1
        continue
      (h, w), (rh, rw) = sizes[e].tolist(), resized[e].tolist()
      if not (0 <= oy <= rh - th and 0 <= ox <= rw - tw):
        invalid += 1
        continue
      o = int(offsets[e])
      img = arena[o:o + h * w * 3].reshape(1, h, w, 3).to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
      proimages[n] = (opre.resize_bilinear_legacy(img, rh, rw)[0, oy:oy + th, ox:ox + tw] - 0.5) / 0.5
      if vectors is not None:
        labels[n] = vectors[e]
        continue
      start, coords, cids = boxes
      b = range(int(start[e]), int(start[e + 1]))
      dense = oweak.bbox_labels([(int(cids[i]),) + tuple(float(v) for v in coords[i]) for i in b
                                 if 0 <= int(cids[i]) < 15], h, w)   # other ids are skipped
      ys = np.minimum(np.floor((np.arange(th) + oy).astype(np.float32) * (np.float32(h) / np.float32(rh))).astype(int), h - 1)
      xs = np.minimum(np.floor((np.arange(tw) + ox).astype(np.float32) * (np.float32(w) / np.float32(rw))).astype(int), w - 1)
      labels[n] = torch.from_numpy(dense[ys][:, xs])
    return proimages, labels
  monkeypatch.setattr(ops, 'weak_train_inputs', weak_train_inputs)


def _refusal(fn):
  from wlseg.dataset_input import DatasetError
  with pytest.raises(DatasetError) as e:
    fn()
  return str(e.value)


def _decode(path):
  return np.array(Image.open(path).convert('RGB'), dtype=np.uint8)


# ------------------------------------------------------------------------------------------------ discovery
@pytest.mark.parametrize('header', [True, False])
def test_the_mid_table_reproduces_the_reference_mid2cid(tmp_path, header):
  from wlseg import weak_input
  gold = np.load(os.path.join(HERE, 'golden', 'reference_run.npz'))
  write_descriptions(str(tmp_path), header=header, case=str.upper)         # display names match case-insensitively
  table = weak_input.weak_class_ids(str(tmp_path))
  got = [table.get(m, -1) for m in ('/m/0k4j', '/m/0k4j', '/m/01bjv', '/m/01g317', '/m/nothing')]
  assert got == gold['rla/cids'].tolist()
  assert len(table) == 14 and '/m/x_tree' not in table


def test_descriptions_without_a_weak_class_are_refused_naming_the_missing(tmp_path):
  from wlseg import hierarchy, weak_input
  names = [hierarchy.weak_display_name(c) for c in range(14) if c not in (6, 12)]
  write_descriptions(str(tmp_path), names=names)
  msg = _refusal(lambda: weak_input.weak_class_ids(str(tmp_path)))
  assert 'class-descriptions-boxable.csv' in msg and 'Person' in msg and 'Traffic sign' in msg and 'Car' not in msg
  msg = _refusal(lambda: weak_input.weak_class_ids(str(tmp_path / 'nowhere')))
  assert 'class-descriptions-boxable.csv' in msg


def test_the_image_level_vector_equals_the_reference():
  from wlseg import weak_input
  gold = np.load(os.path.join(HERE, 'golden', 'reference_run.npz'))
  for cids, want in zip(gold['rla_image/cids'], gold['rla_image/out']):
    present = [int(c) for c in cids if c >= 0]
    if present:                       # an image without a weak class is no example
      assert np.array_equal(weak_input.image_vector(present), want)


def test_examples_counts_and_csr_tables(tmp_path):
  from wlseg import weak_input
  root = str(tmp_path)
  ims = [(f'a{i}', Image.fromarray(_rgb(np.random.default_rng(i), 20 + i, 30))) for i in range(4)]
  boxes = [('a2', 'Car', 0.1, 0.5, 0.2, 0.6), ('a0', 'Person', 0, 1, 0, 1), ('a0', 'Tree', 0, 1, 0, 1),
           ('a0', 'Bus', 0.5, 0.5, 0.25, 0.75), ('gone', 'Car', 0, 1, 0, 1), ('gone', 'Tree', 0, 1, 0, 1),
           ('a3', 'Tree', 0, 1, 0, 1)]
  tags = [('a1', 'Man', 1), ('a1', 'Man', 1), ('a1', 'Girl', 1), ('a2', 'Car', 0), ('a3', 'Dog', 1), ('gone', 'Bus', 1)]
  write_open_images(root, ims, boxes, tags)
  csv_path, labels, absent, no_weak = weak_input.read_part('bbox', root)
  assert csv_path.endswith('train-annotations-bbox.csv') and list(labels) == ['a0', 'a2']
  assert (absent, no_weak) == (2, 2)                          # two rows of 'gone'; a1 and a3 have no weak box
  assert [b[0] for b in labels['a0']] == [6, 1]
  part = weak_input.WeakPart('bbox', root, 1, (8, 12), 0, 1, 0)
  assert part.box_start.tolist() == [0, 2, 3] and part.box_cids.tolist() == [6, 1, 2]
  assert part.box_coords.dtype == np.float32 and part.box_coords[2].tolist() == np.float32([0.1, 0.5, 0.2, 0.6]).tolist()
  assert part.sizes == [(20, 30), (22, 30)] and part.n_boxes == 3
  assert 'absent' in part.summary() and '2 annotation rows' in part.summary() and '2 images without' in part.summary()
  _, labels, absent, no_weak = weak_input.read_part('image', root)
  assert list(labels) == ['a1'] and (absent, no_weak) == (1, 3)
  part = weak_input.WeakPart('image', root, 1, (8, 12), 0, 1, 0)
  assert '2 positive tags' in part.summary()              # Man twice and Girl: two distinct classes
  assert part.vectors.tolist() == [weak_input.image_vector([7, 10]).tolist()]


# ------------------------------------------------------------------------------------------------ refusals
def test_csv_discovery_refusals_name_the_directory_or_file(tmp_path):
  from wlseg import weak_input
  ims = [('a', Image.fromarray(_rgb(np.random.default_rng(0), 10, 10)))]
  root = write_open_images(str(tmp_path / 'none'), ims, bbox_csv=None)
  msg = _refusal(lambda: weak_input.read_part('bbox', root))
  assert root in msg and 'exactly one *annotations-bbox.csv' in msg and 'found 0' in msg
  root = write_open_images(str(tmp_path / 'two'), ims, [('a', 'Car', 0, 1, 0, 1)])
  write_open_images(root, ims, [('a', 'Car', 0, 1, 0, 1)], bbox_csv='validation-annotations-bbox.csv')
  msg = _refusal(lambda: weak_input.read_part('bbox', root))
  assert 'found 2' in msg and 'validation-annotations-bbox.csv' in msg
  root = str(tmp_path / 'cols')
  write_open_images(root, ims, tags_csv=None)
  with open(os.path.join(root, 'x-annotations-human-imagelabels.csv'), 'w') as f:
    f.write('ImageID,Source,LabelName\na,v,/m/0k4j\n')
  msg = _refusal(lambda: weak_input.read_part('image', root))
  assert 'x-annotations-human-imagelabels.csv' in msg and 'Confidence' in msg


@pytest.mark.parametrize('xy', [(0.2, 0.1, 0, 1), (0, 1, 0.6, 0.5), (-0.01, 0.5, 0, 1), (0, 1.5, 0, 1)])
def test_bad_coordinates_are_refused_naming_the_file_and_line(tmp_path, xy):
  from wlseg import weak_input
  ims = [('a', Image.fromarray(_rgb(np.random.default_rng(0), 10, 10)))]
  root = write_open_images(str(tmp_path), ims, [('a', 'Car', 0, 1, 0, 1), ('a', 'Bus') + xy])
  msg = _refusal(lambda: weak_input.read_part('bbox', root))
  assert 'train-annotations-bbox.csv:3' in msg and 'outside [0, 1] or has min > max' in msg


def test_an_image_over_the_box_cap_is_refused_stating_the_cap(tmp_path):
  from wlseg import weak_input
  ims = [('a', Image.fromarray(_rgb(np.random.default_rng(0), 10, 10)))]
  root = write_open_images(str(tmp_path), ims, [('a', 'Car', 0, 1, 0, 1)] * 1025)
  msg = _refusal(lambda: weak_input.read_part('bbox', root))
  assert 'train-annotations-bbox.csv' in msg and '1025 boxes' in msg and '1024' in msg


def test_an_unsupported_image_mode_names_the_file(tmp_path):
  from wlseg import weak_input
  ims = [('a', Image.fromarray(_rgb(np.random.default_rng(0), 10, 10))), ('b', Image.new('CMYK', (12, 8)))]
  root = write_open_images(str(tmp_path), ims, [('a', 'Car', 0, 1, 0, 1), ('b', 'Car', 0, 1, 0, 1)])
  msg = _refusal(lambda: weak_input.WeakPart('bbox', root, 1, (8, 8), 0, 1, 0))
  assert os.path.join(root, 'images', 'b.jpg') in msg and 'CMYK' in msg


def test_a_shard_smaller_than_one_batch_names_the_counts(tmp_path):
  from wlseg import weak_input
  root = random_open_images(str(tmp_path), 5)
  weak_input.WeakPart('bbox', root, 2, (8, 8), 1, 2, 0)
  msg = _refusal(lambda: weak_input.WeakPart('image', root, 3, (8, 8), 1, 2, 0))
  assert '--per_image_split_path' in msg and root in msg and 'holds 5' in msg and 'has 2' in msg and 'batch of 3' in msg


def test_the_budget_covers_all_three_arenas_and_is_refused_before_decoding(tmp_path, monkeypatch):
  from wlseg import dataset_input, train_input, weak_input
  split = cityscapes_train(str(tmp_path / 'cs'), 4)
  root = random_open_images(str(tmp_path / 'oi'), 6)
  st = weak_settings(split, root, root)
  pp = sum(h * w * 4 for h, w in dataset_input.check_pairs(train_input.split_pairs(split, 'cityscapes'))[0])
  need = pp + sum(p.bytes for p in weak_input.parts(st, (24, 40), 0, 1))
  reserves = []

  def budget(device, reserve=train_input.STEP_RESERVE_BYTES):
    reserves.append(reserve)
    return need - 1
  monkeypatch.setattr(train_input, 'device_budget', budget)
  monkeypatch.setattr(dataset_input, '_decode_image', lambda p: pytest.fail('decoded before the budget check'))
  with contextlib.redirect_stdout(io.StringIO()):
    msg = _refusal(lambda: train_input.train_input_fn(None, st))
  assert f'needs {need} bytes' in msg and f'{need - 1} are available' in msg and 'image-level' in msg
  assert reserves == [train_input.MIXED_STEP_RESERVE_BYTES]


# ------------------------------------------------------------------------------------------------ arena
def test_weak_arena_bytes_equal_a_direct_decode(tmp_path):
  from wlseg import weak_input
  root = random_open_images(str(tmp_path), 5)
  part = weak_input.WeakPart('bbox', root, 1, (16, 16), 0, 1, 0)
  with contextlib.redirect_stdout(io.StringIO()):
    part.fill('cpu', workers=2)
  off = 0
  for e, path in enumerate(part.paths):
    im = _decode(path)
    assert int(part.shard.offsets[e]) == off and part.shard.sizes[e].tolist() == list(im.shape[:2])
    assert np.array_equal(part.shard.arena[off:off + im.size].numpy(), im.reshape(-1))
    off += im.size
  assert part.shard.arena.numel() == off


# ------------------------------------------------------------------------------------------------ order
def test_orders_and_crops_are_pure_functions_and_the_per_pixel_order_is_unchanged(tmp_path):
  from wlseg import preprocess, train_input, weak_input
  # the per-pixel generator is still (seed, rank, world, epoch) alone
  want = np.random.default_rng([5, 1, 2, 3]).permutation(len(range(1, 2975, 2)))[:train_input.steps_per_epoch(2975, 2, 4) * 4]
  assert np.array_equal(train_input.epoch_order(5, 1, 2, 2975, 4, 3), want)
  root = random_open_images(str(tmp_path), 11)
  hw = (24, 40)
  a = weak_input.WeakPart('bbox', root, 2, hw, 0, 2, 7)
  b = weak_input.WeakPart('bbox', root, 2, hw, 0, 2, 7)
  i = weak_input.WeakPart('image', root, 2, hw, 0, 2, 7)
  other = weak_input.WeakPart('bbox', root, 2, hw, 1, 2, 7)
  assert a.steps_per_epoch == 11 // 2 // 2
  for e in range(3):
    (oa, ca), (ob, cb) = a.epoch(e), b.epoch(e)
    assert np.array_equal(oa, ob) and np.array_equal(ca, cb) and len(oa) == 4 and len(set(oa.tolist())) == 4
    assert set(oa.tolist()) <= set(range(len(a.ids)))
    for pos, (oy, ox) in zip(oa, ca):
      rh, rw = preprocess.resized_size(*a.sizes[pos], hw, True)
      assert a.resized[pos] == (rh, rw) and 0 <= oy <= rh - hw[0] and 0 <= ox <= rw - hw[1]
    assert not np.array_equal(a.epoch(e)[1][:2], i.epoch(e)[1][:2])
  assert len({tuple(a.epoch(e)[0]) + tuple(a.epoch(e)[1].ravel()) for e in range(4)}) == 4
  assert not np.array_equal(a.epoch(0)[1], other.epoch(0)[1]) or not np.array_equal(a.epoch(0)[0], other.epoch(0)[0])
  assert set(a.ids).isdisjoint(other.ids) and len(a.ids) + len(other.ids) == 11
  steps = [a.batch_at(s) for s in range(4)]
  assert np.array_equal(np.concatenate([s[0] for s in steps]), np.concatenate([a.epoch(0)[0], a.epoch(1)[0]]))


def _take(it, k):
  out = []
  for (f, l), _ in zip(it, range(k)):
    out.append((f['proimages'].clone(), {key: v.clone() for key, v in l.items()}))
  return out


def test_mixed_batches_equal_the_oracle_in_the_stated_order_and_resume_at_any_step(tmp_path, monkeypatch):
  """The 2 + 2 + 1 batch from the arenas: per-pixel rows unchanged, then the bbox rows, then the image-level rows, each
  equal to the oracle at the part's stated (order, crop); a run resumed at step k feeds steps k... of the uninterrupted
  run, across every part's epoch boundary."""
  from tests.test_train_dataset_cpu import _decode as decode_pair, _lut, oracle_example
  from wlseg import train_input, weak_input
  emulated_train_inputs(monkeypatch)
  emulated_weak_train_inputs(monkeypatch)
  split = cityscapes_train(str(tmp_path / 'cs'), 7)
  bb = random_open_images(str(tmp_path / 'bb'), 5, seed=1)
  il = random_open_images(str(tmp_path / 'il'), 4, seed=2, sizes=((30, 80), (61, 37)))
  st = weak_settings(split, bb, il, seed=3)
  hw = (24, 40)
  with contextlib.redirect_stdout(io.StringIO()) as out:
    full = _take(train_input.train_input_fn(None, st), 7)
  text = out.getvalue()
  assert 'bbox part: ' in text and 'image part: ' in text and 'decoded 5 bbox images' in text
  pairs, lut = train_input.split_pairs(split, 'cityscapes'), _lut('cityscapes')
  parts = weak_input.parts(st, hw, 0, 1)
  _, bb_labels, _, _ = weak_input.read_part('bbox', bb)
  for s, (pro, labels) in enumerate(full):
    assert pro.shape == (5, 24, 40, 3) and set(labels) == {'prolabels_per_pixel', 'prolabels_per_bbox',
                                                           'prolabels_per_image'}
    for j, e in enumerate(train_input.batch_at(3, 0, 1, 7, 2, s)):
      want_pro, want_lab = oracle_example(*decode_pair(pairs[e]), lut, max(lut), *hw)
      assert torch.equal(pro[j], want_pro) and torch.equal(labels['prolabels_per_pixel'][j], want_lab)
    row = 2
    for part, key in zip(parts, ('prolabels_per_bbox', 'prolabels_per_image')):
      order, crops = part.batch_at(s)
      for j, (e, off) in enumerate(zip(order, crops)):
        boxes = [(b[0], b[1:]) for b in bb_labels[part.ids[e]]] if part.part == 'bbox' else None
        want_pro, want_lab = oracle_weak_example(_decode(part.paths[e]), boxes,
                                                 part.vectors[e] if boxes is None else None, hw, tuple(off))
        assert torch.equal(pro[row + j], want_pro), (s, key, j)
        assert torch.equal(labels[key][j], want_lab), (s, key, j)
      row += part.Nb
  for k in (1, 2, 5):              # per-pixel epochs of 3 steps, bbox of 2, image-level of 4
    st.initial_global_step = k
    with contextlib.redirect_stdout(io.StringIO()):
      resumed = _take(train_input.train_input_fn(None, st), 7 - k)
    for (pa, la), (pb, lb) in zip(resumed, full[k:]):
      assert torch.equal(pa, pb) and all(torch.equal(la[key], lb[key]) for key in la), k


def test_a_part_without_its_flag_stays_empty(tmp_path, monkeypatch):
  from wlseg import train_input
  emulated_train_inputs(monkeypatch)
  emulated_weak_train_inputs(monkeypatch)
  split = cityscapes_train(str(tmp_path / 'cs'), 4)
  root = random_open_images(str(tmp_path / 'oi'), 4)
  with contextlib.redirect_stdout(io.StringIO()) as out:
    (pro, labels), = _take(train_input.train_input_fn(None, weak_settings(split, image=root)), 1)
  assert pro.shape[0] == 3 and set(labels) == {'prolabels_per_pixel', 'prolabels_per_image'}
  assert 'image part: ' in out.getvalue() and 'bbox part' not in out.getvalue()


def test_the_restated_op_equals_the_oracle_composition_on_ragged_sizes(monkeypatch):
  """Sizes smaller than, taller and wider than the target, odd targets, offsets 0 / max / middle, edge, overlapping
  and degenerate boxes, an unknown cid, an example without a valid box, repeated indices; invalid indices and crops
  are counted and write nothing."""
  from wlseg import ops, preprocess, train_input
  emulated_weak_train_inputs(monkeypatch)
  rng = np.random.default_rng(4)
  th, tw = 23, 37
  shapes = [(11, 19), (97, 40), (30, 150), (23, 37)]
  imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
  boxes = [[(2, (0.0, 1.0, 0.0, 1.0)), (6, (0.2, 0.7, 0.1, 0.9))],
           [(1, (0.5, 0.5, 0.5, 0.5)), (2, (0.0, 0.3, 0.9, 1.0)), (2, (0.1, 0.3, 0.0, 0.4)), (15, (0, 1, 0, 1))],
           [(13, (0.99, 1.0, 0.0, 0.01))],
           [(-1, (0.0, 1.0, 0.0, 1.0))]]
  offsets, _ = train_input.arena_layout(shapes, 3)
  arena = torch.from_numpy(np.concatenate([im.reshape(-1) for im in imgs]))
  resized = [preprocess.resized_size(h, w, (th, tw), True) for h, w in shapes]
  start = np.cumsum([0] + [len(b) for b in boxes]).astype(np.int32)
  flat = [b for bs in boxes for b in bs]
  tables = (torch.from_numpy(start), torch.tensor([b[1] for b in flat], dtype=torch.float32),
            torch.tensor([b[0] for b in flat], dtype=torch.int32))
  index = [0, 1, 2, 3, 1, 2, 1, 5, -1, 0]
  crops = [(0, 0), (resized[1][0] - th, 0), (0, (resized[2][1] - tw) // 2), (0, 0), (7, 0), (0, resized[2][1] - tw),
           (resized[1][0] - th + 1, 0), (0, 0), (0, 0), (1, 0)]
  n = len(index)
  pro, lab = torch.full((n, th, tw, 3), -7.0), torch.full((n, th, tw, 15), -7.0)
  invalid = torch.zeros(1, dtype=torch.int64)
  ops.weak_train_inputs(arena, torch.from_numpy(offsets), torch.tensor(shapes, dtype=torch.int32),
                        torch.tensor(resized, dtype=torch.int32), torch.tensor(index, dtype=torch.int32),
                        torch.tensor(crops, dtype=torch.int32), (th, tw), pro, lab, invalid, boxes=tables)
  assert int(invalid) == 4                 # crop past the end, index 5, index -1, a crop on an axis without room
  for k, (e, off) in enumerate(zip(index, crops)):
    if k in (6, 7, 8, 9):
      assert bool((pro[k] == -7).all()) and bool((lab[k] == -7).all())
      continue
    known = [(c, xy) for c, xy in boxes[e] if 0 <= c < 15]
    want_pro, want_lab = oracle_weak_example(imgs[e], known, None, (th, tw), off)
    assert torch.equal(pro[k], want_pro) and torch.equal(lab[k], want_lab), k
  assert bool((lab[3][..., 14] == 1).all())          # no valid box: void everywhere


# ------------------------------------------------------------------------------------------------ train.py
def _train_main(monkeypatch, tmp_path, extra):
  from tests.test_train_dataset_cpu import _train_main_choice
  return _train_main_choice(monkeypatch, tmp_path, extra)


def test_train_main_refuses_a_weak_flag_without_the_per_pixel_split(monkeypatch, tmp_path):
  root = random_open_images(str(tmp_path / 'oi'), 4)
  for flag in ('--per_bbox_split_path', '--per_image_split_path'):
    with pytest.raises(ValueError) as e:
      _train_main(monkeypatch, tmp_path, [flag, root])
    assert flag in str(e.value) and '--per_pixel_split_path' in str(e.value)


def test_train_main_with_weak_flags_names_each_part(monkeypatch, tmp_path):
  from wlseg import synthetic, train_input
  split = cityscapes_train(str(tmp_path / 'data'), 4)
  root = random_open_images(str(tmp_path / 'oi'), 4)
  fn, out = _train_main(monkeypatch, tmp_path, ['--per_pixel_split_path', split, '--per_bbox_split_path', root])
  assert fn is train_input.train_input_fn
  assert 'bounding-box part from --per_bbox_split_path' in out and 'image-level part empty' in out
  assert 'no Open Images source' not in out
  fn, out = _train_main(monkeypatch, tmp_path, ['--per_pixel_split_path', split, '--per_bbox_split_path', root,
                                                '--per_image_split_path', root, '--synthetic'])
  assert fn is synthetic.train_input_fn and out == ''
  fn, out = _train_main(monkeypatch, tmp_path, ['--per_image_split_path', root, '--synthetic'])
  assert fn is synthetic.train_input_fn and out == ''


def test_the_flags_reach_the_settings():
  from wlseg import settings as wsettings
  st = wsettings.build_parser(wsettings.TRAIN).parse_args(['log', 'cityscapes', '--per_bbox_split_path', 'a',
                                                           '--per_image_split_path', 'b'])
  assert (st.per_bbox_split_path, st.per_image_split_path) == ('a', 'b')


def test_the_weak_classes_have_the_open_images_display_names():
  from wlseg import hierarchy
  assert [hierarchy.weak_display_name(c) for c in range(14)] == [
      'Bicycle', 'Bus', 'Car', 'Motorcycle', 'Train', 'Truck', 'Person', 'Man', 'Woman', 'Boy', 'Girl', 'Traffic light',
      'Traffic sign', 'Stop sign']


def test_a_confidence_that_is_no_number_names_the_file_and_line(tmp_path):
  from wlseg import weak_input
  ims = [('a', Image.fromarray(_rgb(np.random.default_rng(0), 10, 10)))]
  root = write_open_images(str(tmp_path), ims, tags=[('a', 'Car', 1), ('a', 'Bus', 'yes')])
  msg = _refusal(lambda: weak_input.read_part('image', root))
  assert 'train-annotations-human-imagelabels-boxable.csv:3' in msg and "'yes'" in msg
