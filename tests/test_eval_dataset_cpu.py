"""Evaluation on Cityscapes / Vistas splits read from disk (wlseg/dataset_input.py + Estimator.evaluate's packed raw
path + cli.evaluate_main's input choice), on CPU.  ops.eval_inputs is replaced by its contract restated with the oracle
(oracle.preprocess legacy resizes + the label-id gather); the kernel's own bit equality is tests/test_gpu_eval_dataset.py.
"""

import contextlib
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

from tests.test_host_orchestration_cpu import _emulated_eval_tail, _emulated_ops, _host_only_runtime


# ------------------------------------------------------------------------------------------------ split writers
def _rgb(rng, h, w):
  return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


def _lids(rng, h, w, n_lids, block=8):
  """Blocky label-id maps (so that nearest resizing keeps every class around)."""
  small = rng.integers(0, n_lids, (-(-h // block), -(-w // block)), dtype=np.uint8)
  return np.repeat(np.repeat(small, block, 0), block, 1)[:h, :w].copy()


def write_cityscapes(root, examples, split='val'):
  """examples: [(city, stem, PIL image, label array or PIL image)] -> root/leftImg8bit/<split>; returns that path."""
  for city, stem, im, lab in examples:
    for d in ('leftImg8bit', 'gtFine'):
      os.makedirs(os.path.join(root, d, split, city), exist_ok=True)
    im.save(os.path.join(root, 'leftImg8bit', split, city, f'{stem}_leftImg8bit.png'))
    if lab is not None:
      lab = lab if isinstance(lab, Image.Image) else Image.fromarray(lab, mode='L')
      lab.save(os.path.join(root, 'gtFine', split, city, f'{stem}_gtFine_labelIds.png'))
  return os.path.join(root, 'leftImg8bit', split)


def write_vistas(root, examples):
  """examples: [(stem, PIL image, label array)] -> root with images/<stem>.jpg, labels/<stem>.png (palette-indexed)."""
  os.makedirs(os.path.join(root, 'images'), exist_ok=True)
  os.makedirs(os.path.join(root, 'labels'), exist_ok=True)
  for stem, im, lab in examples:
    im.save(os.path.join(root, 'images', f'{stem}.jpg'), quality=90)
    p = Image.fromarray(lab, mode='P')
    p.putpalette([(i * 37) % 256 for i in range(768)])
    p.save(os.path.join(root, 'labels', f'{stem}.png'))
  return root


def mixed_cityscapes(root, n, n_lids=34, seed=0, sizes=((48, 64), (37, 83), (64, 96), (29, 41))):
  rng = np.random.default_rng(seed)
  ex = []
  for i in range(n):
    h, w = sizes[i % len(sizes)]
    ex.append((('bochum', 'aachen')[i % 2], f'c_{i:03d}', Image.fromarray(_rgb(rng, h, w)), _lids(rng, h, w, n_lids)))
  return write_cityscapes(root, ex)


def mixed_vistas(root, n, n_lids=66, seed=1, sizes=((45, 60), (70, 52), (33, 91))):
  rng = np.random.default_rng(seed)
  return write_vistas(root, [(f'v_{i:03d}', Image.fromarray(_rgb(rng, *sizes[i % len(sizes)])),
                              _lids(rng, *sizes[i % len(sizes)], n_lids)) for i in range(n)])


def host_batches(split_dir, steps, Nb, hw, lut):
  """The evaluation contract computed on the host from the files: PIL decode -> u8 * (float)(1/255) -> legacy bilinear
  -> (v - 0.5) / 0.5; label ids -> legacy nearest -> lut.  [(features, labels)] in evaluation order."""
  from oracle import preprocess as opre
  from wlseg import dataset_input
  pairs = dataset_input.list_pairs(split_dir)[:steps * Nb]
  lut = torch.tensor(lut, dtype=torch.int64)
  out = []
  for b in range(steps):
    pro, lab = [], []
    for img_path, lab_path in pairs[b * Nb:(b + 1) * Nb]:
      raw = torch.from_numpy(np.asarray(Image.open(img_path).convert('RGB'), dtype=np.uint8).copy())
      img = raw[None].to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
      pro.append((opre.resize_bilinear_legacy(img, *hw)[0] - 0.5) / 0.5)
      ids = torch.from_numpy(np.asarray(Image.open(lab_path), dtype=np.uint8).copy())
      lab.append(lut[opre.resize_nearest_legacy(ids[None], *hw)[0].long()].to(torch.int32))
    out.append(({'proimages': torch.stack(pro)}, {'prolabels': torch.stack(lab)}))
  return out


def _settings(**kw):
  import argparse
  d = dict(Nb=2, num_eval_steps=2, rank=0, world_size=1)
  d.update(kw)
  return argparse.Namespace(**d)


def _emulated_eval_inputs(monkeypatch):
  """ops.eval_inputs restated: per example the oracle's legacy bilinear / nearest resizes and the label-id gather."""
  from oracle import preprocess as opre
  from wlseg import ops

  def eval_inputs(images, lids, sizes, lut, void_id, target_hw, proimages, prolabels, invalid):
    th, tw = target_hw
    for n in range(images.shape[0]):
      h, w = (int(v) for v in sizes[n])
      if h <= 0 or w <= 0 or h * w * 3 > images.shape[1] or h * w > lids.shape[1]:
        invalid += 1
        continue
      img = images[n, :h * w * 3].reshape(1, h, w, 3).to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
      proimages[n] = (opre.resize_bilinear_legacy(img, th, tw)[0] - 0.5) / 0.5
      ids = opre.resize_nearest_legacy(lids[n, :h * w].reshape(1, h, w), th, tw)[0].long()
      ok = ids < lut.numel()
      invalid += int((~ok).sum())
      prolabels[n] = torch.where(ok, lut[ids.clamp(max=lut.numel() - 1)], torch.tensor(void_id, dtype=torch.int32))
    return proimages, prolabels
  monkeypatch.setattr(ops, 'eval_inputs', eval_inputs)


# ------------------------------------------------------------------------------------------------ discovery
def test_cityscapes_split_is_found_sorted_and_decoded_in_every_image_mode(tmp_path):
  from wlseg import dataset_input
  rng = np.random.default_rng(3)
  rgb = _rgb(rng, 20, 30)
  ims = {'RGB': Image.fromarray(rgb), 'L': Image.fromarray(rgb[..., 0], mode='L'),
         'P': Image.fromarray(rgb).convert('P'), 'RGBA': Image.fromarray(np.dstack([rgb, rgb[..., :1]]), mode='RGBA')}
  lab = _lids(rng, 20, 30, 34)
  pal = Image.fromarray(lab, mode='P')
  pal.putpalette([255 - (i % 256) for i in range(768)])     # the palette must not matter: the index is the id
  ex = [('zurich', 'a_rgb', ims['RGB'], lab), ('aachen', 'b_l', ims['L'], pal), ('aachen', 'a_p', ims['P'], lab),
        ('bochum', 'c_rgba', ims['RGBA'], pal)]
  split = write_cityscapes(str(tmp_path), ex)
  assert dataset_input.detect_layout(split) == 'cityscapes'
  pairs = dataset_input.list_pairs(split)
  assert [os.path.relpath(p[0], split) for p in pairs] == ['aachen/a_p_leftImg8bit.png', 'aachen/b_l_leftImg8bit.png',
                                                           'bochum/c_rgba_leftImg8bit.png', 'zurich/a_rgb_leftImg8bit.png']
  assert pairs[0][1] == os.path.join(str(tmp_path), 'gtFine', 'val', 'aachen', 'a_p_gtFine_labelIds.png')
  batches = list(dataset_input.eval_input_fn(None, _settings(tfrecords_path=split, Nb=2, num_eval_steps=2)))
  assert len(batches) == 2
  order = [ims['P'], ims['L'], ims['RGBA'], ims['RGB']]
  for b, (f, l) in enumerate(batches):
    for j in range(2):
      want = np.asarray(order[2 * b + j].convert('RGB'), dtype=np.uint8)
      assert f['packed_sizes'][j].tolist() == [20, 30]
      assert np.array_equal(f['packed_images'][j, :20 * 30 * 3].numpy(), want.reshape(-1))
      assert np.array_equal(l['packed_lids'][j, :600].numpy(), lab.reshape(-1))


def test_vistas_split_decodes_jpeg_images_and_palette_labels_as_indices(tmp_path):
  from wlseg import dataset_input
  root = mixed_vistas(str(tmp_path / 'validation'), 3)
  assert dataset_input.detect_layout(root) == 'vistas'
  pairs = dataset_input.list_pairs(root)
  assert [os.path.basename(p[0]) for p in pairs] == ['v_000.jpg', 'v_001.jpg', 'v_002.jpg']
  (f, l), = list(dataset_input.eval_input_fn(None, _settings(tfrecords_path=root, Nb=3, num_eval_steps=1)))
  for j, (img_path, lab_path) in enumerate(pairs):
    im = np.asarray(Image.open(img_path).convert('RGB'))
    ids = np.asarray(Image.open(lab_path))
    h, w = ids.shape
    assert f['packed_sizes'][j].tolist() == [h, w] and im.shape[:2] == (h, w)
    assert np.array_equal(f['packed_images'][j, :h * w * 3].numpy(), im.reshape(-1))
    assert np.array_equal(l['packed_lids'][j, :h * w].numpy(), ids.reshape(-1)) and ids.max() > 33


def test_batches_of_a_split_with_mixed_sizes_have_one_shape(tmp_path):
  from wlseg import dataset_input
  split = mixed_cityscapes(str(tmp_path), 8)
  batches = list(dataset_input.eval_input_fn(None, _settings(tfrecords_path=split, Nb=2, num_eval_steps=4)))
  biggest = 64 * 96
  assert {tuple(f['packed_images'].shape) for f, _ in batches} == {(2, biggest * 3)}
  assert {tuple(l['packed_lids'].shape) for _, l in batches} == {(2, biggest)}
  assert {tuple(f['packed_sizes'].shape) for f, _ in batches} == {(2, 2)}
  assert sorted({tuple(s) for f, _ in batches for s in f['packed_sizes'].tolist()}) == [(29, 41), (37, 83), (48, 64), (64, 96)]


def test_ranks_take_disjoint_batches_that_cover_the_evaluation(tmp_path):
  from wlseg import dataset_input
  split = mixed_cityscapes(str(tmp_path), 11)
  steps, Nb, world = 5, 2, 3
  everything = [f['packed_images'] for f, _ in dataset_input.eval_input_fn(
      None, _settings(tfrecords_path=split, Nb=Nb, num_eval_steps=steps))]
  seen = {}
  for rank in range(world):
    got = list(dataset_input.eval_input_fn(None, _settings(tfrecords_path=split, Nb=Nb, num_eval_steps=steps, rank=rank,
                                                           world_size=world)))
    for i, (f, _) in enumerate(got):
      b = rank + i * world                          # batch b goes to rank b % world
      assert b not in seen and torch.equal(f['packed_images'], everything[b])
      seen[b] = rank
  assert sorted(seen) == list(range(steps))


# ------------------------------------------------------------------------------------------------ refused splits
def _err(split, steps=1, Nb=1):
  from wlseg import dataset_input
  with pytest.raises(dataset_input.DatasetError) as e:
    dataset_input.eval_input_fn(None, _settings(tfrecords_path=split, Nb=Nb, num_eval_steps=steps))
  return str(e.value)


def test_missing_label_names_the_file(tmp_path):
  rng = np.random.default_rng(0)
  split = write_cityscapes(str(tmp_path), [('ulm', 'x', Image.fromarray(_rgb(rng, 8, 8)), _lids(rng, 8, 8, 34)),
                                           ('ulm', 'y', Image.fromarray(_rgb(rng, 8, 8)), None)])
  msg = _err(split, steps=2)
  assert 'y_leftImg8bit.png' in msg and 'y_gtFine_labelIds.png' in msg


def test_image_and_label_of_different_sizes_are_refused(tmp_path):
  rng = np.random.default_rng(0)
  split = write_cityscapes(str(tmp_path), [('ulm', 'x', Image.fromarray(_rgb(rng, 8, 10)), _lids(rng, 8, 12, 34))])
  msg = _err(split)
  assert 'x_gtFine_labelIds.png' in msg and '12x8' in msg and '10x8' in msg


@pytest.mark.parametrize('kind', ['rgb', '16bit'])
def test_labels_that_are_not_8bit_indices_are_refused(tmp_path, kind):
  rng = np.random.default_rng(0)
  lab = (Image.fromarray(_rgb(rng, 8, 8)) if kind == 'rgb'
         else Image.fromarray(_lids(rng, 8, 8, 34).astype(np.uint16) * 300))
  split = write_cityscapes(str(tmp_path), [('ulm', 'x', Image.fromarray(_rgb(rng, 8, 8)), lab)])
  msg = _err(split)
  assert 'x_gtFine_labelIds.png' in msg and ('RGB' in msg if kind == 'rgb' else 'I;16' in msg)


def test_unsupported_image_mode_is_refused(tmp_path):
  rng = np.random.default_rng(0)
  split = write_cityscapes(str(tmp_path), [('ulm', 'x', Image.fromarray(_rgb(rng, 8, 8)[..., :2], mode='LA'),
                                            _lids(rng, 8, 8, 34))])
  msg = _err(split)
  assert 'x_leftImg8bit.png' in msg and 'LA' in msg


def test_too_few_files_names_both_numbers(tmp_path):
  split = mixed_cityscapes(str(tmp_path), 5)
  msg = _err(split, steps=3, Nb=2)
  assert '5' in msg and '6' in msg


# ------------------------------------------------------------------------------------------------ evaluate.py
def _cli_on_cpu(monkeypatch):
  from wlseg import cli

  def dist_env(st):
    st.rank, st.world_size, st.device = 0, 1, 'cpu'
    return st
  monkeypatch.setattr(cli, '_dist_env', dist_env)


def _eval_argv(log_dir, split, dataset, ckpt, Neval, Nb, hw):
  from wlseg import problem_defs
  problem_defs.write_all()
  return [str(log_dir), str(Neval), problem_defs.default_path(dataset), str(split), dataset, '--Nb', str(Nb),
          '--height_feature_extractor', str(hw[0]), '--width_feature_extractor', str(hw[1]), '--dtype', 'fp32',
          '--ckpt_path', ckpt]


def _cpu_eval_stack(monkeypatch, dataset):
  from wlseg import hierarchy, problem_defs
  hier = hierarchy.Hierarchy(dataset, problem_defs.GENERATORS[dataset]()['cids2labels'])
  head = _emulated_ops(monkeypatch)
  head.widths, head.dataset = hier.head_widths, dataset
  _emulated_eval_tail(monkeypatch, dataset, hier.head_widths)
  _host_only_runtime(monkeypatch)
  _emulated_eval_inputs(monkeypatch)
  _cli_on_cpu(monkeypatch)


def _checkpoint(tmp_path, dataset):
  import importlib
  from wlseg import checkpoints
  gen = importlib.import_module('tests.golden.make_reference_eval_fixtures')
  return checkpoints.save_file(os.path.join(str(tmp_path), 'model.ckpt-7.pt'), gen.case_params(dataset), 7)


def test_evaluate_main_on_a_cityscapes_split_equals_host_preprocessed_batches(monkeypatch, tmp_path):
  """evaluate.py on a directory: discovery, decoding workers, packed batches, the device conversion (emulated), the
  evaluation step; its confusion matrix equals, entry by entry, Estimator.evaluate's on batches preprocessed on the
  host from the same files, and all_metrics.txt is written."""
  from wlseg import cli, estimator as est, problem_defs, settings as wsettings
  from wlseg.system_factory import SemanticSegmentation
  _cpu_eval_stack(monkeypatch, 'cityscapes')
  split = mixed_cityscapes(str(tmp_path / 'data'), 7)
  ckpt = _checkpoint(tmp_path, 'cityscapes')
  log_dir = tmp_path / 'log'
  log_dir.mkdir()
  hw = (40, 56)
  argv = _eval_argv(log_dir, split, 'cityscapes', ckpt, 6, 2, hw)
  out = io.StringIO()
  with contextlib.redirect_stdout(out):
    got = cli.evaluate_main(argv)
  assert 'Evaluating the cityscapes split' in out.getvalue()
  assert got[0]['steps'] == 3 and got[0]['global_step'] == 7
  assert (log_dir / 'eval_00' / 'all_metrics.txt').read_text().startswith('00007 ')
  lut = est._replacevoids(problem_defs.cityscapes()['lids2cids'])
  batches = host_batches(split, 3, 2, hw, lut)
  st = wsettings.eval_extra_args(wsettings.build_parser(wsettings.EVAL).parse_args(argv))
  st.device, st.rank, st.world_size = 'cpu', 0, 1
  with contextlib.redirect_stdout(io.StringIO()):
    want = SemanticSegmentation({'eval': lambda config, params: iter(batches)}, None, st).evaluate()
  assert want[0]['confusion_matrix_int64'].sum() == 6 * hw[0] * hw[1]
  assert np.array_equal(got[0]['confusion_matrix_int64'], want[0]['confusion_matrix_int64'])
  assert np.array_equal(got[0]['confusion_matrix'], want[0]['confusion_matrix'])


def test_out_of_range_label_id_raises(monkeypatch, tmp_path):
  from wlseg import cli, ops
  _cpu_eval_stack(monkeypatch, 'cityscapes')
  rng = np.random.default_rng(5)
  lab = _lids(rng, 40, 56, 34)
  lab[:8, :8] = 200                                 # Cityscapes has 34 label ids
  split = write_cityscapes(str(tmp_path / 'data'), [('ulm', 'x', Image.fromarray(_rgb(rng, 40, 56)), lab)])
  log_dir = tmp_path / 'log'
  log_dir.mkdir()
  argv = _eval_argv(log_dir, split, 'cityscapes', _checkpoint(tmp_path, 'cityscapes'), 1, 1, (40, 56))
  with contextlib.redirect_stdout(io.StringIO()), pytest.raises(ops.WlsegError, match='^64 label ids'):
    cli.evaluate_main(argv)


@pytest.mark.parametrize('where', ['plain_dir', 'missing', 'tfrecords', 'synthetic_flag'])
def test_other_inputs_still_evaluate_synthetic_data(monkeypatch, tmp_path, where):
  from wlseg import cli, synthetic

  class Stop(Exception):
    pass
  chosen = []

  def fake_system(input_fns, model_fn, settings):
    chosen.append(input_fns['eval'])
    raise Stop()
  _cli_on_cpu(monkeypatch)
  monkeypatch.setattr(cli, 'SemanticSegmentation', fake_system)
  extra = []
  if where == 'plain_dir':
    path = tmp_path / 'somewhere'
    path.mkdir()
    Image.fromarray(np.zeros((4, 4, 3), np.uint8)).save(str(path / 'a.png'))
  elif where == 'missing':
    path = tmp_path / 'nothing_here'
  elif where == 'tfrecords':
    path = 'tfrecords/x.tfrecords'
  else:
    path = mixed_cityscapes(str(tmp_path / 'data'), 2)
    extra = ['--synthetic']
  argv = _eval_argv(tmp_path, path, 'cityscapes', 'unused', 2, 1, (40, 56)) + extra
  out = io.StringIO()
  with contextlib.redirect_stdout(out), pytest.raises(Stop):
    cli.evaluate_main(argv)
  assert chosen == [synthetic.eval_input_fn]
  assert 'Evaluating SYNTHETIC input' in out.getvalue()
