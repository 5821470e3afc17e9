"""Training on Cityscapes / Vistas splits read from disk (wlseg/train_input.py + cli.train_main's input choice), on CPU.
ops.train_inputs is replaced by its contract restated with the oracle's legacy resizes; the kernel's own bit equality is
tests/test_gpu_train_dataset.py."""

import argparse
import contextlib
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

from tests.test_eval_dataset_cpu import _lids, _rgb, write_cityscapes, write_vistas


def cityscapes_train(root, n, sizes=((48, 64), (37, 83), (64, 96), (29, 41)), n_lids=34, seed=0):
  rng = np.random.default_rng(seed)
  ex = [(('bochum', 'aachen', 'zurich')[i % 3], f'c_{i:03d}', Image.fromarray(_rgb(rng, *sizes[i % len(sizes)])),
         _lids(rng, *sizes[i % len(sizes)], n_lids)) for i in range(n)]
  return write_cityscapes(root, ex, split='train')


def vistas_train(root, n, sizes=((45, 60), (70, 52), (33, 91)), n_lids=66, seed=1):
  rng = np.random.default_rng(seed)
  return write_vistas(os.path.join(root, 'training'), [(f'v_{i:03d}', Image.fromarray(_rgb(rng, *sizes[i % len(sizes)])),
                                                        _lids(rng, *sizes[i % len(sizes)], n_lids)) for i in range(n)])


def train_settings(split, dataset='cityscapes', **kw):
  from wlseg import problem_defs
  d = dict(per_pixel_split_path=split, per_pixel_dataset_name=dataset, Nb_per_pixel=2, distribute=False, rank=0,
           world_size=1, device='cpu', Ntrain=2975 if dataset == 'cityscapes' else 18000, seed=0,
           training_problem_def=problem_defs.GENERATORS[dataset](), height_feature_extractor=24,
           width_feature_extractor=40, initial_global_step=0)
  d.update(kw)
  return argparse.Namespace(**d)


def oracle_example(im, ids, lut, void_id, th, tw):
  """The per-pixel training contract of one example on the host: u8 * (float)(1/255) -> legacy bilinear ->
  (v - 0.5) / 0.5; label ids -> legacy nearest -> lut (void_id past its end)."""
  from oracle import preprocess as opre
  img = torch.as_tensor(im)[None].to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
  pro = (opre.resize_bilinear_legacy(img, th, tw)[0] - 0.5) / 0.5
  ids = opre.resize_nearest_legacy(torch.as_tensor(ids)[None], th, tw)[0].long()
  lut = torch.tensor(list(lut) + [void_id], dtype=torch.int32)
  return pro, lut[ids.clamp(max=len(lut) - 1)]


def emulated_train_inputs(monkeypatch):
  """ops.train_inputs restated: per output example the arena example index[n], the oracle's legacy resizes and the
  label-id gather."""
  from oracle import preprocess as opre
  from wlseg import ops

  def train_inputs(arena, offsets, sizes, index, lut, void_id, target_hw, proimages, prolabels, invalid):
    th, tw = target_hw
    for n, e in enumerate(index.tolist()):
      if not 0 <= e < offsets.numel():
        invalid += 1
        continue
      h, w = (int(v) for v in sizes[e])
      o = int(offsets[e])
      img = arena[o:o + h * w * 3].reshape(1, h, w, 3).to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
      proimages[n] = (opre.resize_bilinear_legacy(img, th, tw)[0] - 0.5) / 0.5
      ids = opre.resize_nearest_legacy(arena[o + h * w * 3:o + h * w * 4].reshape(1, h, w), th, tw)[0].long()
      ok = ids < lut.numel()
      invalid += int((~ok).sum())
      prolabels[n] = torch.where(ok, lut[ids.clamp(max=lut.numel() - 1)], torch.tensor(void_id, dtype=torch.int32))
    return proimages, prolabels
  monkeypatch.setattr(ops, 'train_inputs', train_inputs)


def _decode(pair):
  img_path, lab_path = pair
  return np.array(Image.open(img_path).convert('RGB'), dtype=np.uint8), np.array(Image.open(lab_path), dtype=np.uint8)


def _lut(dataset):
  from wlseg import estimator as est, problem_defs
  return est._replacevoids(problem_defs.GENERATORS[dataset]()['lids2cids'])


# ------------------------------------------------------------------------------------------------ discovery
def test_training_splits_are_found_in_path_order(tmp_path):
  from wlseg import train_input
  cs = cityscapes_train(str(tmp_path / 'cs'), 5)
  assert cs.endswith(os.path.join('leftImg8bit', 'train'))
  pairs = train_input.split_pairs(cs, 'cityscapes')
  assert [os.path.relpath(p[0], cs) for p in pairs] == [
      'aachen/c_001_leftImg8bit.png', 'aachen/c_004_leftImg8bit.png', 'bochum/c_000_leftImg8bit.png',
      'bochum/c_003_leftImg8bit.png', 'zurich/c_002_leftImg8bit.png']
  assert pairs[0][1] == os.path.join(str(tmp_path / 'cs'), 'gtFine', 'train', 'aachen', 'c_001_gtFine_labelIds.png')
  vs = vistas_train(str(tmp_path / 'vs'), 3)
  assert [os.path.basename(p[0]) for p in train_input.split_pairs(vs, 'vistas')] == ['v_000.jpg', 'v_001.jpg', 'v_002.jpg']


# ------------------------------------------------------------------------------------------------ refusals
def _refusal(fn):
  from wlseg.dataset_input import DatasetError
  with pytest.raises(DatasetError) as e:
    fn()
  return str(e.value)


def test_a_split_of_the_other_dataset_is_refused_naming_both(tmp_path):
  from wlseg import train_input
  vs = vistas_train(str(tmp_path), 2)
  msg = _refusal(lambda: train_input.train_input_fn(None, train_settings(vs, 'cityscapes')))
  assert vs in msg and 'vistas' in msg and 'cityscapes' in msg
  msg = _refusal(lambda: train_input.split_pairs(str(tmp_path / 'training' / 'images'), 'vistas'))
  assert 'neither' in msg and 'vistas' in msg


def test_missing_label_and_size_mismatch_name_the_file(tmp_path):
  from wlseg import train_input
  rng = np.random.default_rng(0)
  split = write_cityscapes(str(tmp_path / 'a'), [('ulm', 'x', Image.fromarray(_rgb(rng, 8, 8)), _lids(rng, 8, 8, 34)),
                                                 ('ulm', 'y', Image.fromarray(_rgb(rng, 8, 8)), None)], split='train')
  msg = _refusal(lambda: train_input.train_input_fn(None, train_settings(split)))
  assert 'y_leftImg8bit.png' in msg and 'y_gtFine_labelIds.png' in msg
  split = write_cityscapes(str(tmp_path / 'b'), [('ulm', 'x', Image.fromarray(_rgb(rng, 8, 10)), _lids(rng, 8, 12, 34)),
                                                 ('ulm', 'z', Image.fromarray(_rgb(rng, 8, 10)), _lids(rng, 8, 10, 34))],
                           split='train')
  msg = _refusal(lambda: train_input.train_input_fn(None, train_settings(split)))
  assert 'x_gtFine_labelIds.png' in msg and '12x8' in msg and '10x8' in msg


def test_a_shard_smaller_than_one_batch_names_the_counts(tmp_path):
  from wlseg import train_input
  split = cityscapes_train(str(tmp_path), 7)
  # --distribute over 4 ranks: a per-rank batch of 4 / 4 = 1 and shards of at least 1 file.  Two ranks without
  # --distribute each take batches of 4, but the smaller shard holds 7 // 2 = 3 files
  train_input.train_input_fn(None, train_settings(split, Nb_per_pixel=4, distribute=True, world_size=4, rank=3))
  msg = _refusal(lambda: train_input.train_input_fn(None, train_settings(split, Nb_per_pixel=4, world_size=2, rank=1)))
  assert '7' in msg and 'has 3' in msg and 'batch of 4' in msg


def test_an_out_of_range_label_id_names_the_file(tmp_path):
  from wlseg import train_input
  rng = np.random.default_rng(5)
  bad = _lids(rng, 16, 24, 34)
  bad[3, 5] = 34                                    # Cityscapes has 34 label ids: 0..33
  split = write_cityscapes(str(tmp_path), [('ulm', 'a', Image.fromarray(_rgb(rng, 16, 24)), _lids(rng, 16, 24, 34)),
                                           ('ulm', 'b', Image.fromarray(_rgb(rng, 16, 24)), bad)], split='train')
  msg = _refusal(lambda: train_input.train_input_fn(None, train_settings(split)))
  assert 'b_gtFine_labelIds.png' in msg and 'label id 34' in msg and '34 label ids' in msg


def test_an_arena_over_the_budget_is_refused_before_decoding(tmp_path, monkeypatch):
  from wlseg import dataset_input, train_input
  split = cityscapes_train(str(tmp_path), 4)
  pairs = train_input.split_pairs(split, 'cityscapes')
  sizes, _, _ = dataset_input.check_pairs(pairs)
  need = sum(h * w * 4 for h, w in sizes)
  monkeypatch.setattr(dataset_input, '_decode_image', lambda p: pytest.fail('decoded before the budget check'))
  msg = _refusal(lambda: train_input.Shard(pairs, sizes, 34, 'cpu', budget=need - 1))
  assert f'needs {need} bytes' in msg and f'{need - 1} are available' in msg and 'more ranks' in msg
  monkeypatch.setattr(train_input, 'device_budget', lambda device: need - 1)
  msg = _refusal(lambda: train_input.train_input_fn(None, train_settings(split)))
  assert f'needs {need} bytes' in msg


# ------------------------------------------------------------------------------------------------ arena
@pytest.mark.parametrize('dataset', ['cityscapes', 'vistas'])
def test_arena_bytes_and_offsets_equal_a_direct_decode(tmp_path, dataset):
  from wlseg import dataset_input, train_input
  split = cityscapes_train(str(tmp_path), 6) if dataset == 'cityscapes' else vistas_train(str(tmp_path), 5)
  pairs = train_input.split_pairs(split, dataset)
  sizes, _, _ = dataset_input.check_pairs(pairs)
  shard = train_input.Shard(pairs, sizes, len(_lut(dataset)), 'cpu', workers=2)
  assert shard.arena.device.type == 'cpu' and shard.files == len(pairs)
  off = 0
  for e, pair in enumerate(pairs):
    im, ids = _decode(pair)
    h, w = ids.shape
    assert int(shard.offsets[e]) == off and shard.sizes[e].tolist() == [h, w]
    assert np.array_equal(shard.arena[off:off + h * w * 3].numpy(), im.reshape(-1))
    assert np.array_equal(shard.arena[off + h * w * 3:off + h * w * 4].numpy(), ids.reshape(-1))
    off += h * w * 4
  assert shard.arena.numel() == shard.bytes == off


# ------------------------------------------------------------------------------------------------ order
def test_each_epoch_is_a_permutation_of_the_shard_with_the_remainder_dropped():
  from wlseg import train_input
  n, world, Nb = 23, 2, 3                    # shards of 12 and 11; 11 // 3 = 3 batches per epoch on every rank
  assert train_input.steps_per_epoch(n, world, Nb) == 3
  for rank, shard in ((0, 12), (1, 11)):
    orders = [train_input.epoch_order(7, rank, world, n, Nb, e) for e in range(4)]
    for o in orders:
      assert len(o) == 9 and len(set(o.tolist())) == 9 and set(o.tolist()) <= set(range(shard))
    assert len({tuple(o) for o in orders}) == 4
    steps = [train_input.batch_at(7, rank, world, n, Nb, s) for s in range(12)]
    assert np.array_equal(np.concatenate(steps), np.concatenate(orders))


def test_shards_are_disjoint_and_cover_the_split():
  pairs = list(range(29))
  for world in (1, 2, 3, 8):
    shards = [pairs[r::world] for r in range(world)]
    assert sorted(sum(shards, [])) == pairs
    assert all(f % world == r for r, s in enumerate(shards) for f in s)


def test_the_same_seed_gives_the_same_order_and_another_seed_another():
  from wlseg import train_input
  a = train_input.epoch_order(0, 0, 1, 2975, 4, 0)
  assert len(a) == 743 * 4
  assert np.array_equal(a, train_input.epoch_order(0, 0, 1, 2975, 4, 0))
  assert not np.array_equal(a, train_input.epoch_order(1, 0, 1, 2975, 4, 0))
  assert not np.array_equal(a, train_input.epoch_order(0, 0, 1, 2975, 4, 1))
  assert not np.array_equal(train_input.epoch_order(0, 0, 2, 2975, 2, 0), train_input.epoch_order(0, 1, 2, 2975, 2, 0))


def _take(it, k):
  return [(f['proimages'].clone(), l['prolabels_per_pixel'].clone()) for (f, l), _ in zip(it, range(k))]


def test_input_fn_batches_equal_the_oracle_in_the_stated_order_and_resume_at_any_step(tmp_path, monkeypatch):
  """Contract: ragged sizes, each epoch's permutation, the ring of two outputs; a run resumed at step k feeds exactly
  steps k... of the uninterrupted run, across an epoch boundary."""
  from wlseg import train_input
  emulated_train_inputs(monkeypatch)
  split = cityscapes_train(str(tmp_path), 7)
  pairs = train_input.split_pairs(split, 'cityscapes')
  st = train_settings(split, seed=3)
  with contextlib.redirect_stdout(io.StringIO()) as out:
    full = _take(train_input.train_input_fn(None, st), 8)
  assert 'decoded 7 files into' in out.getvalue() and 'Ntrain = 2975' in out.getvalue()
  lut = _lut('cityscapes')
  for s, (pro, lab) in enumerate(full):
    for j, e in enumerate(train_input.batch_at(3, 0, 1, 7, 2, s)):
      want_pro, want_lab = oracle_example(*_decode(pairs[e]), lut, max(lut), 24, 40)
      assert torch.equal(pro[j], want_pro) and torch.equal(lab[j], want_lab), (s, j)
  for k in (1, 3, 5):                        # 3 batches per epoch: 3 starts epoch 1
    st.initial_global_step = k
    with contextlib.redirect_stdout(io.StringIO()):
      resumed = _take(train_input.train_input_fn(None, st), 8 - k)
    assert all(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) for a, b in zip(resumed, full[k:])), k


def test_sharded_input_fn_feeds_only_its_own_files(tmp_path, monkeypatch):
  from wlseg import train_input
  emulated_train_inputs(monkeypatch)
  split = vistas_train(str(tmp_path), 7)
  pairs = train_input.split_pairs(split, 'vistas')
  lut = _lut('vistas')
  for rank in (0, 1):
    st = train_settings(split, 'vistas', Nb_per_pixel=4, distribute=True, world_size=2, rank=rank)
    with contextlib.redirect_stdout(io.StringIO()) as out:
      (pro, lab), = _take(train_input.train_input_fn(None, st), 1)
    assert f'rank {rank}: decoded {len(pairs[rank::2])} files' in out.getvalue()
    for j, e in enumerate(train_input.batch_at(0, rank, 2, 7, 2, 0)):
      want_pro, want_lab = oracle_example(*_decode(pairs[rank::2][e]), lut, max(lut), 24, 40)
      assert torch.equal(pro[j], want_pro) and torch.equal(lab[j], want_lab)


def test_the_restated_contract_equals_the_oracle_on_ragged_sizes_with_repeated_indices(monkeypatch):
  from wlseg import ops, train_input
  emulated_train_inputs(monkeypatch)
  rng = np.random.default_rng(11)
  lut = _lut('vistas')
  shapes = [(31, 45), (97, 211), (20, 17), (64, 128)]
  examples = [(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), rng.integers(0, 66, (h, w), dtype=np.uint8))
              for h, w in shapes]
  offsets, total = train_input.arena_layout(shapes)
  arena = torch.zeros(total, dtype=torch.uint8)
  for (im, ids), o in zip(examples, offsets):
    arena[o:o + im.size] = torch.from_numpy(im.reshape(-1))
    arena[o + im.size:o + im.size + ids.size] = torch.from_numpy(ids.reshape(-1))
  index = torch.tensor([2, 0, 2, 3, 1, 0], dtype=torch.int32)
  pro = torch.zeros(6, 24, 32, 3)
  lab = torch.zeros(6, 24, 32, dtype=torch.int32)
  invalid = torch.zeros(1, dtype=torch.int64)
  ops.train_inputs(arena, torch.from_numpy(offsets), torch.tensor(shapes, dtype=torch.int32), index,
                   torch.tensor(lut, dtype=torch.int32), max(lut), (24, 32), pro, lab, invalid)
  assert int(invalid) == 0
  for n, e in enumerate(index.tolist()):
    want_pro, want_lab = oracle_example(*examples[e], lut, max(lut), 24, 32)
    assert torch.equal(pro[n], want_pro) and torch.equal(lab[n], want_lab)


# ------------------------------------------------------------------------------------------------ train.py
def _train_main_choice(monkeypatch, tmp_path, extra):
  from wlseg import cli

  class Stop(Exception):
    pass
  chosen = []

  def fake_system(input_fns, model_fn, settings):
    chosen.append(input_fns['train'])
    raise Stop()

  def dist_env(st):
    st.rank, st.world_size, st.device = 0, 1, 'cpu'
    return st
  monkeypatch.setattr(cli, '_dist_env', dist_env)
  monkeypatch.setattr(cli, 'SemanticSegmentation', fake_system)
  out = io.StringIO()
  with contextlib.redirect_stdout(out), pytest.raises(Stop):
    cli.train_main([str(tmp_path / 'log'), 'cityscapes'] + extra)
  return chosen[0], out.getvalue()


@pytest.mark.parametrize('extra', ['none', 'synthetic_flag'])
def test_train_main_without_the_split_flag_takes_the_synthetic_input(monkeypatch, tmp_path, extra):
  from wlseg import synthetic
  split = cityscapes_train(str(tmp_path / 'data'), 4)
  argv = [] if extra == 'none' else ['--per_pixel_split_path', split, '--synthetic']
  fn, out = _train_main_choice(monkeypatch, tmp_path, argv)
  assert fn is synthetic.train_input_fn and out == ''


def test_train_main_with_the_split_flag_takes_the_split(monkeypatch, tmp_path):
  from wlseg import train_input
  split = cityscapes_train(str(tmp_path / 'data'), 4)
  fn, out = _train_main_choice(monkeypatch, tmp_path, ['--per_pixel_split_path', split])
  assert fn is train_input.train_input_fn
  assert f'cityscapes split at {split}: 4 image / label pairs' in out and 'no Open Images source' in out


def test_training_from_a_checkpoint_hands_its_step_to_the_input_function(tmp_path, monkeypatch):
  """Estimator.initialize(for_training=True) leaves the restored global step on the settings the input function gets."""
  from tests.test_eval_dataset_cpu import _checkpoint
  from tests.test_host_orchestration_cpu import _emulated_ops
  _emulated_ops(monkeypatch)
  from wlseg import estimator as est, hierarchy, problem_defs, settings as wsettings
  log_dir = tmp_path / 'log'
  log_dir.mkdir()
  _checkpoint(log_dir, 'cityscapes')             # model.ckpt-7.pt
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(
      [str(log_dir), 'cityscapes', '--dtype', 'fp32']))
  hier = hierarchy.Hierarchy('cityscapes', problem_defs.cityscapes()['cids2labels'])
  est.Estimator(st, hier, device='cpu').initialize(log_dir=str(log_dir), for_training=True)
  assert st.initial_global_step == 7
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(
      [str(tmp_path / 'fresh'), 'cityscapes', '--dtype', 'fp32']))
  est.Estimator(st, hier, device='cpu').initialize(log_dir=str(tmp_path / 'fresh'), for_training=True)
  assert st.initial_global_step == 0
