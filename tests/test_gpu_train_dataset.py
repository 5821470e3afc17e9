"""wlseg_train_inputs (csrc/preproc.cu) against the oracle and wlseg_eval_inputs, bit for bit, and train.py on Cityscapes
/ Vistas training splits read from disk against the same training fed batches preprocessed on the host."""

import contextlib
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

from tests.test_eval_dataset_cpu import _lids, _rgb, write_cityscapes
from tests.test_gpu_eval_dataset import _bits_equal, _pack
from tests.test_train_dataset_cpu import _decode, _lut, oracle_example, vistas_train

pytestmark = pytest.mark.gpu


def _arena(cuda, examples):
  from wlseg import train_input
  shapes = [lab.shape for _, lab in examples]
  offsets, total = train_input.arena_layout(shapes)
  arena = torch.zeros(total, dtype=torch.uint8)
  for (im, lab), o in zip(examples, offsets):
    arena[o:o + im.size] = torch.from_numpy(im.reshape(-1))
    arena[o + im.size:o + im.size + lab.size] = torch.from_numpy(lab.reshape(-1))
  return arena.to(cuda), torch.from_numpy(offsets).to(cuda), torch.tensor(shapes, dtype=torch.int32).to(cuda)


def _run(cuda, examples, index, lut, th, tw):
  from wlseg import ops
  arena, offsets, sizes = _arena(cuda, examples)
  n = len(index)
  pro = torch.full((n, th, tw, 3), -7.0, dtype=torch.float32, device=cuda)
  lab = torch.full((n, th, tw), -7, dtype=torch.int32, device=cuda)
  invalid = torch.zeros(1, dtype=torch.int64, device=cuda)
  ops.train_inputs(arena, offsets, sizes, torch.tensor(index, dtype=torch.int32, device=cuda),
                   torch.tensor(lut, dtype=torch.int32, device=cuda), max(lut), (th, tw), pro, lab, invalid)
  torch.cuda.synchronize()
  return pro.cpu(), lab.cpu(), int(invalid.item())


def _eval_kernel(cuda, examples, lut, th, tw):
  from wlseg import ops
  images, lids, sizes = _pack(examples)
  n = len(examples)
  pro = torch.empty((n, th, tw, 3), dtype=torch.float32, device=cuda)
  lab = torch.empty((n, th, tw), dtype=torch.int32, device=cuda)
  invalid = torch.zeros(1, dtype=torch.int64, device=cuda)
  ops.eval_inputs(images.to(cuda), lids.to(cuda), sizes.to(cuda), torch.tensor(lut, dtype=torch.int32, device=cuda),
                  max(lut), (th, tw), pro, lab, invalid)
  torch.cuda.synchronize()
  return pro.cpu(), lab.cpu()


# (dataset, target, [example sizes], index): ragged and odd sizes, one smaller than the target, a full-size
# 1024 x 2048 -> 512 x 1024 batch, repeated and permuted indices
CASES = [
    ('cityscapes', (64, 128), [(97, 211), (64, 128), (31, 45)], [2, 0, 1, 0]),
    ('vistas', (61, 85), [(150, 201), (45, 60), (257, 129), (19, 23)], [3, 3, 1, 2, 0]),
    ('cityscapes', (512, 1024), [(1024, 2048)] * 3, [1, 2, 0, 1]),
]


@pytest.mark.parametrize('case', range(len(CASES)))
def test_train_inputs_is_bit_equal_to_the_oracle_and_to_eval_inputs(cuda, case):
  dataset, (th, tw), shapes, index = CASES[case]
  lut = _lut(dataset)
  rng = np.random.default_rng(200 + case)
  examples = [(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), rng.integers(0, len(lut), (h, w), dtype=np.uint8))
              for h, w in shapes]
  pro, lab, invalid = _run(cuda, examples, index, lut, th, tw)
  assert invalid == 0
  eval_pro, eval_lab = _eval_kernel(cuda, [examples[e] for e in index], lut, th, tw)
  assert _bits_equal(pro, eval_pro) and torch.equal(lab, eval_lab)
  for e in sorted(set(index)):
    want_pro, want_lab = oracle_example(*examples[e], lut, max(lut), th, tw)
    for n in [n for n, i in enumerate(index) if i == e]:
      assert _bits_equal(pro[n], want_pro), (n, float((pro[n] - want_pro).abs().max()))
      assert torch.equal(lab[n], want_lab), n


def test_out_of_range_indices_and_label_ids_are_counted(cuda):
  lut = _lut('cityscapes')
  rng = np.random.default_rng(8)
  a = rng.integers(0, 34, (40, 56), dtype=np.uint8)
  b = rng.integers(0, 34, (29, 77), dtype=np.uint8)
  a[3:7, 10:15] = 34                       # first id past the 34-entry table: 20 sampled pixels at 40 x 56
  ims = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in (a.shape, b.shape)]
  pro, lab, invalid = _run(cuda, [(ims[0], a), (ims[1], b)], [1, -1, 0, 2], lut, 40, 56)
  assert invalid == 2 + 20
  for n in (1, 3):                         # indices -1 and 2 (past the 2 arena examples) write nothing
    assert bool((pro[n] == -7.0).all()) and bool((lab[n] == -7).all())
  for n, (im, ids) in ((0, (ims[1], b)), (2, (ims[0], a))):
    want_pro, want_lab = oracle_example(im, ids, lut, max(lut), 40, 56)
    assert _bits_equal(pro[n], want_pro) and torch.equal(lab[n], want_lab)
  assert int((lab[2] == max(lut)).sum()) >= 20


def _cityscapes_split(root, n, h, w):
  rng = np.random.default_rng(21)
  return write_cityscapes(root, [(('aachen', 'bochum')[i % 2], f't_{i:03d}', Image.fromarray(_rgb(rng, h, w)),
                                  _lids(rng, h, w, 34, block=32)) for i in range(n)], split='train')


def _host_batches(pairs, dataset, steps, Nb, seed, hw):
  """The batches train_input feeds at steps 0..steps-1, preprocessed on the host from the same files."""
  from wlseg import train_input
  lut = _lut(dataset)
  out = []
  for s in range(steps):
    ex = [oracle_example(*_decode(pairs[e]), lut, max(lut), *hw) for e in train_input.batch_at(seed, 0, 1, len(pairs), Nb, s)]
    out.append(({'proimages': torch.stack([p for p, _ in ex])}, {'prolabels_per_pixel': torch.stack([l for _, l in ex])}))
  return out


def test_train_main_on_a_cityscapes_split_equals_host_preprocessed_batches(cuda, tmp_path, monkeypatch):
  """train.py --per_pixel_split_path on 16 pairs, 4 x 512 x 1024 (bf16 product path), 6 steps across an epoch
  boundary, against the same training fed the host-preprocessed batches in the same order.  What every step consumes
  (captured on the step's stream as Trainer.step is entered, after the next batch's gather is already enqueued) equals
  the host batches bit for bit.  Step 1 sees bit-equal inputs and weights: its losses agree to 1e-6.  Later steps start
  from weights that went through float atomics in the loss and gradient sums, and from random init this network
  amplifies that (two runs of one build agree to 1e-2 on the losses, bench.py --dump-outputs): the total loss is held to
  1e-2.  Measured on a B200 over steps 2-6 in two runs: total 4e-4 and 1.2e-3, while the l2 human / vehicle losses,
  averaged over few pixels, moved by up to 5 %."""
  from wlseg import cli, settings as wsettings, trainer as wtrainer
  from wlseg.system_factory import SemanticSegmentation
  split = _cityscapes_split(str(tmp_path / 'data'), 16, 384, 768)
  log_dir = tmp_path / 'log'
  argv = [str(log_dir), 'cityscapes', '--per_pixel_split_path', split, '--steps', '6', '--seed', '5']
  consumed = []
  step = wtrainer.Trainer.step

  def capturing_step(self, features, labels, lr):
    consumed.append((features['proimages'].clone(), labels['prolabels_per_pixel'].clone()))
    return step(self, features, labels, lr)
  monkeypatch.setattr(wtrainer.Trainer, 'step', capturing_step)
  out = io.StringIO()
  with contextlib.redirect_stdout(out):
    got = cli.train_main(argv)
  monkeypatch.setattr(wtrainer.Trainer, 'step', step)
  assert 'cityscapes split at' in out.getvalue() and 'decoded 16 files' in out.getvalue()
  assert got.shape == (6, 6) and np.isfinite(got).all()
  assert os.path.isfile(str(log_dir / 'model.ckpt-6.pt'))
  from wlseg import train_input
  pairs = train_input.split_pairs(split, 'cityscapes')
  batches = _host_batches(pairs, 'cityscapes', 6, 4, 5, (512, 1024))
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(
      [str(tmp_path / 'log_host'), 'cityscapes', '--steps', '6', '--seed', '5']))
  st.device, st.rank, st.world_size = str(cuda), 0, 1
  with contextlib.redirect_stdout(io.StringIO()):
    want = SemanticSegmentation({'train': lambda config, params: iter(batches)}, None, st).train()
  assert len(consumed) == 6
  for i, ((pro, lab), (f, l)) in enumerate(zip(consumed, batches)):
    assert _bits_equal(pro.cpu(), f['proimages']) and torch.equal(lab.cpu(), l['prolabels_per_pixel']), i
  print('from the arena', got.tolist(), 'host-preprocessed', want.tolist())
  np.testing.assert_allclose(got[0], want[0], rtol=1e-6, atol=1e-7)
  np.testing.assert_allclose(got[1:, 0], want[1:, 0], rtol=1e-2)


def _vistas_estimator(cuda, tmp_path, dtype, split, tf_params):
  from wlseg import estimator as est, hierarchy, settings as wsettings, system_factory
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(
      [str(tmp_path), 'vistas', '--per_pixel_split_path', split, '--dtype', dtype, '--learning_rate_values', '0.01',
       '0.01', '0.01', '0.01']))
  st.Nb_per_pixel = st.Nb = 1
  st.device, st.rank, st.world_size, st.save_checkpoints = str(cuda), 0, 1, False
  system_factory.attach_problem_definitions(st)
  hier = hierarchy.Hierarchy('vistas', st.training_problem_def['cids2labels'])
  e = est.Estimator(st, hier, device=cuda)
  e.initialize(for_training=True)
  e.params.load_tf_dict(tf_params)
  return st, e


def test_vistas_step_at_621x855_equals_the_oracle(cuda, tmp_path):
  """One Vistas step at train.py's size 621 x 855 (no multiple of 8) through the arena input, per-rank batch of 1, fp32
  check mode: the five losses equal oracle/train.py on the same preprocessed example (1e-4).  The bf16 step is finite."""
  from oracle import network as onet
  from oracle import train as otrain
  from wlseg import train_input
  split = vistas_train(str(tmp_path / 'data'), 2, sizes=((700, 1000), (480, 640)))
  tf_params = onet.init_params('vistas', seed=4, randomize_bn=True, tame=True)
  st, e = _vistas_estimator(cuda, tmp_path / 'fp32', 'fp32', split, tf_params)
  with contextlib.redirect_stdout(io.StringIO()):
    got = e.train(train_input.train_input_fn(None, st), 1)[0]
  pairs = train_input.split_pairs(split, 'vistas')
  (features, labels), = _host_batches(pairs, 'vistas', 1, 1, st.seed, (621, 855))
  state = otrain.TrainState(tf_params, ema_decay=st.ema_decay, optimizer=st.optimizer)
  ref = otrain.train_step(state, features['proimages'], labels, 'vistas', 0.01, momentum=st.momentum,
                          nesterov=st.use_nesterov, regularization_weight=st.regularization_weight,
                          bn_decay=st.batch_norm_decay)
  want = [ref[k] for k in ('total', 'l1_segmentation', 'l2_vehicle_segmentation', 'l2_human_segmentation', 'regularization')]
  print('fp32', got.tolist(), 'oracle', want)
  np.testing.assert_allclose(got[[0, 2, 3, 4, 5]], want, rtol=1e-4, atol=1e-6)
  st, e = _vistas_estimator(cuda, tmp_path / 'bf16', 'bf16', split, tf_params)
  with contextlib.redirect_stdout(io.StringIO()):
    got = e.train(train_input.train_input_fn(None, st), 2)
  assert np.isfinite(got).all()
