"""wlseg_eval_inputs (csrc/preproc.cu) against the oracle, bit for bit, and evaluate.py on Cityscapes / Vistas splits
read from disk against the same evaluation fed batches preprocessed on the host."""

import contextlib
import io

import numpy as np
import pytest
import torch

from tests.test_eval_dataset_cpu import _checkpoint, _eval_argv, host_batches, mixed_cityscapes, mixed_vistas

pytestmark = pytest.mark.gpu


def _lut(dataset):
  from wlseg import estimator as est, problem_defs
  return est._replacevoids(problem_defs.GENERATORS[dataset]()['lids2cids'])


def _pack(examples, cap_img=None, cap_lab=None):
  """[(uint8 [H, W, 3], uint8 [H, W])] -> packed rows (as wlseg.dataset_input builds them) + sizes."""
  cap_img = cap_img or max(im.size for im, _ in examples)
  cap_lab = cap_lab or max(lab.size for _, lab in examples)
  images = torch.zeros((len(examples), cap_img), dtype=torch.uint8)
  lids = torch.zeros((len(examples), cap_lab), dtype=torch.uint8)
  for n, (im, lab) in enumerate(examples):
    images[n, :im.size] = torch.from_numpy(im.reshape(-1))
    lids[n, :lab.size] = torch.from_numpy(lab.reshape(-1))
  sizes = torch.tensor([lab.shape for _, lab in examples], dtype=torch.int32)
  return images, lids, sizes


def _oracle(im, lab, lut, void_id, th, tw):
  from oracle import preprocess as opre
  img = torch.from_numpy(im)[None].to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
  pro = (opre.resize_bilinear_legacy(img, th, tw)[0] - 0.5) / 0.5
  ids = opre.resize_nearest_legacy(torch.from_numpy(lab)[None], th, tw)[0].long()
  lut = torch.tensor(lut + [void_id], dtype=torch.int32)
  return pro, lut[ids.clamp(max=len(lut) - 1)]


def _run(cuda, examples, lut, void_id, th, tw, cap_img=None, cap_lab=None, sizes=None):
  from wlseg import ops
  images, lids, packed_sizes = _pack(examples, cap_img, cap_lab)
  sizes = packed_sizes if sizes is None else sizes
  n = len(examples)
  pro = torch.full((n, th, tw, 3), -7.0, dtype=torch.float32, device=cuda)
  lab = torch.full((n, th, tw), -7, dtype=torch.int32, device=cuda)
  invalid = torch.zeros(1, dtype=torch.int64, device=cuda)
  ops.eval_inputs(images.to(cuda), lids.to(cuda), sizes.to(cuda), torch.tensor(lut, dtype=torch.int32, device=cuda),
                  void_id, (th, tw), pro, lab, invalid)
  torch.cuda.synchronize()
  return pro.cpu(), lab.cpu(), int(invalid.item())


def _bits_equal(a, b):
  return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# (dataset, target, [example sizes]): ragged batches, odd sizes, down- and up-scaling, N = 1..4
CASES = [
    ('cityscapes', (64, 128), [(1024 // 8, 2048 // 8)]),
    ('cityscapes', (64, 128), [(97, 211), (64, 128), (31, 45)]),
    ('cityscapes', (33, 67), [(128, 256), (37, 83), (200, 101), (33, 67)]),
    ('vistas', (61, 85), [(150, 201), (45, 60)]),
    ('vistas', (64, 96), [(621 // 4, 855 // 4), (19, 23), (64, 96), (257, 129)]),
]


@pytest.mark.parametrize('case', range(len(CASES)))
def test_eval_inputs_is_bit_equal_to_the_oracle(cuda, case):
  dataset, (th, tw), shapes = CASES[case]
  lut = _lut(dataset)
  rng = np.random.default_rng(100 + case)
  examples = [(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), rng.integers(0, len(lut), (h, w), dtype=np.uint8))
              for h, w in shapes]
  pro, lab, invalid = _run(cuda, examples, lut, max(lut), th, tw)
  assert invalid == 0
  for n, (im, ids) in enumerate(examples):
    want_pro, want_lab = _oracle(im, ids, lut, max(lut), th, tw)
    assert _bits_equal(pro[n], want_pro), (n, float((pro[n] - want_pro).abs().max()))
    assert torch.equal(lab[n], want_lab), n


def test_eval_inputs_matches_the_predict_pipeline(cuda):
  """The image half is wlseg/image_input.py's _predict_preprocess restatement, bit for bit."""
  from wlseg import image_input
  lut = _lut('cityscapes')
  rng = np.random.default_rng(7)
  im = rng.integers(0, 256, (123, 301, 3), dtype=np.uint8)
  pro, _, _ = _run(cuda, [(im, np.zeros((123, 301), np.uint8))], lut, max(lut), 64, 128)
  img = torch.from_numpy(im).to(torch.float32) * torch.tensor(1.0 / 255.0, dtype=torch.float32)
  assert _bits_equal(pro[0], (image_input.resize_bilinear_legacy(img, 64, 128) - 0.5) / 0.5)


def test_out_of_range_label_ids_are_counted_and_written_as_void(cuda):
  lut = _lut('cityscapes')
  rng = np.random.default_rng(8)
  a = rng.integers(0, 34, (40, 56), dtype=np.uint8)
  b = rng.integers(0, 34, (29, 77), dtype=np.uint8)
  a[3:7, 10:15] = 34                       # first id past the 34-entry table
  b[:, 41] = 255                           # a sampled column: x = 30 reads floor(30 * 77 / 56) = 41
  ims = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in (a.shape, b.shape)]
  pro, lab, invalid = _run(cuda, [(ims[0], a), (ims[1], b)], lut, max(lut), 40, 56)
  want = [_oracle(im, ids, lut, max(lut), 40, 56) for im, ids in zip(ims, (a, b))]
  from oracle import preprocess as opre
  bad_b = int((opre.resize_nearest_legacy(torch.from_numpy(b)[None], 40, 56) >= 34).sum())
  assert bad_b > 0 and invalid == 20 + bad_b
  assert torch.equal(lab[0], want[0][1]) and torch.equal(lab[1], want[1][1])
  assert int((lab[0] == max(lut)).sum()) >= 20


def test_a_size_row_that_does_not_fit_its_buffers_is_rejected(cuda):
  lut = _lut('vistas')
  rng = np.random.default_rng(9)
  examples = [(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), rng.integers(0, 66, (h, w), dtype=np.uint8))
              for h, w in ((30, 40), (20, 25), (31, 41))]
  sizes = torch.tensor([[30, 40], [20, 25], [31, 41]], dtype=torch.int32)
  # the rows hold 30 x 40 pixels at most: the third example claims more
  pro, lab, invalid = _run(cuda, examples[:2] + [(examples[2][0][:30, :40], examples[2][1][:30, :40])], lut, max(lut),
                           24, 32, sizes=sizes)
  assert invalid == 1
  assert bool((pro[2] == -7.0).all()) and bool((lab[2] == -7).all())
  for n in range(2):
    want_pro, want_lab = _oracle(*examples[n], lut, max(lut), 24, 32)
    assert _bits_equal(pro[n], want_pro) and torch.equal(lab[n], want_lab)
  # a non-positive size is refused the same way
  _, _, invalid = _run(cuda, examples[:1], lut, max(lut), 24, 32, sizes=torch.tensor([[0, 40]], dtype=torch.int32))
  assert invalid == 1


@pytest.mark.parametrize('dataset', ['cityscapes', 'vistas'])
def test_evaluate_main_on_a_split_equals_host_preprocessed_batches(cuda, tmp_path, dataset):
  """evaluate.py on a directory with images of mixed sizes, --Nb 2, 4 steps (the evaluation step graph is captured on
  the second step and replayed after it): the confusion matrix equals, entry by entry, that of the same evaluation fed
  batches preprocessed on the host from the same files."""
  from wlseg import cli, settings as wsettings
  from wlseg.system_factory import SemanticSegmentation
  hw = (64, 128) if dataset == 'cityscapes' else (64, 96)
  if dataset == 'cityscapes':
    split = mixed_cityscapes(str(tmp_path / 'data'), 9, sizes=((128, 256), (97, 211), (48, 64), (200, 300)))
  else:
    split = mixed_vistas(str(tmp_path / 'data'), 9, sizes=((150, 201), (45, 60), (99, 131)))
  log_dir = tmp_path / 'log'
  log_dir.mkdir()
  argv = _eval_argv(log_dir, split, dataset, _checkpoint(tmp_path, dataset), 8, 2, hw)
  argv = [a for a in argv if a not in ('--dtype', 'fp32')]      # the bf16 product path
  with contextlib.redirect_stdout(io.StringIO()):
    got = cli.evaluate_main(argv)
  assert got[0]['steps'] == 4 and (log_dir / 'eval_00' / 'all_metrics.txt').exists()
  batches = host_batches(split, 4, 2, hw, _lut(dataset))
  st = wsettings.eval_extra_args(wsettings.build_parser(wsettings.EVAL).parse_args(argv))
  st.device, st.rank, st.world_size = str(cuda), 0, 1
  with contextlib.redirect_stdout(io.StringIO()):
    want = SemanticSegmentation({'eval': lambda config, params: iter(batches)}, None, st).evaluate()
  assert want[0]['confusion_matrix_int64'].sum() == 8 * hw[0] * hw[1]
  assert np.array_equal(got[0]['confusion_matrix_int64'], want[0]['confusion_matrix_int64'])
