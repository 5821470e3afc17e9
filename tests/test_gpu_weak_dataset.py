"""wlseg_weak_train_inputs (csrc/preproc.cu) against wlseg_resize_crop of wlseg_rasterize_bbox_labels, against
wlseg_tile_image_labels and against the oracle, bit for bit; the CSV loader against the reference's `_generate_rla`; and
train.py on a Cityscapes split plus an Open Images split against the same training fed host-built batches."""

import contextlib
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

from tests.test_eval_dataset_cpu import _rgb
from tests.test_gpu_eval_dataset import _bits_equal
from tests.test_gpu_train_dataset import _cityscapes_split, _host_batches
from tests.test_weak_dataset_cpu import HERE, _decode, oracle_weak_example, random_open_images, write_open_images

pytestmark = pytest.mark.gpu


def _launch(cuda, imgs, boxes, vectors, index, crops, th, tw):
  """-> (proimages, labels, invalid) of one wlseg_weak_train_inputs launch; boxes: per example [(cid, (x0, x1, y0, y1))]
  (bbox part) or None (image part, `vectors` [E, 15])."""
  from wlseg import ops, preprocess, train_input
  shapes = [im.shape[:2] for im in imgs]
  offsets, _ = train_input.arena_layout(shapes, 3)
  arena = torch.from_numpy(np.concatenate([im.reshape(-1) for im in imgs])).to(cuda)
  resized = [preprocess.resized_size(h, w, (th, tw), True) for h, w in shapes]
  kw = {}
  if boxes is not None:
    start = np.cumsum([0] + [len(b) for b in boxes]).astype(np.int32)
    flat = [b for bs in boxes for b in bs]
    kw['boxes'] = (torch.from_numpy(start).to(cuda),
                   torch.tensor([b[1] for b in flat], dtype=torch.float32).reshape(-1, 4).to(cuda),
                   torch.tensor([b[0] for b in flat], dtype=torch.int32).to(cuda))
  else:
    kw['vectors'] = torch.from_numpy(np.asarray(vectors, dtype=np.float32)).to(cuda)
  n = len(index)
  pro = torch.full((n, th, tw, 3), -7.0, device=cuda)
  lab = torch.full((n, th, tw, 15), -7.0, device=cuda)
  invalid = torch.zeros(1, dtype=torch.int64, device=cuda)
  ops.weak_train_inputs(arena, torch.from_numpy(offsets).to(cuda), torch.tensor(shapes, dtype=torch.int32).to(cuda),
                        torch.tensor(resized, dtype=torch.int32).to(cuda), torch.tensor(index, dtype=torch.int32).to(cuda),
                        torch.tensor(crops, dtype=torch.int32).reshape(-1, 2).to(cuda), (th, tw), pro, lab, invalid, **kw)
  torch.cuda.synchronize()
  return pro.cpu(), lab.cpu(), int(invalid.item()), resized


# target, example sizes (smaller than, taller and wider than the target, equal to it, odd), boxes per example: edge,
# overlapping, degenerate (one pixel, zero width), unknown cids (-1, 15), an example without a valid box
TARGETS = [(23, 37), (64, 128), (61, 85)]
SHAPES = [(11, 19), (97, 40), (30, 150), (64, 128), (301, 257)]
BOXES = [[(2, (0.0, 1.0, 0.0, 1.0)), (6, (0.2, 0.7, 0.1, 0.9))],
         [(1, (0.5, 0.5, 0.5, 0.5)), (2, (0.0, 0.3, 0.9, 1.0)), (2, (0.1, 0.3, 0.0, 0.4)), (15, (0, 1, 0, 1))],
         [(13, (0.99, 1.0, 0.0, 0.01)), (7, (0.25, 0.25, 0.0, 1.0)), (7, (0.0, 1.0, 0.3, 0.3))],
         [(-1, (0.0, 1.0, 0.0, 1.0))],
         [(c % 14, (0.01 * c, 0.5 + 0.01 * c, 0.02 * c, 0.3 + 0.02 * c)) for c in range(30)]]


@pytest.mark.parametrize('target', TARGETS)
def test_weak_train_inputs_is_bit_equal_to_rasterise_resize_crop_tile_and_the_oracle(cuda, target):
  from wlseg import ops
  th, tw = target
  rng = np.random.default_rng(th)
  imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in SHAPES]
  vectors = [np.float32([1.0 if c in cs else 0.0 for c in range(15)]) / len(cs)
             for cs in ({0}, {3, 9}, {1, 2, 13}, {6}, {4, 5, 11, 12})]
  index = [0, 1, 2, 3, 4, 1, 4, 2]
  _, _, _, resized = _launch(cuda, imgs, None, vectors, [0], [(0, 0)], th, tw)
  # offsets 0, max and middle on the axis with room
  crops = []
  for k, e in enumerate(index):
    extra = (resized[e][0] - th, resized[e][1] - tw)
    crops.append(tuple((0, x, x // 2)[k % 3] for x in extra))
  pro, lab, invalid, _ = _launch(cuda, imgs, BOXES, None, index, crops, th, tw)
  vpro, vlab, vinvalid, _ = _launch(cuda, imgs, None, vectors, index, crops, th, tw)
  assert invalid == 0 and vinvalid == 0
  assert _bits_equal(pro, vpro)                        # the image arithmetic does not depend on the part
  for k, (e, off) in enumerate(zip(index, crops)):
    h, w = SHAPES[e]
    coords = torch.tensor([[b[1] for b in BOXES[e]]], dtype=torch.float32, device=cuda)
    cids = torch.tensor([[b[0] for b in BOXES[e]]], dtype=torch.int32, device=cuda)
    dense = ops.rasterize_bbox_labels(coords, cids, h, w)
    want = ops.resize_crop(dense, resized[e], off, (th, tw), 'nearest')[0].cpu()
    assert torch.equal(lab[k], want), k
    tiled = ops.tile_image_labels(torch.from_numpy(vectors[e])[None].to(cuda), th, tw)[0].cpu()
    assert torch.equal(vlab[k], tiled), k
    known = [(c, xy) for c, xy in BOXES[e] if 0 <= c < 15]
    want_pro, want_lab = oracle_weak_example(imgs[e], known, None, (th, tw), off)
    assert _bits_equal(pro[k], want_pro), (k, float((pro[k] - want_pro).abs().max()))
    assert torch.equal(lab[k], want_lab), k
  assert bool((lab[index.index(3)][..., 14] == 1).all())        # no valid box: void everywhere


def test_invalid_indices_and_crops_are_counted_and_write_nothing(cuda):
  rng = np.random.default_rng(3)
  imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ((40, 90), (80, 50))]
  boxes = [[(2, (0.1, 0.6, 0.1, 0.6))], [(6, (0.0, 1.0, 0.0, 1.0))]]
  th, tw = 32, 48
  _, _, _, resized = _launch(cuda, imgs, boxes, None, [0], [(0, 0)], th, tw)
  index = [0, 2, -1, 1, 0, 1]
  crops = [(0, 0), (0, 0), (0, 0), (resized[1][0] - th + 1, 0), (0, resized[0][1] - tw + 1), (-1, 0)]
  for kw in ({'boxes': boxes, 'vectors': None}, {'boxes': None, 'vectors': [np.eye(15, dtype=np.float32)[2]] * 2}):
    pro, lab, invalid, _ = _launch(cuda, imgs, kw['boxes'], kw['vectors'], index, crops, th, tw)
    assert invalid == 5
    assert not bool((pro[0] == -7).all()) and not bool((lab[0] == -7).all())
    for k in range(1, 6):
      assert bool((pro[k] == -7).all()) and bool((lab[k] == -7).all()), k


def test_an_example_over_the_box_cap_is_counted_and_writes_nothing(cuda):
  """The loader refuses images with more than 1024 boxes; the kernel counts such an example and leaves it alone."""
  rng = np.random.default_rng(5)
  imgs = [rng.integers(0, 256, (40, 60, 3), dtype=np.uint8)] * 2
  boxes = [[(2, (0.1, 0.6, 0.1, 0.6))] * 1024, [(6, (0.0, 1.0, 0.0, 1.0))] * 1025]
  pro, lab, invalid, _ = _launch(cuda, imgs, boxes, None, [0, 1], [(0, 0), (0, 0)], 32, 48)
  assert invalid == 1
  assert float(lab[0][..., 2].max()) == 1.0
  assert bool((pro[1] == -7).all()) and bool((lab[1] == -7).all())


def test_the_csv_loader_and_the_kernel_reproduce_generate_rla(cuda, tmp_path):
  """The reference's `_generate_rla` on five boxes of Car, Car, Bus, Person and an unknown MID at 20 x 28
  (tests/golden/reference_run.npz): read from an Open Images CSV split and gathered at identity size."""
  from wlseg import weak_input
  gold = np.load(os.path.join(HERE, 'golden', 'reference_run.npz'))
  h, w = (int(x) for x in gold['rla/size'])
  names = ['Car', 'Car', 'Bus', 'Person', 'Nothing']
  boxes = [('x', n) + tuple(float(v) for v in xy) for n, xy in zip(names, gold['rla/coords'])]
  root = write_open_images(str(tmp_path), [('x', Image.fromarray(_rgb(np.random.default_rng(0), h, w)))], boxes)
  part = weak_input.WeakPart('bbox', root, 1, (h, w), 0, 1, 0)
  assert part.resized == [(h, w)] and part.box_cids.tolist() == [2, 2, 1, 6]
  with contextlib.redirect_stdout(io.StringIO()):
    part.fill(cuda)
  pro = torch.empty((1, h, w, 3), device=cuda)
  lab = torch.empty((1, h, w, 15), device=cuda)
  part.gather(0, pro, lab)
  torch.cuda.synchronize()
  assert int(part.invalid.item()) == 0
  assert np.array_equal(lab[0].cpu().numpy(), gold['rla/out'])


def _mixed_host_batches(pairs, parts, labels, steps, seed, hw):
  """The mixed batches train_input feeds at steps 0..steps-1, built on the host from the same files."""
  out = []
  for s, (f, l) in enumerate(_host_batches(pairs, 'cityscapes', steps, 4, seed, hw)):
    pro = [f['proimages']]
    for part in parts:
      order, crops = part.batch_at(s)
      ex = []
      for e, off in zip(order, crops):
        image_id = part.ids[e]
        boxes = [(b[0], b[1:]) for b in labels['bbox'][image_id]] if part.part == 'bbox' else None
        ex.append(oracle_weak_example(_decode(part.paths[e]), boxes, None if boxes else part.vectors[e], hw, tuple(off)))
      pro.append(torch.stack([p for p, _ in ex]))
      l[part.label_key] = torch.stack([d for _, d in ex])
    f['proimages'] = torch.cat(pro)
    out.append((f, l))
  return out


def test_train_main_on_cityscapes_and_open_images_equals_host_built_batches(cuda, tmp_path, monkeypatch):
  """train.py --per_pixel_split_path + --per_bbox_split_path + --per_image_split_path (one Open Images directory),
  4 + 8 + 4 at 512 x 1024 (bf16 product path), 6 steps across every part's epoch boundary, against the same training fed
  the host-built batches.  Every step's inputs are bit-equal; step 1 sees bit-equal inputs and weights, so its losses
  agree to 1e-6; later total losses to 1e-2, as tests/test_gpu_train_dataset.py explains.  The L2 vehicle and human
  losses are not zero: the weak labels reach the loss."""
  from wlseg import cli, settings as wsettings, train_input, trainer as wtrainer, weak_input
  from wlseg.system_factory import SemanticSegmentation
  split = _cityscapes_split(str(tmp_path / 'data'), 16, 384, 768)
  oi = random_open_images(str(tmp_path / 'oi'), 13, seed=9, sizes=((480, 640), (640, 480), (360, 900), (512, 1024)),
                          max_boxes=8)
  argv = [str(tmp_path / 'log'), 'cityscapes', '--per_pixel_split_path', split, '--per_bbox_split_path', oi,
          '--per_image_split_path', oi, '--steps', '6', '--seed', '5']
  consumed = []
  step = wtrainer.Trainer.step

  def capturing_step(self, features, labels, lr):
    consumed.append((features['proimages'].clone(), {k: v.clone() for k, v in labels.items()}))
    return step(self, features, labels, lr)
  monkeypatch.setattr(wtrainer.Trainer, 'step', capturing_step)
  out = io.StringIO()
  with contextlib.redirect_stdout(out):
    got = cli.train_main(argv)
  monkeypatch.setattr(wtrainer.Trainer, 'step', step)
  assert 'bbox part: ' in out.getvalue() and 'image part: ' in out.getvalue()
  assert got.shape == (6, 6) and np.isfinite(got).all()
  hw = (512, 1024)
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(argv[:2] + argv[2:8] + ['--seed', '5']))
  parts = weak_input.parts(st, hw, 0, 1)
  assert [p.Nb for p in parts] == [8, 4] and parts[0].steps_per_epoch == 1 and parts[1].steps_per_epoch == 3
  labels = {'bbox': weak_input.read_part('bbox', oi)[1]}
  batches = _mixed_host_batches(train_input.split_pairs(split, 'cityscapes'), parts, labels, 6, 5, hw)
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(
      [str(tmp_path / 'log_host'), 'cityscapes', '--steps', '6', '--seed', '5']))
  st.device, st.rank, st.world_size = str(cuda), 0, 1
  with contextlib.redirect_stdout(io.StringIO()):
    want = SemanticSegmentation({'train': lambda config, params: iter(batches)}, None, st).train()
  assert len(consumed) == 6
  for i, ((pro, lab), (f, l)) in enumerate(zip(consumed, batches)):
    assert _bits_equal(pro.cpu(), f['proimages']), i
    assert set(lab) == set(l) and all(torch.equal(lab[k].cpu(), l[k]) for k in l), i
  print('from the arenas', got.tolist(), 'host-built', want.tolist())
  np.testing.assert_allclose(got[0], want[0], rtol=1e-6, atol=1e-7)
  np.testing.assert_allclose(got[1:, 0], want[1:, 0], rtol=1e-2)
  assert (got[:, 3] > 0).all() and (got[:, 4] > 0).all()


def test_mixed_step_at_an_odd_size_equals_the_oracle(cuda, tmp_path):
  """One 1 + 1 + 1 Cityscapes + Open Images step at 201 x 299 (no multiple of 8) through the arenas, fp32 check mode:
  the five losses equal oracle/train.py on the same inputs (1e-4)."""
  from oracle import network as onet
  from oracle import train as otrain
  from wlseg import estimator as est, hierarchy, settings as wsettings, system_factory, train_input
  split = _cityscapes_split(str(tmp_path / 'data'), 2, 256, 320)
  oi = random_open_images(str(tmp_path / 'oi'), 2, seed=4, sizes=((300, 420), (250, 260)), max_boxes=6)
  st = wsettings.train_extra_args(wsettings.build_parser(wsettings.TRAIN).parse_args(
      [str(tmp_path / 'fp32'), 'cityscapes', '--per_pixel_split_path', split, '--per_bbox_split_path', oi,
       '--per_image_split_path', oi, '--dtype', 'fp32', '--learning_rate_values', '0.01', '0.01', '0.01', '0.01']))
  st.Nb_per_pixel = st.Nb = st.Nb_per_bbox = st.Nb_per_image = 1
  st.height_feature_extractor, st.width_feature_extractor = 201, 299
  st.device, st.rank, st.world_size, st.save_checkpoints = str(cuda), 0, 1, False
  system_factory.attach_problem_definitions(st)
  hier = hierarchy.Hierarchy('cityscapes', st.training_problem_def['cids2labels'])
  e = est.Estimator(st, hier, device=cuda)
  e.initialize(for_training=True)
  tf_params = onet.init_params('cityscapes', seed=4, randomize_bn=True, tame=True)
  e.params.load_tf_dict(tf_params)
  inputs = []
  it = train_input.train_input_fn(None, st)

  def first(it):
    f, l = next(it)
    inputs.append((f['proimages'].clone().cpu(), {k: v.clone().cpu() for k, v in l.items()}))
    yield f, l
  with contextlib.redirect_stdout(io.StringIO()):
    got = e.train(first(it), 1)[0]
  images, labels = inputs[0]
  assert images.shape == (3, 201, 299, 3) and labels['prolabels_per_bbox'].shape == (1, 201, 299, 15)
  state = otrain.TrainState(tf_params, ema_decay=st.ema_decay, optimizer=st.optimizer)
  ref = otrain.train_step(state, images, labels, 'cityscapes', 0.01, momentum=st.momentum, nesterov=st.use_nesterov,
                          regularization_weight=st.regularization_weight, bn_decay=st.batch_norm_decay)
  want = [ref[k] for k in ('total', 'l1_segmentation', 'l2_vehicle_segmentation', 'l2_human_segmentation', 'regularization')]
  print('fp32', got.tolist(), 'oracle', want)
  np.testing.assert_allclose(got[[0, 2, 3, 4, 5]], want, rtol=1e-4, atol=1e-6)
