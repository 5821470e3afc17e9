"""Entry points of train.py / evaluate.py / predict.py (code/train.py:24-40, code/evaluate.py:25-67,
code/predict.py:22-169)."""

import os
import pickle
from datetime import datetime

import numpy as np

from wlseg import metrics, settings as wsettings, synthetic
from wlseg.system_factory import SemanticSegmentation


def _dist_env(st):
  """One process per GPU (torchrun): rank / world size from the environment."""
  import torch
  st.rank = int(os.environ.get('RANK', '0'))
  st.world_size = int(os.environ.get('WORLD_SIZE', '1'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  st.device = f'cuda:{local}'
  if torch.cuda.is_available():
    torch.cuda.set_device(local)
  if st.world_size > 1:
    import torch.distributed as dist
    if not dist.is_initialized():
      dist.init_process_group('nccl' if torch.cuda.is_available() else 'gloo')
  return st


def _dist_shutdown(st, system):
  """Multi-rank exit: the step graph holds captured NCCL collectives, so it is dropped and the device
  drained before the process group goes away (destroying the group under a live graph can hang)."""
  if getattr(st, 'world_size', 1) <= 1:
    return
  import torch
  import torch.distributed as dist
  tr = getattr(getattr(system, 'estimator', None), 'trainer', None)
  if tr is not None:
    tr._graphs.clear()
  torch.cuda.synchronize()
  if dist.is_initialized():
    dist.barrier()
    torch.cuda.synchronize()
    dist.destroy_process_group()


def train_main(argv):
  ss = wsettings.build_parser(wsettings.TRAIN)
  st = ss.parse_args(argv)
  # upstream insists on an ImageNet checkpoint path (train.py:31-33); none exists here, so training
  # starts from the random initialisation unless log_dir holds a checkpoint
  wsettings.train_extra_args(st)
  _dist_env(st)
  if st.world_size > 1 and not st.distribute:
    # one process per GPU: without --distribute every rank would train its own unsynchronised model and only rank
    # 0's would be saved.  The reference is one process for all GPUs and needs the flag to use more than one.
    raise ValueError(f'WORLD_SIZE={st.world_size} but --distribute is not set: launch one process, or pass --distribute '
                     'for data-parallel training.')
  input_fn = synthetic.train_input_fn
  weak = [f for f in ('per_bbox_split_path', 'per_image_split_path') if getattr(st, f)]
  if weak and not st.per_pixel_split_path and not st.synthetic:
    raise ValueError(f'--{weak[0]} needs --per_pixel_split_path: the weak parts of the batch are trained with per-pixel '
                     'examples (training on weak labels alone is not supported).')
  if st.per_pixel_split_path and not st.synthetic:
    from wlseg import train_input
    pairs = train_input.split_pairs(st.per_pixel_split_path, st.per_pixel_dataset_name)
    if weak:
      parts = ('the bounding-box part from --per_bbox_split_path' if st.per_bbox_split_path else
               'the bounding-box part empty (no --per_bbox_split_path)',
               'the image-level part from --per_image_split_path' if st.per_image_split_path else
               'the image-level part empty (no --per_image_split_path)')
      weak_note = f'{parts[0]}, {parts[1]}.'
    else:
      weak_note = 'the bounding-box and image-level parts of the batch are empty (there is no Open Images source).'
    print(f'Training on the {st.per_pixel_dataset_name} split at {st.per_pixel_split_path}: {len(pairs)} image / label '
          f'pairs, {len(pairs[st.rank::st.world_size])} on this rank; {weak_note}', flush=True)
    input_fn = train_input.train_input_fn
  system = SemanticSegmentation({'train': input_fn}, None, st)
  out = system.train()
  _dist_shutdown(st, system)
  return out


def evaluate_main(argv):
  np.set_printoptions(formatter={'float': '{:>5.2f}'.format}, nanstr=u'nan', linewidth=10000)
  ss = wsettings.build_parser(wsettings.EVAL)
  st = wsettings.eval_extra_args(ss.parse_args(argv))
  _dist_env(st)
  # real images from the split directory tfrecords_path names unless --synthetic or it is no split in a known layout
  from wlseg import dataset_input
  layout = None if getattr(st, 'synthetic', False) else dataset_input.detect_layout(st.tfrecords_path)
  if layout:
    print(f'Evaluating the {layout} split at {st.tfrecords_path}.')
  else:
    why = ('--synthetic is given' if getattr(st, 'synthetic', False) else
           f'{st.tfrecords_path} is not a Cityscapes leftImg8bit/<split> or Vistas split (images/ + labels/) directory')
    print(f'Evaluating SYNTHETIC input: {why}.')
  system = SemanticSegmentation({'eval': dataset_input.eval_input_fn if layout else synthetic.eval_input_fn}, None, st)
  labels = system.settings.evaluation_problem_def['cids2labels']
  void_exists = -1 in system.settings.evaluation_problem_def['lids2cids']
  if void_exists and not system.settings.train_void_class:
    labels = labels[:-1]
  all_metrics = system.evaluate()
  if st.rank == 0:
    mr_filename = os.path.join(system.settings.eval_res_dir, 'all_metrics.txt')
    with open(mr_filename, 'w') as f:
      for m in all_metrics:
        print(f"{m['global_step']:>05} ", end='', file=f)
        metrics.print_metrics_from_confusion_matrix(m['confusion_matrix'], labels, printfile=f)
    with open(os.path.join(system.settings.eval_res_dir, 'all_metrics.p'), 'wb') as f:
      pickle.dump([{k: m[k] for k in ('global_step', 'loss', 'confusion_matrix')} for m in all_metrics], f)
  _dist_shutdown(st, system)
  return all_metrics


def predict_main(argv):
  ss = wsettings.build_parser(wsettings.PREDICT)
  st = wsettings.predict_extra_args(ss.parse_args(argv))
  _dist_env(st)
  for flag in ('plotting', 'plotting_overlapped'):
    if getattr(st, flag, False):
      raise NotImplementedError(f'--{flag}: live matplotlib plotting is outside the B200 hot path')
  # real images from predict_dir (dataset-agnostic pipeline) unless --synthetic or the directory does not exist
  from wlseg import image_input
  real = not getattr(st, 'synthetic', False) and st.predict_dir and os.path.isdir(st.predict_dir)
  system = SemanticSegmentation({'predict': image_input.predict_input_fn if real else synthetic.predict_input_fn}, None, st)
  s = system.settings
  exporting = any(getattr(s, f, False) for f in ('export_lids_images', 'export_color_decisions',
                                                 'export_overlapped_color_decisions'))
  if exporting:
    # code/predict.py:213-219 (_validate_settings) and :78-83 (palettes from the inference problem definition)
    if not s.results_dir or not os.path.isdir(s.results_dir):
      raise ValueError('results_dir must be an existing directory when an export flag is given.')
    idspalette = np.array(s.inference_problem_def.get('cids2lids', []), dtype=np.uint8)
    colorpalette = np.array(s.inference_problem_def['cids2colors'], dtype=np.uint8)
  start = total = datetime.now()
  n = 0
  for outputs in system.predict():
    n += 1
    print(f"\nTime per image (input pipeline + network): {datetime.now() - start}", outputs['decisions'].shape)
    if exporting:
      export_outputs(outputs, s, idspalette, colorpalette)
    start = datetime.now()
  print('\nTotal time (input pipeline + network):', datetime.now() - total, 'for', n, 'image(s)')


def export_outputs(outputs, s, idspalette, colorpalette):
  """code/predict.py:137-164: label-id PNG, colour PNG, and the colour map blended 50:50 over the raw image.
  Host-side palette look-ups on the decisions `SemanticSegmentation.predict()` already returned."""
  from PIL import Image
  decs = outputs['decisions']
  path = outputs['rawimagespaths']
  stem = os.path.splitext(os.path.basename(path.decode() if isinstance(path, bytes) else str(path)))[0]

  def save(arr, suffix):
    out_fname = os.path.join(s.results_dir, stem + suffix)
    assert not os.path.exists(out_fname), f'Output filename ({out_fname}) already exists.'
    Image.fromarray(arr).save(out_fname)
  if s.export_lids_images:
    save(idspalette[decs], '_result_lids.png')
  if s.export_color_decisions:
    save(colorpalette[decs], '_result_color.png')
  if s.export_overlapped_color_decisions:
    raw = outputs['rawimages']
    col = colorpalette[decs]
    if raw.shape[:2] != col.shape[:2]:
      raise ValueError(f'raw image {raw.shape[:2]} and decisions {col.shape[:2]} differ in size')
    save((0.5 * raw + 0.5 * col).astype(np.uint8), '_result_overlapped_color.png')
