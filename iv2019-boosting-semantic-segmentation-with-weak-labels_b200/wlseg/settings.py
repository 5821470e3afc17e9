"""Command-line surface: the reference's flags with the same names, defaults and positional order.

Mirrors code/utils/utils.py:7-174 (`SemanticSegmentationArguments`), the model flags of
code/models/resnet50_extended_model_hierarchical.py:228-269 (`add_model_arguments`), the input
flags the scripts add (code/input_pipelines/cityscapes/input_cityscapes.py:294-319,
code/input_pipelines/dataset_agnostic/dataset_agnostic_predict_input.py:156-164), the predict UI
flags (code/predict.py:171-197) and the per-script hard overrides (`_add_extra_args`:
code/train.py:42-68, code/evaluate.py:69-79, code/predict.py:199-211).

Additive flags of this implementation (absent upstream): --synthetic, --dtype, --steps, --seed, and for train.py
--per_pixel_split_path, --per_bbox_split_path and --per_image_split_path.
"""

import argparse

TRAIN, EVAL, PREDICT = 'train', 'eval', 'infer'  # tf.estimator.ModeKeys values


class SemanticSegmentationArguments(object):
  """Collects the arguments of one mode exactly as the reference does."""

  def __init__(self, mode=None):
    self._parser = argparse.ArgumentParser()
    self._mode = mode
    self.add_system_arguments()
    self.add_tf_arguments()
    if mode == PREDICT:
      self.add_inference_arguments()
    elif mode == TRAIN:
      self.add_train_arguments()
    elif mode == EVAL:
      self.add_evaluate_arguments()
    self.add_b200_arguments()

  @property
  def argparser(self):
    return self._parser

  def parse_args(self, argv):
    self.args = self._parser.parse_args(argv)
    return self.args

  def add_system_arguments(self):
    p = self._parser
    p.add_argument('--height_system', type=int, default=None)
    p.add_argument('--width_system', type=int, default=None)
    p.add_argument('--height_feature_extractor', type=int, default=512)
    p.add_argument('--width_feature_extractor', type=int, default=1024)

  def add_tf_arguments(self):
    # kept for command-line compatibility; there is no XLA here (hand-written kernels + CUDA graphs)
    self._parser.add_argument('--enable_xla', action='store_true')

  def add_b200_arguments(self):
    p = self._parser
    p.add_argument('--synthetic', action='store_true',
                   help='Use the on-device synthetic generator instead of an input pipeline.')
    p.add_argument('--dtype', type=str, default='bf16', choices=['bf16', 'fp32'],
                   help='bf16: tcgen05 product path; fp32: check mode (direct fp32 convolutions).')
    p.add_argument('--steps', type=int, default=None, help='Stop after this many steps.')
    p.add_argument('--seed', type=int, default=0)
    if self._mode == TRAIN:
      p.add_argument('--per_pixel_split_path', type=str, default=None, metavar='DIR',
                     help='Training split of the per-pixel dataset (a Cityscapes leftImg8bit/<split> directory or a Vistas '
                          'split directory with images/ + labels/), decoded once into device memory.')
      p.add_argument('--per_bbox_split_path', type=str, default=None, metavar='DIR',
                     help='Open Images directory (class-descriptions-boxable.csv, one *annotations-bbox.csv, '
                          'images/<ImageID>.jpg) of the bounding-box part of the batch, decoded once into device memory. '
                          'Needs --per_pixel_split_path; may name the same directory as --per_image_split_path.')
      p.add_argument('--per_image_split_path', type=str, default=None, metavar='DIR',
                     help='Open Images directory (class-descriptions-boxable.csv, one '
                          '*annotations-human-imagelabels*.csv, images/<ImageID>.jpg) of the image-level part of the '
                          'batch, decoded once into device memory.  Needs --per_pixel_split_path.')

  def add_train_arguments(self):
    p = self._parser
    p.add_argument('log_dir', type=str)
    p.add_argument('per_pixel_dataset_name', type=str, choices=['cityscapes', 'vistas'])
    p.add_argument('--Ntrain', type=int, default=2975)
    p.add_argument('--init_ckpt_path', type=str, default='/media/panos/data/pretrained/resnet_v1_50_official.ckpt')
    p.add_argument('--training_problem_def_path', type=str)
    p.add_argument('--save_checkpoints_steps', type=int, default=None)
    p.add_argument('--save_summaries_steps', type=int, default=120)
    p.add_argument('--train_void_class', action='store_true')
    p.add_argument('--Ne', type=int, default=17)
    p.add_argument('--Nb', type=int, default=4)
    p.add_argument('--learning_rate_schedule', type=str, default='piecewise_constant',
                   choices=['piecewise_constant', 'polynomial_decay'])
    p.add_argument('--learning_rate_initial', type=float, default=0.01)
    p.add_argument('--learning_rate_boundaries', type=int, default=[8, 15, 17], nargs='*')
    grp = p.add_mutually_exclusive_group()
    grp.add_argument('--learning_rate_decay', type=float)
    grp.add_argument('--learning_rate_values', type=float, nargs='*')
    p.add_argument('--learning_rate_decay_steps', type=float, default=0.5)
    p.add_argument('--learning_rate_final', type=float, default=0.5)
    p.add_argument('--learning_rate_power', type=float, default=0.9)
    p.add_argument('--optimizer', type=str, default='SGDM', choices=['SGD', 'SGDM'])
    p.add_argument('--ema_decay', type=float, default=0.9)
    p.add_argument('--regularization_weight', type=float, default=0.00017)
    p.add_argument('--bootstrapping_percentage', type=int, default=-1)
    p.add_argument('--momentum', type=float, default=0.9)
    p.add_argument('--use_nesterov', action='store_true')
    p.add_argument('--distribute', action='store_true')

  def add_inference_arguments(self):
    p = self._parser
    p.add_argument('log_dir', type=str, default=None)
    p.add_argument('--ckpt_path', type=str, default=None)
    p.add_argument('training_problem_def_path', type=str)
    p.add_argument('predict_dir', type=str, default=None)
    p.add_argument('--inference_problem_def_path', type=str, default=None)
    p.add_argument('--replace_voids', action='store_true')
    p.add_argument('--Nb', type=int, default=1)
    p.add_argument('--restore_emas', action='store_true')
    p.add_argument('--train_void_class', action='store_true')

  def add_evaluate_arguments(self):
    p = self._parser
    p.add_argument('log_dir', type=str, default=None)
    p.add_argument('--eval_all_ckpts', action='store_true')
    p.add_argument('--ckpt_path', type=str, default=None)
    p.add_argument('Neval', type=int)
    p.add_argument('training_problem_def_path', type=str)
    p.add_argument('--evaluation_problem_def_path', type=str, default=None)
    p.add_argument('--replace_voids', action='store_true')
    p.add_argument('--train_void_class', action='store_true')
    p.add_argument('--Nb', type=int, default=1)
    p.add_argument('--restore_emas', action='store_true')


def add_model_arguments(argparser):
  """code/models/resnet50_extended_model_hierarchical.py:228-269."""
  a = argparser.add_argument
  a('--stride_feature_extractor', type=int, default=8)
  a('--name_feature_extractor', type=str, default='resnet_v1_50', choices=['resnet_v1_50', 'resnet_v1_101'])
  a('--feature_dims_decreased', type=int, default=256)
  a('--fov_expansion_kernel_size', type=int, default=0)
  a('--fov_expansion_kernel_rate', type=int, default=0)
  a('--upsampling_method', type=str, default='bilinear', choices=['no', 'bilinear', 'hybrid'])
  a('--psp_module', action='store_true')
  a('--norm_layer', type=str, default='batch', choices=['batch', 'group'])
  a('--cross_replica_norm', action='store_true')
  a('--norm_train_variables', action='store_true')
  a('--batch_norm_accumulate_statistics', action='store_true')
  a('--batch_norm_decay', type=float, default=0.9)


def add_train_input_pipeline_arguments(argparser):
  """per_pixel_per_bbox_per_image.add_train_input_pipeline_arguments adds nothing upstream."""
  return argparser


def add_evaluate_input_pipeline_arguments(argparser):
  """code/input_pipelines/cityscapes/input_cityscapes.py:318 (positional tfrecords_path)."""
  argparser.add_argument('tfrecords_path', type=str,
                         default='/media/panos/data/datasets/cityscapes/tfrecords/valFine.tfrecords')  # as upstream
  argparser.add_argument('--preserve_aspect_ratio', action='store_true')


def add_predict_input_pipeline_arguments(argparser):
  """code/input_pipelines/dataset_agnostic/dataset_agnostic_predict_input.py:156-164."""
  argparser.add_argument('--preserve_aspect_ratio', action='store_true')


def add_predict_ui_arguments(argparser):
  """code/predict.py:171-197 (plotting / export flags; accepted, the UI itself is out of scope)."""
  a = argparser.add_argument
  a('--plotting', action='store_true')
  a('--plotting_overlapped', action='store_true')
  a('--plot_l1_confidence', action='store_true')
  a('--plot_l2_confidence', action='store_true')
  a('--timeout', type=float, default=10.0)
  a('--export_color_decisions', action='store_true')
  a('--export_overlapped_color_decisions', action='store_true')
  a('--export_lids_images', action='store_true')
  a('--results_dir', type=str, default=None)


def add_dataset_positional(argparser):
  """code/evaluate.py:29-33, code/predict.py:28-32."""
  argparser.add_argument('per_pixel_dataset_name', type=str, choices=['vistas', 'cityscapes'],
                         help='During evaluation, it must be given the training dataset name.')


def train_extra_args(settings):
  """code/train.py:42-68."""
  from wlseg import problem_defs
  settings.norm_train_variables = True
  settings.batch_norm_accumulate_statistics = True
  if settings.per_pixel_dataset_name == 'vistas':
    settings.Ntrain = 18000
    settings.height_feature_extractor = 621
    settings.width_feature_extractor = 855
  elif settings.per_pixel_dataset_name == 'cityscapes':
    settings.Ntrain = 2975
    settings.height_feature_extractor = 512
    settings.width_feature_extractor = 1024
  if not getattr(settings, 'training_problem_def_path', None):
    settings.training_problem_def_path = problem_defs.default_path(settings.per_pixel_dataset_name)
  settings.Nb_per_pixel = 4
  settings.Nb_per_bbox = 8
  settings.Nb_per_image = 4
  settings.Nb = settings.Nb_per_pixel
  settings.preserve_aspect_ratio_per_pixel = False
  settings.preserve_aspect_ratio_per_bbox = True
  settings.preserve_aspect_ratio_per_image = True
  return settings


def eval_extra_args(settings):
  """code/evaluate.py:69-73."""
  settings.regularization_weight = 0.0
  settings.batch_norm_decay = 1.0
  return settings


def predict_extra_args(settings):
  """code/predict.py:199-211."""
  settings.regularization_weight = 0.0
  settings.batch_norm_decay = 1.0
  settings.predict_keys = ['decisions', 'l1_probabilities', 'l2_vehicle_probabilities', 'rawimages', 'rawimagespaths']
  return settings


def build_parser(mode):
  """Parser for one of the three scripts, arguments added in the reference's order."""
  ss = SemanticSegmentationArguments(mode=mode)
  if mode == TRAIN:
    add_train_input_pipeline_arguments(ss.argparser)
    add_model_arguments(ss.argparser)
  elif mode == EVAL:
    add_evaluate_input_pipeline_arguments(ss.argparser)
    add_model_arguments(ss.argparser)
    add_dataset_positional(ss.argparser)
  elif mode == PREDICT:
    add_predict_input_pipeline_arguments(ss.argparser)
    add_model_arguments(ss.argparser)
    add_dataset_positional(ss.argparser)
    add_predict_ui_arguments(ss.argparser)
  return ss
