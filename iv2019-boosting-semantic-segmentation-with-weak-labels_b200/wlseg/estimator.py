"""Train / eval / predict step drivers: the host-side mirror of the reference's Estimator glue.

Mirrors code/estimator/define_estimator_hierarchical.py:39-239 (`define_estimator` TRAIN / EVAL /
PREDICT branches), :490-528 (`_map_predictions_to_new_cids`), :530-571 (`_resize_predictions`),
code/estimator/define_metrics.py:5-20, code/estimator/define_optimizer.py:3-26 and
code/input_pipelines/utils.py:118-124 (`get_temp_Nb`).  Everything here is launch sequencing and
buffer ownership; the arithmetic lives in libwlseg.
"""

import glob
import os

import numpy as np
import torch

from wlseg import checkpoints, network, ops
from wlseg.dataset_input import PACKED_IMAGES, PACKED_LIDS, PACKED_SIZES


def _replacevoids(mappings):
  """code/utils/utils.py:286-289."""
  max_m = max(mappings)
  return [m if m != -1 else max_m + 1 for m in mappings]


def get_temp_Nb(params, Nb):
  """code/input_pipelines/utils.py:118-124: per-replica batch = Nb / num_towers (must divide)."""
  if getattr(params, 'distribute', False):
    world = max(1, getattr(params, 'world_size', 1))
    div, mod = divmod(Nb, world)
    assert not mod, 'for now Nb must be divisible by the number of available GPUs.'
    return div
  return Nb


def learning_rate(params, global_step):
  """code/estimator/define_optimizer.py:3-13 with the [TF-1.12] schedule semantics."""
  if params.learning_rate_schedule == 'piecewise_constant':
    for b, v in zip(params.learning_rate_boundaries, params.learning_rate_values):
      if global_step <= b:
        return v
    return params.learning_rate_values[-1]
  if params.learning_rate_schedule == 'polynomial_decay':
    t = params.num_training_steps
    s = min(global_step, t)
    return ((params.learning_rate_initial - params.learning_rate_final) * (1.0 - s / t) ** params.learning_rate_power
            + params.learning_rate_final)
  raise ValueError('Unknown option for learning rate schedule.')


def mean_iou_from_cm(cm, num_classes):
  """code/estimator/define_metrics.py:13-20 on an int confusion matrix (training summary); accepts the device
  tensor the histogram kernel accumulates into."""
  if isinstance(cm, torch.Tensor):
    cm = cm.detach().cpu().numpy()
  cm = np.asarray(cm).astype(np.int32)
  inter = np.diagonal(cm).astype(np.float32)
  union = (cm.sum(0) + cm.sum(1) - np.diagonal(cm)).astype(np.float32) + np.float32(1e-9)
  del num_classes
  return float(np.mean(inter / union, dtype=np.float32))


def resize_decisions_nearest(decs, new_h, new_w):
  """`_resize_predictions` for decisions: NEAREST_NEIGHBOR, align_corners=True, roundf
  (define_estimator_hierarchical.py:559-563).  Identity at every BASELINE configuration."""
  return ops.resize_decisions(decs, new_h, new_w)


def resize_predictions(predictions, new_h, new_w):
  """`_resize_predictions` (define_estimator_hierarchical.py:530-571): the three probability maps bilinearly,
  the decisions by nearest neighbour, both with align_corners=True; other keys pass through."""
  out = dict(predictions)
  for k in ('l1_probabilities', 'l2_vehicle_probabilities', 'l2_human_probabilities'):
    if k in out:
      out[k] = ops.resize_probabilities(out[k], new_h, new_w)
  if 'decisions' in out:
    out['decisions'] = ops.resize_decisions(out['decisions'], new_h, new_w)
  return out


_PROB_KEYS = ('l1_probabilities', 'l2_vehicle_probabilities', 'l2_human_probabilities')


class _Prefetcher:
  """Host -> device staging: batch i+1 is copied (pinned memory, side stream) while batch i computes, into a
  ring of `depth` device buffers per input, so the consumer sees a few RECURRING addresses (network.EvalStep
  replays a CUDA graph per address set without copying) and nothing is allocated per step.  A ring slot is
  overwritten only after the step that read it has finished (event on the consumer's stream).  Device-resident
  batches pass through untouched."""

  def __init__(self, it, device, depth=3, rings=None):
    self.it = iter(it)
    self.device = device
    # one copy stream per Estimator (kept with the rings): creating a stream per call is not free
    holder = {} if rings is None else rings
    self.stream = holder.get('__stream__')
    if self.stream is None:
      self.stream = holder['__stream__'] = torch.cuda.Stream(device=device)
    self.h2d_bytes = 0
    self.depth = depth
    self.rings = {} if rings is None else rings   # shared across calls by the Estimator: addresses stay put
    self.count = 0
    self.next = None
    self._advance(None)

  def _to_dev(self, key, t, slot):
    if not torch.is_tensor(t) or t.is_cuda:
      return t
    if not t.is_pinned():
      t = t.pin_memory()
    self.h2d_bytes += t.numel() * t.element_size()
    ring = self.rings.setdefault((key, tuple(t.shape), t.dtype), [None] * self.depth)
    if ring[slot] is None:
      ring[slot] = torch.empty(t.shape, dtype=t.dtype, device=self.device)
    ring[slot].copy_(t, non_blocking=True)
    return ring[slot]

  def _advance(self, consumed):
    try:
      features, labels = next(self.it)
    except StopIteration:
      self.next = None
      return
    slot = self.count % self.depth
    self.count += 1
    if consumed is not None:
      self.stream.wait_event(consumed)   # every step that read this ring slot has completed
    with torch.cuda.stream(self.stream):
      f = {k: self._to_dev(('f', k), v, slot) for k, v in features.items()}
      l = None if labels is None else {k: self._to_dev(('l', k), v, slot) for k, v in labels.items()}
      ev = torch.cuda.Event()
      ev.record(self.stream)
    self.next = (f, l, ev)

  def __iter__(self):
    return self

  def __next__(self):
    if self.next is None:
      raise StopIteration
    f, l, ev = self.next
    cur = torch.cuda.current_stream()
    # the consumer has enqueued every earlier step by now: the copy of the NEXT batch (into the slot the batch
    # depth - 1 steps back used) may start once all of that has run
    consumed = torch.cuda.Event()
    consumed.record(cur)
    cur.wait_event(ev)
    self._advance(consumed)
    return f, l


class Estimator:
  """Owns the parameters and runs the three modes for `SemanticSegmentation`."""

  def __init__(self, params, hier, device='cuda'):
    self.settings = params
    self.hier = hier
    self.device = torch.device(device)
    self.dtype = torch.bfloat16 if getattr(params, 'dtype', 'bf16') == 'bf16' else torch.float32
    self.params = network.Params(hier, self.device, getattr(params, 'stride_feature_extractor', 8),
                                 psp=getattr(params, 'psp_module', False),
                                 fov=(getattr(params, 'fov_expansion_kernel_size', 0),
                                      getattr(params, 'fov_expansion_kernel_rate', 0)),
                                 upsampling=getattr(params, 'upsampling_method', 'bilinear'),
                                 norm=getattr(params, 'norm_layer', 'batch'))
    self.global_step = 0
    self.net = None
    self.last_h2d_bytes = 0
    self.last_d2h_bytes = 0

  # ---- checkpoints ({TF variable name: tensor} files, wlseg/checkpoints.py) ---------------------------
  def latest_checkpoint(self, log_dir):
    cands = glob.glob(os.path.join(log_dir, 'model.ckpt-*.pt'))
    if not cands:
      return None
    return max(cands, key=lambda p: int(p.rsplit('-', 1)[1].split('.')[0]))

  def save(self, log_dir):
    """train_saver (code/estimator/define_savers.py:3-36): every global variable - model variables, Momentum
    slots, EMA shadows, global_step - under its TF name."""
    path = os.path.join(log_dir, f'model.ckpt-{self.global_step}.pt')
    return checkpoints.save_file(path, checkpoints.export_train_state(self.params, getattr(self, 'trainer', None)),
                                 self.global_step)

  def restore(self, path, for_training=False):
    """EVAL / PREDICT: predict_saver (define_savers.py:38-66; --restore_emas reads the EMA shadows into the
    model variables).  TRAIN: continue from log_dir with the optimizer / EMA slots."""
    variables, step = checkpoints.load_file(path)
    if for_training:
      self._resume = variables   # slots are imported once the trainer exists
      self.params.load_tf_dict(variables)
    else:
      self.params.load_tf_dict(checkpoints.select_for_predict(
          self.params, variables, restore_emas=bool(getattr(self.settings, 'restore_emas', False))))
    self.global_step = step

  def initialize(self, ckpt_path=None, log_dir=None, seed=0, for_training=False):
    """TRAIN: latest checkpoint of log_dir, else warm start from --init_ckpt_path when that file exists
    (replace_initializers, code/estimator/define_initializers.py:72-131), else random init.  EVAL / PREDICT:
    --ckpt_path or the latest checkpoint of log_dir."""
    path = ckpt_path or (self.latest_checkpoint(log_dir) if log_dir else None)
    self._resume = None
    if path:
      self.restore(path, for_training=for_training)
    else:
      if not for_training and not getattr(self.settings, 'synthetic', False):
        # tf.estimator raises when EVAL / PREDICT find nothing to restore; metrics or PNGs of a random-init network
        # must never be produced silently.  --synthetic (benchmarks, BASELINE configs) opts into random weights.
        raise ValueError(f'Could not find trained model in model_dir: {log_dir} (no --ckpt_path and no '
                         'model.ckpt-*.pt); pass --synthetic to evaluate / predict with random-init weights.')
      self.params.init_random(seed)  # BASELINE configs use random weights
      init = getattr(self.settings, 'init_ckpt_path', None)
      if for_training and init and os.path.isfile(init):
        variables, _ = checkpoints.load_file(init)
        mapping = checkpoints.warm_start(self.params, variables, psp_module=getattr(self.settings, 'psp_module', False))
        print(f'initialised {len(mapping)} variables from {init}', flush=True)
    if for_training:
      # the step training continues from: an input function that follows a data order (wlseg.train_input) resumes there
      self.settings.initial_global_step = self.global_step
    self.__dict__.pop('_eval_steps', None)   # graphs captured for a previous network object
    # group norm has no folded inference form: its evaluation forward is the training forward (network.py)
    cls = network.TrainNetwork if self.params.norm == 'group' else network.Network
    self.net = cls(self.params, dtype=self.dtype, bn_decay=getattr(self.settings, 'batch_norm_decay', 0.9))
    return path

  # ---- TRAIN --------------------------------------------------------------------------------------
  def train(self, batches, max_steps, log_every=0):
    """define_estimator TRAIN branch driven for `max_steps` steps (create_train_op + the
    MonitoredTrainingSession loop, define_estimator_hierarchical.py:77-159).  `batches` yields
    (features, labels) with host or device tensors in the reference's contract (SURVEY.md 3.5).
    Returns the per-step loss vectors [total, segmentation, l1, l2_vehicle, l2_human, regularization]
    as one host array (read back once per step, asynchronously)."""
    from wlseg import trainer as wtrainer
    s = self.settings
    dev = self.device
    if getattr(self, 'trainer', None) is None:
      self.trainer = wtrainer.Trainer(self.params, s, dtype=self.dtype, rank=getattr(s, 'rank', 0),
                                      world_size=getattr(s, 'world_size', 1) if getattr(s, 'distribute', False) else 1)
      self.trainer.global_step = self.global_step
      if getattr(self, '_resume', None) is not None:
        checkpoints.import_train_state(self.params, self.trainer, self._resume)
        self._resume = None
    tr = self.trainer
    pre = _Prefetcher(batches, dev, rings=self.__dict__.setdefault('_rings', {}))
    host = torch.zeros((max(1, max_steps), 6), dtype=torch.float32).pin_memory()
    steps = 0
    last_saved = None
    save_every = getattr(s, 'save_checkpoints_steps', None)
    for features, labels in pre:
      if steps >= max_steps:
        break
      lr = learning_rate(s, tr.global_step)
      out = tr.step(features, {k: v for k, v in labels.items() if v is not None}, lr)
      host[steps].copy_(out, non_blocking=True)
      steps += 1
      self.global_step = tr.global_step
      if log_every and steps % log_every == 0 and getattr(s, 'rank', 0) == 0:
        torch.cuda.synchronize(dev)
        print(f'step {tr.global_step}: total loss {float(host[steps - 1, 0]):.4f} lr {lr:g}', flush=True)
      if save_every and getattr(s, 'rank', 0) == 0 and tr.global_step % save_every == 0 and getattr(s, 'save_checkpoints', True):
        self.save(s.log_dir)
        last_saved = tr.global_step
    torch.cuda.synchronize(dev)
    # tf.estimator always writes a checkpoint when train() ends (CheckpointSaverHook.end): with --steps, or a cadence
    # that does not divide the step count, the trained weights would otherwise be lost
    if (steps and getattr(s, 'rank', 0) == 0 and getattr(s, 'save_checkpoints', True) and getattr(s, 'log_dir', None)
            and os.path.isdir(s.log_dir) and last_saved != tr.global_step):
      self.save(s.log_dir)
    self.last_h2d_bytes = pre.h2d_bytes
    self.last_d2h_bytes = steps * 6 * 4
    return host[:steps].numpy().copy()

  # ---- EVAL ---------------------------------------------------------------------------------------
  def evaluate(self, batches, num_classes, lut=None):
    """define_estimator EVAL branch: forward, remap cids, resize to label size, streaming confusion
    matrix.  `batches` yields (features, labels) with host or device tensors, as proimages / prolabels or in the
    packed raw form of wlseg.dataset_input (converted on the device by `_raw_eval_inputs`).  Returns the
    reference's metrics dict {'confusion_matrix': np.int32[C, C], 'loss': 0.0, 'global_step'}."""
    dev = self.device
    lut_t = None if lut is None else torch.tensor(lut, dtype=torch.int32, device=dev)
    replace_voids = bool(getattr(self.settings, 'replace_voids', False))
    # forward + decisions + confusion-matrix update, replayed as one CUDA graph per input shape (network.EvalStep);
    # kept across calls (the graphs are), counters zeroed
    cache = self.__dict__.setdefault('_eval_steps', {})
    key = (id(self.net), num_classes, None if lut is None else tuple(lut), replace_voids)
    step = cache.get(key)
    if step is None:
      step = cache[key] = network.EvalStep(self.net, num_classes, lut_t, replace_voids, self.hier.void_cid)
    step.reset()
    cm, invalid = step.cm, step.invalid
    pre = _Prefetcher(batches, dev, rings=self.__dict__.setdefault('_rings', {}))
    steps = 0
    host_cm = self.__dict__.setdefault('_host_cm', {}).get(num_classes)
    if host_cm is None:   # pinned once: cudaHostAlloc per call costs more than a step's worth of launches
      host_cm = self._host_cm[num_classes] = torch.zeros((num_classes, num_classes), dtype=torch.int64).pin_memory()
    raw = None
    for features, labels in pre:
      if PACKED_IMAGES in features:
        if raw is None:
          raw = self._raw_eval_inputs()
        features, labels = raw(features, labels)
      lab = labels['prolabels']
      if tuple(lab.shape[1:3]) == tuple(features['proimages'].shape[1:3]) and self.params.upsampling != 'no':
        step(features['proimages'], lab)
      else:
        # labels at another size: EVAL order of the reference, (cid map ->) _replace_voids -> _resize_predictions
        out = self.net.predict(features['proimages'], want=('decisions',) + (_PROB_KEYS if replace_voids else ()))
        if replace_voids:
          ops.replace_voids(self.net.hstruct, *(out[k] for k in _PROB_KEYS), out['decisions'], self.hier.void_cid)
        decs = resize_decisions_nearest(out['decisions'], lab.shape[1], lab.shape[2])
        ops.confmat_accumulate(lab.contiguous(), decs, num_classes, cm, lut_t, invalid)
      # the step's result (running metric) goes back to the host every step, asynchronously
      host_cm.copy_(cm, non_blocking=True)
      steps += 1
    torch.cuda.synchronize(dev)
    self.last_h2d_bytes = pre.h2d_bytes
    self.last_d2h_bytes = steps * host_cm.numel() * 8
    if raw is not None and int(raw.invalid.item()):
      raise ops.WlsegError(f'{int(raw.invalid.item())} label ids outside the evaluation problem definition\'s lids2cids '
                           'table, or examples larger than their batch rows')
    if int(invalid.item()):
      raise ops.WlsegError(f'{int(invalid.item())} (label, decision) pairs outside [0, {num_classes})')
    total = cm.cpu().numpy()
    # the reference exposes tf.to_int32(total_cm)
    return {'confusion_matrix': total.astype(np.int32), 'confusion_matrix_int64': total, 'loss': 0.0,
            'global_step': self.global_step, 'steps': steps}

  def _raw_eval_inputs(self):
    """Converter of batches in packed raw form (wlseg.dataset_input) into the evaluation contract on the device
    (ops.eval_inputs).  Results go to one estimator-owned (proimages, prolabels) pair per (N, TH, TW), so EvalStep sees
    recurring addresses and replays its graph without copying.  The label-id table of the evaluation problem definition
    is uploaded once per call; `.invalid` counts what the kernel rejected."""
    s = self.settings
    table = _replacevoids(s.evaluation_problem_def['lids2cids'])
    lut = torch.tensor(table, dtype=torch.int32, device=self.device)
    th, tw = s.height_feature_extractor, s.width_feature_extractor
    outs = self.__dict__.setdefault('_raw_eval_outputs', {})
    invalid = torch.zeros(1, dtype=torch.int64, device=self.device)

    def convert(features, labels):
      images = features[PACKED_IMAGES]
      key = (images.shape[0], th, tw)
      if key not in outs:
        outs[key] = (torch.empty(key + (3,), dtype=torch.float32, device=self.device),
                     torch.empty(key, dtype=torch.int32, device=self.device))
      pro, lab = outs[key]
      ops.eval_inputs(images, labels[PACKED_LIDS], features[PACKED_SIZES], lut, max(table), (th, tw), pro, lab, invalid)
      return {'proimages': pro}, {'prolabels': lab}
    convert.invalid = invalid
    return convert

  # ---- PREDICT ------------------------------------------------------------------------------------
  def predict(self, batches, predict_keys):
    """define_estimator PREDICT branch (define_estimator_hierarchical.py:204-237): yields one dict per example
    with the requested keys, resized to (height_system, width_system) - or, when either is unset, to the size
    of the raw image (:219-229) - and, with --replace_voids, void decisions replaced afterwards (:232-233)."""
    want = tuple(k for k in predict_keys if k not in ('rawimages', 'rawimagespaths'))
    s = self.settings
    replace_voids = bool(getattr(s, 'replace_voids', False))
    need = tuple(dict.fromkeys(want + (_PROB_KEYS + ('decisions',) if replace_voids else ())))
    for features, _ in batches:
      pro = features['proimages']
      if not pro.is_cuda:
        pro = pro.to(self.device, non_blocking=True)
      out = self.net.predict(pro, want=need)
      new_size = (getattr(s, 'height_system', None), getattr(s, 'width_system', None))
      if not all(new_size):
        new_size = tuple(features['rawimages'].shape[1:3]) if 'rawimages' in features else tuple(pro.shape[1:3])
      out = resize_predictions(out, int(new_size[0]), int(new_size[1]))
      if replace_voids:
        ops.replace_voids(self.net.hstruct, *(out[k] for k in _PROB_KEYS), out['decisions'], self.hier.void_cid)
      host = {k: out[k].cpu().numpy() for k in want}
      n = pro.shape[0]
      for i in range(n):
        ex = {k: v[i] for k, v in host.items()}
        if 'rawimages' in predict_keys and 'rawimages' in features:
          ex['rawimages'] = features['rawimages'][i].cpu().numpy()
        if 'rawimagespaths' in predict_keys and 'rawimagespaths' in features:
          ex['rawimagespaths'] = features['rawimagespaths'][i]
        yield ex
