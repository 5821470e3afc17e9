"""The 2-level class hierarchy as ONE validated table object per dataset.

The reference hard-codes the hierarchy three times as literal integer lists
(code/estimator/define_losses_hierarchical.py:38-93,
 code/models/resnet50_extended_model_hierarchical.py:81-83,95-117,
 code/estimator/define_estimator_hierarchical.py:323-337).  Here the tables are DERIVED from the
class names of the problem definition plus three facts:

  * which strong classes are vehicles / humans (they collapse into one L1 super-class each,
    placed where the first of them sat; the void class stays last),
  * which weak (Open Images) class corresponds to which strong class name,
  * all weak human-like classes supervise the first human class ("person").

`Hierarchy.validate()` checks the round trip strong cid -> (L1, L2) -> common cid for every id;
tests/test_hierarchy.py compares every derived table with the reference's literals.
"""

import ctypes

from wlseg import ops

WEAK_CLASSES = ('bicycle', 'bus', 'car', 'motorcycle', 'train', 'truck',
                'human', 'man', 'woman', 'boy', 'girl',
                'traffic light', 'traffic sign', 'stop sign', 'void')
WEAK_HUMANS = ('human', 'man', 'woman', 'boy', 'girl')
# Open Images display names (class-descriptions-boxable.csv) of the weak classes whose name here differs
WEAK_DISPLAY_NAMES = {'human': 'Person'}


def weak_display_name(cid):
  """Open Images display name of weak class `cid` (compared case-insensitively)."""
  name = WEAK_CLASSES[cid]
  return WEAK_DISPLAY_NAMES.get(name, name[0].upper() + name[1:])

_DATASETS = {
    'cityscapes': dict(
        vehicles=('car', 'truck', 'bus', 'train', 'motorcycle', 'bicycle'),
        humans=('person', 'rider'),
        weak2strong={'bicycle': 'bicycle', 'bus': 'bus', 'car': 'car', 'motorcycle': 'motorcycle',
                     'train': 'train', 'truck': 'truck'},
        weak_l1={'traffic light': None, 'traffic sign': None, 'stop sign': None},
    ),
    'vistas': dict(
        vehicles=('Bicycle', 'Boat', 'Bus', 'Car', 'Caravan', 'Motorcycle', 'On Rails', 'Other Vehicle',
                  'Trailer', 'Truck', 'Wheeled Slow'),
        humans=('Person', 'Bicyclist', 'Motorcyclist', 'Other Rider'),
        weak2strong={'bicycle': 'Bicycle', 'bus': 'Bus', 'car': 'Car', 'motorcycle': 'Motorcycle',
                     'train': 'On Rails', 'truck': 'Truck'},
        weak_l1={'traffic light': None, 'traffic sign': None, 'stop sign': None},
    ),
}


class Hierarchy:
  """Tables for one per-pixel dataset.  `labels` = cids2labels of the problem definition
  (void last)."""

  def __init__(self, dataset, labels):
    if dataset not in _DATASETS:
      raise ValueError(f'unknown per_pixel_dataset_name {dataset!r}')
    spec = _DATASETS[dataset]
    self.dataset = dataset
    self.labels = list(labels)
    n = len(self.labels)
    self.num_classes = n
    void = n - 1
    veh = [self.labels.index(v) for v in spec['vehicles']]
    hum = [self.labels.index(v) for v in spec['humans']]
    assert veh == sorted(veh) and hum == sorted(hum)
    # --- strong cid -> L1 cid: walk the strong ids, collapsing each super-class at its first member
    self.pp2l1 = [0] * n
    self.l1_2common = []
    seen = {}
    for cid in range(n):
      group = 'vehicle' if cid in veh else 'human' if cid in hum else None
      if group is not None and group in seen:
        self.pp2l1[cid] = seen[group]
        continue
      l1 = len(self.l1_2common)
      self.pp2l1[cid] = l1
      self.l1_2common.append(cid)
      if group is not None:
        seen[group] = l1
    self.cid_l1_vehicle = seen['vehicle']
    self.cid_l1_human = seen['human']
    # --- strong cid -> L2 cids (void = last id of each head)
    self.pp2veh = [veh.index(c) if c in veh else len(veh) for c in range(n)]
    self.pp2hum = [hum.index(c) if c in hum else len(hum) for c in range(n)]
    self.veh2common = veh + [void]
    self.hum2common = hum + [void]
    # --- weak cid -> L2 cids
    self.bb2veh, self.bb2hum, self.bb2l1 = [], [], []
    for wname in WEAK_CLASSES:
      strong = spec['weak2strong'].get(wname)
      self.bb2veh.append(veh.index(self.labels.index(strong)) if strong is not None else len(veh))
      self.bb2hum.append(0 if wname in WEAK_HUMANS else len(hum))
      if strong is not None:
        self.bb2l1.append(self.cid_l1_vehicle)
      elif wname in WEAK_HUMANS:
        self.bb2l1.append(self.cid_l1_human)
      else:
        self.bb2l1.append(len(self.l1_2common) - 1)
    self.C1, self.Cv, self.Ch = len(self.l1_2common), len(veh) + 1, len(hum) + 1
    self.validate()

  @property
  def head_widths(self):
    return self.C1, self.Cv, self.Ch

  @property
  def void_cid(self):
    """Common (strong-label) id of the void class: the last one."""
    return self.num_classes - 1

  @property
  def total_channels(self):
    return self.C1 + self.Cv + self.Ch

  @property
  def logits_pitch(self):
    """Channel pitch of the low-resolution logits buffer (multiple of 8 for the vector kernels)."""
    return (self.total_channels + 7) // 8 * 8

  def compose(self, l1, l2v, l2h):
    """Scalar restatement of the decision rule (host-side checks only)."""
    if l1 == self.cid_l1_vehicle:
      return self.veh2common[l2v]
    if l1 == self.cid_l1_human:
      return self.hum2common[l2h]
    return self.l1_2common[l1]

  def validate(self):
    n = self.num_classes
    assert max(self.pp2l1) + 1 == self.C1 and max(self.pp2veh) + 1 == self.Cv and max(self.pp2hum) + 1 == self.Ch
    assert self.C1 <= 64 and self.Cv <= 16 and self.Ch <= 8 and n <= 80
    for cid in range(n):
      got = self.compose(self.pp2l1[cid], self.pp2veh[cid], self.pp2hum[cid])
      assert got == cid, f'hierarchy round trip failed for strong cid {cid}: {got}'

  def as_struct(self):
    h = ops.Hierarchy()
    h.C1, h.Cv, h.Ch = self.C1, self.Cv, self.Ch
    h.cid_l1_vehicle, h.cid_l1_human = self.cid_l1_vehicle, self.cid_l1_human
    h.num_classes = self.num_classes

    def fill(dst, src):
      for i, v in enumerate(src):
        dst[i] = v
    fill(h.l1_to_common, self.l1_2common)
    fill(h.veh_to_common, self.veh2common)
    fill(h.hum_to_common, self.hum2common)
    fill(h.pp_to_l1, self.pp2l1)
    fill(h.pp_to_veh, self.pp2veh)
    fill(h.pp_to_hum, self.pp2hum)
    fill(h.bb_to_veh, self.bb2veh)
    fill(h.bb_to_hum, self.bb2hum)
    return h


_ = ctypes  # (ctypes structs are created through ops.Hierarchy)
