"""Writes tests/golden/oracle_small.json: small seeded input -> output vectors of the ORACLE.

The reference itself (TensorFlow 1.12) cannot be imported in this container (SURVEY.md section 8c),
so these vectors are produced by the oracle restatement, not by the reference: they freeze the
oracle (drift guard) and give the GPU tests committed targets.  Run:  python -m tests.golden.make_golden
"""

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

from oracle import losses as olosses  # noqa: E402
from oracle import metrics as ometrics  # noqa: E402
from oracle import network as onet  # noqa: E402
from oracle import tfops  # noqa: E402
from oracle import weak_labels as oweak  # noqa: E402


def inputs():
  g = torch.Generator().manual_seed(1234)
  low = [torch.randn(2, 3, 4, c, generator=g) * 2 for c in (14, 7, 3)]
  strong = torch.randint(0, 20, (1, 24, 32), generator=g, dtype=torch.int32)
  bbox = torch.from_numpy(oweak.bbox_labels([(2, 0.1, 0.6, 0.2, 0.9), (6, 0.3, 0.8, 0.1, 0.5), (1, 0.5, 0.9, 0.5, 0.9)],
                                            24, 32))[None]
  images = torch.rand(1, 32, 64, 3, generator=g) * 2 - 1
  return low, strong, bbox, images


def compute():
  low, strong, bbox, images = inputs()
  full = [tfops.resize_bilinear(z, 24, 32) for z in low]
  pred = onet.compose_predictions(*full, 'cityscapes')
  loss = olosses.define_losses(pred, {'prolabels_per_pixel': strong, 'prolabels_per_bbox': bbox}, 'cityscapes')
  cm = ometrics.confusion_matrix(strong.numpy(), pred['decisions'][:1].numpy(), 20)
  # the network runs in float64: in float32 its logits depend on the CPU's convolution kernels (their summation order)
  # by up to 7e-6 after 57 batch-norm layers, above the tolerance the pin is checked with; in float64 the same code
  # agrees with itself across machines and thread counts to 1e-14
  params = {k: v.double() for k, v in onet.init_params('cityscapes', seed=0, randomize_bn=True, tame=True).items()}
  net = onet.Net(params, 'cityscapes')
  lowres = torch.cat(net.lowres_logits(images.double()), -1)
  return {
      'full_l1_logits_row0': full[0][0, 0, :, :].reshape(-1).tolist(),
      'decisions': pred['decisions'].reshape(-1).tolist(),
      'l1_probabilities_pixel': pred['l1_probabilities'][1, 5, 7].tolist(),
      'losses': [float(loss[k]) for k in ('l1_segmentation', 'l2_vehicle_segmentation', 'l2_human_segmentation',
                                          'segmentation')],
      'counts': [float(loss['counts'][k]) for k in ('l1', 'l2_vehicle', 'l2_human')],
      'confusion_matrix': cm.reshape(-1).tolist(),
      'network_lowres_logits': lowres.reshape(-1).tolist(),
  }


if __name__ == '__main__':
  out = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'oracle_small.json')
  with open(out, 'w') as fp:
    json.dump(compute(), fp)
  print(out, os.path.getsize(out), 'bytes')
