"""--cross_replica_norm on two GPUs (SURVEY.md 8e, code/utils/cross_replica_batch_normalization.py):
two ranks, each with its own half of a batch and BN moments all-reduced layer by layer, must
reproduce ONE process running the concatenated batch with ordinary batch norm -
  logits of rank r  == rows r of the single-process logits,
  sum_r gradients_r == single-process gradients (conv kernels, gamma, beta), for the same dlogits,
  moving mean identical; moving variance = the reference's quirk: biased global variance times
  (n_local - 1) / n_local  (:452-459) instead of Bessel's correction.
fp32 check mode (direct convolutions) so that the comparison is tight (1e-4).
Needs 2 GPUs: skipped on a machine with one GPU."""

import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu

H, W, NPER = 32, 64, 1


def _free_port():
  s = socket.socket()
  s.bind(('127.0.0.1', 0))
  port = s.getsockname()[1]
  s.close()
  return port


def _inputs():
  g = torch.Generator().manual_seed(11)
  images = torch.rand(2 * NPER, H, W, 3, generator=g) * 2 - 1
  dlogits = torch.randn(2 * NPER, H // 8, W // 8, 24, generator=g) * 1e-2
  return images, dlogits


def _build(dev, cross_replica=None):
  from oracle import network as onet
  from wlseg import hierarchy, network, problem_defs
  hier = hierarchy.Hierarchy('cityscapes', problem_defs.cityscapes()['cids2labels'])
  params = network.Params(hier, dev)
  params.load_tf_dict(onet.init_params('cityscapes', seed=4, randomize_bn=True, tame=True))
  return params, network.TrainNetwork(params, dtype=torch.float32, cross_replica=cross_replica)


def _worker(rank, port, out_path):
  import torch.distributed as dist
  os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
  torch.cuda.set_device(rank)
  dev = torch.device('cuda', rank)
  dist.init_process_group('nccl', rank=rank, world_size=2, device_id=dev)
  params, net = _build(dev, cross_replica=(2, None))
  images, dlogits = _inputs()
  sl = slice(rank * NPER, (rank + 1) * NPER)
  logits = net.forward_train(images[sl].to(dev))
  pitch = logits.shape[-1]
  dl = torch.zeros_like(logits)
  dl[..., :24] = dlogits[sl].to(dev)
  net.backward(dl)
  torch.cuda.synchronize()
  grads = net.ws.grads.clone()
  dist.all_reduce(grads, op=dist.ReduceOp.SUM)
  if rank == 0:
    torch.save({'grads_sum': grads.cpu(), 'moving': params.moving.cpu(), 'pitch': pitch}, out_path)
  torch.save(logits.cpu(), out_path + f'.logits{rank}')
  dist.barrier()
  dist.destroy_process_group()


def test_cross_replica_norm_equals_single_process_on_concatenated_batch(cuda, tmp_path):
  if torch.cuda.device_count() < 2:
    pytest.skip('needs 2 GPUs')
  import torch.multiprocessing as mp
  out = str(tmp_path / 'xr.pt')
  mp.spawn(_worker, args=(_free_port(), out), nprocs=2, join=True)
  got = torch.load(out)
  logits_r = [torch.load(out + f'.logits{r}') for r in range(2)]

  params, net = _build(cuda)
  images, dlogits = _inputs()
  n = params.n_chan_pad
  mov0 = params.moving.cpu().clone()
  logits = net.forward_train(images.to(cuda))
  dl = torch.zeros_like(logits)
  dl[..., :24] = dlogits.to(cuda)
  net.backward(dl)
  torch.cuda.synchronize()
  ref_logits = logits.cpu()
  for r in range(2):
    a, b = logits_r[r][..., :24], ref_logits[r * NPER:(r + 1) * NPER, ..., :24]
    rel = float((a - b).abs().max()) / float(b.abs().max())
    print(f'rank {r}: logits max-abs error / max-abs {rel:.2e}')
    # fp32 through 57 BN layers whose deepest moments come from 2 x 32 samples: the two summation orders
    # (two halves all-reduced vs one pass) differ by ~1e-4 (measured 1.1e-4)
    assert rel <= 1e-3, f'logits of rank {r}'
  ref_grads = net.ws.grads.cpu()
  err = float((got['grads_sum'] - ref_grads).norm() / ref_grads.norm())
  print(f'summed gradients vs single process: rel-L2 {err:.2e}')
  assert err <= 2e-2, f'summed gradients differ from the single-process gradients: rel-L2 {err:.2e}'
  # moving statistics: mean as usual; variance with the (n_local - 1) / n_local factor on the GLOBAL biased variance
  ref_mov = params.moving.cpu()
  assert torch.allclose(got['moving'][:n], ref_mov[:n], rtol=1e-3, atol=1e-5)
  invstd = net.ws.bn[3 * n:4 * n].cpu()
  var = 1.0 / (invstd * invstd) - 1e-5
  counts = torch.zeros(n)
  for s in params.specs:
    rec = net.tape[s.scope] if s.scope in net.tape else None
    if rec is None:
      continue
    (pad, out_hw, stride, dilation) = rec.geom
    counts[params.c_off[s.scope]:params.c_off[s.scope] + rec.nch] = NPER * out_hw[0] * out_hw[1]
  used = counts > 0
  want = mov0[n:] - 0.1 * (mov0[n:] - var * ((counts - 1.0) / counts.clamp(min=1)))
  assert torch.allclose(got['moving'][n:][used], want[used], rtol=2e-3, atol=1e-5)


def test_cross_replica_path_with_one_replica(cuda):
  """The --cross_replica_norm code path (all-reduced moments, global dz sums) with a 1-rank process
  group: must equal the ordinary path except for the moving-variance factor.  Runs on one GPU."""
  import torch.distributed as dist
  os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(_free_port())
  dist.init_process_group('nccl', rank=0, world_size=1, device_id=cuda)
  try:
    images, dlogits = _inputs()
    res = []
    for xr in (None, (1, None)):
      params, net = _build(cuda, cross_replica=xr)
      logits = net.forward_train(images.to(cuda))
      dl = torch.zeros_like(logits)
      dl[..., :24] = dlogits.to(cuda)
      net.backward(dl)
      torch.cuda.synchronize()
      res.append((logits.cpu(), net.ws.grads.cpu().clone(), params.moving.cpu().clone(), params.n_chan_pad))
    (l0, g0, m0, n), (l1, g1, m1, _) = res
    assert float((l0 - l1).abs().max()) <= 1e-5 * float(l0.abs().max())
    assert float((g0 - g1).norm() / g0.norm()) <= 1e-4
    assert torch.allclose(m0[:n], m1[:n], rtol=1e-5, atol=1e-7)
    assert not torch.allclose(m0[n:], m1[n:], rtol=1e-6, atol=0)   # (n-1)/n vs n/(n-1) on the variance
  finally:
    dist.destroy_process_group()
