"""2-rank NCCL test of the training path's exchange step (SURVEY 8e): a discriminator step with the R1 penalty, data-parallel over
two B200s through DistributedDataParallel (bucketed gradient all-reduce over NVLink), every convolution on the sm_100a
kernels.  The averaged gradients must equal the single-GPU step on the concatenated batch.  Needs two GPUs; skipped on a machine
with one."""
import importlib
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup():
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from conftest import load_pkg
    load_pkg()
    return importlib.import_module('pgpp_b200.training.discriminator')


def _build(device):
    disc = _setup()
    torch.manual_seed(0)
    D = disc.Discriminator(c_dim=0, img_resolution=64, img_channels=3, channel_base=2048, channel_max=64,
                           epilogue_kwargs=dict(mbstd_group_size=2)).train().to(device)
    imgs = torch.randn(8, 3, 64, 64, generator=torch.Generator().manual_seed(2)).clamp(-1, 1).to(device)
    return D, imgs


def _d_loss(D, img):
    cg = importlib.import_module('pgpp_b200.torch_utils.ops.conv2d_gradfix')
    img = img.detach().requires_grad_(True)
    logits = D(img, None)
    with cg.no_weight_gradients():
        gx, = torch.autograd.grad(logits.sum(), [img], create_graph=True)
    return (torch.nn.functional.softplus(-logits).squeeze(1) + 5.0 * gx.square().sum([1, 2, 3])).mean()


def _worker(rank, world, port, out_path):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    device = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=device)
    D, imgs = _build(device)
    custom_ops = importlib.import_module('pgpp_b200.torch_utils.custom_ops')
    before = custom_ops.launch_count()
    ddp = torch.nn.parallel.DistributedDataParallel(D, device_ids=[device], broadcast_buffers=False, find_unused_parameters=True)
    per = imgs.shape[0] // world
    _d_loss(ddp, imgs[rank * per:(rank + 1) * per]).backward()
    torch.cuda.synchronize()
    assert custom_ops.launch_count() - before >= 50
    if rank == 0:
        torch.save({n: p.grad.cpu() for n, p in D.named_parameters()}, out_path)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_rank_nccl_ddp_d_step_with_r1_equals_single_gpu(tmp_path):
    out_path = str(tmp_path / 'grads.pt')
    port = 33500 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, out_path), nprocs=2, join=True)
    D, imgs = _build('cuda:0')
    # minibatch-std groups of 2 stay inside a rank's shard of 4, so the mean of the two shard losses is the global loss
    (0.5 * (_d_loss(D, imgs[:4]) + _d_loss(D, imgs[4:]))).backward()
    got = torch.load(out_path)
    for n, p in D.named_parameters():
        scale = max(p.grad.abs().max().item(), 1e-8)
        assert (got[n] - p.grad.cpu()).abs().max().item() <= 1e-4 * scale, n
