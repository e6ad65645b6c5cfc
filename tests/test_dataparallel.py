"""world_size-2 gloo (CPU) tests of the data-parallel plumbing (SURVEY.md section 8e): the bucketed gradient exchange
must reproduce the single-process gradient of the concatenated batch, whatever the bucket size."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _net():
    torch.manual_seed(7)
    return nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 8, 3, padding=1), nn.ReLU(),
                         nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(8, 5))


def _data():
    g = torch.Generator().manual_seed(11)
    return torch.randn(8, 3, 12, 12, generator=g), (torch.rand(8, 5, generator=g) < 0.3).float()


def _worker(rank, world, port, bucket_mb, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from chexpert_b200.dataparallel import GradientBuckets
    net = _net()
    if rank == 1:                         # replicas must be re-synchronised from rank 0 by the constructor
        with torch.no_grad():
            for p in net.parameters():
                p.add_(1.0)
    gb = GradientBuckets(net, bucket_mb=bucket_mb)
    x, t = _data()
    xs, ts = x.chunk(world)[rank], t.chunk(world)[rank]
    grads = []
    for _ in range(2):                    # two steps: reset() must really clear the buckets
        gb.reset()
        loss = nn.functional.binary_cross_entropy_with_logits(net(xs), ts, reduction='none').sum(1).mean(0)
        loss.backward()
        gb.finish()
        grads = [p.grad.clone() for p in net.parameters()]
    torch.save({'grads': grads, 'nb': len(gb.buckets), 'params': [p.detach().clone() for p in net.parameters()]},
               os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


@pytest.mark.parametrize('bucket_mb', [25.0, 0.0005])
def test_bucketed_allreduce_matches_full_batch(tmp_path, bucket_mb):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), bucket_mb, str(tmp_path)), nprocs=world, join=True)
    net = _net()
    x, t = _data()
    nn.functional.binary_cross_entropy_with_logits(net(x), t, reduction='none').sum(1).mean(0).backward()
    want = [p.grad for p in net.parameters()]
    r0, r1 = (torch.load(tmp_path / f'r{r}.pt') for r in range(world))
    if bucket_mb < 1:
        assert r0['nb'] > 1               # the tiny cap really splits the parameters into several buckets
    for a, b in zip(r0['params'], r1['params']):
        assert torch.equal(a, b)
    for g0, g1, w in zip(r0['grads'], r1['grads'], want):
        assert torch.equal(g0, g1)
        assert torch.allclose(g0, w, rtol=1e-5, atol=1e-7)


def test_single_process_is_a_noop():
    from chexpert_b200.dataparallel import GradientBuckets
    net = _net()
    gb = GradientBuckets(net)
    x, t = _data()
    gb.reset()
    nn.functional.binary_cross_entropy_with_logits(net(x), t).backward()
    gb.finish()
    ref = _net()
    nn.functional.binary_cross_entropy_with_logits(ref(x), t).backward()
    for p, q in zip(net.parameters(), ref.parameters()):
        assert torch.allclose(p.grad, q.grad)


def test_finish_without_reset_is_an_error():
    """finish() twice, or a backward() after finish() without reset(), would average gradients that are already averaged: the
    next finish() raises instead."""
    from chexpert_b200.dataparallel import GradientBuckets
    net = _net()
    gb = GradientBuckets(net)
    x, t = _data()
    loss = lambda: nn.functional.binary_cross_entropy_with_logits(net(x), t)   # noqa: E731
    gb.reset()
    loss().backward()
    gb.finish()
    with pytest.raises(RuntimeError, match='finish'):
        gb.finish()
    loss().backward()
    with pytest.raises(RuntimeError, match='without reset'):
        gb.finish()


def test_backward_calls_between_reset_and_finish_add_up():
    from chexpert_b200.dataparallel import GradientBuckets
    net, ref = _net(), _net()
    gb = GradientBuckets(net, bucket_mb=0.0005)
    x, t = _data()
    f = nn.functional.binary_cross_entropy_with_logits
    gb.reset()
    f(net(x[:4]), t[:4]).backward()
    f(net(x[4:]), t[4:]).backward()
    gb.finish()
    (f(ref(x[:4]), t[:4]) + f(ref(x[4:]), t[4:])).backward()
    for p, q in zip(net.parameters(), ref.parameters()):
        assert torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-7)


def _worker_unused(rank, world, port, out_dir):
    """Rank 1 never uses `b`: it has no gradient there and contributes zeros, yet the collectives must pair up."""
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from chexpert_b200.dataparallel import GradientBuckets
    torch.manual_seed(3)
    a, b = nn.Linear(6, 6), nn.Linear(6, 6)
    net = nn.ModuleList([a, b])
    gb = GradientBuckets(net, bucket_mb=1e-5)          # one bucket per parameter
    g = torch.Generator().manual_seed(5 + rank)
    x = torch.randn(4, 6, generator=g)
    gb.reset()
    y = a(x) if rank == 1 else b(a(x))                 # rank 1: `b` receives no gradient at all
    y.sum().backward()
    gb.finish()
    torch.save([p.grad.clone() for p in net.parameters()], os.path.join(out_dir, f'u{rank}.pt'))
    dist.destroy_process_group()


def test_collectives_stay_ordered_when_a_rank_skips_parameters(tmp_path):
    world = 2
    mp.spawn(_worker_unused, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    g0, g1 = (torch.load(tmp_path / f'u{r}.pt') for r in range(world))
    for p, q in zip(g0, g1):
        assert torch.equal(p, q)                       # both ranks hold the same averaged gradients
    assert float(g0[2].abs().sum()) > 0                # b.weight: rank 0's contribution / 2


def _worker_nccl(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    from chexpert_b200.train import TrainStep, synthetic_batch
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ts = TrainStep(f'cuda:{rank}', size=64, precision='fp32', lr=1e-2, seed=0)
    ts.model.eval()                        # BatchNorm on running stats: the only cross-sample coupling is then the mean over the batch
    x, t = synthetic_batch(4, size=64, seed=21, device=f'cuda:{rank}')
    xs, tsub = x.chunk(world)[rank], t.chunk(world)[rank]
    loss = ts(xs, tsub)
    torch.cuda.synchronize()
    torch.save({'loss': loss.cpu(), 'params': [p.detach().cpu() for p in ts.model.parameters()]}, os.path.join(out_dir, f'n{rank}.pt'))
    ts.release()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_trainstep_nccl_two_ranks_equal_the_full_batch_step(tmp_path):
    """ADVICE r1: the NCCL whole-model path (bucketed all-reduce under the real TrainStep) against the same step on one rank with
    the concatenated batch.  Needs 2 GPUs (gpurun --gpus 2)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    from chexpert_b200.train import TrainStep, synthetic_batch
    world = 2
    mp.spawn(_worker_nccl, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ts = TrainStep('cuda:0', size=64, precision='fp32', lr=1e-2, seed=0)
    ts.model.eval()
    x, t = synthetic_batch(4, size=64, seed=21, device='cuda:0')
    ts(x, t)
    want = [p.detach().cpu() for p in ts.model.parameters()]
    r0, r1 = (torch.load(tmp_path / f'n{r}.pt') for r in range(world))
    for a, b, w in zip(r0['params'], r1['params'], want):
        assert torch.equal(a, b)                                          # replicas stay identical
        assert torch.allclose(a, w, rtol=2e-4, atol=2e-6), float((a - w).abs().max())
