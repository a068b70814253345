"""world_size-2 gloo tests (CPU) for the host-side multi-GPU logic: clip sharding and the LFQ batch-entropy
all-reduce (the only collective on the path, SURVEY.md 8e / Appendix A.1 step 7)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from magvit2_pytorch_b200.dist import allreduce_mean_, entropy_from_avg_prob, shard_clips, shard_range


def test_shard_range_partitions_exactly():
    for n in (1, 4, 7, 32, 33):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for (a, b), (c, d) in zip(spans, spans[1:]):
                assert b == c and a <= b
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle.restated import lfq_train_losses
    g = torch.Generator().manual_seed(0)
    presign = torch.randn(8, 40, 10, generator=g) * 0.7          # (clips, tokens, bits) -- the full batch
    local = shard_clips(presign)                                  # this rank's clips
    assert local.shape[0] == 4

    def reduce(avg):
        avg = avg.clone()
        allreduce_mean_(avg)
        return avg

    ps, be, cm, aux, avg = lfq_train_losses(local, 10, world_reduce=reduce)
    # a tensor would travel as a shared-memory handle that the parent can only open while this process is alive;
    # a numpy array is pickled by value
    q.put((rank, ps.item(), be.item(), cm.item(), aux.item(), avg.numpy()))
    dist.barrier()
    dist.destroy_process_group()


def test_lfq_batch_entropy_allreduce_world2_gloo():
    from oracle.restated import lfq_train_losses
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    g = torch.Generator().manual_seed(0)
    presign = torch.randn(8, 40, 10, generator=g) * 0.7
    ps_all, be_all, cm_all, _, avg_all = lfq_train_losses(presign, 10)
    # batch entropy comes from the GLOBAL mean code probability -> identical on both ranks and equal to the
    # single-process value on the whole batch; per-sample entropy / commitment are per-rank means
    for rank, ps, be, cm, aux, avg in res:
        avg = torch.from_numpy(avg)
        assert abs(be - be_all.item()) < 1e-5
        assert torch.allclose(avg, avg_all, atol=1e-6)
        assert abs(be - entropy_from_avg_prob(avg).item()) < 1e-6
    assert abs((res[0][1] + res[1][1]) / 2 - ps_all.item()) < 1e-5
    assert abs((res[0][3] + res[1][3]) / 2 - cm_all.item()) < 1e-5


def _grad_worker(rank, world, port, q):
    """Per rank: gradient of the LFQ auxiliary loss wrt this rank's encoder output, (a) with an autograd-aware all-reduce of the mean
    code probability (the reference's semantics, SURVEY Appendix A.1 step 7) and (b) with the training path's formulation
    avg_local + (avg_global - avg_local).detach() (train._lfq_train), where avg_global comes from a plain all-reduce."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import torch.distributed.nn.functional as dnn
    import torch.nn.functional as F
    from magvit2_pytorch_b200 import modules as M
    from magvit2_pytorch_b200 import train as T
    torch.manual_seed(0)
    qz = M.LFQ(16, 16, 0.1, 1.0, 2.5, 10.)
    with torch.no_grad():
        for p in qz.parameters():
            p.copy_(torch.randn(p.shape, generator=torch.Generator().manual_seed(3)) * 0.4)
    x = torch.randn(2, 3, 4, 4, 16, generator=torch.Generator().manual_seed(10 + rank))      # this rank's clips, channels-last

    def aux_reference(xr):
        p = (F.linear(xr, qz.project_in.weight, qz.project_in.bias) / 10.).tanh() * 10.
        p = p.reshape(-1, 4).float()
        codebook = ((torch.arange(16)[:, None] & qz.mask) != 0).float() * 2 - 1
        prob = (200. * (p @ codebook.t())).softmax(dim=-1)
        per_sample = T._entropy(prob).mean()
        avg = dnn.all_reduce(prob.mean(dim=0)) / world                         # autograd-aware SUM, then / world
        qd = torch.where(p > 0, torch.ones_like(p), -torch.ones_like(p))
        return (per_sample - 2.5 * T._entropy(avg)) * 0.1 + ((p - qd) ** 2).mean() * 1.0, avg.detach()

    xa = x.clone().requires_grad_(True)
    aux_a, avg_global = aux_reference(xa)
    ga, = torch.autograd.grad(aux_a, xa)
    xb = x.clone().requires_grad_(True)
    _, aux_b = T._lfq_train(xb, qz, avg_global)
    gb, = torch.autograd.grad(aux_b, xb)
    q.put((rank, aux_a.item(), aux_b.item(), float((ga - gb).abs().max()), float(ga.abs().max())))
    dist.barrier()
    dist.destroy_process_group()


def test_training_path_cross_rank_entropy_gradient_world2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_grad_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, aux_a, aux_b, err, scale in res:
        assert abs(aux_a - aux_b) < 1e-6, (rank, aux_a, aux_b)
        assert err <= 1e-6 * max(1.0, scale), (rank, err, scale)
