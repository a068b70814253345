"""world_size-2 NCCL test on two GPUs of one box: the README-layer tokenizer in ``model.train()`` mode, batch sharded
by clip, with the one collective of the path (LFQ avg_prob all-reduce, SURVEY Appendix A.1 step 7 / reference M:1705)
issued on a side stream under the decoder.  Checked against the CPU oracle on the GLOBAL batch.
Run with two GPUs:  gpurun --gpus 2 -- python -m pytest tests/test_dist_gpu.py -m gpu"""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q, dtype_name):
    import torch.distributed as dist
    from magvit2_pytorch_b200.dist import shard_clips
    from tests.util import build_product, golden_video, load_golden
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g = load_golden("mini")
    dtype = getattr(torch, dtype_name)
    model = build_product(g["kwargs"], g["wseed"]).to(f"cuda:{rank}").to(dtype)
    video = golden_video(g)                                   # the full batch (2 clips)
    local = shard_clips(video).to(f"cuda:{rank}")             # this rank's clip(s)
    model.train()
    for graphs in (False, True, True, True):                  # eager, then warm-up / capture / replay of the graph path
        model.cuda_graphs = graphs
        codes, recon = model(local, return_codes=True, return_recon=True)
        ps, be, cm = model.quantizer_loss_breakdown
        torch.cuda.synchronize()
    # numpy arrays are pickled by value; a tensor would travel as a shared-memory handle that the parent can only open
    # while this process is alive
    q.put((rank, codes.cpu().numpy(), recon.float().cpu().numpy(), ps.item(), be.item(), cm.item(),
           model.quantizer_aux_loss.item()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("dtype_name", ["float32", "bfloat16"])
def test_train_mode_forward_world2_nccl(dtype_name):
    assert torch.cuda.is_available()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (gpurun --gpus 2)")
    from oracle.restated import lfq_train_losses
    from tests.util import build_oracle, build_product, golden_video, load_golden
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, dtype_name)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    g = load_golden("mini")
    codes = torch.cat([torch.from_numpy(r[1]) for r in res])
    recon = torch.cat([torch.from_numpy(r[2]) for r in res])
    cpu_model = build_product(g["kwargs"], g["wseed"])
    orc = build_oracle(cpu_model, g["kwargs"])
    ref_codes, pre = orc.tokenize(golden_video(g), return_presign=True)
    ps_all, be_all, cm_all, aux_all, _ = lfq_train_losses(pre, 10)
    if dtype_name == "float32":
        assert torch.equal(codes, g["codes"]) and torch.equal(codes, ref_codes)       # identical in train and eval mode
        assert (recon - g["recon"]).abs().max().item() < 1e-5                          # decoder fed q (== straight-through value)
        tol = 2e-4
    else:
        assert (codes != g["codes"]).float().mean().item() <= 0.0834
        tol = 0.05                                            # bf16 encoder: pre-sign values deviate by ~2e-2
    # batch entropy comes from the GLOBAL mean code probability: identical on both ranks, equal to the single-process value
    assert abs(res[0][4] - res[1][4]) < 1e-6
    assert abs(res[0][4] - be_all.item()) <= tol * max(1.0, abs(be_all.item()))
    # per-sample entropy / commitment are per-rank means over equal shards
    assert abs((res[0][3] + res[1][3]) / 2 - ps_all.item()) <= tol * max(1.0, abs(ps_all.item()))
    assert abs((res[0][5] + res[1][5]) / 2 - cm_all.item()) <= tol * max(1.0, abs(cm_all.item()))
