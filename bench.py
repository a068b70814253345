"""bench.py -- headline metric of BASELINE.json: video frames/s through tokenize + decode_from_code_indices,
17x128x128 clips, bf16, README config (BASELINE.json configs[1]), data-parallel over N GPUs of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch of 4 synthetic clips per GPU (weak scaling: the batch
is sharded by clip, no data-path collective in eval -- SURVEY.md 8e).  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/codes.npy (float64, exact code indices)
and DIR/recon.npy (float32).  Weights and inputs are seeded, so two builds run with the same arguments can be
compared output for output.

--impl reference times the reference's own CPU implementation of the path: the reference is pure Python and
cannot travel to the GPU box, so this arm runs the restated oracle (oracle/restated.py, pinned bit-for-bit to
the reference's goldens) -- the same torch-eager CPU ops the reference dispatches -- on all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

README_LAYERS = (
    "residual", "compress_space", ("consecutive_residual", 2), "compress_space",
    ("consecutive_residual", 2), "linear_attend_space", "compress_space",
    ("consecutive_residual", 2), "attend_space", "compress_time",
    ("consecutive_residual", 2), "compress_time", ("consecutive_residual", 2), "attend_time",
)
README_KW = dict(image_size=128, init_dim=64, max_dim=512, codebook_size=1024, layers=README_LAYERS)
# the other BASELINE.json configs (not the headline; `--workload cfg4|fsq` for the record)
WORKLOADS = {
    "readme": dict(kw=README_KW, clips=4, size=128, flop_clip=1.512e12,
                   name="README VideoTokenizer (BASELINE configs[1]): tokenize + decode_from_code_indices, "
                        "4 clips of 3x17x128x128 per GPU, batch sharded by clip"),
    "cfg3": dict(kw=README_KW, clips=4, size=128, flop_clip=1.512e12, train_mode=True,
                 name="BASELINE configs[2]: README VideoTokenizer in model.train(): forward(return_codes, return_recon) with the LFQ "
                      "entropy terms and their cross-rank avg_prob all-reduce (NCCL, side stream, overlapped with the decoder), "
                      "4 clips of 3x17x128x128 per GPU, batch sharded by clip"),
    "cfg4": dict(kw=dict(image_size=256, init_dim=64, max_dim=1024, codebook_size=1024, layers=README_LAYERS), clips=3,
                 size=256, flop_clip=8.944e12,
                 name="BASELINE configs[3]: image_size=256 max_dim=1024, tokenize + decode, 3 clips of 3x17x256x256 per GPU"),
    "fsq": dict(kw=dict(image_size=128, init_dim=64, max_dim=512, use_fsq=True, fsq_levels=[8, 5, 5, 5], layers=README_LAYERS),
                clips=4, size=128, flop_clip=1.512e12,
                name="BASELINE configs[4]: FSQ [8,5,5,5] variant, tokenize + decode_from_code_indices round trip, "
                     "4 clips of 3x17x128x128 per GPU"),
}
CLIPS_PER_GPU = 4
FRAMES = 17
# SURVEY.md 8d / BASELINE.md 3 (forward hooks on the reference's own modules, 2 FLOP per MAC)
FLOP_PER_CLIP_CONV_PATH = 1.2787e12       # causal Conv3d path only (k>1 Conv3d)
FLOP_PER_CLIP_ALL = 1.512e12              # conv + linear + attention einsums
METRIC = "video-frames/sec tokenize+decode, 17x128x128 bf16"


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []          # (host monotonic time of arrival, csv line)
        self.t0 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.monotonic(), ln.strip()))

    def begin(self):
        """Marks the start of the timed region: only samples that arrive between begin() and stop() are used.  (nvidia-smi takes
        100 - 300 ms to start streaming, longer than a 20-step timed region, so it is started before the warm-up.)"""
        self.t0 = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t1 = time.monotonic()
        window = [ln for (ts, ln) in self.lines if self.t0 is None or self.t0 <= ts <= t1]
        for ln in window:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _best_cpu_threads():
    """Host threads the CPU arm should use.  os.cpu_count() over-reports inside the container (the GPU boxes show 128
    logical CPUs but a cgroup share: 128 torch threads run 10x slower than 16), so a 1-second conv3d calibration
    picks the fastest of a few thread counts."""
    import torch
    import torch.nn.functional as F
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    x = torch.randn(1, 64, 8, 64, 64)
    w = torch.randn(64, 64, 3, 3, 3)
    best, best_t = 1, float("inf")
    for nt in sorted({min(avail, c) for c in (4, 8, 16, 32, 64, avail)}):
        torch.set_num_threads(nt)
        F.conv3d(x, w, padding=1)
        t0 = time.perf_counter()
        F.conv3d(x, w, padding=1)
        dt = time.perf_counter() - t0
        if dt < best_t * 0.95:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return best


def _cpu_oracles():
    """The CPU arm's two arithmetic flavours (fp32 and bf16 storage, as ``model.float()`` / ``model.bfloat16()`` of the
    reference would run on the host), weights identical to the GPU arm's."""
    import torch
    import synth_data as Wt
    from oracle.restated import OracleTokenizer
    from magvit2_pytorch_b200 import VideoTokenizer
    torch.manual_seed(0)
    model = VideoTokenizer(**README_KW)
    Wt.fill_state_dict_(model, 0)
    sd = {k: v for k, v in model.state_dict().items()}
    del model
    return {"f32": OracleTokenizer(sd, dtype=torch.float32, **README_KW),
            "bf16": OracleTokenizer(sd, dtype=torch.bfloat16, **README_KW)}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, codes, recon):
    """The arrays a caller of the timed path receives, as .npy files of at most DUMP_MAX_BYTES in all (the largest
    workload writes 40 MB).  A reconstruction that does not fit is replaced by a fixed, seeded sample of its elements:
    a 1-D array of the values at sorted flat indices, the same indices for the same shape."""
    import numpy as np
    arrays = {"codes": codes.detach().cpu().double().numpy(), "recon": recon.detach().float().cpu().numpy()}
    if sum(a.nbytes for a in arrays.values()) > DUMP_MAX_BYTES:
        r = arrays["recon"]
        keep = (DUMP_MAX_BYTES - arrays["codes"].nbytes) // r.itemsize
        idx = np.sort(np.random.default_rng(0).choice(r.size, size=keep, replace=False))
        arrays["recon"] = r.reshape(-1)[idx]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _cpu_time_step(orc, video):
    t0 = time.perf_counter()
    orc.decode_from_code_indices(orc.tokenize(video))
    return time.perf_counter() - t0


def _cpu_pick_dtype(orcs, video1):
    """One warm-up + one timed 1-clip pass per dtype; returns (name of the faster one, {name: seconds per clip}).
    Host cores with AMX / AVX512-BF16 run the bf16 path ~2x faster than fp32, older cores ~10x slower."""
    import torch
    secs = {}
    for name, orc in orcs.items():
        v = video1.to(torch.bfloat16) if name == "bf16" else video1
        _cpu_time_step(orc, v)
        secs[name] = _cpu_time_step(orc, v)
    return min(secs, key=secs.get), secs


def run_reference_arm(args):
    """CPU baseline: the reference's torch-eager CPU path (restated oracle), all host threads, bounded sample:
    fp32 or bf16 storage (whichever these host cores run faster), 4 clips per step like the GPU arm when the
    K + W passes fit in ~3 minutes, else 1 clip (and a 5-frame clip if even that does not fit).
    With --dump-outputs the sample is fixed instead (fp32, one 17-frame clip), so that the dumped arrays do not depend
    on the speed of the host.  CPU kernels still differ between instruction sets, so dumps from different hosts agree
    to fp32 round-off, not bit for bit."""
    import torch
    import synth_data as Wt

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _best_cpu_threads()
    orcs = _cpu_oracles()
    frames = FRAMES
    if args.dump_outputs:
        dt_name, secs, sample_clips = "f32", {}, 1
    else:
        dt_name, secs = _cpu_pick_dtype(orcs, Wt.synth_video(1, 3, FRAMES, 128, seed=1))
        passes = args.steps + max(args.warmup, 0)
        sample_clips = CLIPS_PER_GPU
        if secs[dt_name] * sample_clips * passes > 180.0:
            sample_clips = 1
        if secs[dt_name] * sample_clips * passes > 180.0:
            frames = 5
    orc = orcs[dt_name]

    def mk(nclips):
        v = Wt.synth_video(nclips, 3, frames, 128, seed=1)
        return v.to(torch.bfloat16) if dt_name == "bf16" else v

    video = mk(sample_clips)
    if sample_clips > 1 and _cpu_time_step(orc, video) / sample_clips > secs[dt_name]:
        sample_clips = 1                       # these host cores run the single clip at a higher frame rate: time that
        video = mk(1)
    for _ in range(max(args.warmup, 0)):
        _cpu_time_step(orc, video)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        codes = orc.tokenize(video)
        recon = orc.decode_from_code_indices(codes)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, codes, recon)
    fps = sample_clips * frames * args.steps / dt
    probe = "1-clip probe: " + ", ".join(f"{k} {v:.2f} s" for k, v in secs.items()) if secs else "fixed for --dump-outputs"
    out = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dt_name, "data": "synthetic",
        "config": {"workload": "README VideoTokenizer (BASELINE configs[1]), tokenize+decode, CPU torch eager",
                   "clips_per_step": sample_clips},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{sample_clips} clip(s) ({frames}x128x128) per step, {dt_name} ({probe}), "
                                   f"{cores} threads, oracle/restated.py (torch CPU eager, same ATen ops the reference dispatches)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def cpu_baseline_sample():
    """Bounded CPU sample for the product arm's cpu_baseline object (rank 0, N=1 only): 1 clip and 4 clips, fp32 and
    bf16 storage; `value` is the best of them."""
    import torch
    import synth_data as Wt

    cores = _best_cpu_threads()
    orcs = _cpu_oracles()
    dt_name, secs = _cpu_pick_dtype(orcs, Wt.synth_video(1, 3, FRAMES, 128, seed=1))
    orc = orcs[dt_name]
    v4 = Wt.synth_video(CLIPS_PER_GPU, 3, FRAMES, 128, seed=1)
    if dt_name == "bf16":
        v4 = v4.to(torch.bfloat16)
    t4 = min(_cpu_time_step(orc, v4) for _ in range(2)) if secs[dt_name] * CLIPS_PER_GPU * 2 < 60.0 else None
    rates = {f"B=1 {k}": FRAMES / v for k, v in secs.items()}
    if t4 is not None:
        rates[f"B={CLIPS_PER_GPU} {dt_name}"] = CLIPS_PER_GPU * FRAMES / t4
    best = max(rates, key=rates.get)
    return {"value": rates[best], "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": "tokenize+decode of 17x128x128 clips, oracle/restated.py (torch CPU eager), frames/s: "
                      + ", ".join(f"{k}: {v:.2f}" for k, v in rates.items()) + f"; value = {best}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # default: 400 timed steps (~3 s, long enough to reach the power-limited clocks), 3 for the CPU arm
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)     # default: 5, 1 for the CPU arm
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="readme", choices=sorted(WORKLOADS))
    # consecutive steps (independent batches) are issued round-robin on this many CUDA streams, each replaying its own
    # CUDA-graph instances (magvit2_pytorch_b200.StreamLanes); 1 = strictly serial steps
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("MV2_LANES", "3")))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)
    args = ap.parse_args()
    cpu_arm = args.impl == "reference"
    if args.steps is None:
        args.steps = 3 if cpu_arm else 400
    if args.warmup is None:
        args.warmup = 1 if cpu_arm else 5
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if cpu_arm:
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import synth_data as Wt
    from magvit2_pytorch_b200 import VideoTokenizer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    args.warmup = max(args.warmup, 3)

    wl = WORKLOADS[args.workload]
    global CLIPS_PER_GPU, FLOP_PER_CLIP_ALL
    CLIPS_PER_GPU, FLOP_PER_CLIP_ALL = wl["clips"], wl["flop_clip"]
    torch.manual_seed(0)
    model = VideoTokenizer(**wl["kw"])
    Wt.fill_state_dict_(model, 0)
    model = model.to(dev).bfloat16().eval()
    model.cuda_graphs = True            # public opt-in: replay the static launch plan as one CUDA graph per entry point
    model.pdl = os.environ.get("MV2_PDL", "0") == "1"   # public opt-in: programmatic dependent launch between kernels
    eng = model.engine

    # inputs: NB distinct batches per rank so consecutive steps never re-read the same input from L2
    NB = 12
    if args.workload == "cfg4":
        NB = 4
    host_batches = [Wt.synth_video(CLIPS_PER_GPU, 3, FRAMES, wl["size"], seed=1000 + rank * NB + i).pin_memory() for i in range(NB)]
    dev_batches = [hb.to(dev, non_blocking=True) for hb in host_batches]
    torch.cuda.synchronize()

    train_mode = bool(wl.get("train_mode"))
    if train_mode:
        model.train()

    def step(v):
        if train_mode:           # reference M:1705 in training mode: the LFQ aux terms + their all-reduce run inside the call
            return model(v, return_codes=True, return_recon=True)
        codes = model.tokenize(v)
        return codes, model.decode_from_code_indices(codes)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from magvit2_pytorch_b200 import HostRoundTrip, StreamLanes
    nl = max(1, args.lanes)
    if args.workload == "cfg4" and "MV2_LANES" not in os.environ and args.lanes == 3:
        nl = 1     # measured (profiles/r02_bench_cfg4*.json): the 256^2 step is power limited (SM clock 1635 MHz with 3 lanes); 1 lane is faster
    lanes = StreamLanes(model, nl)
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()                      # streaming by the time the timed region begins (begin() below marks its start)
    for i in range(max(args.warmup, 3 * nl)):       # every lane: plain call, graph capture, first replay
        lanes.run(step, dev_batches[i % NB])
    lanes.join()
    # ---------------- timed region: inputs resident in HBM ----------------
    barrier()
    if rank == 0:
        clk.begin()
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last, _ = lanes.run(step, dev_batches[i % NB])
    lanes.join()                         # the timing stream waits for every lane: all K steps end inside the timed region
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launches - l0
    clocks = clk.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        # copied before any later call: with CUDA graphs the results live in the lane's static output buffers
        dump_outputs(args.dump_outputs, *last)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = t.item()
    frames_total = world * CLIPS_PER_GPU * FRAMES * args.steps
    value = frames_total / (ms_max / 1e3)

    # ---------------- e2e: host (pinned) buffers in, host buffers out, copies inside the timed region ----
    fm = wl["size"] // 8
    out_codes = torch.empty((CLIPS_PER_GPU, 5, fm, fm), dtype=torch.int32 if wl["kw"].get("use_fsq") else torch.int64).pin_memory()
    out_video = torch.empty((CLIPS_PER_GPU, 3, FRAMES, wl["size"], wl["size"]), dtype=torch.bfloat16).pin_memory()

    # two result buffers alternate so a step never overwrites host results whose copy may still be in flight;
    # HostRoundTrip (the package's pinned-host front end) runs copy-in / kernels / copy-out on three streams, so the
    # copies of neighbouring steps overlap this step's kernels -- every step still copies its own input and results
    out_bufs = [(out_codes, out_video), (torch.empty_like(out_codes).pin_memory(), torch.empty_like(out_video).pin_memory())]
    depth = max(2, nl)           # one staging slot per lane (two per lane measured 2 % slower: profiles/README.md)
    out_bufs += [(torch.empty_like(out_codes).pin_memory(), torch.empty_like(out_video).pin_memory()) for _ in range(depth - 2)]
    hrt = HostRoundTrip(model, depth=depth, train_mode_forward=train_mode, lanes=nl)
    cur = torch.cuda.current_stream()

    def step_e2e(i):
        oc, ov = out_bufs[i % depth]
        return hrt.submit(host_batches[i % NB], oc, ov)

    for i in range(3 * depth):
        step_e2e(i)
    barrier()
    e0.record()
    for i in range(args.steps):
        step_e2e(i)
    hrt.join()                           # every device->host copy (all slots) is inside the timed region
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = frames_total / (t.item() / 1e3)
    h2d = host_batches[0].numel() * host_batches[0].element_size()
    d2h = out_codes.numel() * out_codes.element_size() + out_video.numel() * 2

    # ---------------- roofline of the dominant kernel (tcgen05 implicit-GEMM conv), timed live ----------
    # instrumented pass: CUDA events around every conv launch of one step, on the launching stream
    peaks, peaks_src = _peaks()
    roofline = None
    model.cuda_graphs = False            # the instrumented pass needs one event pair per launch
    prof = eng.profile_convs(lambda: step(dev_batches[0]), steps=3)
    model.cuda_graphs = True
    if prof.get("conv3d"):
        ms3, n3, fl3 = prof["conv3d"]
        msa, na, fla = prof["all"]
        ach = fl3 / (ms3 / 1e3) / 1e12
        # which measured peak applies (B200_PROFILING.md): the burst figure while the SM clock holds its maximum (short
        # timed region, no power cap seen), the sustained one once the run is long enough to be power limited
        pk_burst, pk_sus = peaks["bf16_tflops"], peaks["bf16_tflops_sustained"]
        sm_now, sm_max = (clocks or {}).get("sm_mhz"), (clocks or {}).get("sm_max_mhz")
        # (sw_power_cap shows up within milliseconds on this path, but the clock only dips ~2 %: the cuBLAS "sustained" figure
        #  was taken at a 1387 MHz median and does not describe that regime, so the decision is made on the clock itself)
        power_limited = bool(sm_now and sm_max and sm_now < 0.90 * sm_max)
        pk = pk_sus if power_limited else pk_burst
        traffic = None
        try:     # dram__bytes_read + write per conv3d launch, from the committed ncu capture of one step (profiles/)
            if args.workload == "readme":
                traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_step_metrics_summary.json")))["conv3d"]["avg_dram_bytes"]
        except Exception:
            traffic = None
        roofline = {"bound": "tensor", "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk, "traffic": traffic,
                    "frac_of_burst_peak": ach / pk_burst, "frac_of_sustained_peak": ach / pk_sus,
                    "kernel": "tc_slab_kernel on the causal 3x3x3 Conv3d layers (82% of the step's FLOPs)",
                    "launches_per_step": n3, "kernel_ms_per_step": ms3, "flop_per_launch_avg": fl3 / max(n3, 1),
                    "flops": "algorithmic: 2*B*T*H*W*Co*Ci*kt*kh*kw per launch (conv_in counted with its 3x7x7x7 taps, not the padded K)",
                    "peak_source": f"MEASURED_PEAKS.json {'bf16_tflops_sustained (SM clock fell below 90% of max: power-limited run)' if power_limited else 'bf16_tflops (burst figure: the SM clock stayed within 10% of its maximum during the timed region)'} ({peaks_src})",
                    "all_tcgen05_launches": {"launches_per_step": na, "ms_per_step": msa,
                                             "achieved": fla / (msa / 1e3) / 1e12, "frac": fla / (msa / 1e3) / 1e12 / pk},
                    "whole_step_frac": (FLOP_PER_CLIP_ALL * CLIPS_PER_GPU * world * args.steps / (ms_max / 1e3) / 1e12)
                                       / (pk * world)}

    if world > 1:
        dist.barrier()
    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["name"],
                       "global_batch": CLIPS_PER_GPU * world, "parallelism": f"dp{world}",
                       "lanes": f"{nl} CUDA stream lane(s) per GPU: consecutive steps (independent batches) overlap on the device; "
                                "ms_per_step = timed region / steps",
                       "l2": f"inputs rotate over {NB} distinct batches per rank ({NB * h2d / 1e6:.0f} MB > 126 MB L2); "
                             "per-step activation working set ~2 GB"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "magvit2_pytorch_b200.HostRoundTrip.submit(pinned video, pinned codes out, pinned video out): "
                           f"H2D / kernels / D2H on separate streams, {depth} device staging slots, {nl} compute lane(s); every step "
                           "copies its own fp32 input in and its codes + bf16 reconstruction out"},
            "gpu_launches": launches,
            "roofline": roofline,
        }
        if world == 1 and not args.no_cpu_baseline and args.workload == "readme":
            out["cpu_baseline"] = cpu_baseline_sample()
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
