"""bench.py's reference arm (the CPU leg the driver runs as `bench.py --impl reference`) prints exactly one JSON line
with the contract's keys.  CPU only; one 1-clip step of the oracle (~10 s)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "frames/s" and d["higher_is_better"] is True and d["steps"] == 1
    assert d["value"] > 0 and abs(d["value"] - d["cpu_baseline"]["value"]) < 1e-9
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]
    codes, recon = np.load(tmp_path / "codes.npy"), np.load(tmp_path / "recon.npy")
    assert codes.dtype == np.float64 and recon.dtype == np.float32
    # the sample is fixed when dumping, whatever the speed of the host: fp32, one 17x128x128 clip
    assert d["dtype"] == "f32" and codes.shape == (1, 5, 16, 16) and recon.shape == (1, 3, 17, 128, 128)
    assert np.isfinite(recon).all()


def test_dump_outputs_samples_a_reconstruction_over_the_size_cap(tmp_path, monkeypatch):
    """Outputs above bench.DUMP_MAX_BYTES are written as a fixed, seeded sample: within the cap, the same elements on
    every call, each one a value of the reconstruction; the codes stay whole."""
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4096)
    codes = torch.arange(24).reshape(2, 3, 4)
    recon = torch.randn(2, 3, 5, 16, 16, generator=torch.Generator().manual_seed(0)).bfloat16()
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), codes, recon)
    c = np.load(tmp_path / "a" / "codes.npy")
    ra, rb = np.load(tmp_path / "a" / "recon.npy"), np.load(tmp_path / "b" / "recon.npy")
    assert np.array_equal(c, codes.double().numpy())
    assert ra.dtype == np.float32 and ra.ndim == 1 and 4096 - 4 < c.nbytes + ra.nbytes <= 4096
    assert np.array_equal(ra, rb)
    assert np.isin(ra, recon.float().numpy()).all()


@pytest.mark.gpu
def test_dump_outputs_are_what_the_last_timed_step_returned(tmp_path):
    """--dump-outputs after --steps 2 holds exactly what tokenize + decode_from_code_indices return for the second seeded
    batch (bench.py: step i reads batch i % 12, seed 1000 + i), called directly on a model with the same weights."""
    import torch
    import synth_data as Wt
    from bench import FRAMES, README_KW
    from magvit2_pytorch_b200 import VideoTokenizer
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    codes, recon = np.load(tmp_path / "codes.npy"), np.load(tmp_path / "recon.npy")
    assert codes.dtype == np.float64 and recon.dtype == np.float32

    torch.manual_seed(0)
    model = VideoTokenizer(**README_KW)
    Wt.fill_state_dict_(model, 0)
    model = model.cuda().bfloat16().eval()
    video = Wt.synth_video(4, 3, FRAMES, 128, seed=1001).cuda()
    want_codes = model.tokenize(video)
    want_recon = model.decode_from_code_indices(want_codes)
    assert np.array_equal(codes, want_codes.cpu().double().numpy())
    assert np.array_equal(recon, want_recon.float().cpu().numpy())


def test_own_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: without CUDA the product arm must exit non-zero instead of timing the oracle."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("needs a machine without a GPU")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-cpu-baseline"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert not any(l.startswith("{") and '"value"' in l for l in out.stdout.splitlines())
