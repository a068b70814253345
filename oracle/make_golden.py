"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.pt by running the UNMODIFIED
reference (imported from /root/reference through oracle/ref_loader.py) on CPU.
Runs only in the build container:   python -m oracle.make_golden [names...]

Each fixture pins, for one constructor config + synthetic-weight seed + input
seed: the reference's code indices, the quantiser's pre-sign/bounded values
(captured with a forward hook on the reference's own project_in), the
reconstructed video (full for small configs, a strided sample for the README
config) and a strided sample of every encoder/decoder layer output (forward
hooks on the reference's own modules) for bisecting.

Third-party arithmetic caveat: LFQ/FSQ/Taylor attention come from
oracle/shims (restated; the real PyPI packages are not installable here).
"""
from __future__ import annotations

import os
import sys
import time

import torch

from oracle import weights as W
from oracle.ref_loader import build_reference_tokenizer

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

README_LAYERS = (
    "residual", "compress_space", ("consecutive_residual", 2), "compress_space",
    ("consecutive_residual", 2), "linear_attend_space", "compress_space",
    ("consecutive_residual", 2), "attend_space", "compress_time",
    ("consecutive_residual", 2), "compress_time", ("consecutive_residual", 2), "attend_time",
)

CONFIGS = {
    # BASELINE.json configs[0]
    "cfg1": dict(kwargs=dict(image_size=32, init_dim=16, codebook_size=1024,
                             layers=("residual", "compress_space")),
                 video=(1, 3, 5, 32, 32), wseed=0, vseed=1243, full=True),
    # every layer type of the README spec at toy size (tdf=4 -> 9 frames)
    "mini": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, layers=README_LAYERS),
                 video=(2, 3, 9, 32, 32), wseed=0, vseed=1234, full=True),
    "mini_fsq": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, use_fsq=True, fsq_levels=[8, 5, 5, 5],
                                 layers=README_LAYERS),
                     video=(2, 3, 9, 32, 32), wseed=0, vseed=1234, full=True),
    # BASELINE.json configs[1] (README), one clip.  Tap channel stride 32 (readme / readme_bf16 and cfg4 / cfg4_bf16) keeps
    # each fixture under 1 MB; an fp32 golden and its bf16 twin must use the same strides
    "readme": dict(kwargs=dict(image_size=128, init_dim=64, max_dim=512, codebook_size=1024, layers=README_LAYERS),
                   video=(1, 3, 17, 128, 128), wseed=0, vseed=1234, full=False, cs=32, ss=8),
    # SURVEY 8f N1: the one conditioned layer type that runs in the reference (cond_residual = ResidualUnitMod /
    # Conv3DMod, M:680-753, M:946-988).  Conditioned layers must be the trailing ones (has_cond is never reset, M:1153).
    "mini_cond": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, dim_cond=12,
                                  layers=("residual", "compress_space", "compress_time", "cond_residual", "cond_residual")),
                      video=(2, 3, 5, 32, 32), wseed=0, vseed=1249, cseed=77, full=True),   # vseed chosen for min |pre-sign| = 2.3e-4
    # SURVEY 8f N3: separate_first_frame_encoding (M:1113-1120, M:1553-1561, M:1633-1639)
    # --- reference run as model.bfloat16() (SURVEY 8d parity protocol (ii)): the bf16 product path is judged against the
    #     reference's OWN bf16 deviation from fp32, layer by layer.  Decode is run on the fp32 golden's codes ("identical
    #     codes fed to both sides"); the tokenize side stores the bf16 reference's own codes / pre-sign values.
    "readme_bf16": dict(kwargs=dict(image_size=128, init_dim=64, max_dim=512, codebook_size=1024, layers=README_LAYERS),
                        video=(1, 3, 17, 128, 128), wseed=0, vseed=1234, full=False, cs=32, ss=8, dtype="bf16",
                        codes_from="readme"),
    "mini_bf16": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, layers=README_LAYERS),
                      video=(2, 3, 9, 32, 32), wseed=0, vseed=1234, full=True, dtype="bf16", codes_from="mini"),
    # BASELINE.json configs[3]: image 256, max_dim 1024 (attention-heavy: space-attention seq 1024, linear-attention seq 4096)
    "cfg4": dict(kwargs=dict(image_size=256, init_dim=64, max_dim=1024, codebook_size=1024, layers=README_LAYERS),
                 video=(1, 3, 17, 256, 256), wseed=0, vseed=1234, full=False, cs=32, ss=16, rs=8),
    "cfg4_bf16": dict(kwargs=dict(image_size=256, init_dim=64, max_dim=1024, codebook_size=1024, layers=README_LAYERS),
                      video=(1, 3, 17, 256, 256), wseed=0, vseed=1234, full=False, cs=32, ss=16, rs=8, dtype="bf16",
                      codes_from="cfg4"),
    # BASELINE.json configs[4]: FSQ variant of the README config, levels [8,5,5,5] (SURVEY 8d)
    "fsq": dict(kwargs=dict(image_size=128, init_dim=64, max_dim=512, use_fsq=True, fsq_levels=[8, 5, 5, 5], layers=README_LAYERS),
                video=(1, 3, 17, 128, 128), wseed=0, vseed=1234, full=False, cs=16, ss=8),
    "fsq_bf16": dict(kwargs=dict(image_size=128, init_dim=64, max_dim=512, use_fsq=True, fsq_levels=[8, 5, 5, 5], layers=README_LAYERS),
                     video=(1, 3, 17, 128, 128), wseed=0, vseed=1234, full=False, cs=16, ss=8, dtype="bf16", codes_from="fsq"),
    # video_contains_first_frame=False (M:1528-1537, M:1646-1647, M:1691): 8 frames, no front padding, no crop
    "mini_noff": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, layers=README_LAYERS),
                      video=(2, 3, 8, 32, 32), wseed=0, vseed=1235, full=True, first_frame=False),
    # pad_mode of conv_in / conv_out (M:925-927, M:1109, M:1127): F.pad modes other than 'constant'
    "pad_reflect": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, pad_mode="reflect",
                                    layers=("residual", "compress_space", "compress_time", "residual")),
                        video=(2, 3, 9, 32, 32), wseed=0, vseed=1236, full=True),
    "pad_replicate": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, pad_mode="replicate",
                                      layers=("residual", "compress_space", "compress_time", "residual")),
                          video=(2, 3, 9, 32, 32), wseed=0, vseed=1236, full=True),
    "pad_circular": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, pad_mode="circular",
                                     layers=("residual", "compress_space", "compress_time", "residual")),
                         video=(2, 3, 9, 32, 32), wseed=0, vseed=1236, full=True),
    # SURVEY 8f N3: gateloop_time (M:1216-1222; SimpleGateLoopLayer through oracle/shims/gateloop.py)
    "mini_gateloop": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024,
                                      layers=("residual", "compress_space", "gateloop_time", "compress_time", "gateloop_time", "residual")),
                          video=(2, 3, 9, 32, 32), wseed=0, vseed=1237, full=True),
    # num_codebooks > 1 (M:1057 -> M:1367 / M:1381) and lfq_spherical (M:1070 -> M:1372): indices keep a trailing codebook axis
    "mini_mc": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=256, num_codebooks=2, lfq_spherical=True,
                                layers=("residual", "compress_space", "compress_time", "residual")),
                    video=(2, 3, 5, 32, 32), wseed=0, vseed=1238, full=True),
    "mini_mc_fsq": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, use_fsq=True, fsq_levels=[8, 5, 5], num_codebooks=2,
                                    layers=("residual", "compress_space", "compress_time", "residual")),
                        video=(2, 3, 5, 32, 32), wseed=0, vseed=1238, full=True),
    "mini_sff": dict(kwargs=dict(image_size=32, init_dim=16, max_dim=64, codebook_size=1024, separate_first_frame_encoding=True,
                                 layers=("residual", "compress_space", "compress_time", "residual")),
                     video=(2, 3, 5, 32, 32), wseed=0, vseed=1234, full=True),
}


def _sample(t: torch.Tensor, cs: int = 7, ss: int = 5) -> torch.Tensor:
    """Strided sample of a (B,C,T,H,W) tensor: all b, every cs-th channel, all t, every ss-th row/col."""
    return t[:, ::cs, :, ::ss, ::ss].contiguous().clone()


def make(name: str):
    cfg = CONFIGS[name]
    kwargs = dict(cfg["kwargs"])
    torch.manual_seed(0)
    model = build_reference_tokenizer(**kwargs)
    W.fill_state_dict_(model, cfg["wseed"])
    model.eval()
    video = W.synth_video(*cfg["video"][:3], cfg["video"][3], seed=cfg["vseed"])
    bf16 = cfg.get("dtype") == "bf16"
    if bf16:
        model = model.bfloat16()
        video = video.bfloat16()

    taps = {}
    hooks = []

    def tap(nm):
        def fn(mod, inp, out):
            taps[nm] = _sample(out.detach().float(), cfg.get("cs", 7), cfg.get("ss", 5))
        return fn

    hooks.append(model.conv_in.register_forward_hook(tap("conv_in")))
    n_layers = len(kwargs["layers"])
    for i in range(n_layers):
        hooks.append(model.encoder_layers[i].register_forward_hook(tap(f"enc{i}")))
        hooks.append(model.decoder_layers[i].register_forward_hook(tap(f"dec{i}")))
    presign = {}

    def grab_proj(mod, inp, out):
        presign["proj"] = out.detach().clone()

    hooks.append(model.quantizers.project_in.register_forward_hook(grab_proj))

    cond = None
    if kwargs.get("dim_cond") is not None:
        g = torch.Generator(device="cpu")
        g.manual_seed(cfg["cseed"])
        cond = torch.randn(cfg["video"][0], kwargs["dim_cond"], generator=g)
        hooks.append(model.encoder_cond_in.register_forward_hook(lambda m, i, o: taps.__setitem__("enc_cond_in", o.detach().clone())))
    t0 = time.time()
    with torch.no_grad():
        # tokenize() does not forward ``cond`` (M:1651-1654): conditioned specs use forward(return_codes=True)
        ff = cfg.get("first_frame", True)
        if not ff:
            codes = model(video, return_codes=True, video_contains_first_frame=False)
        else:
            codes = model.tokenize(video) if cond is None else model(video, cond=cond, return_codes=True)
        t1 = time.time()
        codes_dec = codes
        if cfg.get("codes_from"):      # decode the fp32 golden's codes, so both dtypes decode identical tokens
            codes_dec = torch.load(os.path.join(GOLDEN_DIR, cfg["codes_from"] + ".pt"), weights_only=False)["codes"]
        recon = model.decode_from_code_indices(codes_dec, cond=cond, video_contains_first_frame=ff).float()
        t2 = time.time()
        if not bf16 and ff:
            # README.md:85-90 round-trip statement
            recon_fwd = model(video, cond=cond, return_recon=True)
            assert torch.equal(recon, recon_fwd), "reference round-trip (README.md:87-90) does not hold"
    for h in hooks:
        h.remove()

    proj = presign["proj"].float()
    if kwargs.get("use_fsq", False):
        pre = proj   # raw project_in output; bounding is re-derived by the checker
    else:
        pre = (proj / 10.).tanh() * 10.
        if kwargs.get("lfq_spherical"):
            nc_ = kwargs.get("num_codebooks", 1)
            pre = torch.nn.functional.normalize(pre.reshape(*pre.shape[:-1], nc_, -1), dim=-1).reshape(pre.shape)
    out = dict(
        name=name, kwargs=kwargs, video_shape=tuple(cfg["video"]), wseed=cfg["wseed"], vseed=cfg["vseed"],
        codes=codes.clone(), presign=pre.clone(),
        taps=taps, tap_strides=(cfg.get("cs", 7), cfg.get("ss", 5)),
        recon_sample=recon[:, :, :, ::cfg.get("rs", 4), ::cfg.get("rs", 4)].contiguous().clone(), recon_stride=cfg.get("rs", 4),
        recon_mean=recon.mean(dim=(3, 4)).clone(),
        ref_seconds=dict(tokenize=t1 - t0, decode=t2 - t1),
        torch_version=torch.__version__,
        cond=cond,
        # generator state_dict layout of the reference (key -> shape; integer buffers by value): lets a checker rebuild the
        # synthetic weights (oracle/weights.py) for specs the product does not construct yet
        sd_shapes={k: tuple(v.shape) for k, v in model.state_dict().items() if W.is_generator_key(k) and v.is_floating_point()},
        sd_buffers={k: v.clone() for k, v in model.state_dict().items() if W.is_generator_key(k) and not v.is_floating_point()},
        dtype="bf16" if bf16 else "fp32", codes_decoded=codes_dec.clone(), first_frame=ff,
        reference_commit="a00519fa (v0.5.1)",
        third_party="oracle/shims (restated LFQ/FSQ/TaylorSeriesLinearAttn; real packages unavailable)",
    )
    if cfg["full"]:
        out["recon"] = recon.clone()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    path = os.path.join(GOLDEN_DIR, f"{name}.pt")
    torch.save(out, path)
    amin = pre.abs().min().item()
    print(f"[golden] {name}: codes {tuple(codes.shape)} {codes.dtype}, min|presign|={amin:.3e}, "
          f"recon absmax={recon.abs().max().item():.3f}, tokenize {t1 - t0:.2f}s decode {t2 - t1:.2f}s, "
          f"{os.path.getsize(path) / 1e3:.0f} KB")


if __name__ == "__main__":
    names = sys.argv[1:] or list(CONFIGS)
    for n in names:
        make(n)
