"""The training forward runs the inference path's own steps (conv_in, the stages, the quantiser, conv_out), so its
reconstruction and codes equal those of an eval-mode forward on the same weights and clip, bit for bit."""
import pytest
import torch

from magvit2_pytorch_b200 import train as T
from tests.util import build_product, golden_video, load_golden

pytestmark = pytest.mark.gpu


def _train_vs_eval(name, dtype=torch.float32, **engine_flags):
    assert torch.cuda.is_available()
    g = load_golden(name)
    model = build_product(g["kwargs"], g["wseed"]).cuda().to(dtype)
    video = golden_video(g).cuda().to(dtype)
    cond = g["cond"].cuda() if g.get("cond") is not None else None
    model.train()
    recon, _, codes, _ = T.train_forward(model, video, cond=cond)
    model.eval()
    for k, v in engine_flags.items():
        setattr(model.engine, k, v)
    with torch.no_grad():
        if cond is None:
            want_recon = model(video, return_recon=True)
            want_codes = model.tokenize(video)
        else:
            want_recon = model(video, cond=cond, return_recon=True)
            want_codes = model(video, cond=cond, return_codes=True)
    assert recon.dtype == want_recon.dtype and torch.equal(recon.detach(), want_recon), name
    assert torch.equal(codes, want_codes), name


@pytest.mark.parametrize("name", ["mini_train", "mini_fsq_train", "mini_sff_train", "pad_reflect_train", "mini_cond_train",
                                  "mini_gateloop_train"])
def test_fp32_training_forward_equals_inference(name):
    _train_vs_eval(name)


def test_bf16_training_forward_equals_inference():
    """The training forward runs each ResidualUnit unfused (its backward needs the intermediate activations), so the
    eval-mode forward it is compared with does too."""
    _train_vs_eval("mini_train", torch.bfloat16, fuse_ru=False)
