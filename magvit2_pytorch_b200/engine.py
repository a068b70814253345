"""Host-side executor: walks the VideoTokenizer layer schedule and launches the sm_100a
kernels of libmagvit2_b200.so through the C ABI (ctypes).  PyTorch is used only for device
memory (caching allocator), streams and parameter storage.

Activations are channels-last (B, T, H, W, C) tensors in the compute dtype (fp32 -> CUDA-core
path, bf16 -> tcgen05 tensor-core path for the dense contractions).  There is no eager / CPU
fallback: every op is a library call and a missing library is an error.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib
from ._lib import (ACT_ELU, ACT_NONE, ACT_SILU, MV2_BF16, MV2_F32, MV2_U8, SHUFFLE_NONE, SHUFFLE_SPACE,
                   SHUFFLE_TIME, AttnArgs, ConvArgs, TcConvArgs, TcRuArgs, check)


def _dt(t: torch.dtype) -> int:
    if t == torch.float32:
        return MV2_F32
    if t == torch.bfloat16:
        return MV2_BF16
    raise TypeError(f"unsupported dtype {t} (only float32 and bfloat16)")


def _src_dt(t: torch.dtype) -> int:
    """dtype code of a layout-in SOURCE tensor: uint8 frames are accepted there (normalised x / 255 on the fly)."""
    return MV2_U8 if t == torch.uint8 else _dt(t)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


@dataclass
class ConvPack:
    """One convolution's parameters in kernel layout."""
    w: torch.Tensor              # [taps][Ci][Co] in the compute dtype (CUDA-core path)
    bias: Optional[torch.Tensor]  # fp32 [Co]
    k: Tuple[int, int, int]
    Ci: int
    Co: int
    w_tc: Optional[torch.Tensor] = None      # [Co][taps*Ci] bf16, K-major (tcgen05 path); rows permuted for shuffles
    bias_tc: Optional[torch.Tensor] = None   # bias in w_tc's row order
    Ci_tc: int = 0                           # GEMM dims of the tcgen05 call (may be padded / re-paired)
    Co_tc: int = 0
    epi_mode: int = 0                        # 1: fused GEGLU (output has Co_tc // 2 channels)
    k_tc: Optional[Tuple[int, int, int]] = None
    macs: int = 0                            # algorithmic multiply-accumulates per output position (Co * Ci * taps, unpadded)
    w_down: Optional[torch.Tensor] = None    # SpatialDownsample2x pack for mv2_tc_down_space_forward ([Co][6][2*Ci] bf16)


def pack_conv(weight: torch.Tensor, bias: Optional[torch.Tensor], dtype, k=None, shuffle_q: int = 1) -> ConvPack:
    """weight: torch layout (Co, Ci, *kernel).  Kernel dims are mapped onto (kt, kh, kw) by `k`.
    shuffle_q = 4 / 2 for the depth-to-space / depth-to-time up-samplers: the tcgen05 kernel wants output
    rows ordered (q, c) instead of the reference's (c, q) so shuffled stores are channel-contiguous."""
    Co, Ci = weight.shape[:2]
    if k is None:
        ks = tuple(weight.shape[2:])
        k = (1,) * (3 - len(ks)) + ks
    w3 = weight.detach().reshape(Co, Ci, -1)
    w = w3.permute(2, 1, 0).contiguous().to(dtype)
    b = None if bias is None else bias.detach().float().contiguous()
    pk = ConvPack(w=w, bias=b, k=tuple(int(v) for v in k), Ci=int(Ci), Co=int(Co))
    pk.macs = int(Co) * int(Ci) * int(w3.shape[2])
    if dtype == torch.bfloat16:
        wt = w3.permute(0, 2, 1).reshape(Co, -1)                      # [Co][tap*Ci + ci]
        bt = b
        if shuffle_q > 1:
            cy = Co // shuffle_q
            wt = wt.reshape(cy, shuffle_q, -1).permute(1, 0, 2).reshape(Co, -1)
            bt = None if b is None else b.reshape(cy, shuffle_q).t().reshape(Co).contiguous()
        pk.w_tc = wt.contiguous().to(torch.bfloat16)
        pk.bias_tc = bt
        pk.Ci_tc, pk.Co_tc, pk.k_tc = pk.Ci, pk.Co, pk.k
    return pk


def pack_conv_down_space(pk: ConvPack, weight):
    """SpatialDownsample2x (M:768: Conv2d k3 s2 p1) for mv2_tc_down_space_forward: w[co][tap'][2*Ci], tap' = dh * 2 + q,
    q = 0 -> [zeros | w[:, :, dh, 0]] (the column left of the pair), q = 1 -> [w[:, :, dh, 1] | w[:, :, dh, 2]]."""
    Co, Ci, kh, kw = weight.shape
    if (kh, kw) != (3, 3) or Ci % 64 != 0 or Co % 32 != 0:
        return
    w = weight.detach().float()
    wd = torch.zeros((Co, 3, 2, 2 * Ci), device=w.device)
    wd[:, :, 0, Ci:] = w[:, :, :, 0].permute(0, 2, 1)
    wd[:, :, 1, :Ci] = w[:, :, :, 1].permute(0, 2, 1)
    wd[:, :, 1, Ci:] = w[:, :, :, 2].permute(0, 2, 1)
    pk.w_down = wd.reshape(Co, 6 * 2 * Ci).contiguous().to(torch.bfloat16)


def _round_up(v, m):
    return (v + m - 1) // m * m


def pack_ff(fc1_w, fc1_b, fc2_w, fc2_b, dtype):
    """FeedForward weights (reference M:492-496).  tcgen05 layout: the hidden width I is padded to a multiple of 64,
    fc1's rows are re-paired as [8 x-rows, their 8 gate-rows] per group of 16 so GEGLU (M:466-469) fuses into fc1's
    epilogue, and fc2's K is zero-padded to match."""
    fc1 = pack_conv(fc1_w, fc1_b, dtype)
    fc2 = pack_conv(fc2_w, fc2_b, dtype)
    if dtype == torch.bfloat16:
        two_i, C_ = fc1_w.shape[:2]
        I = two_i // 2
        Ip = _round_up(I, 64)
        w1 = fc1_w.detach().reshape(two_i, C_).float()
        b1 = fc1_b.detach().float()
        wx = torch.zeros((Ip, C_), device=w1.device)
        wg = torch.zeros((Ip, C_), device=w1.device)
        bx = torch.zeros((Ip,), device=w1.device)
        bg = torch.zeros((Ip,), device=w1.device)
        wx[:I], wg[:I], bx[:I], bg[:I] = w1[:I], w1[I:], b1[:I], b1[I:]
        wp = torch.stack((wx.reshape(Ip // 8, 8, C_), wg.reshape(Ip // 8, 8, C_)), dim=1).reshape(2 * Ip, C_)
        bp = torch.stack((bx.reshape(Ip // 8, 8), bg.reshape(Ip // 8, 8)), dim=1).reshape(2 * Ip)
        fc1.w_tc, fc1.bias_tc = wp.contiguous().to(torch.bfloat16), bp.contiguous()
        fc1.Ci_tc, fc1.Co_tc, fc1.epi_mode = int(C_), 2 * Ip, 1
        w2 = fc2_w.detach().reshape(fc2_w.shape[0], I).float()
        w2p = torch.zeros((w2.shape[0], Ip), device=w2.device)
        w2p[:, :I] = w2
        fc2.w_tc = w2p.contiguous().to(torch.bfloat16)
        fc2.Ci_tc, fc2.Co_tc = Ip, int(w2.shape[0])
    return fc1, fc2


def pack_conv_in_kwpack(weight, bias, cpack=32):
    """conv_in (M:1109) for the tcgen05 path: (Co, Cin, kt, kh, kw) -> [Co][(dt, dh)][dw * Cin + c], zero padded to
    `cpack` channels -- pairs with mv2_ingest_kwpack."""
    Co, Cin, kt, kh, kw = weight.shape
    if Cin * kw > cpack:
        return None
    w = weight.detach().float().permute(0, 2, 3, 4, 1).reshape(Co, kt * kh, kw * Cin)
    wp = torch.zeros((Co, kt * kh, cpack), device=w.device)
    wp[:, :, :kw * Cin] = w
    pk = ConvPack(w=None, bias=None, k=(kt, kh, 1), Ci=cpack, Co=int(Co))
    pk.w_tc = wp.reshape(Co, kt * kh * cpack).contiguous().to(torch.bfloat16)
    pk.bias_tc = None if bias is None else bias.detach().float().contiguous()
    pk.Ci_tc, pk.Co_tc, pk.k_tc = cpack, int(Co), (kt, kh, 1)
    pk.kw_orig, pk.cin_orig = int(kw), int(Cin)
    pk.macs = int(Co) * int(Cin) * int(kt * kh * kw)          # the padded K (cpack x kt x kh) is not algorithmic work
    return pk


def stage_modules(st, mod, decoder: bool) -> dict:
    """Where a stage's parameters sit inside its layer module `mod` (the reference's nesting, M:1138-1318), by role.  Read by
    Engine.prepare, which packs them, and by the training path, which differentiates them."""
    if st.kind == "residual":       # Residual(Sequential(CausalConv3d, ELU, Conv3d 1x1x1, ELU, SqueezeExcite)) (M:930-944)
        return dict(units=[dict(conv3=ru.fn[0].conv, conv1=ru.fn[2], se=ru.fn[4]) for ru in (list(mod) if st.nested else [mod])])
    if st.kind == "cond_residual":
        return dict(unit=mod)
    if st.kind in ("compress_space", "compress_time"):
        return dict(conv=mod.net[0] if decoder else mod.conv)
    if st.kind in ("attend_space", "linear_attend_space"):      # Residual(attention), Residual(FeedForward)
        return dict(attn=mod[0].fn, ff=mod[1].fn)
    if st.kind == "attend_time":                               # Residual(TokenShift(...)) for both blocks
        return dict(attn=mod[0].fn.fn, ff=mod[1].fn.fn)
    if st.kind == "gateloop_time":                             # ToTimeSequence(Residual(SimpleGateLoopLayer))
        return dict(gateloop=mod.fn.fn)
    raise ValueError(st.kind)


class Engine:
    """Executes the inference path of one VideoTokenizer on its parameters' device/dtype."""

    def __init__(self, model):
        self.model = model
        self.lib = _lib.load()
        self._packs: Dict[str, object] = {}
        self._sig = None
        self._sig_id = 0             # bumped whenever parameters are re-packed (invalidates cached CUDA graphs)
        self.launches = 0            # kernels launched through the C ABI (bench's gpu_launches)
        self.use_tc = True           # bf16: dense contractions on tcgen05 (False -> CUDA-core cross-check path)
        self.tc_variant = "auto"     # "auto" | "tap" (tc_conv.cu only) | "slab" (prefer tc_slab.cu)
        self.fuse_ru = True          # bf16: conv3x3x3 + ELU + conv1x1x1 + ELU + SE pool partials in one tcgen05 launch (C = 64 / 128)
        self.fused_ru_calls = 0
        # bf16, small frames: SE pool + gate MLP + gate/residual in ONE launch (mv2_se_tail).  Off by default: measured 38 us per
        # unit at C = 512 / 16x16 (one CTA per frame is instruction-issue bound: ncu issue-active 49 %, 7.7 k warp instructions
        # per warp) against 36 us for the four small launches under graph replay (profiles/r02_se_tail.json)
        self.se_tail = False
        self.se_tail_calls = 0
        self.fuse_conv_out = True    # bf16: conv_out stores torch's (B,C,T,H,W) directly and skips the time_padding frames
        self.tc_calls = 0
        self.slab_calls = 0
        self.simt_conv_calls = 0
        self.taps: Optional[dict] = None  # when set, per-stage activations are recorded (tests)
        self._prof: Optional[list] = None  # when set, (event0, event1, flops) per tcgen05 conv launch
        self.conv_log: Optional[list] = None  # when set, one shape record per tcgen05 conv launch (tools/step_breakdown.py)

    # ------------------------------------------------------------------ parameters
    def _signature(self):
        ps = list(self.model.parameters())
        return (tuple((p.data_ptr(), p._version) for p in ps), ps[0].dtype, ps[0].device)

    def prepare(self):
        """(Re)pack parameters into kernel layouts when they changed (load_state_dict, .to(), ...)."""
        sig = self._signature()
        if sig == self._sig:
            return
        m = self.model
        p0 = m.conv_in.conv.weight
        if p0.device.type != "cuda":
            raise RuntimeError("magvit2_pytorch_b200.VideoTokenizer runs on CUDA (sm_100a) only; "
                               "move the model with .cuda() -- there is no CPU fallback")
        if p0.dtype not in (torch.float32, torch.bfloat16):
            raise TypeError("parameters must be float32 or bfloat16")
        arch = self.lib.mv2_device_arch()
        if arch < 100:
            raise RuntimeError(f"libmagvit2_b200.so targets sm_100a; device reports sm_{arch}")
        self.dtype = p0.dtype
        self.device = p0.device
        dt = self.dtype
        P: Dict[str, object] = {}
        P["conv_in"] = pack_conv(m.conv_in.conv.weight, m.conv_in.conv.bias, dt)
        P["conv_in_tc"] = pack_conv_in_kwpack(m.conv_in.conv.weight, m.conv_in.conv.bias) if dt == torch.bfloat16 else None
        P["conv_out"] = pack_conv(m.conv_out.conv.weight, m.conv_out.conv.bias, dt)
        if m.separate_first_frame_encoding:       # SameConv2d (M:887-890): a (1, kh, kw) conv on the single first frame
            P["conv_in_ff"] = pack_conv(m.conv_in_first_frame.weight, m.conv_in_first_frame.bias, dt)
            P["conv_out_ff"] = pack_conv(m.conv_out_first_frame.weight, m.conv_out_first_frame.bias, dt)

        def f32(t):
            return t.detach().float().contiguous()

        def pack_ru(u, key):
            se, c1 = u["se"], u["conv1"]
            C_ = c1.weight.shape[0]
            P[key] = dict(
                conv3=pack_conv(u["conv3"].weight, u["conv3"].bias, dt),
                conv1=pack_conv(c1.weight, c1.bias, dt),
                wk=f32(se.to_k.weight.reshape(-1)), bk=float(se.to_k.bias.detach().float().item()),
                w1=f32(se.net[0].weight.reshape(se.net[0].weight.shape[0], C_)), b1=f32(se.net[0].bias),
                w2=f32(se.net[2].weight.reshape(C_, -1)), b2=f32(se.net[2].bias),
                hidden=int(se.net[0].weight.shape[0]),
            )
            if dt == torch.bfloat16:      # bf16 copies of the gate MLP for the one-launch SE tail (exact: the parameters are bf16)
                P[key]["w1b"] = P[key]["w1"].to(torch.bfloat16).contiguous()
                P[key]["w2b"] = P[key]["w2"].to(torch.bfloat16).contiguous()

        def pack_ffn(ff, key):
            fc1, fc2 = pack_ff(ff.net[0].weight, ff.net[0].bias, ff.net[2].weight, ff.net[2].bias, dt)
            P[key] = dict(gamma=f32(ff.norm.gamma.reshape(-1)), fc1=fc1, fc2=fc2, inner=ff.dim_inner)

        def pack_attn(at, key):
            P[key] = dict(gamma=f32(at.norm.gamma), qkv=pack_conv(at.to_qkv[0].weight[:, :, None, None, None], None, dt),
                          out=pack_conv(at.to_out[1].weight[:, :, None, None, None], None, dt),
                          mem_kv=at.mem_kv.detach().to(dt).float().contiguous(),
                          heads=at.heads, dim_head=at.dim_head, n_mem=int(at.mem_kv.shape[2]))

        def pack_lin(la, key):
            P[key] = dict(gamma=f32(la.norm.gamma),
                          q=pack_conv(la.attn.to_q[0].weight[:, :, None, None, None], None, dt),
                          kv=pack_conv(la.attn.to_kv[0].weight[:, :, None, None, None], None, dt),
                          out=pack_conv(la.attn.to_out[0].weight[:, :, None, None, None], None, dt),
                          heads=la.heads, dim_head=la.dim_head)

        for side, layers in (("enc", m.encoder_layers), ("dec", m.decoder_layers)):
            decoder = side == "dec"
            stages = m.stages if not decoder else list(reversed(m.stages))
            for i, st in enumerate(stages):
                parts = stage_modules(st, layers[i], decoder)
                key = f"{side}{i}"
                if st.kind == "residual":
                    for j, u in enumerate(parts["units"]):
                        pack_ru(u, f"{key}.{j}")
                elif st.kind == "cond_residual":
                    mod = parts["unit"]
                    w = mod.conv.weights
                    wq = w.detach().to(dt).float()                  # the weights as the module holds them in this dtype
                    P[key] = dict(conv3=pack_conv(w, None, dt), conv1=pack_conv(mod.conv_out.weight, mod.conv_out.bias, dt),
                                  S=(wq * wq).sum(dim=(2, 3, 4)).contiguous(), eps=float(mod.conv.eps),
                                  wc=f32(mod.to_cond.weight), bc=f32(mod.to_cond.bias))
                elif st.kind == "compress_space":
                    conv = parts["conv"]
                    if not decoder:
                        P[key] = pack_conv(conv.weight, conv.bias, dt)                 # (Co,Ci,3,3) -> k=(1,3,3)
                        if dt == torch.bfloat16:
                            pack_conv_down_space(P[key], conv.weight)
                    else:
                        P[key] = pack_conv(conv.weight, conv.bias, dt, shuffle_q=4)    # (4Co,Ci,1,1)
                elif st.kind == "compress_time":
                    conv = parts["conv"]
                    if not decoder:
                        P[key] = pack_conv(conv.weight, conv.bias, dt, k=(3, 1, 1))             # Conv1d (Co,Ci,3)
                    else:
                        P[key] = pack_conv(conv.weight, conv.bias, dt, k=(1, 1, 1), shuffle_q=2)  # Conv1d (2Co,Ci,1)
                elif st.kind in ("attend_space", "attend_time"):
                    pack_attn(parts["attn"], key + ".attn")
                    pack_ffn(parts["ff"], key + ".ff")
                elif st.kind == "linear_attend_space":
                    pack_lin(parts["attn"], key + ".attn")
                    pack_ffn(parts["ff"], key + ".ff")
                elif st.kind == "gateloop_time":
                    gl = parts["gateloop"]
                    P[key] = dict(gamma=f32(gl.norm.gamma), qkva=pack_conv(gl.to_qkva[0].weight[:, :, None, None, None], None, dt))
        if m.has_cond:
            for side, stem in (("enc", m.encoder_cond_in), ("dec", m.decoder_cond_in)):
                P[f"{side}_cond_in"] = dict(w=f32(stem[0].weight), b=f32(stem[0].bias))
        q = m.quantizers
        # the reference applies the projections in the module dtype (bf16 weights in bf16 mode)
        P["quant"] = dict(win=q.project_in.weight.detach().to(dt).float().contiguous(), bin=q.project_in.bias.detach().to(dt).float().contiguous(),
                          wout=q.project_out.weight.detach().to(dt).float().contiguous(), bout=q.project_out.bias.detach().to(dt).float().contiguous())
        self._packs = P
        self._sig = sig
        self._sig_id += 1

    # ------------------------------------------------------------------ primitive ops
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _new(self, shape, dtype=None):
        return torch.empty(shape, device=self.device, dtype=dtype or self.dtype)

    def _tc_launch(self, entry, args, kind, k, out, macs, **shape):
        """Launches the tcgen05 conv entry point `entry` (kind "slab" | "tap") on an output of `out` = (B, T, H, W) positions.
        Under profile_convs CUDA events bracket the launch; when conv_log is set, the launch's shape is recorded there."""
        if self._prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        check(getattr(self.lib, entry)(C.byref(args), self._stream()), entry)
        if self._prof is not None:
            e1.record()
            self._prof.append((e0, e1, 2.0 * out[0] * out[1] * out[2] * out[3] * macs, kind, k[0] * k[1] * k[2]))
        if self.conv_log is not None:
            self.conv_log.append(dict(kind=kind, k=tuple(k), out=out, **shape))
        self.tc_calls += 1
        self.slab_calls += int(kind == "slab")

    def conv(self, x, pk: ConvPack, *, stride=(1, 1, 1), pad=None, out_spatial=None, act=ACT_NONE,
             res=None, shuffle=SHUFFLE_NONE, token_shift=False, out_cf=False, oscale=None):
        """x: (B,T,H,W,Ci) channels-last.  `pad` = leading (pt,ph,pw); causal default (kt-1, kh//2, kw//2).
        out_cf (tcgen05 slab path, Co % 8 != 0 only): write torch's (B,Co,To,Ho,Wo) layout directly."""
        B, Ti, Hi, Wi, Ci = x.shape
        tc_ok = (self.dtype == torch.bfloat16 and self.use_tc and pk.w_tc is not None and not token_shift
                 and Ci == pk.Ci_tc)
        kt, kh, kw = pk.k_tc if (tc_ok and pk.k_tc) else pk.k
        if pad is None:
            pad = (kt - 1, kh // 2, kw // 2)
        if out_spatial is None:
            out_spatial = (Ti, Hi, Wi)
        To, Ho, Wo = out_spatial
        if tc_ok:
            co_gemm = pk.Co_tc
            co_out = co_gemm // 2 if pk.epi_mode == 1 else co_gemm
            if shuffle == SHUFFLE_SPACE:
                y = self._new((B, To, 2 * Ho, 2 * Wo, co_out // 4))
            elif shuffle == SHUFFLE_TIME:
                y = self._new((B, 2 * To, Ho, Wo, co_out // 2))
            elif out_cf:
                y = self._new((B, co_out, To, Ho, Wo))
            else:
                y = self._new((B, To, Ho, Wo, co_out))
            if res is not None:
                assert res.shape == y.shape and res.dtype == y.dtype and res.is_contiguous()
            ta = TcConvArgs(x=_ptr(x), w=_ptr(pk.w_tc), bias=_ptr(pk.bias_tc), res=_ptr(res), y=_ptr(y),
                            B=B, Ti=Ti, Hi=Hi, Wi=Wi, Ci=Ci, To=To, Ho=Ho, Wo=Wo, Co=co_gemm,
                            kt=kt, kh=kh, kw=kw, st=stride[0], sh=stride[1], sw=stride[2],
                            pt=pad[0], ph=pad[1], pw=pad[2], act=act, shuffle=shuffle, epi_mode=pk.epi_mode,
                            oscale=_ptr(oscale), out_layout=int(out_cf))
            # measured policy (profiles/r01_sweep_slab_v*.json): the persistent slab kernel wins on every layer it supports
            # (incl. the 64-byte-row conv_in once it runs 4 M-tiles and 7 taps per weight stage); the tap-wise kernel
            # keeps the strided down-samplers.  tc_variant = "tap" forces the tap-wise kernel (tests / sweeps).
            use_slab = self.tc_variant != "tap" and bool(self.lib.mv2_tc_slab_supported(C.byref(ta)))
            use_down = (not use_slab and self.tc_variant != "tap" and pk.w_down is not None and stride == (1, 2, 2)
                        and bool(self.lib.mv2_tc_down_space_supported(C.byref(ta))))
            if use_down:
                ta.w = _ptr(pk.w_down)
                use_slab = True
            if use_slab or self.lib.mv2_tc_conv_supported(C.byref(ta)):
                entry = "mv2_tc_down_space_forward" if use_down else "mv2_tc_slab_forward" if use_slab else "mv2_tc_conv_forward"
                self._tc_launch(entry, ta, "slab" if use_slab else "tap", pk.k, (B, To, Ho, Wo), pk.macs, Ci=Ci, Co=co_out,
                                geglu=pk.epi_mode == 1, shuffle=shuffle, res=res is not None)
                self.launches += 1
                return y
            assert not out_cf, "channels-first output is a tcgen05 slab-kernel feature"
            assert pk.w is not None and pk.epi_mode == 0 and Ci == pk.Ci, "tcgen05-only weight pack has no CUDA-core fallback"
            kt, kh, kw = pk.k
        assert Ci == pk.Ci, (Ci, pk.Ci)
        assert pk.w is not None and not out_cf
        if shuffle == SHUFFLE_SPACE:
            y = self._new((B, To, 2 * Ho, 2 * Wo, pk.Co // 4))
        elif shuffle == SHUFFLE_TIME:
            y = self._new((B, 2 * To, Ho, Wo, pk.Co // 2))
        else:
            y = self._new((B, To, Ho, Wo, pk.Co))
        if res is not None:
            assert res.shape == y.shape and res.dtype == y.dtype and res.is_contiguous()
        self.simt_conv_calls += 1
        a = ConvArgs(x=_ptr(x), w=_ptr(pk.w), bias=_ptr(pk.bias), res=_ptr(res), y=_ptr(y), dtype=_dt(self.dtype),
                     B=B, Ti=Ti, Hi=Hi, Wi=Wi, Ci=Ci, To=To, Ho=Ho, Wo=Wo, Co=pk.Co,
                     kt=kt, kh=kh, kw=kw, st=stride[0], sh=stride[1], sw=stride[2],
                     pt=pad[0], ph=pad[1], pw=pad[2], act=act, shuffle=shuffle, x_token_shift=int(token_shift),
                     oscale=_ptr(oscale))
        check(self.lib.mv2_conv_forward(C.byref(a), self._stream()), "mv2_conv_forward")
        self.launches += 1
        return y

    def residual_unit(self, x, p):
        """ResidualUnit (reference M:930-944): x + SE(ELU(conv1(ELU(causal_conv3(x)))))."""
        B, T, H, W, Cc = x.shape
        F_, Pn = B * T, H * W
        st = self._stream()
        c3, c1 = p["conv3"], p["conv1"]
        if self.dtype == torch.bfloat16 and self.use_tc and self.fuse_ru and c3.w_tc is not None and self.tc_variant != "tap":
            ra = TcRuArgs(x=_ptr(x), w3=_ptr(c3.w_tc), b3=_ptr(c3.bias_tc), w1=_ptr(c1.w_tc), b1=_ptr(c1.bias_tc),
                          se_wk=_ptr(p["wk"]), se_bk=p["bk"], y=None, se_ws=None, B=B, T=T, H=H, W=W, C=Cc,
                          kt=c3.k[0], kh=c3.k[1], kw=c3.k[2])
            if self.lib.mv2_tc_ru_supported(C.byref(ra)):
                y = self._new(x.shape)
                ws = self._new((self.lib.mv2_tc_ru_workspace_bytes(C.byref(ra)) // 4,), torch.float32)
                ra.y, ra.se_ws = _ptr(y), _ptr(ws)
                nrec = self.lib.mv2_tc_ru_records(C.byref(ra))
                self._tc_launch("mv2_tc_ru_forward", ra, "slab", c3.k, (B, T, H, W), c3.macs + c1.macs, Ci=Cc, Co=Cc, geglu=False,
                                shuffle=0, res=False, fused_ru=True)
                gates = self._new((F_, Cc), torch.float32)
                check(self.lib.mv2_se_gate_records(_ptr(ws), nrec, F_, Cc, p["hidden"], _ptr(p["w1"]), _ptr(p["b1"]), _ptr(p["w2"]),
                                                   _ptr(p["b2"]), _ptr(gates), st), "mv2_se_gate_records")
                out = self._new(x.shape)
                check(self.lib.mv2_gate_residual(_ptr(y), _ptr(x), _ptr(gates), _ptr(out), _dt(self.dtype), F_, Pn, Cc, st),
                      "mv2_gate_residual")
                self.launches += 4
                self.fused_ru_calls += 1
                return out
        if not (self.dtype == torch.bfloat16 and self.se_tail and "w1b" in p
                and self.lib.mv2_se_tail_supported(F_, Pn, Cc, p["hidden"])):
            return self.residual_unit_unfused(x, p)[0]
        h = self.conv(x, c3, act=ACT_ELU)
        y = self.conv(h, c1, act=ACT_ELU)
        out = self._new(x.shape)
        check(self.lib.mv2_se_tail(_ptr(y), _ptr(x), _ptr(out), F_, Pn, Cc, p["hidden"], _ptr(p["wk"]), p["bk"],
                                   _ptr(p["w1b"]), _ptr(p["b1"]), _ptr(p["w2b"]), _ptr(p["b2"]), st), "mv2_se_tail")
        self.launches += 1
        self.se_tail_calls += 1
        return out

    def residual_unit_unfused(self, x, p):
        """ResidualUnit on separate launches: h = ELU(conv3(x)), y = ELU(conv1(h)), SE pool, gate MLP, gate + residual.
        Returns (out, h, y); the training backward differentiates through the intermediate h and y."""
        B, T, H, W, Cc = x.shape
        F_, Pn = B * T, H * W
        st, dt = self._stream(), _dt(self.dtype)
        h = self.conv(x, p["conv3"], act=ACT_ELU)
        y = self.conv(h, p["conv1"], act=ACT_ELU)
        ws = self._new((self.lib.mv2_se_workspace_bytes(F_, Pn, Cc) // 4,), torch.float32)
        gates = self._new((F_, Cc), torch.float32)
        check(self.lib.mv2_se_pool(_ptr(y), dt, F_, Pn, Cc, _ptr(p["wk"]), p["bk"], _ptr(ws), st), "mv2_se_pool")
        check(self.lib.mv2_se_gate(_ptr(ws), dt, F_, Pn, Cc, p["hidden"], _ptr(p["w1"]), _ptr(p["b1"]), _ptr(p["w2"]),
                                   _ptr(p["b2"]), _ptr(gates), st), "mv2_se_gate")
        out = self._new(x.shape)
        check(self.lib.mv2_gate_residual(_ptr(y), _ptr(x), _ptr(gates), _ptr(out), dt, F_, Pn, Cc, st), "mv2_gate_residual")
        self.launches += 3
        return out, h, y

    def dense_small(self, x, w, b, act=ACT_NONE):
        """fp32 y[b][n] = act(x[b] . w[n] + bias[n]) (cond stems M:1344-1352, to_cond M:983)."""
        Bx, K = x.shape
        N = w.shape[0]
        y = self._new((Bx, N), torch.float32)
        check(self.lib.mv2_dense_small(_ptr(x), _ptr(w), _ptr(b), _ptr(y), Bx, K, N, act, self._stream()), "mv2_dense_small")
        self.launches += 1
        return y

    def cond_stem(self, cond, side):
        p = self._packs[f"{side}_cond_in"]
        return self.dense_small(cond.float().contiguous(), p["w"], p["b"], ACT_SILU)

    def residual_unit_mod(self, x, p, cond_e):
        """ResidualUnitMod (M:978-988): x + ELU(conv_out(ELU(Conv3DMod(x, to_cond(cond))))).  The per-clip modulated weights
        are never built: input channels are scaled by (cond + 1), the shared-weight conv runs unchanged and the demodulation
        rsqrt(sum w_b^2) multiplies the accumulator per (clip, output channel) in the epilogue (include/magvit2_b200.h)."""
        B, T, H, W, Cc = x.shape
        c = self.dense_small(cond_e, p["wc"], p["bc"])
        scale_in = self._new((B, Cc), torch.float32)
        inv_norm = self._new((B, Cc), torch.float32)
        st = self._stream()
        check(self.lib.mv2_mod_prepare(_ptr(c), _ptr(p["S"]), p["eps"], _ptr(scale_in), _ptr(inv_norm), B, Cc, Cc, st), "mv2_mod_prepare")
        xs = self._new(x.shape)
        check(self.lib.mv2_scale_channels(_ptr(x), _ptr(scale_in), _ptr(xs), _dt(self.dtype), B, T * H * W, Cc, st), "mv2_scale_channels")
        self.launches += 2
        h = self.conv(xs, p["conv3"], act=ACT_ELU, oscale=inv_norm)
        return self.conv(h, p["conv1"], act=ACT_ELU, res=x)

    def rmsnorm(self, x, gamma, token_shift=False):
        B, T, H, W, Cc = x.shape
        out = self._new(x.shape)
        check(self.lib.mv2_rmsnorm(_ptr(x), _ptr(out), _dt(self.dtype), _ptr(gamma), B, T, H * W, Cc,
                                   int(token_shift), self._stream()), "mv2_rmsnorm")
        self.launches += 1
        return out

    def feed_forward(self, x, p, token_shift=False):
        """Residual(FeedForward) (M:471-508, M:1191): x + fc2(geglu(fc1(rmsnorm(shift(x)))))."""
        B, T, H, W, Cc = x.shape
        xn = self.rmsnorm(x, p["gamma"], token_shift)
        # fused fc1 + GEGLU pack is tcgen05-only (K = C must be a multiple of 16); other widths take the unfused
        # CUDA-core convs + mv2_geglu below, like the fp32 path
        if self.dtype == torch.bfloat16 and self.use_tc and p["fc1"].epi_mode == 1 and Cc % 16 == 0:
            g = self.conv(xn, p["fc1"])                       # fc1 + bias + GEGLU fused, hidden width padded to 64
            return self.conv(g, p["fc2"], res=x)
        fc1 = p["fc1"]
        hdn = self._conv_simt_only(xn, fc1)
        I = p["inner"]
        g = self._new((B, T, H, W, I))
        check(self.lib.mv2_geglu(_ptr(hdn), _ptr(g), _dt(self.dtype), B * T * H * W, I, self._stream()), "mv2_geglu")
        self.launches += 1
        return self._conv_simt_only(g, p["fc2"], res=x)

    def _conv_simt_only(self, x, pk, **kw):
        use, self.use_tc = self.use_tc, False
        try:
            return self.conv(x, pk, **kw)
        finally:
            self.use_tc = use

    def attention(self, x, p, axis: str):
        """Residual(SpaceAttention) / Residual(TokenShift(TimeAttention)) (M:444-464, M:1190, M:1235)."""
        B, T, H, W, Cc = x.shape
        time_axis = axis == "time"
        xn = self.rmsnorm(x, p["gamma"], token_shift=time_axis)
        qkv = self.conv(xn, p["qkv"])
        heads, dh = p["heads"], p["dim_head"]
        o = self._new((B, T, H, W, heads * dh))
        HW = H * W
        if time_axis:
            a = AttnArgs(qkv=_ptr(qkv), out=_ptr(o), mem_kv=_ptr(p["mem_kv"]), dtype=_dt(self.dtype), heads=heads,
                         dim_head=dh, n_mem=p["n_mem"], causal=1, n_outer=B, n_inner=HW, L=T,
                         outer_stride=T * HW, inner_stride=1, tok_stride=HW)
        else:
            a = AttnArgs(qkv=_ptr(qkv), out=_ptr(o), mem_kv=_ptr(p["mem_kv"]), dtype=_dt(self.dtype), heads=heads,
                         dim_head=dh, n_mem=p["n_mem"], causal=0, n_outer=B * T, n_inner=1, L=HW,
                         outer_stride=HW, inner_stride=0, tok_stride=1)
        check(self.lib.mv2_attention(C.byref(a), self._stream()), "mv2_attention")
        self.launches += 1
        return self.conv(o, p["out"], res=x)

    def linear_attention(self, x, p):
        """Residual(LinearSpaceAttention) (M:421-442, M:1207)."""
        B, T, H, W, Cc = x.shape
        xn = self.rmsnorm(x, p["gamma"])
        q = self.conv(xn, p["q"])
        kv = self.conv(xn, p["kv"])
        heads, dh = p["heads"], p["dim_head"]
        n_seq, L = B * T, H * W
        ws = self._new((self.lib.mv2_linattn_workspace_bytes(n_seq, heads, L) // 4,), torch.float32)
        o = self._new((B, T, H, W, heads * dh))
        check(self.lib.mv2_linear_attention(_ptr(q), _ptr(kv), _ptr(o), _dt(self.dtype), n_seq, L, heads, dh,
                                            _ptr(ws), self._stream()), "mv2_linear_attention")
        self.launches += 2
        return self.conv(o, p["out"], res=x)

    def gateloop(self, x, p):
        """ToTimeSequence(Residual(SimpleGateLoopLayer)) (M:178-191, M:1216-1222): RMSNorm, Linear(dim, 3 dim), then the gated
        recurrence over time per (pixel, channel) with the residual add fused (mv2_gateloop_scan)."""
        B, T, H, W, Cc = x.shape
        qkva = self.conv(self.rmsnorm(x, p["gamma"]), p["qkva"])
        out = self._new(x.shape)
        check(self.lib.mv2_gateloop_scan(_ptr(qkva), _ptr(x), _ptr(out), _dt(self.dtype), B, T, H * W, Cc, self._stream()),
              "mv2_gateloop_scan")
        self.launches += 1
        return out

    def profile_convs(self, fn, steps: int = 3):
        """Runs fn() `steps` times with CUDA events around every tcgen05 conv launch (on the launching stream).
        A long spin kernel is queued first so the host runs ahead of the GPU and the event pairs bracket pure
        kernel time, not host launch gaps.  Returns {class: (kernel ms per step, launches per step, FLOPs per step)}
        for class in 'conv3d' (taps > 1 convs in tc_slab_kernel: the causal Conv3d path) and 'all' (every tcgen05 launch)."""
        fn()
        torch.cuda.synchronize(self.device)
        self._prof = []
        try:
            for _ in range(steps):
                torch.cuda._sleep(int(40e6))          # ~20 ms of GPU busy-wait: lets the host enqueue the whole step
                fn()
            torch.cuda.synchronize(self.device)
            recs = [(e0.elapsed_time(e1), f, kind, taps) for e0, e1, f, kind, taps in self._prof]
        finally:
            self._prof = None
        out = {}
        for name, sel in (("conv3d", lambda r: r[2] == "slab" and r[3] > 1), ("all", lambda r: True)):
            rs = [r for r in recs if sel(r)]
            if rs:
                out[name] = (sum(r[0] for r in rs) / steps, len(rs) // steps, sum(r[1] for r in rs) / steps)
        return out

    # ------------------------------------------------------------------ stages
    def _stage(self, x, st, key, decoder: bool, cond_e=None):
        P = self._packs
        B, T, H, W, Cc = x.shape
        if st.kind == "residual":
            for j in range(st.count):
                x = self.residual_unit(x, P[f"{key}.{j}"])
        elif st.kind == "cond_residual":
            x = self.residual_unit_mod(x, P[key], cond_e)
        elif st.kind == "compress_space":
            if decoder:   # SpatialUpsample2x (M:838-846)
                x = self.conv(x, P[key], act=ACT_SILU, shuffle=SHUFFLE_SPACE)
            else:         # SpatialDownsample2x (M:770-780): Conv2d k3 s2 p1
                x = self.conv(x, P[key], stride=(1, 2, 2), pad=(0, 1, 1),
                              out_spatial=(T, (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1))
        elif st.kind == "compress_time":
            if decoder:   # TimeUpsample2x (M:875-883)
                x = self.conv(x, P[key], act=ACT_SILU, shuffle=SHUFFLE_TIME)
            else:         # TimeDownsample2x (M:796-807): pad (2, 0), Conv1d k3 s2
                x = self.conv(x, P[key], stride=(2, 1, 1), pad=(2, 0, 0), out_spatial=((T + 2 - 3) // 2 + 1, H, W))
        elif st.kind == "attend_space":
            x = self.attention(x, P[key + ".attn"], "space")
            x = self.feed_forward(x, P[key + ".ff"])
        elif st.kind == "attend_time":
            x = self.attention(x, P[key + ".attn"], "time")
            x = self.feed_forward(x, P[key + ".ff"], token_shift=True)
        elif st.kind == "linear_attend_space":
            x = self.linear_attention(x, P[key + ".attn"])
            x = self.feed_forward(x, P[key + ".ff"])
        elif st.kind == "gateloop_time":
            x = self.gateloop(x, P[key])
        else:
            raise ValueError(st.kind)
        return x

    def _tap(self, name, x):
        if self.taps is not None:
            self.taps[name] = x.permute(0, 4, 1, 2, 3).float().cpu()

    # ------------------------------------------------------------------ layout
    def to_channels_last(self, v: torch.Tensor, t_pad: int = 0):
        """(B,C,T,H,W) torch tensor (fp32, bf16, or uint8 frames: normalised x / 255 as the reference's data loaders do,
        D:103, D:188) -> (B,T+t_pad,H,W,C) compute dtype."""
        if v.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
            v = v.float()
        v = v.contiguous()
        B, Cc, T, H, W = v.shape
        out = self._new((B, T + t_pad, H, W, Cc))
        check(self.lib.mv2_to_channels_last(_ptr(v), _src_dt(v.dtype), _ptr(out), _dt(self.dtype), B, Cc, T, H, W, t_pad,
                                            self._stream()), "mv2_to_channels_last")
        self.launches += 1
        return out

    def ingest_kwpack(self, v: torch.Tensor, t_pad: int, pin):
        """(B,C,T,H,W) -> (B,T+t_pad,H,W,32) bf16 with the k_w taps packed into channels (mv2_ingest_kwpack)."""
        if v.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
            v = v.float()
        v = v.contiguous()
        B, Cc, T, H, W = v.shape
        out = self._new((B, T + t_pad, H, W, pin.Ci_tc), torch.bfloat16)
        check(self.lib.mv2_ingest_kwpack(_ptr(v), _src_dt(v.dtype), _ptr(out), B, Cc, T, H, W, t_pad, pin.kw_orig,
                                         pin.kw_orig // 2, pin.Ci_tc, self._stream()), "mv2_ingest_kwpack")
        self.launches += 1
        return out

    _PAD_MODES = {"reflect": 1, "replicate": 2, "circular": 3}

    def causal_conv_padded(self, x, pk, pad_mode):
        """CausalConv3d with pad_mode != 'constant' (M:925-927): the padding is materialised by mv2_pad_cl, then the conv
        runs without any implicit padding.  As in the reference the mode falls back to 'constant' when time_pad >= T."""
        B, T, H, W, Cc = x.shape
        kt, kh, kw = pk.k
        if pad_mode == "constant" or kt - 1 >= T:
            return self.conv(x, pk)
        xp = self._new((B, T + kt - 1, H + 2 * (kh // 2), W + 2 * (kw // 2), Cc))
        check(self.lib.mv2_pad_cl(_ptr(x), _ptr(xp), _dt(self.dtype), B, T, H, W, Cc, kt - 1, kh // 2, kw // 2,
                                  self._PAD_MODES[pad_mode], self._stream()), "mv2_pad_cl")
        self.launches += 1
        return self.conv(xp, pk, pad=(0, 0, 0), out_spatial=(T, H, W))

    def copy_frames(self, src, t0, n, dst=None, dst_t0=0, zero_front=False):
        """Frames [t0, t0 + n) of a channels-last clip tensor -> a new (B, n, ...) tensor, or into ``dst`` at ``dst_t0``."""
        B, Ts = src.shape[:2]
        if dst is None:
            dst = self._new((B, n) + tuple(src.shape[2:]), src.dtype)
        frame_bytes = src[0, 0].numel() * src.element_size()
        assert dst[0, 0].numel() * dst.element_size() == frame_bytes and src.is_contiguous() and dst.is_contiguous()
        check(self.lib.mv2_copy_frames(_ptr(src), _ptr(dst), B, Ts, dst.shape[1], t0, dst_t0, n, frame_bytes, int(zero_front),
                                       self._stream()), "mv2_copy_frames")
        return dst

    def to_channels_first(self, x: torch.Tensor, t_crop: int = 0, out_dtype=None):
        B, T, H, W, Cc = x.shape
        out_dtype = out_dtype or self.dtype
        out = torch.empty((B, Cc, T - t_crop, H, W), device=self.device, dtype=out_dtype)
        check(self.lib.mv2_to_channels_first(_ptr(x), _dt(x.dtype), _ptr(out), _dt(out_dtype), B, Cc, T, H, W, t_crop,
                                             self._stream()), "mv2_to_channels_first")
        self.launches += 1
        return out

    def mse(self, a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
        """F.mse_loss(a, b) of two same-layout tensors (reference M:1722: video vs reconstruction, both (B,C,T,H,W)) as a 0-d
        fp32 tensor; `a` may hold uint8 frames (x / 255)."""
        assert a.shape == b.shape, (a.shape, b.shape)
        if a.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
            a = a.float()
        a, b = a.contiguous(), b.contiguous()
        ws = self._new((self.lib.mv2_mse_workspace_bytes() // 4,), torch.float32)
        out = self._new((1,), torch.float32)
        check(self.lib.mv2_mse(_ptr(a), _src_dt(a.dtype), _ptr(b), _dt(b.dtype), a.numel(), _ptr(ws), _ptr(out), self._stream()), "mv2_mse")
        self.launches += 2
        return out[0]

    # ------------------------------------------------------------------ the path
    def conv_in_cl(self, video: torch.Tensor, first_frame: bool = True):
        """conv_in (M:1109) of video (B,C,T,H,W) -> (channels-last feature map, saved).  The time_padding zero frames are only
        prepended when the clip starts with a first frame (video_contains_first_frame, M:1534-1537).  `saved` holds the
        channels-last inputs of the causal conv that a weight gradient needs: "rest_in" (frames 1.., first frame encoded
        separately) or "padded_in" (the zero-prepended clip, pad_mode != 'constant')."""
        m = self.model
        t_pad = m.time_padding if first_frame else 0
        pin = self._packs.get("conv_in_tc")
        saved = {}
        if m.separate_first_frame_encoding and first_frame:
            # M:1553-1561: the first frame goes through its own 2-D conv, frames 1.. through the causal conv_in on their own,
            # then the feature map is [time_padding zero frames, first, rest]
            B, _, T, H, W = video.shape
            v_cl = self.to_channels_last(video, 0)
            parts = [(self.conv(self.copy_frames(v_cl, 0, 1), self._packs["conv_in_ff"]), t_pad)]
            if T > 1:
                saved["rest_in"] = self.copy_frames(v_cl, 1, T - 1)
                parts.append((self.causal_conv_padded(saved["rest_in"], self._packs["conv_in"], m.conv_in.pad_mode), t_pad + 1))
            x = self._new((B, T + t_pad, H, W, parts[0][0].shape[-1]))
            for i, (part, t0) in enumerate(parts):
                self.copy_frames(part, 0, part.shape[1], dst=x, dst_t0=t0, zero_front=(i == 0))
        elif m.conv_in.pad_mode != "constant":
            saved["padded_in"] = self.to_channels_last(video, t_pad)
            x = self.causal_conv_padded(saved["padded_in"], self._packs["conv_in"], m.conv_in.pad_mode)
        elif self.dtype == torch.bfloat16 and self.use_tc and pin is not None:
            x = self.ingest_kwpack(video, t_pad, pin)
            x = self.conv(x, pin, pad=(pin.k_tc[0] - 1, pin.k_tc[1] // 2, 0))
        else:
            x = self.to_channels_last(video, t_pad)
            x = self.conv(x, self._packs["conv_in"])
        return x, saved

    def conv_out_cf(self, x: torch.Tensor, first_frame: bool = True):
        """conv_out (M:1127) of the decoder output x (B,T,H,W,C) -> (video (B,3,T,H,W), saved).  The leading time_padding
        frames are dropped only for clips that contain a first frame (M:1646-1647).  `saved` holds "rest_out", the frames
        the causal conv read when the first frame is decoded separately."""
        m = self.model
        pk = self._packs["conv_out"]
        B, T, H, W, Cc = x.shape
        tp = m.time_padding if first_frame else 0
        saved = {}
        if m.separate_first_frame_encoding and first_frame:
            # M:1633-1639: conv_out_first_frame on frame `tp`, the causal conv_out on the frames after it, re-attached
            first = self.conv(self.copy_frames(x, tp, 1), self._packs["conv_out_ff"])
            out = self._new((B, T - tp, H, W, first.shape[-1]))
            self.copy_frames(first, 0, 1, dst=out, dst_t0=0)
            if T - tp > 1:
                saved["rest_out"] = self.copy_frames(x, tp + 1, T - tp - 1)
                rest = self.causal_conv_padded(saved["rest_out"], pk, m.conv_out.pad_mode)
                self.copy_frames(rest, 0, T - tp - 1, dst=out, dst_t0=1)
            return self.to_channels_first(out), saved
        if m.conv_out.pad_mode != "constant":
            return self.to_channels_first(self.causal_conv_padded(x, pk, m.conv_out.pad_mode), t_crop=tp), saved
        if (self.dtype == torch.bfloat16 and self.use_tc and self.tc_variant != "tap" and self.fuse_conv_out and pk.w_tc is not None
                and pk.Co % 8 != 0 and Cc % 64 == 0 and pk.k[2] <= 3 and T > tp):
            # conv_out writes the reconstruction in torch's (B,C,T,H,W) layout itself and never computes the time_padding
            # frames the reference drops afterwards (M:1642-1647)
            return self.conv(x, pk, pad=(pk.k[0] - 1 - tp, pk.k[1] // 2, pk.k[2] // 2), out_spatial=(T - tp, H, W), out_cf=True), saved
        return self.to_channels_first(self.conv(x, pk), t_crop=tp), saved

    def encode_cl(self, video: torch.Tensor, first_frame: bool = True, cond=None):
        """video (B,C,T,H,W) on device -> encoder output, channels-last.  Reference encode M:1523-1576."""
        m = self.model
        x, _ = self.conv_in_cl(video, first_frame)
        self._tap("conv_in", x)
        cond_e = self.cond_stem(cond, "enc") if (m.has_cond and cond is not None) else None     # M:1544-1548
        for i, st in enumerate(m.stages):
            x = self._stage(x, st, f"enc{i}", decoder=False, cond_e=cond_e)
            self._tap(f"enc{i}", x)
        return x

    def decode_cl(self, q: torch.Tensor, first_frame: bool = True, cond=None):
        """quantized channels-last (B,T',H',W',C) -> video (B,3,T,H,W).  Reference decode M:1598-1649."""
        m = self.model
        x = q
        cond_e = self.cond_stem(cond, "dec") if (m.has_cond and cond is not None) else None     # M:1612-1616
        for j, st in enumerate(reversed(m.stages)):
            x = self._stage(x, st, f"dec{j}", decoder=True, cond_e=cond_e)
            self._tap(f"dec{j}", x)
        return self.conv_out_cf(x, first_frame)[0]

    def quantize_cl(self, x, want_quantized=True, want_aux=False):
        """x channels-last -> (quantized channels-last | None, indices (B,T,H,W[,num_codebooks]), aux fp32 [N][D] | None)."""
        m = self.model
        B, T, H, W, Cc = x.shape
        N = B * T * H * W
        P = self._packs["quant"]
        q = self._new(x.shape) if want_quantized else None
        qz = m.quantizers
        d, nc = qz.codebook_dim, qz.num_codebooks
        ishape = (B, T, H, W) if nc == 1 else (B, T, H, W, nc)      # keep_num_codebooks_dim = num_codebooks > 1 (A.1 step 9)
        aux = self._new((N, d * nc), torch.float32) if want_aux else None
        if m.use_fsq:
            idx = torch.empty(ishape, device=self.device, dtype=torch.int32)
            lv = (C.c_int32 * d)(*qz.levels)
            check(self.lib.mv2_fsq_forward(_ptr(x), _dt(self.dtype), N, Cc, d, nc, lv, _ptr(P["win"]), _ptr(P["bin"]),
                                           _ptr(P["wout"]), _ptr(P["bout"]), _ptr(idx), _ptr(q), _ptr(aux),
                                           self._stream()), "mv2_fsq_forward")
        else:
            idx = torch.empty(ishape, device=self.device, dtype=torch.int64)
            clamp = qz.soft_clamp_input_value
            check(self.lib.mv2_lfq_forward(_ptr(x), _dt(self.dtype), N, Cc, d, nc, _ptr(P["win"]), _ptr(P["bin"]),
                                           _ptr(P["wout"]), _ptr(P["bout"]), float(clamp) if clamp else 0.0, int(qz.spherical),
                                           _ptr(idx), _ptr(q), _ptr(aux), self._stream()), "mv2_lfq_forward")
        self.launches += 1
        return q, idx, aux

    def codes_to_quantized_cl(self, codes: torch.Tensor):
        """indices (B,T,H,W[,num_codebooks]) int64/int32 -> quantized channels-last.  LFQ/FSQ.indices_to_codes (M:1593)."""
        m = self.model
        codes = codes.contiguous()
        B, T, H, W = codes.shape[:4]
        qz = m.quantizers
        Cc = qz.dim
        N = B * T * H * W
        P = self._packs["quant"]
        d, nc = qz.codebook_dim, qz.num_codebooks
        q = self._new((B, T, H, W, Cc))
        is64 = int(codes.dtype == torch.int64)
        if m.use_fsq:
            lv = (C.c_int32 * d)(*qz.levels)
            check(self.lib.mv2_fsq_decode(_ptr(codes), is64, N, Cc, d, nc, lv, _ptr(P["wout"]), _ptr(P["bout"]), _ptr(q),
                                          _dt(self.dtype), self._stream()), "mv2_fsq_decode")
        else:
            check(self.lib.mv2_lfq_decode(_ptr(codes), is64, N, Cc, d, nc, _ptr(P["wout"]), _ptr(P["bout"]), _ptr(q),
                                          _dt(self.dtype), self._stream()), "mv2_lfq_decode")
        self.launches += 1
        return q
