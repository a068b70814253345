"""Training-mode forward with gradients (SURVEY.md 8f N2, first slice): ``model.train(); loss, breakdown =
model(video, return_loss=True); loss.backward()`` for tokenizers without the GAN / perceptual branches
(``use_gan=False, perceptual_loss_weight=0``) -- what ``VideoTokenizerTrainer.train_step`` does with the generator loss
(reference trainer.py:356-363).

Division of labour
  * FORWARD: the hand-written sm_100a kernels of the inference path (engine.Engine / libmagvit2_b200.so), with the
    ResidualUnit run unfused so that its intermediate activations exist.  The activations the backward needs are kept as
    they come out of the kernels (channels-last).
  * BACKWARD: the DATA gradient of the stride-1 causal convs (the 3x3x3 and 1x1x1 convs of every ResidualUnit, conv_out: about
    half of the backward's conv FLOPs) runs on the engine's own conv kernels -- a transposed conv is the same implicit GEMM with
    flipped / transposed weights.  The weight / bias gradients of all convs and the strided down-samplers call
    ``aten.convolution_backward`` (cuDNN) directly on the saved activations -- no forward recomputation.  The light blocks (SqueezeExcite gating, attention / linear-attention /
    FeedForward blocks, the two up-samplers, the quantiser with its straight-through estimator and auxiliary losses) are
    differentiated by re-evaluating a torch restatement of the block on its saved input (``_vjp``).
  There are no dedicated backward kernels (wgrad, attention backward) yet; this slice makes the drop-in claim true for the trainer's generator step,
  it is not a speed claim for training.  Gradients are checked against the unmodified reference's autograd on the `mini`
  config (tests/golden/mini_train.pt, tests/test_train_gpu.py).

Reference lines: M: = magvit2_pytorch/magvit2_pytorch.py, A: = attend.py.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Sequence

import torch
import torch.nn.functional as F

from .engine import pack_conv, stage_modules


# --------------------------------------------------------------------------------------------
# torch restatements of the light blocks, channels-last (B, T, H, W, C) -- used for the backward only
# --------------------------------------------------------------------------------------------
def _rmsnorm(x, gamma):
    """RMSNorm (M:275-276): F.normalize over channels * sqrt(C) * gamma."""
    return F.normalize(x, dim=-1) * (x.shape[-1] ** 0.5) * gamma.reshape(-1)


def _token_shift(x):
    """TokenShift (M:250-254): the second chunk of the channels delayed by one frame, zeros at t = 0."""
    a, s = x.chunk(2, dim=-1)
    s = F.pad(s, (0, 0, 0, 0, 0, 0, 1, -1))
    return torch.cat((a, s), dim=-1)


def _squeeze_excite(y, se):
    """SqueezeExcite (M:221-240) on (B,T,H,W,C): per frame, softmax-pooled channel vector -> 2-layer MLP -> sigmoid gate."""
    B, T, H, W, Cc = y.shape
    yf = y.reshape(B * T, H * W, Cc)
    logits = yf @ se.to_k.weight.reshape(Cc) + se.to_k.bias
    attn = logits.float().softmax(dim=-1).to(y.dtype)
    pooled = torch.einsum("fp,fpc->fc", attn, yf)
    hd = se.net[0].weight.shape[0]
    hid = F.leaky_relu(F.linear(pooled, se.net[0].weight.reshape(hd, Cc), se.net[0].bias), 0.1)
    gate = torch.sigmoid(F.linear(hid, se.net[2].weight.reshape(Cc, hd), se.net[2].bias))
    return (yf * gate[:, None, :]).reshape(y.shape)


def _softmax_attention(q, k, v, causal):
    """Attend (A:218-241) with the right-aligned causal mask (A:46-47, A:123-129)."""
    dots = torch.einsum("bhid,bhjd->bhij", q, k) * (q.shape[-1] ** -0.5)
    i, j = dots.shape[-2:]
    if causal and i > 1:
        mask = torch.ones((i, j), dtype=torch.bool, device=q.device).triu(j - i + 1)
        dots = dots.masked_fill(mask, -torch.finfo(dots.dtype).max)
    return torch.einsum("bhij,bhjd->bhid", dots.softmax(dim=-1), v)


def _attention_block(x, at, axis):
    """Residual(SpaceAttention) / Residual(TokenShift(TimeAttention)) (M:327-388, M:444-464, M:1190, M:1235)."""
    B, T, H, W, Cc = x.shape
    xs = _token_shift(x) if axis == "time" else x
    xn = _rmsnorm(xs, at.norm.gamma)
    tok = xn.permute(0, 2, 3, 1, 4).reshape(B * H * W, T, Cc) if axis == "time" else xn.reshape(B * T, H * W, Cc)
    b, n, _ = tok.shape
    qkv = F.linear(tok, at.to_qkv[0].weight).reshape(b, n, 3, at.heads, -1).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    mem = at.mem_kv.to(x.dtype)
    k = torch.cat((mem[0][None].expand(b, -1, -1, -1), k), dim=-2)
    v = torch.cat((mem[1][None].expand(b, -1, -1, -1), v), dim=-2)
    o = _softmax_attention(q, k, v, causal=(axis == "time")).permute(0, 2, 1, 3).reshape(b, n, -1)
    o = F.linear(o, at.to_out[1].weight)
    o = o.reshape(B, H, W, T, Cc).permute(0, 3, 1, 2, 4) if axis == "time" else o.reshape(B, T, H, W, Cc)
    return o + x


def _linear_attention_block(x, la):
    """Residual(LinearSpaceAttention) (M:390-442) with the Taylor-series linear attention of SURVEY Appendix A.3."""
    B, T, H, W, Cc = x.shape
    heads, dh = la.heads, la.dim_head
    tok = _rmsnorm(x, la.norm.gamma).reshape(B * T, H * W, Cc)
    b, n, _ = tok.shape
    q = F.linear(tok, la.attn.to_q[0].weight).reshape(b, n, heads, dh).permute(0, 2, 1, 3) * dh ** -0.5
    kv = F.linear(tok, la.attn.to_kv[0].weight).reshape(b, n, 2, heads, dh).permute(2, 0, 3, 1, 4)
    k, v = kv[0], kv[1]

    def phi(z):
        one = z.new_ones((*z.shape[:-1], 1))
        z2 = (z[..., :, None] * z[..., None, :]) * (0.5 ** 0.5)
        return torch.cat((one, z, z2.reshape(*z.shape[:-1], -1)), dim=-1)

    q, k = phi(q), phi(k)
    kvs = torch.einsum("bhnd,bhne->bhde", k, v)
    num = torch.einsum("bhnd,bhde->bhne", q, kvs)
    den = torch.einsum("bhnd,bhd->bhn", q, k.sum(dim=-2))[..., None]
    o = (num / den.clamp(min=1e-5)).permute(0, 2, 1, 3).reshape(b, n, heads * dh)
    return F.linear(o, la.attn.to_out[0].weight).reshape(x.shape) + x


def _gateloop_block(x, gl):
    """ToTimeSequence(Residual(SimpleGateLoopLayer)) (M:178-191, M:1216-1222): s_t = sigmoid(a_t) s_{t-1} + kv_t, out_t = q_t s_t."""
    q, kv, a = F.linear(_rmsnorm(x, gl.norm.gamma), gl.to_qkva[0].weight).chunk(3, dim=-1)
    a = a.sigmoid()
    s = torch.zeros_like(kv[:, 0])
    outs = []
    for t in range(x.shape[1]):
        s = a[:, t] * s + kv[:, t]
        outs.append(q[:, t] * s)
    return torch.stack(outs, dim=1) + x


def _residual_unit_mod(x, cond_e, mod):
    """ResidualUnitMod (M:946-988) with Conv3DMod (M:718-753): per-clip weights w (cond + 1), demodulated by rsqrt(sum w_b^2),
    one grouped causal conv over the batch; ELU; 1x1x1 conv; ELU; residual.  x (B,T,H,W,C), cond_e (B, dim_cond)."""
    B, T, H, W, Cc = x.shape
    c = F.linear(cond_e.to(x.dtype), mod.to_cond.weight, mod.to_cond.bias)
    w = mod.conv.weights
    o, i, kt, kh, kw = w.shape
    wb = w[None] * (c[:, None, :, None, None, None] + 1.)
    wb = wb * (wb ** 2).sum(dim=(2, 3, 4, 5), keepdim=True).clamp(min=mod.conv.eps).rsqrt()
    xc = x.permute(0, 4, 1, 2, 3)
    xg = F.pad(xc.reshape(1, B * i, T, H, W), (kw // 2, kw // 2, kh // 2, kh // 2, kt - 1, 0))
    y = F.elu(F.conv3d(xg, wb.reshape(B * o, i, kt, kh, kw), groups=B).reshape(B, o, T, H, W))
    y = F.elu(F.conv3d(y, mod.conv_out.weight, mod.conv_out.bias))
    return (y + xc).permute(0, 2, 3, 4, 1)


def _feed_forward_block(x, ff, shift):
    """Residual(FeedForward) / Residual(TokenShift(FeedForward)) (M:466-508, M:1191, M:1236)."""
    xs = _token_shift(x) if shift else x
    xn = _rmsnorm(xs, ff.norm.gamma)
    w1, w2 = ff.net[0].weight, ff.net[2].weight
    hdn = F.linear(xn, w1.reshape(w1.shape[0], -1), ff.net[0].bias)
    a, gate = hdn.chunk(2, dim=-1)
    return F.linear(F.gelu(gate) * a, w2.reshape(w2.shape[0], -1), ff.net[2].bias) + x


def _upsample_space(x, conv):
    """SpatialUpsample2x (M:811-846): 1x1 conv C -> 4 C', SiLU, 'b (c p1 p2) h w -> b c (h p1) (w p2)'."""
    B, T, H, W, _ = x.shape
    w = conv.weight
    o = F.silu(F.linear(x, w.reshape(w.shape[0], -1), conv.bias))
    co = o.shape[-1] // 4
    return o.reshape(B, T, H, W, co, 2, 2).permute(0, 1, 2, 5, 3, 6, 4).reshape(B, T, 2 * H, 2 * W, co)


def _upsample_time(x, conv):
    """TimeUpsample2x (M:848-883): 1x1 conv C -> 2 C', SiLU, 'b (c p) t -> b c (t p)'."""
    B, T, H, W, _ = x.shape
    w = conv.weight
    o = F.silu(F.linear(x, w.reshape(w.shape[0], -1), conv.bias))
    co = o.shape[-1] // 2
    return o.reshape(B, T, H, W, co, 2).permute(0, 1, 5, 2, 3, 4).reshape(B, 2 * T, H, W, co)


def _entropy(p, eps=1e-5):
    return (-p * torch.log(p.clamp(min=eps))).sum(dim=-1)


def _lfq_train(x, qz, avg_global, inv_temperature=100.):
    """LFQ training forward (SURVEY Appendix A.1 steps 2-10) on (B,T,H,W,C): -> (straight-through quantised output, aux loss).
    `avg_global` is the cross-rank mean code probability of the forward pass; the local term enters as
    avg_local + (avg_global - avg_local).detach(), which reproduces the gradient of the reference's autograd-aware
    all-reduce (each rank back-propagates d H / d avg_global into its own tokens)."""
    d, nc = qz.codebook_dim, qz.num_codebooks
    p = F.linear(x, qz.project_in.weight, qz.project_in.bias)
    cv = qz.soft_clamp_input_value
    if cv:
        p = (p / cv).tanh() * cv
    p = p.reshape(-1, nc, d)
    if qz.spherical:
        p = F.normalize(p, dim=-1)
    p = p.float()
    qd = torch.where(p > 0, torch.ones_like(p), -torch.ones_like(p))
    st = (p + (qd - p).detach()).reshape(*x.shape[:-1], nc * d)
    out = F.linear(st.to(x.dtype), qz.project_out.weight, qz.project_out.bias)
    mask = qz.mask.to(p.device)
    codebook = ((torch.arange(2 ** d, device=p.device)[:, None] & mask) != 0).float() * 2 - 1
    prob = (2 * inv_temperature * torch.einsum("tcd,kd->tck", p, codebook)).softmax(dim=-1)      # (tokens, nc, K)
    per_sample = _entropy(prob).mean()
    avg_local = prob.mean(dim=0)                                                                  # (nc, K)
    avg = avg_local + (avg_global.reshape(nc, -1) - avg_local).detach()
    commit = ((p - qd) ** 2).mean()
    aux = (per_sample - qz.diversity_gamma * _entropy(avg).mean()) * qz.entropy_loss_weight + commit * qz.commitment_loss_weight
    return out, aux


def _fsq_train(x, qz):
    """FSQ forward (SURVEY Appendix A.2) with the round() straight-through estimator."""
    lv = torch.tensor(qz.levels * qz.num_codebooks, dtype=torch.int32, device=x.device)     # the levels repeat per codebook
    z = F.linear(x, qz.project_in.weight, qz.project_in.bias).float()
    half_l = (lv - 1) * (1 + 1e-3) / 2
    offset = torch.where(lv % 2 == 0, 0.5, 0.0)
    bounded = (z + (offset / half_l).atanh()).tanh() * half_l - offset
    quant = bounded + (bounded.round() - bounded).detach()
    return F.linear((quant / (lv // 2)).to(x.dtype), qz.project_out.weight, qz.project_out.bias)


# --------------------------------------------------------------------------------------------
# the tape
# --------------------------------------------------------------------------------------------
def _elu_grad(g, y):
    """d ELU(x) / dx from the OUTPUT y = ELU(x): 1 for x > 0 (y > 0), exp(x) = y + 1 otherwise."""
    return g * torch.where(y > 0, torch.ones_like(y), y + 1)


class TrainRunner:
    """One training-mode forward through the engine's kernels, recording what the backward needs."""

    def __init__(self, model):
        m = model
        self.g_cond: Dict[str, torch.Tensor] = {}      # gradient wrt the cond stems' outputs, summed over the cond_residual stages
        self.m = m
        self.eng = m.engine
        self.tape: List[Callable] = []
        self.grads: Dict[torch.nn.Parameter, torch.Tensor] = {}
        self.codes = None
        self.breakdown = None
        self.own_dgrad = True            # data gradient of the stride-1 convs through the engine's own conv kernels
        self.own_dgrad_calls = 0

    # ---- gradient bookkeeping
    def _acc(self, param, g):
        if g is None or not param.requires_grad:
            return
        g = g.reshape(param.shape).to(param.dtype)
        self.grads[param] = g if param not in self.grads else self.grads[param] + g

    def _vjp(self, fn, x, params: Sequence[torch.nn.Parameter], gout, extra=None):
        """Gradient of the block fn at its saved input x: re-evaluates the torch restatement under autograd.  `extra`: further
        leaf tensors (requires_grad) the block reads; their gradients are returned as the second element of a tuple."""
        x_ = x.detach().requires_grad_(True)
        params = [p for p in params if p.requires_grad]
        extra = list(extra or [])
        with torch.enable_grad():
            out = fn(x_)
        outs, gouts = (list(out), list(gout)) if isinstance(out, (tuple, list)) else ([out], [gout])
        gs = torch.autograd.grad(outs, [x_] + params + extra, gouts, allow_unused=True)
        for p, g in zip(params, gs[1:1 + len(params)]):
            self._acc(p, g)
        if extra:
            return gs[0], gs[1 + len(params):]
        return gs[0]

    def _conv_bwd(self, g, x, weight, bias, k, stride=(1, 1, 1), pad=None, need_gx=True, x_is_cf=False):
        """Backward of a conv the engine ran as  y = conv(x; leading pad (pt, ph, pw), stride).
        g: (B,To,Ho,Wo,Co) channels-last grad of the pre-activation output; x: the saved channels-last input (or, x_is_cf,
        a (B,C,T,H,W) tensor).  Returns grad wrt x (channels-last) or None.
          * data gradient of the stride-1 causal convs (every ResidualUnit conv, conv_out): OUR conv kernels -- the transposed
            conv is the same implicit GEMM with the weights flipped in (t, h, w) and transposed in (co, ci), no leading pad in
            time (gx[t] = sum_e W'[e] g[t + e]; frames past the clip are the kernels' out-of-bounds zeros);
          * weight / bias gradients, and the data gradient of the strided down-samplers: aten.convolution_backward (cuDNN).  The
            time axis is padded at the FRONT only (causal, M:913-928): those zero frames are materialised; H / W use the
            symmetric padding natively."""
        kt, kh, kw = k
        causal_default = pad is None
        if pad is None:
            pad = (kt - 1, kh // 2, kw // 2)
        pt, ph, pw = pad
        w5 = weight.reshape(weight.shape[0], weight.shape[1], kt, kh, kw)
        gx = None
        own_dgrad = need_gx and self.own_dgrad and causal_default and tuple(stride) == (1, 1, 1) and not x_is_cf
        if own_dgrad:
            wt = w5.detach().flip(2, 3, 4).transpose(0, 1).contiguous()          # (Ci, Co, kt, kh, kw): dgrad weights
            gx = self.eng.conv(g.contiguous(), pack_conv(wt, None, self.eng.dtype), pad=(0, ph, pw), out_spatial=tuple(x.shape[1:4]))
            self.own_dgrad_calls += 1
        if x_is_cf:
            x_cf = F.pad(x, (0, 0, 0, 0, pt, 0)) if pt > 0 else x
        else:       # pad the (contiguous) channels-last tensor along T, then view it as (B,C,T,H,W) in channels_last_3d strides
            x_cf = (F.pad(x, (0, 0, 0, 0, 0, 0, pt, 0)) if pt > 0 else x).permute(0, 4, 1, 2, 3)
        lib_gx = need_gx and not own_dgrad
        gxl, gw, gb = torch.ops.aten.convolution_backward(
            g.permute(0, 4, 1, 2, 3), x_cf, w5, [w5.shape[0]] if bias is not None else None, list(stride), [0, ph, pw],
            [1, 1, 1], False, [0, 0, 0], 1, [lib_gx, weight.requires_grad, bias is not None and bias.requires_grad])
        self._acc(weight, gw)
        if bias is not None:
            self._acc(bias, gb)
        if not need_gx:
            return None
        if own_dgrad:
            return gx
        return gxl[:, :, pt:].permute(0, 2, 3, 4, 1).contiguous()

    def _conv_bwd_padmode(self, g, x, weight, bias, k, pad_mode, need_gx=True):
        """Backward of Engine.causal_conv_padded (CausalConv3d with pad_mode reflect / replicate / circular, M:925-927): the padding
        is re-applied with F.pad under autograd, the conv backward runs without implicit padding on the padded tensor, and the
        gradient is folded back through the padding.  Falls back to the zero-padded case like the forward (time_pad >= T)."""
        kt, kh, kw = k
        if pad_mode == "constant" or kt - 1 >= x.shape[1]:
            return self._conv_bwd(g, x, weight, bias, k, need_gx=need_gx)
        x_ = x.detach().permute(0, 4, 1, 2, 3).requires_grad_(need_gx)
        with torch.enable_grad():
            xp = F.pad(x_, (kw // 2, kw // 2, kh // 2, kh // 2, kt - 1, 0), mode=pad_mode)
        w5 = weight.reshape(weight.shape[0], weight.shape[1], kt, kh, kw)
        gxp, gw, gb = torch.ops.aten.convolution_backward(
            g.permute(0, 4, 1, 2, 3), xp.detach(), w5, [w5.shape[0]] if bias is not None else None, [1, 1, 1], [0, 0, 0], [1, 1, 1],
            False, [0, 0, 0], 1, [need_gx, weight.requires_grad, bias is not None and bias.requires_grad])
        self._acc(weight, gw)
        if bias is not None:
            self._acc(bias, gb)
        if not need_gx:
            return None
        gx, = torch.autograd.grad(xp, x_, gxp)
        return gx.permute(0, 2, 3, 4, 1).contiguous()

    # ---- forward pieces (engine kernels) that record their backward
    def _residual_unit(self, x, p, u):
        """ResidualUnit (M:930-944) unfused: both conv outputs are kept for the backward."""
        out, h, y = self.eng.residual_unit_unfused(x, p)
        c3m, c1m, se = u["conv3"], u["conv1"], u["se"]
        k3 = tuple(c3m.weight.shape[2:])

        def bwd(g):
            gy = self._vjp(lambda t: _squeeze_excite(t, se), y, list(se.parameters()), g)
            gh = self._conv_bwd(_elu_grad(gy, y), h, c1m.weight, c1m.bias, (1, 1, 1))
            gx = self._conv_bwd(_elu_grad(gh, h), x, c3m.weight, c3m.bias, k3)
            return g + gx

        self.tape.append(bwd)
        return out

    def _block(self, x, run, fn, params):
        """A light block: forward by the engine (`run`), backward by the torch restatement `fn` on the saved input."""
        out = run(x)
        self.tape.append(lambda g: self._vjp(fn, x, params, g))
        return out

    def _stage(self, x, st, key, parts, decoder, cond_e=None):
        """One stage through the engine; `parts` = engine.stage_modules(...) of its layer module."""
        eng = self.eng
        P = eng._packs
        if st.kind == "cond_residual":
            mod = parts["unit"]
            side = "dec" if decoder else "enc"
            xin = x
            out = eng._stage(x, st, key, decoder=decoder, cond_e=cond_e)

            def bwd(g):
                ce = cond_e.detach().requires_grad_(True)
                gx, (gc,) = self._vjp(lambda t: _residual_unit_mod(t, ce, mod), xin, list(mod.parameters()), g, extra=[ce])
                if gc is not None:
                    self.g_cond[side] = gc if side not in self.g_cond else self.g_cond[side] + gc
                return gx

            self.tape.append(bwd)
            return out
        if st.kind == "residual":
            for j, u in enumerate(parts["units"]):
                x = self._residual_unit(x, P[f"{key}.{j}"], u)
            return x
        if st.kind in ("compress_space", "compress_time") and not decoder:
            conv = parts["conv"]
            if st.kind == "compress_space":     # SpatialDownsample2x (M:770-780): Conv2d k3 s2 p1 per frame
                k, stride, pad = (1, 3, 3), (1, 2, 2), (0, 1, 1)
            else:                               # TimeDownsample2x (M:796-807): F.pad (2, 0) + Conv1d k3 s2 per pixel
                k, stride, pad = (3, 1, 1), (2, 1, 1), (2, 0, 0)
            xin = x
            out = eng._stage(x, st, key, decoder=False)
            self.tape.append(lambda g: self._conv_bwd(g, xin, conv.weight, conv.bias, k, stride, pad))
            return out
        run = lambda t: eng._stage(t, st, key, decoder=decoder)       # noqa: E731
        if st.kind == "compress_space":
            conv = parts["conv"]
            return self._block(x, run, lambda t: _upsample_space(t, conv), list(conv.parameters()))
        if st.kind == "compress_time":
            conv = parts["conv"]
            return self._block(x, run, lambda t: _upsample_time(t, conv), list(conv.parameters()))
        if st.kind == "gateloop_time":
            gl = parts["gateloop"]
            return self._block(x, run, lambda t: _gateloop_block(t, gl), list(gl.parameters()))
        if st.kind in ("attend_space", "attend_time", "linear_attend_space"):
            time_axis = st.kind == "attend_time"
            at, ff = parts["attn"], parts["ff"]
            if st.kind == "linear_attend_space":
                x = self._block(x, lambda t: eng.linear_attention(t, P[key + ".attn"]), lambda t: _linear_attention_block(t, at),
                                list(at.parameters()))
            else:
                axis = "time" if time_axis else "space"
                x = self._block(x, lambda t: eng.attention(t, P[key + ".attn"], axis), lambda t: _attention_block(t, at, axis),
                                list(at.parameters()))
            return self._block(x, lambda t: eng.feed_forward(t, P[key + ".ff"], token_shift=time_axis),
                               lambda t: _feed_forward_block(t, ff, time_axis), list(ff.parameters()))
        raise NotImplementedError(f"no training path for layer type {st.kind!r}")

    def forward(self, video, first_frame=True, group=None, cond=None):
        """-> (recon (B,C,T,H,W), aux_loss 0-d fp32); codes / the LFQ breakdown are left in .codes / .breakdown."""
        from .dist import LfqBatchEntropy
        m, eng = self.m, self.eng
        self.cond = cond
        ce_enc = eng.cond_stem(cond, "enc") if m.has_cond else None            # M:1544-1548 (Linear + SiLU stems)
        ce_dec = eng.cond_stem(cond, "dec") if m.has_cond else None            # M:1612-1616
        t_pad = m.time_padding if first_frame else 0
        cin, cout = m.conv_in.conv, m.conv_out.conv
        kin = tuple(cin.weight.shape[2:])
        sff = bool(m.separate_first_frame_encoding and first_frame)
        mode_in, mode_out = m.conv_in.pad_mode, m.conv_out.pad_mode
        x, saved_in = eng.conv_in_cl(video, first_frame)

        def bwd_conv_in(g):     # the video needs no gradient: weight / bias only
            v = (video.float() / 255. if video.dtype == torch.uint8 else video).to(eng.dtype)
            if sff:
                ff = m.conv_in_first_frame
                kff = (1,) + tuple(ff.weight.shape[2:])
                self._conv_bwd(g[:, t_pad:t_pad + 1].contiguous(), v[:, :, 0:1], ff.weight, ff.bias, kff, pad=(0, kff[1] // 2, kff[2] // 2),
                               need_gx=False, x_is_cf=True)
                if v.shape[2] > 1:
                    self._conv_bwd_padmode(g[:, t_pad + 1:].contiguous(), saved_in["rest_in"], cin.weight, cin.bias, kin, mode_in, need_gx=False)
                return None
            if mode_in != "constant":
                self._conv_bwd_padmode(g, saved_in["padded_in"], cin.weight, cin.bias, kin, mode_in, need_gx=False)
                return None
            self._conv_bwd(g, v, cin.weight, cin.bias, kin, pad=(t_pad + kin[0] - 1, kin[1] // 2, kin[2] // 2),
                           need_gx=False, x_is_cf=True)
            return None

        self.tape.append(bwd_conv_in)
        for i, st in enumerate(m.stages):
            x = self._stage(x, st, f"enc{i}", stage_modules(st, m.encoder_layers[i], False), decoder=False, cond_e=ce_enc)

        qz = m.quantizers
        if m.use_fsq:
            xq = x
            q, self.codes, _ = eng.quantize_cl(x)
            aux = torch.zeros((), device=eng.device, dtype=torch.float32)
            self._q_index = len(self.tape)
            self.tape.append(lambda gs: self._vjp(lambda t: _fsq_train(t, qz), xq, list(qz.parameters()), gs[0]))
        else:
            xq = x
            q, self.codes, pre = eng.quantize_cl(x, want_quantized=True, want_aux=True)
            be = LfqBatchEntropy(eng, num_codebooks=qz.num_codebooks)
            be.start(pre, group)
            avg_sum = be.avg_prob_sum
            ps, bent, commit, aux = be.finish(qz.diversity_gamma, qz.entropy_loss_weight, qz.commitment_loss_weight, group)
            world = torch.distributed.get_world_size(group) if (torch.distributed.is_available() and torch.distributed.is_initialized()) else 1
            avg_global = avg_sum / world
            self.breakdown = (ps, bent, commit)
            self._q_index = len(self.tape)
            self.tape.append(lambda gs: self._vjp(lambda t: _lfq_train(t, qz, avg_global), xq, list(qz.parameters()), gs))

        x = q
        for j, st in enumerate(reversed(m.stages)):
            x = self._stage(x, st, f"dec{j}", stage_modules(st, m.decoder_layers[j], True), decoder=True, cond_e=ce_dec)
        xo = x
        kout = tuple(cout.weight.shape[2:])
        recon, saved_out = eng.conv_out_cf(x, first_frame)

        def bwd_conv_out(g_recon):    # (B,C,T,H,W) -> channels-last with zero gradient on the cropped time_padding frames
            g = g_recon.permute(0, 2, 3, 4, 1)
            if sff:
                off = m.conv_out_first_frame
                kff = (1,) + tuple(off.weight.shape[2:])
                gx = torch.zeros_like(xo)
                gx[:, t_pad:t_pad + 1] = self._conv_bwd(g[:, 0:1].contiguous(), xo[:, t_pad:t_pad + 1].contiguous(), off.weight, off.bias, kff,
                                                        pad=(0, kff[1] // 2, kff[2] // 2))
                if xo.shape[1] - t_pad > 1:
                    gx[:, t_pad + 1:] = self._conv_bwd_padmode(g[:, 1:].contiguous(), saved_out["rest_out"], cout.weight, cout.bias, kout, mode_out)
                return gx
            if t_pad:
                g = F.pad(g, (0, 0, 0, 0, 0, 0, t_pad, 0))
            return self._conv_bwd_padmode(g.contiguous(), xo, cout.weight, cout.bias, kout, mode_out)

        self.tape.append(bwd_conv_out)
        self._recon_shape = tuple(recon.shape)
        return recon, aux

    def backward(self, g_recon, g_aux):
        """Runs the tape in reverse; returns {Parameter: grad}.  g_recon (B,C,T,H,W) or None, g_aux 0-d or None."""
        if not self.tape:
            raise RuntimeError("the tokenizer's backward ran already: the saved activations are released after one backward pass "
                               "(call the forward again; retain_graph is not supported by this path)")
        if g_recon is None:
            g_recon = torch.zeros(self._recon_shape, device=self.eng.device, dtype=self.eng.dtype)
        g = g_recon.to(self.eng.dtype)
        n = len(self.tape)
        q_index = self._q_index                  # the quantiser's entry sits between the encoder and decoder entries
        with torch.no_grad():
            for i in range(n - 1, -1, -1):
                if i == q_index:
                    if self.m.use_fsq:
                        g = self.tape[i]((g,))
                    else:
                        ga = g_aux if g_aux is not None else torch.zeros((), device=self.eng.device)
                        g = self.tape[i]((g, ga.float()))
                else:
                    g = self.tape[i](g)
            for side, stem in (("enc", self.m.encoder_cond_in), ("dec", self.m.decoder_cond_in)):
                if side in self.g_cond:       # cond stems (M:1344-1352): Linear + SiLU of the raw cond vector
                    lin = stem[0]
                    self._vjp(lambda t, lin=lin: F.silu(F.linear(t, lin.weight.float(), lin.bias.float())), self.cond.float(),
                              list(lin.parameters()), self.g_cond[side].float())
        self.tape = []
        return self.grads


class _TokenizerTrainFn(torch.autograd.Function):
    """(video, *parameters) -> (recon, aux_loss): forward by the engine kernels, backward by TrainRunner's tape."""

    @staticmethod
    def forward(ctx, runner, first_frame, cond, video, *params):
        recon, aux = runner.forward(video, first_frame, cond=cond)
        ctx.runner, ctx.params = runner, params
        return recon, aux

    @staticmethod
    def backward(ctx, g_recon, g_aux):
        grads = ctx.runner.backward(g_recon, g_aux)
        # every parameter handed to the Function gets a gradient tensor (zeros if this call did not touch it, e.g. conv_in of a
        # one-frame clip with separate_first_frame_encoding): DistributedDataParallel waits for the hook of every parameter it can
        # reach from the outputs
        return (None, None, None, None) + tuple(grads[p] if p in grads else torch.zeros_like(p) for p in ctx.params)


def live_parameters(model, first_frame=True):
    """The parameters a forward can reach.  Left out, exactly like in the reference's graph (so DistributedDataParallel must be
    built with find_unused_parameters=True there as here): the final LayerNorm of the encoder, which is constructed but never
    executed (M:1322-1326, M:1565), and the first-frame convs unless separate_first_frame_encoding applies to this call."""
    dead = {id(p) for p in model.encoder_layers[len(model.stages)].parameters()}
    if not (model.separate_first_frame_encoding and first_frame):
        dead |= {id(p) for mod in (model.conv_in_first_frame, model.conv_out_first_frame) for p in mod.parameters()}
    return [p for p in model.parameters() if p.requires_grad and id(p) not in dead]


def train_forward(model, video, first_frame=True, cond=None):
    """-> (recon with grad_fn, aux_loss with grad_fn, codes, lfq breakdown | None)."""
    runner = TrainRunner(model)
    params = live_parameters(model, first_frame)
    recon, aux = _TokenizerTrainFn.apply(runner, first_frame, cond, video, *params)
    return recon, aux, runner.codes, runner.breakdown
