"""TEST INFRASTRUCTURE ONLY -- the oracle for the VGen sampling hot path.

A plain-PyTorch (fp32 by default) restatement of what the reference computes on the path
    DiffusionDDIM.ddim_sample_loop -> UNetSD_T2VBase / UNetSD_I2VGen (+ VideoLCM / SR600 / HiGen variants)
    forward -> AutoencoderKL.decode,
written from the reference's arithmetic, not from its module tree: every function works directly on a
reference-format state_dict (dict name -> tensor) and derives the block structure from the key names.
Each function cites the reference lines it follows (paths relative to the reference root).

Pinning: the reference has no tests or golden vectors for this path (SURVEY.md section 4), so the
oracle is pinned against the reference ITSELF, imported on CPU through oracle/refload.py:
oracle/make_golden.py and oracle/make_golden_pin.py run the reference classes next to every function
here and freeze their outputs into tests/golden/, which tests/test_oracle_golden.py and
tests/test_oracle_pin.py compare with, so the pin holds where the reference is absent.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.  The product (vgen_b200/) never does.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


# ------------------------------------------------------------------------------------ schedules
def cosine_betas(num_timesteps=1000, cosine_s=0.008):
    """tools/modules/diffusions/schedules.py:72-79 (python-float loop, clamp 0.999, fp64)."""
    def abar(u):
        return math.cos((u + cosine_s) / (1 + cosine_s) * math.pi / 2) ** 2
    vals = []
    for i in range(num_timesteps):
        vals.append(min(1.0 - abar((i + 1) / num_timesteps) / abar(i / num_timesteps), 0.999))
    return torch.tensor(vals, dtype=torch.float64)


def linear_sd_betas(num_timesteps, init_beta, last_beta):
    """schedules.py:62-63."""
    return torch.linspace(init_beta ** 0.5, last_beta ** 0.5, num_timesteps, dtype=torch.float64) ** 2


def zero_terminal_snr(betas):
    """schedules.py:143-165: shift/scale sqrt(alpha_bar) so the last step has zero SNR."""
    sab = (1 - betas).cumprod(0).sqrt()
    first, last = sab[0].clone(), sab[-1].clone()
    sab = (sab - last) * (first / (first - last))
    ab = sab ** 2
    alphas = torch.cat([ab[0:1], ab[1:] / ab[:-1]])
    return 1 - alphas


def make_betas(schedule="cosine", num_timesteps=1000, zero_terminal_snr_flag=False, **kw):
    """schedules.py:5-21."""
    if schedule == "cosine":
        b = cosine_betas(num_timesteps, kw.get("cosine_s", 0.008))
    elif schedule == "linear_sd":
        b = linear_sd_betas(num_timesteps, kw["init_beta"], kw["last_beta"])
    else:
        raise ValueError(schedule)
    if zero_terminal_snr_flag and abs(b.max() - 1.0) > 0.0001:
        b = zero_terminal_snr(b)
    return b


def ddim_tables(betas):
    """diffusion_ddim.py:46-78 -- the fp64 tables the DDIM path reads."""
    ab = torch.cumprod(1 - betas, dim=0)
    return {
        "alphas_cumprod": ab,
        "sqrt_alphas_cumprod": torch.sqrt(ab),
        "sqrt_one_minus_alphas_cumprod": torch.sqrt(1.0 - ab),
        "sqrt_recip_alphas_cumprod": torch.sqrt(1.0 / ab),
        "sqrt_recipm1_alphas_cumprod": torch.sqrt(1.0 / ab - 1),
    }


def ddim_steps(num_timesteps, ddim_timesteps):
    """diffusion_ddim.py:250."""
    return (1 + torch.arange(0, num_timesteps, num_timesteps // ddim_timesteps)).clamp(0, num_timesteps - 1).flip(0)


def ddim_sample_loop(noise, model, model_kwargs, betas, guide_scale, ddim_timesteps, eta=0.0, mean_type="v",
                     autocast_cfg=False, trace=None, max_steps=None):
    """diffusion_ddim.py:244-254 (loop), :209-241 (ddim_sample), :147-206 (p_mean_variance) for
    var_type fixed_small, mean_type v|eps, clamp/percentile/condition_fn None.

    model(xt, t, **kwargs) -> tensor shaped like xt.  With autocast_cfg the classifier-free mix is done
    in the model's output dtype (fp16 under the reference's autocast); table entries are cast to xt's
    dtype exactly like _i() (:10-16).  max_steps (test aid): stop after that many steps of the schedule."""
    T = len(betas)
    tab = ddim_tables(betas)
    stride = T // ddim_timesteps
    xt = noise
    b = noise.size(0)

    def pick(name, t):
        return tab[name].to(xt.device)[t].view(b, *([1] * (xt.ndim - 1))).to(xt)

    for n_done, step in enumerate(ddim_steps(T, ddim_timesteps)):
        if max_steps is not None and n_done >= max_steps:
            break
        t = torch.full((b,), int(step), dtype=torch.long, device=xt.device)
        if guide_scale is None:
            out = model(xt, t, **model_kwargs)
        else:
            y_out = model(xt, t, **model_kwargs[0])
            u_out = model(xt, t, **model_kwargs[1])
            if not autocast_cfg:
                y_out, u_out = y_out.to(xt.dtype), u_out.to(xt.dtype)
            out = u_out + guide_scale * (y_out - u_out)
        if mean_type == "v":
            x0 = pick("sqrt_alphas_cumprod", t) * xt - pick("sqrt_one_minus_alphas_cumprod", t) * out
        elif mean_type == "eps":
            x0 = pick("sqrt_recip_alphas_cumprod", t) * xt - pick("sqrt_recipm1_alphas_cumprod", t) * out
        else:
            raise ValueError(mean_type)
        eps = (pick("sqrt_recip_alphas_cumprod", t) * xt - x0) / pick("sqrt_recipm1_alphas_cumprod", t)
        a_t = pick("alphas_cumprod", t)
        a_prev = pick("alphas_cumprod", (t - stride).clamp(0))
        sigma = eta * torch.sqrt((1 - a_prev) / (1 - a_t) * (1 - a_t / a_prev))
        noise_t = torch.randn_like(xt)  # drawn even when eta == 0 (:237)
        mask = t.ne(0).float().view(b, *([1] * (xt.ndim - 1)))
        xt = torch.sqrt(a_prev) * x0 + torch.sqrt(1 - a_prev - sigma ** 2) * eps + mask * sigma * noise_t
        if trace is not None:
            trace.append(xt.clone())
    return xt


# ------------------------------------------------------------------------------------ primitives
def sinusoidal_embedding(t, dim):
    """tools/modules/unet/util.py:178-190 (cos first, then sin)."""
    half = dim // 2
    t = t.float()
    freqs = torch.pow(10000, -torch.arange(half).to(t).div(half))
    ang = torch.outer(t, freqs)
    return torch.cat([torch.cos(ang), torch.sin(ang)], dim=1)


class _SD:
    """state_dict view with a prefix."""

    def __init__(self, sd, prefix=""):
        self.sd, self.p = sd, prefix

    def sub(self, name):
        return _SD(self.sd, f"{self.p}{name}.")

    def __getitem__(self, name):
        return self.sd[self.p + name]

    def has(self, name):
        return (self.p + name) in self.sd

    def get(self, name):
        return self.sd.get(self.p + name)


def _gn(x, s, eps):
    return F.group_norm(x, 32, s["weight"], s["bias"], eps)


def _ln(x, s):
    return F.layer_norm(x, (x.shape[-1],), s["weight"], s["bias"], 1e-5)


def _lin(x, s):
    return F.linear(x, s["weight"], s.get("bias"))


def _attention(x, ctx, s, heads):
    """MemoryEfficientCrossAttention, util.py:231-269: softmax(q k^T / sqrt(d)) v per head."""
    ctx = x if ctx is None else ctx
    q, k, v = _lin(x, s.sub("to_q")), _lin(ctx, s.sub("to_k")), _lin(ctx, s.sub("to_v"))
    b, lq, inner = q.shape
    d = inner // heads

    def split(t):
        return t.reshape(b, t.shape[1], heads, d).permute(0, 2, 1, 3)

    o = F.scaled_dot_product_attention(split(q), split(k), split(v))
    o = o.permute(0, 2, 1, 3).reshape(b, lq, inner)
    return _lin(o, s.sub("to_out.0"))


def _basic_block(x, ctx, s, heads):
    """BasicTransformerBlock.forward, util.py:700-704 (attn2 is self-attention when ctx is None);
    FeedForward/GEGLU :707-741 (exact erf GELU)."""
    x = _attention(_ln(x, s.sub("norm1")), None, s.sub("attn1"), heads) + x
    x = _attention(_ln(x, s.sub("norm2")), ctx, s.sub("attn2"), heads) + x
    h = _ln(x, s.sub("norm3"))
    val, gate = _lin(h, s.sub("ff.net.0.proj")).chunk(2, dim=-1)
    x = _lin(val * F.gelu(gate), s.sub("ff.net.2")) + x
    return x


def _temporal_conv(x5, s, woimg=False):
    """TemporalConvBlock_v2.forward, util.py:1686-1697.  x5: [b, c, f, h, w]; GroupNorm statistics
    span all frames; conv is (3,1,1) with zero padding over f.  woimg: TemporalConvBlock_v2WoImg
    (unet_higen.py:71-85) multiplies the branch by 0.0 when there is a single frame."""
    h = x5
    for name, widx in (("conv1", 2), ("conv2", 3), ("conv3", 3), ("conv4", 3)):
        c = s.sub(name)
        h = F.silu(F.group_norm(h, 32, c["0.weight"], c["0.bias"], 1e-5))
        h = F.conv3d(h, c[f"{widx}.weight"], c[f"{widx}.bias"], padding=(1, 0, 0))
    if woimg and x5.size(2) == 1:
        return x5 + 0.0 * h
    return x5 + h


def _res_block(x, emb, s, batch, woimg=False):
    """ResBlock._forward, util.py:900-927 (use_scale_shift_norm False, no up/down).  x: [(b f), c, h, w]."""
    h = F.conv2d(F.silu(_gn(x, s.sub("in_layers.0"), 1e-5)), s["in_layers.2.weight"], s["in_layers.2.bias"], padding=1)
    e = _lin(F.silu(emb), s.sub("emb_layers.1")).type(h.dtype)
    h = h + e[:, :, None, None]
    h = F.conv2d(F.silu(_gn(h, s.sub("out_layers.0"), 1e-5)), s["out_layers.3.weight"], s["out_layers.3.bias"], padding=1)
    skip = x if not s.has("skip_connection.weight") else F.conv2d(x, s["skip_connection.weight"], s["skip_connection.bias"])
    h = skip + h
    bf, c, hh, ww = h.shape
    h5 = h.reshape(batch, bf // batch, c, hh, ww).permute(0, 2, 1, 3, 4)
    h5 = _temporal_conv(h5, s.sub("temopral_conv"), woimg)  # (sic) the typo is part of the checkpoint format
    return h5.permute(0, 2, 1, 3, 4).reshape(bf, c, hh, ww)


def _spatial_transformer(x, ctx, s, head_dim):
    """SpatialTransformer.forward (use_linear=True), util.py:354-373."""
    bf, c, hh, ww = x.shape
    h = _gn(x, s.sub("norm"), 1e-6).permute(0, 2, 3, 1).reshape(bf, hh * ww, c)
    h = _lin(h, s.sub("proj_in"))
    h = _basic_block(h, ctx, s.sub("transformer_blocks.0"), h.shape[-1] // head_dim)
    h = _lin(h, s.sub("proj_out"))
    return h.reshape(bf, hh, ww, c).permute(0, 3, 1, 2) + x


def _temporal_transformer(x, s, head_dim, batch, woimg=False):
    """TemporalTransformer.forward (use_linear=False, only_self_att=True), util.py:1240-1286.
    x: [(b f), c, h, w]; tokens are the f frames of one pixel; both attentions are self-attention."""
    bf, c, hh, ww = x.shape
    f = bf // batch
    x5 = x.reshape(batch, f, c, hh, ww).permute(0, 2, 1, 3, 4)           # b c f h w
    h = F.group_norm(x5, 32, s["norm.weight"], s["norm.bias"], 1e-6)
    h = h.permute(0, 3, 4, 2, 1).reshape(batch * hh * ww, f, c)          # (b h w) f c
    h = F.linear(h, s["proj_in.weight"][:, :, 0], s["proj_in.bias"])     # Conv1d k=1 == per-token linear
    h = _basic_block(h, None, s.sub("transformer_blocks.0"), h.shape[-1] // head_dim)
    h = F.linear(h, s["proj_out.weight"][:, :, 0], s["proj_out.bias"])
    h = h.reshape(batch, hh, ww, f, c).permute(0, 3, 4, 1, 2).reshape(bf, c, hh, ww)
    if woimg and f == 1:                                                 # TemporalTransformerWoImg, unet_higen.py:146-149
        return 0.0 * h + x
    return h + x


def _run_block(x, s, emb, ctx, head_dim, batch, woimg=False, sr600=False):
    """One entry of input_blocks / middle_block / output_blocks: dispatch on the parameters present
    (the reference dispatches on module type, unet_t2v.py:280-348)."""
    if s.has("in_layers.0.weight"):
        return _res_block(x, emb, s, batch, woimg)
    if s.has("transformer_blocks.0.norm1.weight"):
        if s["proj_in.weight"].ndim == 2:
            return _spatial_transformer(x, ctx, s, head_dim)
        return _temporal_transformer(x, s, head_dim, batch, woimg)
    if s.has("op.weight"):                                    # Downsample: conv3x3 stride 2, util.py:946
        # UNetSD_SR600 pads the height by 2 (unet_sr600.py:151-153) so that odd heights survive the round trip
        return F.conv2d(x, s["op.weight"], s["op.bias"], stride=2, padding=(2, 1) if sr600 else 1)
    if s.has("conv.weight"):                                  # Upsample: nearest x2 then conv, util.py:761-771
        up = F.interpolate(x, scale_factor=2, mode="nearest")
        if sr600:                                             # UpsampleSR600 drops the first and last row, util.py:799-801
            up = up[..., 1:-1, :]
        return F.conv2d(up, s["conv.weight"], s["conv.bias"], padding=1)
    if s.has("weight"):                                       # the first plain conv
        return F.conv2d(x, s["weight"], s["bias"], padding=1)
    raise KeyError(f"unrecognised block at {s.p}")


def _children(sd, prefix):
    idx = set()
    n = len(prefix)
    for k in sd:
        if k.startswith(prefix):
            idx.add(int(k[n:].split(".", 1)[0]))
    return sorted(idx)


def fourier_filter(x, threshold, scale):
    """Fourier_filter, unet_sr600.py:30-49: scale the (2*threshold)^2 centre bins of the shifted 2-D
    spectrum of every [H, W] plane, keep the real part of the inverse transform."""
    dtype = x.dtype
    xf = torch.fft.fftshift(torch.fft.fftn(x.float(), dim=(-2, -1)), dim=(-2, -1))
    hh, ww = xf.shape[-2:]
    mask = torch.ones(xf.shape, dtype=torch.float32, device=x.device)
    crow, ccol = hh // 2, ww // 2
    mask[..., crow - threshold:crow + threshold, ccol - threshold:ccol + threshold] = scale
    xf = torch.fft.ifftshift(xf * mask, dim=(-2, -1))
    return torch.fft.ifftn(xf, dim=(-2, -1)).real.to(dtype)


def _unet_trunk(sd, x, emb, ctx, head_dim, batch, woimg=False, conv_in_add=None, sr600=False):
    """encoder / middle / decoder with skip concatenation, unet_t2v.py:257-277.
    conv_in_add: tensor added right after the first conv (HiGen img_embedding, unet_higen.py:544-547);
    sr600: backbone scaling + Fourier-filtered skips on the first two decoder blocks (unet_sr600.py:269-285)."""
    root = _SD(sd)
    skips = []
    for i in _children(sd, "input_blocks."):
        blk = root.sub(f"input_blocks.{i}")
        if blk.has("op.weight"):
            x = _run_block(x, blk, emb, ctx, head_dim, batch, woimg, sr600)
        else:
            for j in _children(sd, blk.p):
                x = _run_block(x, blk.sub(str(j)), emb, ctx, head_dim, batch, woimg, sr600)
                if i == 0 and j == 0 and conv_in_add is not None:
                    x = x + conv_in_add
        skips.append(x)
    for j in _children(sd, "middle_block."):
        x = _run_block(x, root.sub(f"middle_block.{j}"), emb, ctx, head_dim, batch, woimg)
    for n, i in enumerate(_children(sd, "output_blocks.")):
        skip = skips.pop()
        if sr600 and n < 2:
            half = x.shape[1] // 2
            x = torch.cat([x[:, :half] * (1.1, 1.2)[n], x[:, half:]], dim=1)
            skip = fourier_filter(skip, 1, (0.6, 0.4)[n])
        x = torch.cat([x, skip], dim=1)
        blk = root.sub(f"output_blocks.{i}")
        for j in _children(sd, blk.p):
            x = _run_block(x, blk.sub(str(j)), emb, ctx, head_dim, batch, woimg, sr600)
    x = F.conv2d(F.silu(_gn(x, root.sub("out.0"), 1e-5)), sd["out.2.weight"], sd["out.2.bias"], padding=1)
    return x


def _mlp(x, s):
    return _lin(F.silu(_lin(x, s.sub("0"))), s.sub("2"))


def unet_t2v_forward(sd, x, t, y, fps=None, head_dim=64, use_fps_condition=False):
    """UNetSD_T2VBase.forward, unet_t2v.py:210-277.  x [b,4,f,h,w]; t [b]; y [b,L,1024]."""
    b, c, f, h, w = x.shape
    dim = sd["time_embed.0.weight"].shape[1]
    root = _SD(sd)
    emb = _mlp(sinusoidal_embedding(t, dim).to(x.dtype), root.sub("time_embed"))
    if use_fps_condition and fps is not None:
        emb = emb + _mlp(sinusoidal_embedding(fps, dim).to(x.dtype), root.sub("fps_embedding"))
    emb = emb.repeat_interleave(f, dim=0)
    ctx = y.repeat_interleave(f, dim=0)
    xx = x.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
    out = _unet_trunk(sd, xx, emb, ctx, head_dim, b)
    return out.reshape(b, f, -1, h, w).permute(0, 2, 1, 3, 4)


def unet_videolcm_forward(sd, x, t, y, fps=None, head_dim=64, use_fps_condition=False):
    """UNetSD_VideoLCM.forward with video_compositions == ['text'] (configs/videolcm_t2v_infer.yaml:67),
    unet_videolcm.py:541-760: `concat` stays all-zero (:598), pre_image is an empty Sequential (:409,705),
    the context is y alone (:713-726)."""
    b, c, f, h, w = x.shape
    dim = sd["time_embed.0.weight"].shape[1]
    root = _SD(sd)
    concat_dim = sd["input_blocks.0.0.weight"].shape[1] - c
    xx = torch.cat([x, x.new_zeros(b, concat_dim, f, h, w)], dim=1)
    emb = _mlp(sinusoidal_embedding(t, dim).to(x.dtype), root.sub("time_embed"))
    if use_fps_condition and fps is not None:
        emb = emb + _mlp(sinusoidal_embedding(fps, dim).to(x.dtype), root.sub("fps_embedding"))
    emb = emb.repeat_interleave(f, dim=0)
    ctx = y.repeat_interleave(f, dim=0)
    xx = xx.permute(0, 2, 1, 3, 4).reshape(b * f, c + concat_dim, h, w)
    out = _unet_trunk(sd, xx, emb, ctx, head_dim, b)
    return out.reshape(b, f, -1, h, w).permute(0, 2, 1, 3, 4)


def unet_sr600_forward(sd, x, t, y, head_dim=64):
    """UNetSD_SR600.forward, unet_sr600.py:220-299."""
    b, c, f, h, w = x.shape
    dim = sd["time_embed.0.weight"].shape[1]
    emb = _mlp(sinusoidal_embedding(t, dim).to(x.dtype), _SD(sd).sub("time_embed")).repeat_interleave(f, dim=0)
    ctx = y.repeat_interleave(f, dim=0)
    xx = x.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
    out = _unet_trunk(sd, xx, emb, ctx, head_dim, b, sr600=True)
    return out.reshape(b, f, -1, h, w).permute(0, 2, 1, 3, 4)


def _context_block_higen(x, ctx, s, heads):
    """BasicTransformerBlock with disable_self_attn=True (util.py:700-704): attn1 is cross attention too."""
    x = _attention(_ln(x, s.sub("norm1")), ctx, s.sub("attn1"), heads) + x
    x = _attention(_ln(x, s.sub("norm2")), ctx, s.sub("attn2"), heads) + x
    h = _ln(x, s.sub("norm3"))
    val, gate = _lin(h, s.sub("ff.net.0.proj")).chunk(2, dim=-1)
    return _lin(val * F.gelu(gate), s.sub("ff.net.2")) + x


def unet_higen_forward(sd, x, t, y, spat_prior, motion_cond, appearance_cond, fps=None, head_dim=64,
                       use_fps_condition=False):
    """UNetSD_HiGen.forward, unet_higen.py:401-467.
    embeddings (:436-443): per-frame time + motion (:387-396, linear interpolation of f-1 embeddings to f
    frames) + appearance (:398-399); context (:444-445): TextContextCrossTransformerMultiLayer :154-172;
    spat_prior enters through img_embedding right after the first conv (:544-547)."""
    b, c, f, h, w = x.shape
    dim = sd["time_embed.0.weight"].shape[1]
    root = _SD(sd)
    emb = _mlp(sinusoidal_embedding(t, dim).to(x.dtype), root.sub("time_embed"))
    if use_fps_condition and fps is not None:
        emb = emb + _mlp(sinusoidal_embedding(fps, dim).to(x.dtype), root.sub("fps_embedding"))
    emb = emb.repeat_interleave(f, dim=0)
    if f > 1:
        if motion_cond.size(1) != f:
            me = sinusoidal_embedding(motion_cond.flatten(0, 1), dim).view(b, f - 1, dim)
            me = F.interpolate(me.transpose(1, 2), size=f, mode="linear").transpose(1, 2)
        else:
            me = sinusoidal_embedding(motion_cond.flatten(0, 1), dim).view(b, f, dim)
        me = _mlp(me.to(x.dtype), root.sub("msim_embedding")).flatten(0, 1)
    else:
        me = _mlp(sinusoidal_embedding(motion_cond, dim).to(x.dtype), root.sub("msim_embedding"))
    emb = emb + me
    emb = emb + _mlp(appearance_cond.to(x.dtype), root.sub("asim_embedding")).flatten(0, 1)
    ce = root.sub("context_embedding")
    yy = _lin(y, ce.sub("input_mapping"))
    tok = sd["context_embedding.tokens"].to(x.dtype).repeat(b, 1, 1)
    for d in _children(sd, "context_embedding.context_transformer."):
        tok = _context_block_higen(tok, yy, ce.sub(f"context_transformer.{d}"), 8)
    ctx = _lin(tok, ce.sub("output_mapping")).repeat_interleave(f, dim=0)
    img = F.conv2d(spat_prior, sd["img_embedding.weight"], sd["img_embedding.bias"], padding=1).repeat_interleave(f, dim=0)
    xx = x.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
    out = _unet_trunk(sd, xx, emb, ctx, head_dim, b, woimg=True, conv_in_add=img)
    return out.reshape(b, f, -1, h, w).permute(0, 2, 1, 3, 4)


def _local_temporal_encoder(tok, s):
    """TransformerV2(heads=2, dim=4, dim_head=4, mlp_dim=4, depth=1), util.py:1396-1452:
    x = Attention(LN(x)) + x ; x = FF(x) + x with FF = Linear, GELU, Linear (non-gated)."""
    a = s.sub("layers.0.0")
    h = _ln(tok, a.sub("norm"))
    qkv = F.linear(h, a["fn.to_qkv.weight"])
    q, k, v = qkv.chunk(3, dim=-1)
    heads = 2
    bsz, n, inner = q.shape
    d = inner // heads

    def split(u):
        return u.reshape(bsz, n, heads, d).permute(0, 2, 1, 3)

    att = torch.softmax(torch.einsum("bhid,bhjd->bhij", split(q), split(k)) * d ** -0.5, dim=-1)
    o = torch.einsum("bhij,bhjd->bhid", att, split(v)).permute(0, 2, 1, 3).reshape(bsz, n, inner)
    tok = _lin(o, a.sub("fn.to_out.0")) + tok
    ff = s.sub("layers.0.1.net")
    tok = _lin(F.gelu(_lin(tok, ff.sub("0.0"))), ff.sub("2")) + tok
    return tok


def unet_i2vgen_forward(sd, x, t, y, image, local_image, fps, head_dim=64):
    """UNetSD_I2VGen.forward, unet_i2vgen.py:243-346."""
    b, c, f, h, w = x.shape
    dim = sd["time_embed.0.weight"].shape[1]
    root = _SD(sd)
    if local_image.ndim == 5 and local_image.size(2) > 1:
        local_image = local_image[:, :, :1]
    elif local_image.ndim != 5:
        local_image = local_image.unsqueeze(2)
    # [Concat] :281-295 -- first-frame latent + position planes (tpos+1)/(f-1)
    if f > 1:
        planes = [torch.ones_like(local_image[:, :, :1]) * ((tp + 1) / (f - 1)) for tp in range(f - 1)]
        ximg = torch.cat([local_image[:, :, :1]] + planes, dim=2)
    else:
        ximg = local_image
    ximg = ximg.permute(0, 2, 1, 3, 4).reshape(b * ximg.shape[2], -1, h, w)
    lc = root.sub("local_image_concat")
    ximg = F.conv2d(ximg, lc["0.weight"], lc["0.bias"], padding=1)
    ximg = F.conv2d(F.silu(ximg), lc["2.weight"], lc["2.bias"], padding=1)
    ximg = F.conv2d(F.silu(ximg), lc["4.weight"], lc["4.bias"], padding=1)
    cc = ximg.shape[1]
    tok = ximg.reshape(b, f, cc, h, w).permute(0, 3, 4, 1, 2).reshape(b * h * w, f, cc)
    tok = _local_temporal_encoder(tok, root.sub("local_temporal_encoder"))
    ximg = tok.reshape(b, h, w, f, cc).permute(0, 4, 3, 1, 2)
    concat = ximg + ximg  # "concat += _ximg" twice, :294-295 (acknowledged upstream bug, reproduced)
    # [Embeddings] :298-299
    emb = _mlp(sinusoidal_embedding(t, dim).to(x.dtype), root.sub("time_embed")) + \
        _mlp(sinusoidal_embedding(fps, dim).to(x.dtype), root.sub("fps_embedding"))
    emb = emb.repeat_interleave(f, dim=0)
    # [Context] :301-323 -- text tokens, 64 local-image tokens, num_tokens global-image tokens
    le = root.sub("local_image_embedding")
    li = local_image.permute(0, 2, 1, 3, 4).reshape(b, -1, h, w)
    li = F.silu(F.conv2d(li, le["0.weight"], le["0.bias"], padding=1))
    li = F.adaptive_avg_pool2d(li, (32, 32))
    li = F.silu(F.conv2d(li, le["3.weight"], le["3.bias"], stride=2, padding=1))
    li = F.conv2d(li, le["5.weight"], le["5.bias"], stride=2, padding=1)
    li = li.flatten(2).permute(0, 2, 1)
    ctx = torch.cat([y, li], dim=1)
    if image is not None:
        ce = _mlp(image, root.sub("context_embedding"))
        ctx = torch.cat([ctx, ce.view(b, -1, y.shape[-1])], dim=1)
    ctx = ctx.repeat_interleave(f, dim=0)
    xx = torch.cat([x, concat], dim=1).permute(0, 2, 1, 3, 4).reshape(b * f, -1, h, w)
    out = _unet_trunk(sd, xx, emb, ctx, head_dim, b)
    return out.reshape(b, f, -1, h, w).permute(0, 2, 1, 3, 4)


# ------------------------------------------------------------------------------------ VAE decode
def _vae_resnet(x, s):
    """ResnetBlock.forward, autoencoder.py:315-335 (temb None; GroupNorm eps 1e-6; swish)."""
    h = F.conv2d(F.silu(_gn(x, s.sub("norm1"), 1e-6)), s["conv1.weight"], s["conv1.bias"], padding=1)
    h = F.conv2d(F.silu(_gn(h, s.sub("norm2"), 1e-6)), s["conv2.weight"], s["conv2.bias"], padding=1)
    if s.has("nin_shortcut.weight"):
        x = F.conv2d(x, s["nin_shortcut.weight"], s["nin_shortcut.bias"])
    return x + h


def _vae_attn(x, s):
    """AttnBlock.forward, autoencoder.py:365-389: single-head softmax(q k^T / sqrt(c)) v over h*w."""
    b, c, hh, ww = x.shape
    h = _gn(x, s.sub("norm"), 1e-6)
    q = F.conv2d(h, s["q.weight"], s["q.bias"]).flatten(2).permute(0, 2, 1)
    k = F.conv2d(h, s["k.weight"], s["k.bias"]).flatten(2)
    v = F.conv2d(h, s["v.weight"], s["v.bias"]).flatten(2)
    att = torch.softmax(torch.bmm(q, k) * (int(c) ** -0.5), dim=2)
    o = torch.bmm(v, att.permute(0, 2, 1)).reshape(b, c, hh, ww)
    return x + F.conv2d(o, s["proj_out.weight"], s["proj_out.bias"])


def vae_decode(sd, z):
    """AutoencoderKL.decode, autoencoder.py:100-103 -> Decoder.forward :653-686.  z [n,4,h,w] -> [n,3,8h,8w]."""
    root = _SD(sd)
    z = F.conv2d(z, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
    d = root.sub("decoder")
    h = F.conv2d(z, d["conv_in.weight"], d["conv_in.bias"], padding=1)
    h = _vae_resnet(h, d.sub("mid.block_1"))
    h = _vae_attn(h, d.sub("mid.attn_1"))
    h = _vae_resnet(h, d.sub("mid.block_2"))
    levels = _children(sd, "decoder.up.")
    for lvl in reversed(levels):
        u = d.sub(f"up.{lvl}")
        for j in _children(sd, u.p + "block."):
            h = _vae_resnet(h, u.sub(f"block.{j}"))
        if u.has("upsample.conv.weight"):
            h = F.conv2d(F.interpolate(h, scale_factor=2.0, mode="nearest"), u["upsample.conv.weight"],
                         u["upsample.conv.bias"], padding=1)
    h = F.silu(_gn(h, d.sub("norm_out"), 1e-6))
    return F.conv2d(h, d["conv_out.weight"], d["conv_out.bias"], padding=1)


def vae_encode_moments(sd, x):
    """Encoder.forward (autoencoder.py:549-578) + quant_conv (:87).  x [n,3,H,W] -> moments [n, 2*zc, H/8, W/8]."""
    root = _SD(sd)
    e = root.sub("encoder")
    h = F.conv2d(x, e["conv_in.weight"], e["conv_in.bias"], padding=1)
    levels = _children(sd, "encoder.down.")
    for lvl in levels:
        dn = e.sub(f"down.{lvl}")
        for j in _children(sd, dn.p + "block."):
            h = _vae_resnet(h, dn.sub(f"block.{j}"))
        if dn.has("downsample.conv.weight"):
            h = F.conv2d(F.pad(h, (0, 1, 0, 1)), dn["downsample.conv.weight"], dn["downsample.conv.bias"], stride=2)
    h = _vae_resnet(h, e.sub("mid.block_1"))
    h = _vae_attn(h, e.sub("mid.attn_1"))
    h = _vae_resnet(h, e.sub("mid.block_2"))
    h = F.conv2d(F.silu(_gn(h, e.sub("norm_out"), 1e-6)), e["conv_out.weight"], e["conv_out.bias"], padding=1)
    return F.conv2d(h, sd["quant_conv.weight"], sd["quant_conv.bias"])


def vae_encode_first_stage(sd, x, scale_factor):
    """AutoencoderKL.encode_firsr_stage (autoencoder.py:85-90) with DiagonalGaussianDistribution.sample (:211-225):
    the noise comes from the global CPU generator, shape of the mean."""
    mean, logvar = torch.chunk(vae_encode_moments(sd, x), 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    noise = torch.randn(mean.shape).to(device=x.device)
    return scale_factor * (mean + torch.exp(0.5 * logvar) * noise)
