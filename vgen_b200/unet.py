"""B200-native UNetSD_T2VBase / UNetSD_I2VGen / UNetSD_VideoLCM / UNetSD_TFT2V / UNetSD_SR600 / UNetSD_HiGen: same
constructor arguments, state_dict keys and forward signatures as the reference classes (tools/modules/unet/unet_t2v.py:19-277,
unet_i2vgen.py:19-346, unet_videolcm.py:188-760, unet_tf2tv.py:188-843, unet_sr600.py:52-299, unet_higen.py:175-467), but
the forward is a fixed-layout graph of libvgen_b200.so kernels.

Design (not a port of the reference's module tree):
  * activations stay fp16 channels-last [(b f), h, w, C] for the whole forward; the reference's dozens
    of '(b f) c h w <-> b c f h w' / '(b h w) f c' permute+contiguous copies (unet_t2v.py:294-296,
    util.py:1251-1280,923-926) do not exist: temporal kernels address frames by stride.
  * weights are repacked once per load into GEMM-ready fp16 [out][taps*in] matrices; q/k/v projections
    are fused into one GEMM; GEGLU value/gate rows are interleaved for the fused epilogue; the cross
    attention K/V of the (frame-invariant) context are computed once per video, not once per frame.
  * bias, timestep-embedding add, residual adds and GEGLU run in the GEMM epilogues.
Numerics follow the reference under fp16 autocast: fp16 operands, fp32 accumulation and fp32
norm/softmax statistics, fp16 rounding where the reference materialises an fp16 tensor.
"""
from __future__ import annotations

import os

import torch

from . import arch, ops
from .graph import graphed
from .params import SpecModule


def _f16(t, dev):
    return t.detach().to(device=dev, dtype=torch.float16).contiguous()


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _pack_conv3x3(w, dev, cin_pad=None):
    """[n, c, 3, 3] -> [n, 9*c'] with k = (ky*3+kx)*c' + ci (c' = c or the padded channel count),
    K padded with zeros to a multiple of 64 for the tap-GEMM."""
    n, c = w.shape[0], w.shape[1]
    cp = cin_pad or c
    wp = torch.zeros(n, 3, 3, cp, dtype=torch.float32)
    wp[..., :c] = w.detach().float().cpu().permute(0, 2, 3, 1)
    wp = wp.reshape(n, 9 * cp)
    kpad = ((9 * cp + 63) // 64) * 64
    if kpad != 9 * cp:
        wp = torch.cat([wp, torch.zeros(n, kpad - 9 * cp)], dim=1)
    return wp.to(device=dev, dtype=torch.float16).contiguous()


def _geglu_bn(n):
    for bn in (256, 192, 128, 64):
        if n % bn == 0:
            return bn
    raise ValueError(f"GEGLU width {n} is not a multiple of 64")


class _UNetBase(SpecModule):
    KIND = "t2v"
    cfg_batch = True  # samplers may evaluate the cond / uncond CFG branches as one batch-2b forward (diffusion.cfg_forward)
    WOIMG = False     # HiGen: temporal branches contribute 0 when a single frame is sampled
    SR600 = False     # SR600: (2,1)-padded downsampling, row-cropped upsampling, filtered skips
    # nn.LayerNorm folded into the projection that follows it (vgen_row_stats + vgen_epilogue.row_stats / col_sum: the normalised
    # tokens are never written).  OFF by default: on config 2 it halves the LayerNorm family (8.5 -> 4.3 ms / step) but the k = 320
    # projections that consume it are epilogue-bound and pay for the extra per-column terms (+6.3 ms), a wash within run-to-run
    # noise (profiles/r02r_bench_i2vgen_lnfold{0,1}.json).  VGEN_LN_FOLD=1, or FOLD_LN = True on a module followed by
    # invalidate_packed(), turns it on; parity is the same (tests/test_gpu_parity.py).
    FOLD_LN = os.environ.get("VGEN_LN_FOLD", "0") == "1"

    def __init__(self, config=None, in_dim=4, dim=512, y_dim=512, context_dim=512, hist_dim=156, dim_condition=4,
                 out_dim=6, num_tokens=4, dim_mult=[1, 2, 3, 4], num_heads=None, head_dim=64, num_res_blocks=3,
                 attn_scales=[1 / 2, 1 / 4, 1 / 8], use_scale_shift_norm=True, dropout=0.1, temporal_attn_times=1,
                 temporal_attention=True, use_checkpoint=False, use_image_dataset=False, use_sim_mask=False,
                 training=True, inpainting=True, use_fps_condition=False, p_all_zero=0.1, p_all_keep=0.1, zero_y=None,
                 adapter_transformer_layers=1, concat_dim=8, context_embedding_depth=4, **kwargs):
        super().__init__()
        self.cfg = config
        if head_dim != 64:
            raise NotImplementedError("vgen_b200: head_dim must be 64 (all released VGen checkpoints)")
        if use_image_dataset:
            raise NotImplementedError("vgen_b200: use_image_dataset (training-time flag) is not supported")
        if adapter_transformer_layers != 1:
            raise NotImplementedError("vgen_b200: adapter_transformer_layers != 1 is not supported")
        # arguments that would change the reference's graph must not be swallowed silently (dropout / use_checkpoint /
        # training / inpainting / p_all_* only matter for training and are accepted as no-ops)
        if temporal_attn_times != 1:
            raise NotImplementedError("vgen_b200: temporal_attn_times != 1 (extra TemporalTransformers per block) is not "
                                      "used by any released config and is not supported")
        if use_sim_mask:
            raise NotImplementedError("vgen_b200: use_sim_mask=True (masked temporal attention) is not supported")
        self.plan = arch.unet_plan(self.KIND, in_dim=in_dim, dim=dim, y_dim=y_dim, context_dim=context_dim, out_dim=out_dim,
                                   num_tokens=num_tokens, dim_mult=tuple(dim_mult), num_heads=num_heads, head_dim=head_dim,
                                   num_res_blocks=num_res_blocks, attn_scales=tuple(attn_scales),
                                   temporal_attention=temporal_attention, use_fps_condition=use_fps_condition,
                                   concat_dim=concat_dim, context_embedding_depth=context_embedding_depth,
                                   compositions=self._compositions(config), inpainting=inpainting)
        # attributes the reference exposes and engines read
        self.in_dim, self.dim, self.y_dim, self.context_dim, self.out_dim = in_dim, dim, y_dim, context_dim, out_dim
        self.embed_dim, self.num_tokens, self.head_dim = dim * 4, num_tokens, head_dim
        self.zero_y = zero_y
        self.use_fps_condition = self.plan.use_fps_condition
        self._build_params(arch.unet_spec(self.plan), arch.unet_zero_init)

    @staticmethod
    def _compositions(config):
        """config.video_compositions of the VideoComposer-capable classes; () for the others."""
        return ()

    # ------------------------------------------------------------------------------ weight packing
    def _pack(self):
        sd = {k: v for k, v in self.state_dict().items()}
        dev = self.device
        if dev.type != "cuda":
            raise ops._l.VgenError("vgen_b200 UNet forward needs the module on a CUDA device (no CPU path exists)")
        W = {}

        def lin(p, bias=True):
            w = sd[p + "weight"]
            W[p + "w"] = _f16(w.reshape(w.shape[0], -1), dev)
            if bias:
                W[p + "b"] = _f32(sd[p + "bias"], dev)

        def norm(p):
            W[p + "g"] = _f32(sd[p + "weight"], dev)
            W[p + "b"] = _f32(sd[p + "bias"], dev)

        def conv3(p, cin_pad=None):
            W[p + "w"] = _pack_conv3x3(sd[p + "weight"], dev, cin_pad)
            W[p + "b"] = _f32(sd[p + "bias"], dev)

        def tconv(p):
            w = sd[p + "weight"]  # [n, c, 3, 1, 1] -> [n, 3*c], k = kt*c + ci
            W[p + "w"] = _f16(w[:, :, :, 0, 0].permute(0, 2, 1).reshape(w.shape[0], -1), dev)
            W[p + "b"] = _f32(sd[p + "bias"], dev)

        def fold(key, wmat, bias, nrm):
            """LayerNorm `nrm` folded into the linear `key` that consumes it (ops.fold_layer_norm)."""
            wf, cs, lb = ops.fold_layer_norm(wmat, bias, sd[nrm + "weight"], sd[nrm + "bias"])
            W[key], W[key + ".cs"], W[key + ".lb"] = _f16(wf, dev), _f32(cs, dev), _f32(lb, dev)

        def block(p, cross, cross1=False):
            a1, a2 = p + "attn1.", p + "attn2."
            ln_fold = self.FOLD_LN and not cross1
            if cross1:   # disable_self_attn=True: attn1 attends to the context as well (util.py:700-702)
                W[a1 + "q"] = _f16(sd[a1 + "to_q.weight"], dev)
                W[a1 + "kv"] = _f16(torch.cat([sd[a1 + "to_k.weight"], sd[a1 + "to_v.weight"]], 0), dev)
            else:
                W[a1 + "qkv"] = _f16(torch.cat([sd[a1 + "to_q.weight"], sd[a1 + "to_k.weight"], sd[a1 + "to_v.weight"]], 0), dev)
            lin(a1 + "to_out.0.")
            if cross:
                W[a2 + "q"] = _f16(sd[a2 + "to_q.weight"], dev)
                W[a2 + "kv"] = _f16(torch.cat([sd[a2 + "to_k.weight"], sd[a2 + "to_v.weight"]], 0), dev)
            else:
                W[a2 + "qkv"] = _f16(torch.cat([sd[a2 + "to_q.weight"], sd[a2 + "to_k.weight"], sd[a2 + "to_v.weight"]], 0), dev)
            lin(a2 + "to_out.0.")
            for nm in ("norm1.", "norm2.", "norm3."):
                norm(p + nm)
            gw, gb = sd[p + "ff.net.0.proj.weight"].detach().float(), sd[p + "ff.net.0.proj.bias"].detach().float()
            bn = _geglu_bn(gw.shape[0])
            if ln_fold:
                # norm1 -> attn1.qkv, norm2 -> attn2.q (cross) / attn2.qkv, norm3 -> GEGLU projection
                fold(a1 + "qkv", torch.cat([sd[a1 + "to_q.weight"], sd[a1 + "to_k.weight"], sd[a1 + "to_v.weight"]], 0), None, p + "norm1.")
                if cross:
                    fold(a2 + "q", sd[a2 + "to_q.weight"], None, p + "norm2.")
                else:
                    fold(a2 + "qkv", torch.cat([sd[a2 + "to_q.weight"], sd[a2 + "to_k.weight"], sd[a2 + "to_v.weight"]], 0), None, p + "norm2.")
                g3, b3 = sd[p + "norm3.weight"].detach().float(), sd[p + "norm3.bias"].detach().float()
                gb = gb + gw @ b3
                gw = gw * g3[None, :]
            wp, bp = ops.pack_geglu_weight(gw, gb, bn)
            W[p + "ff.geglu.w"], W[p + "ff.geglu.b"], W[p + "ff.geglu.bn"] = _f16(wp, dev), _f32(bp, dev), bn
            if ln_fold:
                W[p + "ff.geglu.cs"] = _f32(W[p + "ff.geglu.w"].double().sum(1), dev)
            lin(p + "ff.net.2.")

        def layer(L):
            p = L.prefix
            if L.kind == "conv_in":
                conv3(p, cin_pad=((L.cin + 7) // 8) * 8)
            elif L.kind == "res":
                norm(p + "in_layers.0."), conv3(p + "in_layers.2.")
                lin(p + "emb_layers.1.")
                norm(p + "out_layers.0."), conv3(p + "out_layers.3.")
                if L.cin != L.cout:
                    lin(p + "skip_connection.")
                for name, widx in (("conv1", 2), ("conv2", 3), ("conv3", 3), ("conv4", 3)):
                    q = f"{p}temopral_conv.{name}."
                    norm(q + "0."), tconv(f"{q}{widx}.")
            elif L.kind == "spatial":
                norm(p + "norm."), lin(p + "proj_in."), block(p + "transformer_blocks.0.", True), lin(p + "proj_out.")
            elif L.kind == "temporal":
                norm(p + "norm."), lin(p + "proj_in."), block(p + "transformer_blocks.0.", False), lin(p + "proj_out.")
            elif L.kind == "down":
                conv3(p + "op.")
            elif L.kind == "up":
                conv3(p + "conv.")

        for pre in ("time_embed.0.", "time_embed.2."):
            lin(pre)
        if self.plan.use_fps_condition:
            lin("fps_embedding.0."), lin("fps_embedding.2.")
        if self.KIND == "i2vgen":
            lin("context_embedding.0."), lin("context_embedding.2.")
            conv3("local_image_concat.0.", cin_pad=8), conv3("local_image_concat.2."), conv3("local_image_concat.4.")
            e = "local_temporal_encoder.layers.0."
            norm(e + "0.norm."), lin(e + "0.fn.to_qkv.", bias=False), lin(e + "0.fn.to_out.0.")
            lin(e + "1.net.0.0."), lin(e + "1.net.2.")
            conv3("local_image_embedding.0.", cin_pad=8), conv3("local_image_embedding.3."), conv3("local_image_embedding.5.")
        if self.plan.compositions:
            if "image" in self.plan.compositions:
                lin("pre_image_condition.0."), lin("pre_image_condition.2.")
            for comp, stem, after, _cin in arch.ADAPTERS:
                if comp not in self.plan.compositions:
                    continue
                if comp != "mask" or self.plan.inpainting:
                    W[stem + ".0.w"] = _f16(ops.pack_cond_stem_weight(sd[stem + ".0.weight"]), dev)
                    W[stem + ".0.b"] = _f32(sd[stem + ".0.bias"], dev)
                    conv3(stem + ".3."), conv3(stem + ".5.")
                e = after + ".layers.0."
                norm(e + "0.norm."), lin(e + "0.fn.to_qkv.", bias=False), lin(e + "0.fn.to_out.0.")
                lin(e + "1.net.0.0."), lin(e + "1.net.2.")
        if self.KIND == "higen":
            W["context_embedding.tokens"] = _f16(sd["context_embedding.tokens"][0], dev)
            for d in range(self.plan.context_embedding_depth):
                block(f"context_embedding.context_transformer.{d}.", True, cross1=True)
            lin("context_embedding.input_mapping."), lin("context_embedding.output_mapping.")
            for pre in ("asim_embedding.", "msim_embedding."):
                lin(pre + "0."), lin(pre + "2.")
            conv3("img_embedding.", cin_pad=8)
        for blk in self.plan.input_blocks:
            for L in blk:
                layer(L)
        for L in self.plan.middle:
            layer(L)
        for blk in self.plan.output_blocks:
            for L in blk:
                layer(L)
        norm("out.0."), conv3("out.2.")
        self._packed = W
        return W

    # ------------------------------------------------------------------------------ building blocks
    def _conv3x3_any(self, x, W, p, **epi):
        """3x3 stride-1 conv: TMA tap-GEMM when C % 64 == 0, otherwise im2col + GEMM."""
        n, h, w, c = x.shape
        wt = W[p + "w"]
        if c % 64 == 0 and wt.shape[1] == 9 * c:
            return ops.conv2d_3x3(x, wt, bias=W[p + "b"], **epi)
        col = ops.im2col(x, 3, 3, 1, 1, 1, h, w, wt.shape[1], act_silu=epi.pop("act_silu", False))
        out = ops.linear(col, wt, bias=W[p + "b"], residual=epi.get("residual"))
        return out.view(n, h, w, wt.shape[0])

    def _conv3x3_s2(self, x, W, p, act_silu=False, pad_h=1):
        n, h, w, c = x.shape
        ho, wo = (h + 2 * pad_h - 3) // 2 + 1, (w - 1) // 2 + 1
        wt = W[p + "w"]
        col = ops.im2col(x, 3, 3, 2, pad_h, 1, ho, wo, wt.shape[1], act_silu=act_silu)
        return ops.linear(col, wt, bias=W[p + "b"]).view(n, ho, wo, wt.shape[0])

    def _res_block(self, x, emb, L, W, b, f):
        """ResBlock._forward + TemporalConvBlock_v2 (util.py:900-927,1686-1697)."""
        p = L.prefix
        n, h, w, _ = x.shape
        # emb is [b, E] (one embedding per video) or [b*f, E] (HiGen: one per frame, unet_higen.py:440-443)
        e = ops.linear_small(emb, W[p + "emb_layers.1.w"], W[p + "emb_layers.1.b"], silu_in=True)  # [b | b*f, cout]
        g = ops.group_norm(x, W[p + "in_layers.0.g"], W[p + "in_layers.0.b"], 1e-5, True)
        hcur = ops.conv2d_3x3(g, W[p + "in_layers.2.w"], bias=W[p + "in_layers.2.b"], group_bias=e,
                              group_div=(b * f) // emb.shape[0])
        g = ops.group_norm(hcur, W[p + "out_layers.0.g"], W[p + "out_layers.0.b"], 1e-5, True)
        if L.cin != L.cout:
            skip = ops.linear(x.view(-1, L.cin), W[p + "skip_connection.w"], bias=W[p + "skip_connection.b"])
        else:
            skip = x
        hcur = ops.conv2d_3x3(g, W[p + "out_layers.3.w"], bias=W[p + "out_layers.3.b"], residual=skip.view(-1, L.cout))
        if self.WOIMG and f == 1:
            return hcur  # TemporalConvBlock_v2WoImg: identity + 0.0 * branch (unet_higen.py:80-83)
        # temporal conv: GroupNorm statistics over all frames of a video, 3-tap conv over frames
        t = hcur
        names = (("conv1", 2), ("conv2", 3), ("conv3", 3), ("conv4", 3))
        for i, (name, widx) in enumerate(names):
            q = f"{p}temopral_conv.{name}."
            g = ops.group_norm(t, W[q + "0.g"], W[q + "0.b"], 1e-5, True, n=b)
            last = i == len(names) - 1
            # all videos of the batch in one launch (the frame taps are zero-padded per video)
            t = ops.tconv3(g.view(b, f, h * w, L.cout), W[f"{q}{widx}.w"], bias=W[f"{q}{widx}.b"],
                           residual=hcur.view(b, f, h * w, L.cout) if last else None).view(hcur.shape)
        return t

    @staticmethod
    def _ln_linear(t, W, key, nrm):
        """nn.LayerNorm `nrm` followed by the bias-free projection `key` (util.py:694-704): when the pack folded the norm into
        the weights (key.cs present) only the row statistics are computed and the GEMM epilogue applies them."""
        if key + ".cs" in W:
            return ops.linear(t, W[key], bias=W[key + ".lb"], ln=(ops.row_stats(t), W[key + ".cs"]))
        return ops.linear(ops.layer_norm(t, W[nrm + "g"], W[nrm + "b"]), W[key])

    def _self_attn_spatial(self, t, W, p, nrm, heads, n, hw, inner):
        qkv = self._ln_linear(t, W, p + "qkv", nrm)             # [M, 3*inner]
        v3 = qkv.view(n, hw, 3 * inner)
        return ops.attention_d64(v3[:, :, :inner], v3[:, :, inner:2 * inner], v3[:, :, 2 * inner:], heads)

    def _basic_block_spatial(self, t, ctx_tokens, W, p, heads, n, hw, inner, f):
        """BasicTransformerBlock on tokens t [M, inner] (M = n*hw); ctx_tokens [b, L, ctx_dim] fp16."""
        a = self._self_attn_spatial(t, W, p + "attn1.", p + "norm1.", heads, n, hw, inner)
        t = ops.linear(a.view(-1, inner), W[p + "attn1.to_out.0.w"], bias=W[p + "attn1.to_out.0.b"], residual=t)
        q = self._ln_linear(t, W, p + "attn2.q", p + "norm2.").view(n, hw, inner)
        bctx, lctx, cdim = ctx_tokens.shape
        kv = ops.linear(ctx_tokens.view(-1, cdim), W[p + "attn2.kv"]).view(bctx, lctx, 2 * inner)
        a = ops.attention_d64(q, kv[:, :, :inner], kv[:, :, inner:], heads, kv_batch_div=f)
        t = ops.linear(a.view(-1, inner), W[p + "attn2.to_out.0.w"], bias=W[p + "attn2.to_out.0.b"], residual=t)
        return self._feed_forward(t, W, p)

    def _feed_forward(self, t, W, p):
        if p + "ff.geglu.cs" in W:   # norm3 folded into the GEGLU projection
            gg = ops.linear(t, W[p + "ff.geglu.w"], bias=W[p + "ff.geglu.b"], geglu=True, bn=W[p + "ff.geglu.bn"],
                            ln=(ops.row_stats(t), W[p + "ff.geglu.cs"]))
        else:
            xn = ops.layer_norm(t, W[p + "norm3.g"], W[p + "norm3.b"])
            gg = ops.linear(xn, W[p + "ff.geglu.w"], bias=W[p + "ff.geglu.b"], geglu=True, bn=W[p + "ff.geglu.bn"])
        return ops.linear(gg, W[p + "ff.net.2.w"], bias=W[p + "ff.net.2.b"], residual=t)

    def _spatial_transformer(self, x, ctx_tokens, L, W, f):
        """SpatialTransformer.forward, use_linear=True (util.py:354-373)."""
        p = L.prefix
        n, h, w, c = x.shape
        g = ops.group_norm(x, W[p + "norm.g"], W[p + "norm.b"], 1e-6, False)
        t = ops.linear(g.view(-1, c), W[p + "proj_in.w"], bias=W[p + "proj_in.b"])
        t = self._basic_block_spatial(t, ctx_tokens, W, p + "transformer_blocks.0.", L.heads, n, h * w, L.inner, f)
        out = ops.linear(t, W[p + "proj_out.w"], bias=W[p + "proj_out.b"], residual=x.view(-1, c))
        return out.view(n, h, w, c)

    def _temporal_attn(self, t, W, p, nrm, heads, b, f, hw, inner):
        qkv = self._ln_linear(t, W, p + "qkv", nrm).view(b, f, hw, 3 * inner)
        # all videos of the batch in one launch
        return ops.attention_temporal(qkv[..., :inner], qkv[..., inner:2 * inner], qkv[..., 2 * inner:], heads, 64)

    def _temporal_transformer(self, x, L, W, b, f):
        """TemporalTransformer.forward, only_self_att=True (util.py:1240-1286): both attentions are
        self-attention over the f frames of a pixel; GroupNorm statistics span all frames."""
        if self.WOIMG and f == 1:
            return x  # TemporalTransformerWoImg: 0.0 * branch + x_in (unet_higen.py:146-149)
        p = L.prefix
        n, h, w, c = x.shape
        hw, inner = h * w, L.inner
        g = ops.group_norm(x, W[p + "norm.g"], W[p + "norm.b"], 1e-6, False, n=b)
        t = ops.linear(g.view(-1, c), W[p + "proj_in.w"], bias=W[p + "proj_in.b"])
        q = p + "transformer_blocks.0."
        for att, nrm in (("attn1.", "norm1."), ("attn2.", "norm2.")):
            a = self._temporal_attn(t, W, q + att, q + nrm, L.heads, b, f, hw, inner)
            t = ops.linear(a.view(-1, inner), W[q + att + "to_out.0.w"], bias=W[q + att + "to_out.0.b"], residual=t)
        t = self._feed_forward(t, W, q)
        out = ops.linear(t, W[p + "proj_out.w"], bias=W[p + "proj_out.b"], residual=x.view(-1, c))
        return out.view(n, h, w, c)

    def _run_layer(self, x, L, W, emb, ctx_tokens, b, f, conv_in_residual=None):
        if L.kind == "res":
            return self._res_block(x, emb, L, W, b, f)
        if L.kind == "spatial":
            return self._spatial_transformer(x, ctx_tokens, L, W, f)
        if L.kind == "temporal":
            return self._temporal_transformer(x, L, W, b, f)
        if L.kind == "down":
            # UNetSD_SR600 pads the height by 2 (unet_sr600.py:151-153)
            return self._conv3x3_s2(x, W, L.prefix + "op.", pad_h=2 if self.SR600 else 1)
        if L.kind == "up":
            if self.SR600:   # UpsampleSR600 drops the first and last upsampled row (util.py:799-801)
                up = ops.upsample_nearest2x_rows(x, 1, 2 * x.shape[1] - 2)
            else:
                up = ops.upsample_nearest2x(x)
            return ops.conv2d_3x3(up, W[L.prefix + "conv.w"], bias=W[L.prefix + "conv.b"])
        if L.kind == "conv_in":
            if conv_in_residual is not None:
                return self._conv3x3_any(x, W, L.prefix, residual=conv_in_residual)
            return self._conv3x3_any(x, W, L.prefix)
        raise ValueError(L.kind)

    def _merge_skip(self, x, skip, n):
        """torch.cat([x, xs.pop()], dim=1) of the decoder (unet_t2v.py:269); SR600 overrides it."""
        return ops.concat_channels(x, skip)

    def _trunk(self, x, emb, ctx_tokens, W, b, f, conv_in_residual=None):
        """encoder / middle / decoder with skip concatenation + head (unet_t2v.py:257-277)."""
        skips = []
        for blk in self.plan.input_blocks:
            for L in blk:
                x = self._run_layer(x, L, W, emb, ctx_tokens, b, f, conv_in_residual)
            skips.append(x)
        for L in self.plan.middle:
            x = self._run_layer(x, L, W, emb, ctx_tokens, b, f)
        for n, blk in enumerate(self.plan.output_blocks):
            x = self._merge_skip(x, skips.pop(), n)
            for L in blk:
                x = self._run_layer(x, L, W, emb, ctx_tokens, b, f)
        g = ops.group_norm(x, W["out.0.g"], W["out.0.b"], 1e-5, True)
        return ops.conv2d_3x3(g, W["out.2.w"], bias=W["out.2.b"])

    def _transformer_v2(self, tok, W, e, b, f, hw, cd):
        """Transformer_v2 / TransformerV2(heads=2, dim=cd, dim_head=cd, mlp_dim=cd, depth=1) over the f frames of every pixel
        (unet_videolcm.py:121-141, util.py:1396-1452): x = Attention(LN(x)) + x; x = FF(x) + x with FF = Linear, GELU,
        Linear.  tok: [(b f h w), cd] frame-major per video; e: the prefix of layers.0."""
        xn = ops.layer_norm(tok, W[e + "0.norm.g"], W[e + "0.norm.b"])
        qkv = ops.linear_small(xn, W[e + "0.fn.to_qkv.w"]).view(b, f, hw, 6 * cd)
        att = ops.attention_temporal(qkv[..., :2 * cd], qkv[..., 2 * cd:4 * cd], qkv[..., 4 * cd:], 2, cd)
        tok = ops.linear_small(att.view(-1, 2 * cd), W[e + "0.fn.to_out.0.w"], W[e + "0.fn.to_out.0.b"], residual=tok)
        hid = ops.linear_small(tok, W[e + "1.net.0.0.w"], W[e + "1.net.0.0.b"], gelu_out=True)
        return ops.linear_small(hid, W[e + "1.net.2.w"], W[e + "1.net.2.b"], residual=tok)

    def _mlp(self, x, W, p):
        h = ops.linear_small(x, W[p + "0.w"], W[p + "0.b"])
        return ops.linear_small(h, W[p + "2.w"], W[p + "2.b"], silu_in=True)

    def _time_embedding(self, t, fps, W):
        emb = self._mlp(ops.sinusoidal_embedding(t, self.dim), W, "time_embed.")
        if self.plan.use_fps_condition and fps is not None:
            emb = ops.eltwise("add", emb, self._mlp(ops.sinusoidal_embedding(fps, self.dim), W, "fps_embedding."))
        return emb

    @staticmethod
    def _to_f16_rows(t):
        """[b, L, C] (fp32 or fp16) -> contiguous fp16 [b, L, C] through the cast kernel."""
        b, L, c = t.shape
        if t.dtype == torch.float16 and t.is_contiguous():
            return t
        return ops.cp_to_pc(t.contiguous().view(b * L, c, 1).float(), b * L, c, 1).view(b, L, c)

    def _check_x(self, x, t):
        if not x.is_cuda:
            raise ops._l.VgenError("vgen_b200 UNet: inputs must be CUDA tensors (no CPU path exists)")
        if x.dim() != 5:
            raise ValueError("x must be [b, c, f, h, w]")
        if t.numel() != x.shape[0]:
            raise ValueError("t must have one entry per batch element")


class UNetSD_T2VBase(_UNetBase):
    """Drop-in for tools/modules/unet/unet_t2v.py:19-20 (registered as MODEL 'UNetSD_T2VBase')."""
    KIND = "t2v"

    @graphed
    @torch.no_grad()
    def forward(self, x, t, y=None, fps=None, masked=None, video_mask=None, focus_present_mask=None,
                prob_focus_present=0., mask_last_frame_num=0, **kwargs):
        self._check_x(x, t)
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        emb = self._time_embedding(t, fps, W)
        if y is None:
            if self.zero_y is None:
                raise ValueError("y is None and no zero_y was given")
            y = self.zero_y.to(x.device).repeat(b, 1, 1)[:, :1, :]
        ctx = self._to_f16_rows(y)
        xin = ops.cp_to_pc(x.contiguous(), b, c, f * h * w, c_pad=8).view(b * f, h, w, 8)
        out = self._trunk(xin, emb, ctx, W, b, f)                     # [(b f), h, w, out_dim]
        return ops.pc_to_cp(out.view(b, f * h * w, self.out_dim), b, self.out_dim, f * h * w).view(b, self.out_dim, f, h, w)


class UNetSD_I2VGen(_UNetBase):
    """Drop-in for tools/modules/unet/unet_i2vgen.py:19-20 (registered as MODEL 'UNetSD_I2VGen')."""
    KIND = "i2vgen"

    def _small_conv(self, x, W, p, stride=1, act_silu=False):
        n, h, w, c = x.shape
        if stride == 2:
            return self._conv3x3_s2(x, W, p, act_silu=act_silu)
        wt = W[p + "w"]
        col = ops.im2col(x, 3, 3, 1, 1, 1, h, w, wt.shape[1], act_silu=act_silu)
        return ops.linear(col, wt, bias=W[p + "b"]).view(n, h, w, wt.shape[0])

    def _local_concat(self, local_first, W, b, f, h, w):
        """[Concat] branch, unet_i2vgen.py:281-295.  local_first: [b, 4, 1, h, w] (first-frame latent)."""
        dev = local_first.device
        if f > 1:
            pos = (torch.arange(1, f, device=dev, dtype=torch.float32) / (f - 1)).view(1, 1, f - 1, 1, 1)
            ximg = torch.cat([local_first.float(), pos.expand(b, local_first.shape[1], f - 1, h, w)], dim=2)
        else:
            ximg = local_first.float()
        ximg = ops.cp_to_pc(ximg.contiguous(), b, ximg.shape[1], f * h * w, c_pad=8).view(b * f, h, w, 8)
        ximg = self._small_conv(ximg, W, "local_image_concat.0.")
        ximg = self._small_conv(ximg, W, "local_image_concat.2.", act_silu=True)
        ximg = self._small_conv(ximg, W, "local_image_concat.4.", act_silu=True)      # [(b f), h, w, cd]
        cd = ximg.shape[-1]
        # TransformerV2(heads=2, dim=cd, dim_head=cd): tokens are the f frames of one pixel (util.py:1396-1452)
        tok = self._transformer_v2(ximg.view(-1, cd), W, "local_temporal_encoder.layers.0.", b, f, h * w, cd)
        return ops.eltwise("scale", tok, s=2.0)   # "concat += _ximg" twice (:294-295), exact in fp16

    def _local_tokens(self, local_first, W, b, h, w):
        """local_image_embedding, unet_i2vgen.py:126-132,312-316 -> [b, 64, 1024] context tokens."""
        x = ops.cp_to_pc(local_first.float().contiguous(), b, local_first.shape[1], h * w, c_pad=8).view(b, h, w, 8)
        x = self._small_conv(x, W, "local_image_embedding.0.")
        x = ops.adaptive_avgpool(x, 32, 32, silu_in=True)
        x = self._small_conv(x, W, "local_image_embedding.3.", stride=2)
        x = self._small_conv(x, W, "local_image_embedding.5.", stride=2, act_silu=True)
        return x.view(b, -1, x.shape[-1])

    @graphed
    @torch.no_grad()
    def forward(self, x, t, y=None, image=None, local_image=None, masked=None, fps=None, video_mask=None,
                focus_present_mask=None, prob_focus_present=0., mask_last_frame_num=0, **kwargs):
        self._check_x(x, t)
        if local_image is None or fps is None:
            raise ValueError("UNetSD_I2VGen.forward needs local_image and fps")
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        if local_image.ndim == 5 and local_image.size(2) > 1:
            local_image = local_image[:, :, :1]
        elif local_image.ndim != 5:
            local_image = local_image.unsqueeze(2)
        cd = self.plan.concat_dim
        concat = self._local_concat(local_image, W, b, f, h, w)                    # [(b f h w), cd]
        emb = self._time_embedding(t, fps, W)
        if y is None:
            if self.zero_y is None:
                raise ValueError("y is None and no zero_y was given")
            y = self.zero_y.to(x.device).repeat(b, 1, 1)[:, :1, :]
        y16 = self._to_f16_rows(y)
        loc = self._local_tokens(local_image[:, :, 0], W, b, h, w)               # [b, 64, 1024]
        parts = [y16, loc]
        if image is not None:
            img = self._to_f16_rows(image).view(-1, image.shape[-1])
            ce = self._mlp(img, W, "context_embedding.")
            parts.append(ce.view(b, self.num_tokens, self.context_dim))
        ltot = sum(p.shape[1] for p in parts)
        ctx = torch.empty(b, ltot, self.context_dim, device=x.device, dtype=torch.float16)
        off, cdim = 0, self.context_dim
        ctx_rows = ctx.view(b, ltot * cdim)
        for part in parts:                      # one strided copy per part (rows = videos)
            lp = part.shape[1]
            ops.copy2d(part.reshape(b, lp * cdim), ctx_rows[:, off * cdim:(off + lp) * cdim])
            off += lp
        xin = ops.cp_to_pc(x.contiguous(), b, c, f * h * w, c_pad=c + cd).view(-1, c + cd)
        ops.copy2d(concat, xin[:, c:])
        out = self._trunk(xin.view(b * f, h, w, c + cd), emb, ctx, W, b, f)
        return ops.pc_to_cp(out.view(b, f * h * w, self.out_dim), b, self.out_dim, f * h * w).view(b, self.out_dim, f, h, w)


def _cfg_get(config, name, default=None):
    if config is None:
        return default
    if isinstance(config, dict):
        return config.get(name, default)
    return getattr(config, name, default)


class UNetSD_VideoLCM(_UNetBase):
    """Drop-in for tools/modules/unet/unet_videolcm.py:188-189 (MODEL 'UNetSD_VideoLCM').

    Text-to-video (configs/videolcm_t2v_infer.yaml, video_compositions == ['text']): `concat` stays all-zero (:598),
    pre_image is an empty Sequential (:409,:705) and the context is the text tokens (:713-726).

    VideoComposer (configs/videolcm_vcomposer_infer.yaml, tft2v_vcomposer_*.yaml): one adapter per spatial composition
    (depthmap, motion, canny, mask, sketch, single_sketch, local_image; :294-372) fills the concat channels of the first
    conv (:598-703), and 'image' appends pre_image_condition(image) as num_tokens context tokens (:743-745).  The
    conditions do not depend on x, t or y, and the engines pass the same tensors to every step of a video, so:
      * the adapter stage runs eagerly, outside the CUDA graph, and its [b*f*h*w, concat_dim] fp16 result is memoised
        (strong reference + version counter + shape / stride / dtype of every condition tensor); a graph replay never
        copies a full-resolution condition;
      * a condition tensor that both CFG branches share is passed once (cfg_shared_kwargs, diffusion.cfg_forward) and
        its concat rows are applied to both halves of the batch-2b forward.
    `histogram` and `use_text_clip_vip_model` are not supported and raise."""
    KIND = "videolcm"
    COMPOSITIONS = ("text", "image") + tuple(a[0] for a in arch.ADAPTERS)
    # forward keyword -> composition, in the order the reference adds the adapters to `concat` (:599-699)
    CONDITIONS = (("depth", "depthmap"), ("local_image", "local_image"), ("motion", "motion"), ("canny", "canny"),
                  ("sketch", "sketch"), ("single_sketch", "single_sketch"), ("masked", "mask"))
    cfg_shared_kwargs = frozenset(k for k, _ in CONDITIONS)
    _POSITIONAL = ("y", "depth", "image", "motion", "local_image", "single_sketch", "masked", "canny", "sketch", "histogram",
                   "fps", "video_mask", "focus_present_mask", "prob_focus_present", "mask_last_frame_num")

    @staticmethod
    def _compositions(config):
        comps = tuple(_cfg_get(config, "video_compositions", None) or ["text"])
        bad = [c for c in comps if c not in UNetSD_VideoLCM.COMPOSITIONS]
        if "histogram" in comps:
            raise NotImplementedError("vgen_b200 UNetSD_VideoLCM: the 'histogram' composition is not supported")
        if bad:
            raise NotImplementedError(f"vgen_b200 UNetSD_VideoLCM: unknown video_compositions {bad}")
        if _cfg_get(config, "use_text_clip_vip_model", False):
            raise NotImplementedError("vgen_b200 UNetSD_VideoLCM: use_text_clip_vip_model is not supported")
        return comps

    def __init__(self, config=None, *args, **kwargs):
        super().__init__(config, *args, **kwargs)
        self.video_compositions = list(self.plan.compositions)
        self.concat_dim = self.plan.concat_dim
        self.inpainting = self.plan.inpainting
        res = _cfg_get(config, "resolution", None)
        self.resolution = list(res) if res is not None else None
        if set(self.video_compositions) & {a[0] for a in arch.ADAPTERS} and self.resolution is None:
            raise ValueError("UNetSD_VideoLCM: config.resolution is required for the spatial compositions (:270,:299)")
        self.adapter_runs = 0      # adapter stages computed (memo misses), for tests and benchmarks

    def forward(self, x, t, *args, **kwargs):
        if len(args) > len(self._POSITIONAL):
            raise TypeError("forward: too many positional arguments")
        bound = dict(zip(self._POSITIONAL, args))
        if bound.keys() & kwargs.keys():
            raise TypeError(f"forward: multiple values for {sorted(bound.keys() & kwargs.keys())}")
        bound.update(kwargs)
        if bound.get("histogram") is not None:
            raise NotImplementedError("vgen_b200 UNetSD_VideoLCM: the 'histogram' condition is not supported")
        conds = [(k, comp, bound[k]) for k, comp in self.CONDITIONS if bound.get(k) is not None]
        if not conds and bound.get("image") is None:
            return self._forward_text(x, t, *args, **kwargs)
        return self._forward_vcomposer(x, t, bound, conds)

    @graphed(key="forward")
    @torch.no_grad()
    def _forward_text(self, x, t, y=None, depth=None, image=None, motion=None, local_image=None, single_sketch=None,
                      masked=None, canny=None, sketch=None, histogram=None, fps=None, video_mask=None,
                      focus_present_mask=None, prob_focus_present=0., mask_last_frame_num=0, **kwargs):
        self._check_x(x, t)
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        emb = self._time_embedding(t, fps, W)
        if y is None:
            if self.zero_y is None:
                raise ValueError("y is None and no zero_y was given")
            y = self.zero_y.to(x.device).repeat(b, 1, 1)            # all tokens (:724-725), unlike T2VBase
        ctx = self._to_f16_rows(y)
        cin = self.plan.input_blocks[0][0].cin                      # in_dim + concat_dim; the concat channels are 0
        cpad = ((cin + 7) // 8) * 8
        xin = ops.cp_to_pc(x.contiguous(), b, c, f * h * w, c_pad=cpad).view(b * f, h, w, cpad)
        out = self._trunk(xin, emb, ctx, W, b, f)
        return ops.pc_to_cp(out.view(b, f * h * w, self.out_dim), b, self.out_dim, f * h * w).view(b, self.out_dim, f, h, w)

    # ------------------------------------------------------------------------------ VideoComposer path
    def _latent_of_resolution(self):
        """Latent size the adapters produce: AdaptiveAvgPool2d((res[1]//2, res[0]//2)) then two stride-2 convs."""
        ph, pw = self.resolution[1] // 2, self.resolution[0] // 2
        s2 = lambda n: (n - 1) // 2 + 1  # noqa: E731
        return ph, pw, s2(s2(ph)), s2(s2(pw))

    def _check_conditions(self, x, conds, image):
        b, _, f, h, w = x.shape
        comps = set(self.video_compositions)
        cb = None
        for name, comp, v in conds:
            if comp not in comps:
                raise ValueError(f"UNetSD_VideoLCM: condition '{name}' given but '{comp}' is not in video_compositions")
            if comp == "mask" and not self.inpainting:
                raise ValueError("UNetSD_VideoLCM: 'masked' given to a model built with inpainting=False (:563)")
            cin = next(a[3] for a in arch.ADAPTERS if a[0] == comp)
            if not torch.is_tensor(v) or v.dim() != 5 or v.shape[1] != cin or v.shape[2] != f:
                raise ValueError(f"UNetSD_VideoLCM: condition '{name}' must be [b, {cin}, {f}, H, W], got "
                                 f"{tuple(v.shape) if torch.is_tensor(v) else type(v)}")
            if not v.is_cuda or v.dtype not in (torch.float32, torch.float16):
                raise ValueError(f"UNetSD_VideoLCM: condition '{name}' must be a CUDA fp32 or fp16 tensor")
            if cb is None:
                cb = v.shape[0]
            if v.shape[0] != cb or b % cb:
                raise ValueError(f"UNetSD_VideoLCM: condition batches must agree and divide the batch of x ({b})")
        if conds:
            _, _, lh, lw = self._latent_of_resolution()
            if (lh, lw) != (h, w):
                raise ValueError(f"UNetSD_VideoLCM: config.resolution {self.resolution} reduces the conditions to {lh}x{lw}, "
                                 f"but the latent is {h}x{w}")
        if image is not None:
            if "image" not in comps:
                raise ValueError("UNetSD_VideoLCM: condition 'image' given but 'image' is not in video_compositions")
            if not torch.is_tensor(image) or image.shape[-1] != self.context_dim or image.numel() != b * self.context_dim:
                raise ValueError(f"UNetSD_VideoLCM: image must hold one {self.context_dim}-wide embedding per video")

    def _adapter(self, v, comp, W, f, hw):
        _, stem, after, _ = next(a for a in arch.ADAPTERS if a[0] == comp)
        ph, pw, _, _ = self._latent_of_resolution()
        cd = self.concat_dim
        z = ops.cond_stem(v.contiguous(), W[stem + ".0.w"], W[stem + ".0.b"], ph, pw)   # conv + SiLU + pool, [(b f), ph, pw, 4cd]
        z = self._conv3x3_s2(z, W, stem + ".3.")
        z = self._conv3x3_s2(z, W, stem + ".5.", act_silu=True)                       # [(b f), h, w, cd]
        return self._transformer_v2(z.view(-1, cd), W, after + ".layers.0.", v.shape[0], f, hw, cd)

    @staticmethod
    def _memo_key(conds):
        """Identity of the condition tensors: None when one cannot be tracked (inference-mode tensors have no version
        counter), so such calls always recompute."""
        key = []
        for name, _, v in conds:
            if v.is_inference():
                return None
            key.append((name, v, v._version, tuple(v.shape), v.stride(), v.dtype))
        return key

    @staticmethod
    def _memo_hit(memo, key):
        if memo is None or key is None or len(memo[0]) != len(key):
            return False
        return all(a[0] == b[0] and a[1] is b[1] and a[2:] == b[2:] for a, b in zip(memo[0], key))

    @torch.no_grad()
    def _adapter_concat(self, conds, W, f, hw):
        """sum of the adapter outputs in the reference's order, fp32 accumulation, one fp16 rounding: [cb*f*hw, concat_dim]."""
        key = self._memo_key(conds)
        memo = W.get("__cond_memo__")
        if self._memo_hit(memo, key):
            return memo[1]
        W.pop("__cond_memo__", None)
        outs = [self._adapter(v, comp, W, f, hw) for _, comp, v in conds]
        concat = outs[0] if len(outs) == 1 else ops.cond_sum(outs)
        self.adapter_runs += 1
        if key is not None:
            W["__cond_memo__"] = (key, concat)
        return concat

    def _forward_vcomposer(self, x, t, bound, conds):
        self._check_x(x, t)
        image = bound.get("image")
        self._check_conditions(x, conds, image)
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        concat = self._adapter_concat(conds, W, f, h * w) if conds else None
        return self._forward_cond(x, t, concat=concat, y=bound.get("y"), image=image, fps=bound.get("fps"))

    @graphed(key="forward_vcomposer")
    @torch.no_grad()
    def _forward_cond(self, x, t, concat=None, y=None, image=None, fps=None):
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        emb = self._time_embedding(t, fps, W)
        if y is None:
            if self.zero_y is None:
                raise ValueError("y is None and no zero_y was given")
            y = self.zero_y.to(x.device).repeat(b, 1, 1)
        ctx = self._to_f16_rows(y)
        if image is not None:                  # context = [y, pre_image_condition(image) as num_tokens tokens] (:743-745)
            img = self._to_f16_rows(image.reshape(1, b, self.context_dim)).view(b, self.context_dim)
            tok = self._mlp(img, W, "pre_image_condition.")                     # [b, num_tokens * context_dim]
            ly, cdim = ctx.shape[1], self.context_dim
            full = torch.empty(b, (ly + self.num_tokens) * cdim, device=x.device, dtype=torch.float16)
            ops.copy2d(ctx.reshape(b, ly * cdim), full[:, :ly * cdim])
            ops.copy2d(tok, full[:, ly * cdim:])
            ctx = full.view(b, ly + self.num_tokens, cdim)
        cin = self.plan.input_blocks[0][0].cin
        cpad = ((cin + 7) // 8) * 8
        xin = ops.cp_to_pc(x.contiguous(), b, c, f * h * w, c_pad=cpad).view(-1, cpad)
        if concat is not None:                 # the condition rows of cb videos, applied to every group of cb videos of x
            n, cd = concat.shape
            for j in range(xin.shape[0] // n):
                ops.copy2d(concat, xin[j * n:(j + 1) * n, c:c + cd])
        out = self._trunk(xin.view(b * f, h, w, cpad), emb, ctx, W, b, f)
        return ops.pc_to_cp(out.view(b, f * h * w, self.out_dim), b, self.out_dim, f * h * w).view(b, self.out_dim, f, h, w)


class UNetSD_TFT2V(UNetSD_VideoLCM):
    """Drop-in for tools/modules/unet/unet_tf2tv.py:188-189 (MODEL 'UNetSD_TFT2V', configs/tft2v_*_infer.yaml): the same
    trunk, adapters and parameters as UNetSD_VideoLCM.  Its misc_dropout(y) (:727) is the identity at inference; a `t_w`
    keyword is accepted and ignored."""

    def forward(self, x, t, *args, t_w=None, **kwargs):
        return super().forward(x, t, *args, **kwargs)


class UNetSD_SR600(_UNetBase):
    """Drop-in for tools/modules/unet/unet_sr600.py:52-53 (MODEL 'UNetSD_SR600'): the T2V trunk with
    (2,1)-padded downsampling, row-cropped upsampling, and -- on the first two decoder blocks -- the
    backbone half scaled by 1.1 / 1.2 and the skip passed through Fourier_filter(threshold=1, 0.6 / 0.4)
    (:269-285).  The filter and the scaling are fused into the channel concat."""
    KIND = "sr600"
    SR600 = True
    _BACKBONE_SCALE = (1.1, 1.2)
    _SKIP_SCALE = (0.6, 0.4)

    def _merge_skip(self, x, skip, n):
        if n >= 2:
            return ops.concat_channels(x, skip)
        cx, cs = x.shape[-1], skip.shape[-1]
        out = torch.empty(*x.shape[:-1], cx + cs, device=x.device, dtype=torch.float16)
        o2, x2 = out.view(-1, cx + cs), x.view(-1, cx)
        half = cx // 2
        ops.scale_copy2d(x2[:, :half], o2[:, :half], self._BACKBONE_SCALE[n])
        ops.copy2d(x2[:, half:], o2[:, half:cx])
        ops.fourier_lowfreq_filter(skip, self._SKIP_SCALE[n], out=o2[:, cx:])
        return out

    @graphed
    @torch.no_grad()
    def forward(self, x, t, y, x_lr=None, fps=None, video_mask=None, focus_present_mask=None, prob_focus_present=0.,
                mask_last_frame_num=0, **kwargs):
        self._check_x(x, t)
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        if h % 2:
            raise ValueError("UNetSD_SR600: latent height must be even (UpsampleSR600 restores 2*h'-2 rows)")
        emb = self._time_embedding(t, None, W)
        ctx = self._to_f16_rows(y)
        xin = ops.cp_to_pc(x.contiguous(), b, c, f * h * w, c_pad=8).view(b * f, h, w, 8)
        out = self._trunk(xin, emb, ctx, W, b, f)
        return ops.pc_to_cp(out.view(b, f * h * w, self.out_dim), b, self.out_dim, f * h * w).view(b, self.out_dim, f, h, w)


class UNetSD_HiGen(_UNetBase):
    """Drop-in for tools/modules/unet/unet_higen.py:175-176 (MODEL 'UNetSD_HiGen'), both stages of
    inference_higen_entrance.py (:198-203 one-frame spatial stage, :221-229 32-frame temporal stage):
      * per-frame embeddings = time + motion-similarity + appearance-similarity (:436-443,:387-399);
      * context = 16 learned tokens cross-attending to the projected text (:154-172);
      * the spatial prior enters through img_embedding right after the first conv (:544-547);
      * every temporal branch is multiplied by 0 when f == 1 (:80-83,:146-149) -- skipped here."""
    KIND = "higen"
    WOIMG = True

    def _context_tokens(self, y16, W, b):
        """TextContextCrossTransformerMultiLayer.forward (unet_higen.py:167-172) -> [b, num_tokens, context_dim]."""
        p = "context_embedding."
        E, T = self.embed_dim, self.num_tokens
        yy = ops.linear(y16.view(-1, y16.shape[-1]), W[p + "input_mapping.w"], bias=W[p + "input_mapping.b"]).view(b, -1, E)
        tok = torch.empty(b, T * E, device=y16.device, dtype=torch.float16)
        ops.copy2d(W[p + "tokens"].view(1, T * E).expand(b, T * E), tok)          # broadcast over the batch (row stride 0)
        tok = tok.view(b * T, E)
        heads = 8
        for d in range(self.plan.context_embedding_depth):
            q = f"{p}context_transformer.{d}."
            for att, nrm in (("attn1.", "norm1."), ("attn2.", "norm2.")):
                xn = ops.layer_norm(tok, W[q + nrm + "g"], W[q + nrm + "b"])
                qq = ops.linear(xn, W[q + att + "q"]).view(b, T, E)
                kv = ops.linear(yy.view(-1, E), W[q + att + "kv"]).view(b, -1, 2 * E)
                a = ops.attention_cross_small(qq, kv[:, :, :E], kv[:, :, E:], heads)
                tok = ops.linear(a.view(-1, E), W[q + att + "to_out.0.w"], bias=W[q + att + "to_out.0.b"], residual=tok)
            tok = self._feed_forward(tok, W, q)
        out = ops.linear(tok, W[p + "output_mapping.w"], bias=W[p + "output_mapping.b"])
        return out.view(b, T, self.context_dim)

    def _frame_embeddings(self, t, fps, motion_cond, appearance_cond, W, b, f):
        """[b*f, embed_dim]: time (+fps) embedding of the video repeated per frame + motion + appearance."""
        tt = t.reshape(-1).repeat_interleave(f)                   # index plumbing; the MLP is row-wise
        emb = self._time_embedding(tt, None if fps is None else fps.reshape(-1).repeat_interleave(f), W)
        if f > 1:
            if motion_cond.size(1) != f:
                me = ops.sinusoidal_embedding(motion_cond.reshape(-1), self.dim).view(b, f - 1, self.dim)
                me = ops.interp_linear_rows(me, f)
            else:
                me = ops.sinusoidal_embedding(motion_cond.reshape(-1), self.dim)
            me = self._mlp(me.view(b * f, self.dim), W, "msim_embedding.")
        else:
            me = self._mlp(ops.sinusoidal_embedding(motion_cond.reshape(-1), self.dim), W, "msim_embedding.")
        emb = ops.eltwise("add", emb, me)
        ac = self._to_f16_rows(appearance_cond.reshape(b, f, -1))
        return ops.eltwise("add", emb, self._mlp(ac.view(b * f, -1), W, "asim_embedding."))

    @graphed
    @torch.no_grad()
    def forward(self, x, t, y=None, fps=None, masked=None, video_mask=None, spat_prior=None, motion_cond=None,
                appearance_cond=None, focus_present_mask=None, prob_focus_present=0., mask_last_frame_num=0, **kwargs):
        self._check_x(x, t)
        if y is None or spat_prior is None or motion_cond is None or appearance_cond is None:
            raise ValueError("UNetSD_HiGen.forward needs y, spat_prior, motion_cond and appearance_cond")
        W = self._packed or self._pack()
        b, c, f, h, w = x.shape
        emb = self._frame_embeddings(t, fps, motion_cond, appearance_cond, W, b, f)
        ctx = self._context_tokens(self._to_f16_rows(y), W, b)
        # img_embedding(spat_prior) repeated over the frames, added to the first conv (residual epilogue)
        sp = ops.cp_to_pc(spat_prior.contiguous().float(), b, spat_prior.shape[1], h * w, c_pad=8).view(b, h, w, 8)
        img = self._conv3x3_any(sp, W, "img_embedding.").view(b, h * w, self.dim)
        img_rep = torch.empty(b, f, h * w, self.dim, device=x.device, dtype=torch.float16)
        for bi in range(b):                     # broadcast over the frames of a video (row stride 0): b launches, not b*f
            ops.copy2d(img[bi].reshape(1, -1).expand(f, -1), img_rep[bi].view(f, -1))
        xin = ops.cp_to_pc(x.contiguous(), b, c, f * h * w, c_pad=8).view(b * f, h, w, 8)
        out = self._trunk(xin, emb, ctx, W, b, f, conv_in_residual=img_rep.view(-1, self.dim))
        return ops.pc_to_cp(out.view(b, f * h * w, self.out_dim), b, self.out_dim, f * h * w).view(b, self.out_dim, f, h, w)
