"""TEST INFRASTRUCTURE ONLY -- the VideoComposer (condition-adapter) cases of UNetSD_VideoLCM / UNetSD_TFT2V.

  * VCOMPOSER_CASES: constructor, composition set, weight seed and input recipe of each case;
  * make_vcomposer_inputs: deterministic inputs (numpy PCG64 keyed by tensor name, like oracle/synth.py);
  * unet_vcomposer_forward: a PyTorch restatement of the reference forward with conditions
    (tools/modules/unet/unet_videolcm.py:598-760; unet_tf2tv.py is the same arithmetic at inference): the adapters, then the
    trunk of oracle/vgen_oracle.py.

tools/make_golden_vcomposer.py runs the REAL reference classes on CPU on these cases, checks this restatement against
them and freezes the outputs into tests/golden/vc_*.npz; the GPU tests replay them.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle import synth, vgen_oracle as vo
from oracle.cases import _LCM_TINY, _FULL_UNET

# forward keyword -> (composition, adapter module, Transformer_v2 module, channels), in the order the reference adds the
# adapters to `concat` (:599-699)
CONDITIONS = (
    ("depth", "depthmap", "depth_embedding", "depth_embedding_after", 1),
    ("local_image", "local_image", "local_image_embedding", "local_image_embedding_after", 3),
    ("motion", "motion", "motion_embedding", "motion_embedding_after", 2),
    ("canny", "canny", "canny_embedding", "canny_embedding_after", 1),
    ("sketch", "sketch", "sketch_embedding", "sketch_embedding_after", 1),
    ("single_sketch", "single_sketch", "single_sketch_embedding", "single_sketch_embedding_after", 1),
    ("masked", "mask", "masked_embedding", "mask_embedding_after", 4),
)
ALL_CONDS = tuple(c[0] for c in CONDITIONS)
ALL_COMPS = ["text", "mask", "depthmap", "sketch", "motion", "image", "local_image", "single_sketch", "canny"]
# scale and value range of each synthetic condition (depth / edges in [0, 1], motion vectors and images signed)
_COND_RECIPE = {"depth": (0.5, True), "local_image": (0.5, False), "motion": (1.0, False), "canny": (0.5, True),
                "sketch": (0.5, True), "single_sketch": (0.5, True), "masked": (0.5, False)}

VCOMPOSER_CASES = {
    # (a) every spatial composition plus the image tokens
    "vc_tft2v_all": dict(cls="UNetSD_TFT2V", ctor=_LCM_TINY, comps=ALL_COMPS, inpainting=True, seed=31, b=1, f=4, h=8, w=12,
                         ntok=5, t=[501], conds=ALL_CONDS, image=True, ddim=dict(steps=4, guide_scale=9.0)),
    # (b) the text-only TF-T2V configs declare ['text', 'image'] and are called without image
    "vc_tft2v_textimg": dict(cls="UNetSD_TFT2V", ctor=_LCM_TINY, comps=["text", "image"], inpainting=True, seed=32, b=1, f=3,
                             h=8, w=12, ntok=6, t=[301], conds=(), image=False),
    # (c) two videos, a subset of the adapters, no inpainting (mask_embedding_after exists, masked_embedding does not)
    "vc_videolcm_b2": dict(cls="UNetSD_VideoLCM", ctor=_LCM_TINY, comps=["text", "depthmap", "sketch"], inpainting=False,
                           seed=33, b=2, f=3, h=8, w=6, ntok=5, t=[751, 99], conds=("depth", "sketch"), image=False),
}

# full-size TF-T2V (configs/tft2v_vcomposer_infer.yaml: the 1.41 B UNet, 16 frames at 448x256)
FULL_VCOMPOSER = dict(cls="UNetSD_TFT2V", ctor=dict(_FULL_UNET, concat_dim=8, num_tokens=4), comps=ALL_COMPS, inpainting=True,
                      seed=34, b=1, f=16, h=32, w=56, ntok=77, t=[759], conds=ALL_CONDS, image=True)


def resolution(case):
    """config.resolution ([W, H] in pixels) whose adapters reduce to the case's latent h x w."""
    return [8 * case["w"], 8 * case["h"]]


def config(case):
    return dict(video_compositions=list(case["comps"]), resolution=resolution(case))


def ctor(case):
    return dict(case["ctor"], inpainting=case["inpainting"])


def make_vcomposer_inputs(case):
    s = case["seed"] + 1000
    b, f, h, w, L = case["b"], case["f"], case["h"], case["w"], case["ntok"]
    H, W = 8 * h, 8 * w
    d = {
        "x": synth.tensor("x", (b, 4, f, h, w), 1.0, s),
        "t": torch.tensor(case["t"], dtype=torch.long),
        "y": synth.tensor("y", (b, L, 1024), 1.0, s),
        "y_neg": synth.tensor("y_neg", (b, L, 1024), 1.0, s),
    }
    for name, _, _, _, cin in CONDITIONS:
        if name in case["conds"]:
            scale, unit = _COND_RECIPE[name]
            v = synth.tensor(name, (b, cin, f, H, W), scale, s)
            d[name] = v.abs().clamp(0, 1) if unit else v
    if case["image"]:
        d["image"] = synth.tensor("image", (b, 1, 1024), 1.0, s)
    return d


def cond_kwargs(inp):
    """The condition keywords present in an input dict (reference keyword names)."""
    return {k: inp[k] for k in ALL_CONDS + ("image",) if k in inp}


def _adapter(v, sd, stem, after, res):
    """<stem>(rearrange(v, 'b c f h w -> (b f) c h w')) then <after> over the frames of each pixel (:599-607)."""
    b, cin, f, H, W = v.shape
    z = v.permute(0, 2, 1, 3, 4).reshape(b * f, cin, H, W)
    z = F.silu(F.conv2d(z, sd[stem + ".0.weight"], sd[stem + ".0.bias"], padding=1))
    z = F.adaptive_avg_pool2d(z, (res[1] // 2, res[0] // 2))
    z = F.silu(F.conv2d(z, sd[stem + ".3.weight"], sd[stem + ".3.bias"], stride=2, padding=1))
    z = F.conv2d(z, sd[stem + ".5.weight"], sd[stem + ".5.bias"], stride=2, padding=1)
    cc, hh, ww = z.shape[1:]
    tok = z.reshape(b, f, cc, hh, ww).permute(0, 3, 4, 1, 2).reshape(b * hh * ww, f, cc)
    tok = vo._local_temporal_encoder(tok, vo._SD(sd).sub(after))     # Transformer_v2: same arithmetic as TransformerV2
    return tok.reshape(b, hh, ww, f, cc).permute(0, 4, 3, 1, 2)      # b c f h w


def unet_vcomposer_forward(sd, x, t, y, res, image=None, fps=None, head_dim=64, use_fps_condition=False, **conds):
    """UNetSD_VideoLCM / UNetSD_TFT2V forward at inference (unet_videolcm.py:541-760) with conditions."""
    b, c, f, h, w = x.shape
    dim = sd["time_embed.0.weight"].shape[1]
    root = vo._SD(sd)
    concat_dim = sd["input_blocks.0.0.weight"].shape[1] - c
    concat = x.new_zeros(b, concat_dim, f, h, w)
    for name, _, stem, after, _ in CONDITIONS:
        v = conds.get(name)
        if v is not None:
            concat = concat + _adapter(v, sd, stem, after, res)
    xx = torch.cat([x, concat], dim=1)
    emb = vo._mlp(vo.sinusoidal_embedding(t, dim).to(x.dtype), root.sub("time_embed"))
    if use_fps_condition and fps is not None:
        emb = emb + vo._mlp(vo.sinusoidal_embedding(fps, dim).to(x.dtype), root.sub("fps_embedding"))
    emb = emb.repeat_interleave(f, dim=0)
    ctx = y
    if image is not None:
        tok = vo._mlp(image, root.sub("pre_image_condition"))
        tok = tok.view(b, -1, y.shape[-1])                               # .view(-1, num_tokens, context_dim) (:744)
        ctx = torch.cat([ctx, tok], dim=1)
    ctx = ctx.repeat_interleave(f, dim=0)
    xx = xx.permute(0, 2, 1, 3, 4).reshape(b * f, c + concat_dim, h, w)
    out = vo._unet_trunk(sd, xx, emb, ctx, head_dim, b)
    return out.reshape(b, f, -1, h, w).permute(0, 2, 1, 3, 4)
