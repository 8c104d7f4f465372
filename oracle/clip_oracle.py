"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the CLIP conditioning path the reference's embedders run
(tools/modules/clip_embedder.py:183-199 `FrozenOpenCLIPTextVisualEmbedder.forward / encode_with_transformer /
text_transformer_forward`; the model itself is open_clip's `CLIP`, of which the reference vendors a copy under
utils/reward/open_clip/: `transformer.py` ResidualAttentionBlock :189-244, VisionTransformer :323-520, `model.py` CLIP).

Functional, driven by an open_clip-format state_dict (the format of `open_clip_pytorch_model.bin`).  Pinned against the
vendored open_clip `CLIP` class itself (oracle/make_golden_clip.py compares it with that class and freezes its outputs
into tests/golden/clip_tiny.npz).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _n_layers(sd, prefix):
    idx = set()
    for k in sd:
        if k.startswith(prefix):
            idx.add(int(k[len(prefix):].split(".", 1)[0]))
    return len(idx)


def _block(x, sd, p, heads, causal):
    """ResidualAttentionBlock.forward (pre-LN; nn.MultiheadAttention with a fused in_proj; MLP c_fc -> GELU(erf) -> c_proj)."""
    b, L, W = x.shape
    d = W // heads
    h = F.layer_norm(x, (W,), sd[p + "ln_1.weight"], sd[p + "ln_1.bias"], 1e-5)
    qkv = F.linear(h, sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"])
    q, k, v = qkv.chunk(3, dim=-1)

    def sp(t):
        return t.reshape(b, L, heads, d).permute(0, 2, 1, 3)

    o = F.scaled_dot_product_attention(sp(q), sp(k), sp(v), is_causal=causal)
    o = o.permute(0, 2, 1, 3).reshape(b, L, W)
    x = x + F.linear(o, sd[p + "attn.out_proj.weight"], sd[p + "attn.out_proj.bias"])
    h = F.layer_norm(x, (W,), sd[p + "ln_2.weight"], sd[p + "ln_2.bias"], 1e-5)
    h = F.linear(F.gelu(F.linear(h, sd[p + "mlp.c_fc.weight"], sd[p + "mlp.c_fc.bias"])), sd[p + "mlp.c_proj.weight"],
                 sd[p + "mlp.c_proj.bias"])
    return x + h


def encode_text(sd, tokens, heads, layer="penultimate"):
    """clip_embedder.py:189-212: token + positional embedding, the first (n - layer_idx) causal blocks, ln_final;
    returns (pooled @ text_projection [b, E], tokens [b, 77, W])."""
    layer_idx = {"last": 0, "penultimate": 1}[layer]
    x = sd["token_embedding.weight"][tokens] + sd["positional_embedding"]
    n = _n_layers(sd, "transformer.resblocks.")
    for i in range(n - layer_idx):
        x = _block(x, sd, f"transformer.resblocks.{i}.", heads, True)
    x = F.layer_norm(x, (x.shape[-1],), sd["ln_final.weight"], sd["ln_final.bias"], 1e-5)
    xt = x[torch.arange(x.shape[0]), tokens.argmax(dim=-1)] @ sd["text_projection"]
    return xt, x


def encode_image(sd, image, head_width):
    """VisionTransformer.forward (transformer.py:455-520; no patch-norm, class-token pooling): [b, 3, H, W] -> [b, E]."""
    w = sd["visual.conv1.weight"]
    patch = w.shape[-1]
    x = F.conv2d(image, w, stride=patch)
    b, W = x.shape[0], x.shape[1]
    x = x.reshape(b, W, -1).permute(0, 2, 1)
    cls = sd["visual.class_embedding"].to(x.dtype) + torch.zeros(b, 1, W, dtype=x.dtype, device=x.device)
    x = torch.cat([cls, x], dim=1) + sd["visual.positional_embedding"]
    x = F.layer_norm(x, (W,), sd["visual.ln_pre.weight"], sd["visual.ln_pre.bias"], 1e-5)
    heads = W // head_width
    for i in range(_n_layers(sd, "visual.transformer.resblocks.")):
        x = _block(x, sd, f"visual.transformer.resblocks.{i}.", heads, False)
    pooled = F.layer_norm(x[:, 0], (W,), sd["visual.ln_post.weight"], sd["visual.ln_post.bias"], 1e-5)
    return pooled @ sd["visual.proj"]
