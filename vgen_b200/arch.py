"""Architecture plans and parameter specs (names + shapes) of the UNets / VAE on the hot path.

The checkpoint format IS the interface: `load_state_dict(strict=True)` must accept the reference's
key names and shapes (1 480 tensors for UNetSD_T2VBase, 1 509 for UNetSD_I2VGen, 248 for
AutoencoderKL).  The plan below is derived from the constructor arguments exactly as the reference
builds its module tree:
    tools/modules/unet/unet_t2v.py:87-208, unet_i2vgen.py:88-240 (block layout),
    tools/modules/unet/util.py:311-353,674-741,807-898,1189-1238,1652-1684 (per-module parameters),
    tools/modules/autoencoder.py:30-62,276-313,338-363,483-547,581-651 (VAE).
tests/test_host_logic.py::test_param_spec_equals_reference pins the generated spec against
tests/golden/*.spec.json (dumped from the reference classes by oracle/make_golden.py).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Tuple

Spec = List[Tuple[str, Tuple[int, ...]]]


# ----------------------------------------------------------------------------------------- UNet
@dataclass
class Layer:
    kind: str                 # conv_in | res | spatial | temporal | down | up
    prefix: str               # state_dict prefix, e.g. "input_blocks.1.0."
    cin: int = 0
    cout: int = 0
    heads: int = 0
    inner: int = 0            # transformer width (heads * head_dim)


@dataclass
class UNetPlan:
    kind: str                               # t2v | i2vgen | videolcm | sr600 | higen
    in_dim: int
    dim: int
    embed_dim: int
    y_dim: int
    context_dim: int
    out_dim: int
    head_dim: int
    num_tokens: int
    concat_dim: int
    use_fps_condition: bool
    context_embedding_depth: int = 0        # higen: depth of TextContextCrossTransformerMultiLayer
    compositions: Tuple[str, ...] = ()      # videolcm / tft2v: config.video_compositions
    inpainting: bool = True                 # videolcm / tft2v: 'mask' builds masked_embedding only when True
    input_blocks: List[List[Layer]] = field(default_factory=list)
    middle: List[Layer] = field(default_factory=list)
    output_blocks: List[List[Layer]] = field(default_factory=list)


def unet_plan(kind, in_dim=4, dim=512, y_dim=512, context_dim=512, out_dim=6, num_tokens=4, dim_mult=(1, 2, 3, 4),
              num_heads=None, head_dim=64, num_res_blocks=3, attn_scales=(1 / 2, 1 / 4, 1 / 8), temporal_attention=True,
              use_fps_condition=False, concat_dim=8, context_embedding_depth=4, compositions=(), inpainting=True,
              **_ignored) -> UNetPlan:
    """Block layout for the given constructor kwargs (defaults are the reference's own)."""
    if not temporal_attention:
        raise NotImplementedError("temporal_attention=False is not on the sampling hot path")
    num_heads = num_heads if num_heads else dim // 32
    embed_dim = dim * 4
    if kind == "i2vgen":
        concat_dim = in_dim  # unet_i2vgen.py:82 overrides the argument
        use_fps_condition = True  # fps_embedding is always built and used (unet_i2vgen.py:104-109,298)
    if kind == "sr600":
        use_fps_condition = False  # UNetSD_SR600 never builds fps_embedding (unet_sr600.py:96-100)
    has_concat = kind in ("i2vgen", "videolcm")  # channels concatenated to x before the first conv
    plan = UNetPlan(kind, in_dim, dim, embed_dim, y_dim, context_dim, out_dim, head_dim, num_tokens,
                    concat_dim if has_concat else 0, use_fps_condition,
                    context_embedding_depth if kind == "higen" else 0,
                    tuple(compositions) if kind == "videolcm" else (), bool(inpainting))
    enc_dims = [dim * u for u in [1] + list(dim_mult)]
    dec_dims = [dim * u for u in [dim_mult[-1]] + list(dim_mult)[::-1]]
    shortcut = []
    scale = 1.0
    first_in = in_dim + plan.concat_dim
    plan.input_blocks.append([
        Layer("conv_in", "input_blocks.0.0.", first_in, dim),
        Layer("temporal", "input_blocks.0.1.", dim, dim, num_heads, num_heads * head_dim),
    ])
    shortcut.append(dim)
    idx = 1
    for i, (cin, cout) in enumerate(zip(enc_dims[:-1], enc_dims[1:])):
        for j in range(num_res_blocks):
            blk = [Layer("res", f"input_blocks.{idx}.0.", cin, cout)]
            if scale in attn_scales:
                blk.append(Layer("spatial", f"input_blocks.{idx}.1.", cout, cout, cout // head_dim, cout))
                blk.append(Layer("temporal", f"input_blocks.{idx}.2.", cout, cout, cout // head_dim, cout))
            cin = cout
            plan.input_blocks.append(blk)
            shortcut.append(cout)
            idx += 1
            if i != len(dim_mult) - 1 and j == num_res_blocks - 1:
                plan.input_blocks.append([Layer("down", f"input_blocks.{idx}.", cout, cout)])
                shortcut.append(cout)
                scale /= 2.0
                idx += 1
    c = enc_dims[-1]
    plan.middle = [
        Layer("res", "middle_block.0.", c, c),
        Layer("spatial", "middle_block.1.", c, c, c // head_dim, c),
        Layer("temporal", "middle_block.2.", c, c, c // head_dim, c),
        Layer("res", "middle_block.3.", c, c),
    ]
    idx = 0
    for i, (cin, cout) in enumerate(zip(dec_dims[:-1], dec_dims[1:])):
        for j in range(num_res_blocks + 1):
            blk = [Layer("res", f"output_blocks.{idx}.0.", cin + shortcut.pop(), cout)]
            k = 1
            if scale in attn_scales:
                blk.append(Layer("spatial", f"output_blocks.{idx}.{k}.", cout, cout, cout // head_dim, cout))
                blk.append(Layer("temporal", f"output_blocks.{idx}.{k + 1}.", cout, cout, cout // head_dim, cout))
                k += 2
            cin = cout
            if i != len(dim_mult) - 1 and j == num_res_blocks:
                blk.append(Layer("up", f"output_blocks.{idx}.{k}.", cout, cout))
                scale *= 2.0
            plan.output_blocks.append(blk)
            idx += 1
    return plan


def _lin(p, n, k, bias=True):
    out = [(p + "weight", (n, k))]
    if bias:
        out.append((p + "bias", (n,)))
    return out


def _norm(p, c):
    return [(p + "weight", (c,)), (p + "bias", (c,))]


def _conv(p, n, c, *ks):
    return [(p + "weight", (n, c) + tuple(ks)), (p + "bias", (n,))]


def _attn(p, dim, ctx):
    return (_lin(p + "to_q.", dim, dim, False) + _lin(p + "to_k.", dim, ctx, False) + _lin(p + "to_v.", dim, ctx, False) +
            _lin(p + "to_out.0.", dim, dim))


def _basic_block(p, dim, ctx):
    """BasicTransformerBlock registration order: attn1, ff, attn2, norm1..3 (util.py:681-696)."""
    return (_attn(p + "attn1.", dim, dim) + _lin(p + "ff.net.0.proj.", dim * 8, dim) + _lin(p + "ff.net.2.", dim, dim * 4) +
            _attn(p + "attn2.", dim, ctx) + _norm(p + "norm1.", dim) + _norm(p + "norm2.", dim) + _norm(p + "norm3.", dim))


def _layer_spec(L: Layer, plan: UNetPlan) -> Spec:
    p = L.prefix
    if L.kind == "conv_in":
        return _conv(p, L.cout, L.cin, 3, 3)
    if L.kind == "res":
        s = _norm(p + "in_layers.0.", L.cin) + _conv(p + "in_layers.2.", L.cout, L.cin, 3, 3)
        s += _lin(p + "emb_layers.1.", L.cout, plan.embed_dim)
        s += _norm(p + "out_layers.0.", L.cout) + _conv(p + "out_layers.3.", L.cout, L.cout, 3, 3)
        if L.cin != L.cout:
            s += _conv(p + "skip_connection.", L.cout, L.cin, 1, 1)
        for name, widx in (("conv1", 2), ("conv2", 3), ("conv3", 3), ("conv4", 3)):
            q = f"{p}temopral_conv.{name}."
            s += _norm(q + "0.", L.cout) + _conv(f"{q}{widx}.", L.cout, L.cout, 3, 1, 1)
        return s
    if L.kind == "spatial":
        # context_dim of the decoder blocks is hard-coded to 1024 upstream (unet_t2v.py:180)
        ctx = 1024 if p.startswith("output_blocks") else plan.context_dim
        return (_norm(p + "norm.", L.cin) + _lin(p + "proj_in.", L.inner, L.cin) +
                _basic_block(p + "transformer_blocks.0.", L.inner, ctx) + _lin(p + "proj_out.", L.inner, L.cin))
    if L.kind == "temporal":
        return (_norm(p + "norm.", L.cin) + _conv(p + "proj_in.", L.inner, L.cin, 1) +
                _basic_block(p + "transformer_blocks.0.", L.inner, L.inner) + _conv(p + "proj_out.", L.cin, L.inner, 1))
    if L.kind == "down":
        return _conv(p + "op.", L.cout, L.cin, 3, 3)
    if L.kind == "up":
        return _conv(p + "conv.", L.cout, L.cin, 3, 3)
    raise ValueError(L.kind)


def _mlp(p, a, b, c):
    return _lin(p + "0.", b, a) + _lin(p + "2.", c, b)


# VideoComposer condition adapters of UNetSD_VideoLCM / UNetSD_TFT2V in the reference's creation order
# (unet_videolcm.py:295-372): composition -> (stem module, Transformer_v2 module, condition channels)
ADAPTERS = (
    ("depthmap", "depth_embedding", "depth_embedding_after", 1),
    ("motion", "motion_embedding", "motion_embedding_after", 2),
    ("canny", "canny_embedding", "canny_embedding_after", 1),
    ("mask", "masked_embedding", "mask_embedding_after", 4),
    ("sketch", "sketch_embedding", "sketch_embedding_after", 1),
    ("single_sketch", "single_sketch_embedding", "single_sketch_embedding_after", 1),
    ("local_image", "local_image_embedding", "local_image_embedding_after", 3),
)


def _transformer_v2(p, cd):
    """Transformer_v2(heads=2, dim=cd, dim_head=cd, mlp_dim=cd, depth=1), unet_videolcm.py:121-141 (Attention :39-67,
    FeedForward util.py:724-741 with mult 4)."""
    e = p + "layers.0."
    return (_norm(e + "0.norm.", cd) + _lin(e + "0.fn.to_qkv.", 2 * cd * 3, cd, False) + _lin(e + "0.fn.to_out.0.", cd, 2 * cd) +
            _lin(e + "1.net.0.0.", cd * 4, cd) + _lin(e + "1.net.2.", cd, cd * 4))


def _vcomposer_spec(plan: UNetPlan) -> Spec:
    cd = plan.concat_dim
    s: Spec = []
    if "image" in plan.compositions:
        s += _mlp("pre_image_condition.", plan.context_dim, plan.context_dim, plan.context_dim * plan.num_tokens)
    for comp, stem, after, cin in ADAPTERS:
        if comp not in plan.compositions:
            continue
        if comp != "mask" or plan.inpainting:   # masked_embedding is None without inpainting, its Transformer_v2 exists
            s += _conv(stem + ".0.", cd * 4, cin, 3, 3) + _conv(stem + ".3.", cd * 4, cd * 4, 3, 3) + _conv(stem + ".5.", cd, cd * 4, 3, 3)
        s += _transformer_v2(after + ".", cd)
    return s


def unet_spec(plan: UNetPlan) -> Spec:
    s: Spec = _mlp("time_embed.", plan.dim, plan.embed_dim, plan.embed_dim)
    if plan.kind == "videolcm":
        s += _vcomposer_spec(plan)
    if plan.kind == "i2vgen":
        cd = plan.concat_dim
        s += _mlp("context_embedding.", plan.y_dim, plan.embed_dim, plan.context_dim * plan.num_tokens)
        s += _mlp("fps_embedding.", plan.dim, plan.embed_dim, plan.embed_dim)
        s += _conv("local_image_concat.0.", cd * 4, 4, 3, 3) + _conv("local_image_concat.2.", cd * 4, cd * 4, 3, 3) + \
            _conv("local_image_concat.4.", cd, cd * 4, 3, 3)
        e = "local_temporal_encoder.layers.0."
        s += _norm(e + "0.norm.", cd) + _lin(e + "0.fn.to_qkv.", 2 * cd * 3, cd, False) + _lin(e + "0.fn.to_out.0.", cd, 2 * cd)
        s += _lin(e + "1.net.0.0.", cd * 4, cd) + _lin(e + "1.net.2.", cd, cd * 4)
        s += _conv("local_image_embedding.0.", cd * 8, 4, 3, 3) + _conv("local_image_embedding.3.", cd * 16, cd * 8, 3, 3) + \
            _conv("local_image_embedding.5.", 1024, cd * 16, 3, 3)
    elif plan.use_fps_condition:
        s += _mlp("fps_embedding.", plan.dim, plan.embed_dim, plan.embed_dim)
    if plan.kind == "higen":
        # TextContextCrossTransformerMultiLayer (unet_higen.py:154-166) + similarity / image embeddings (:271-289)
        ed = plan.embed_dim
        s += [("context_embedding.tokens", (1, plan.num_tokens, ed))]
        for d in range(plan.context_embedding_depth):
            s += _basic_block(f"context_embedding.context_transformer.{d}.", ed, ed)
        s += _lin("context_embedding.input_mapping.", ed, plan.y_dim) + _lin("context_embedding.output_mapping.", plan.context_dim, ed)
        s += _mlp("asim_embedding.", 32, ed, ed) + _mlp("msim_embedding.", plan.dim, ed, ed)
        s += _conv("img_embedding.", plan.dim, plan.in_dim, 3, 3)
    for blk in plan.input_blocks:
        for L in blk:
            s += _layer_spec(L, plan)
    for L in plan.middle:
        s += _layer_spec(L, plan)
    for blk in plan.output_blocks:
        for L in blk:
            s += _layer_spec(L, plan)
    last = plan.output_blocks[-1][0].cout
    s += _norm("out.0.", last) + _conv("out.2.", plan.out_dim, last, 3, 3)
    return s


# Tensors the reference zero-initialises (zero_module util.py:716-722; nn.init.zeros_ :873-875,
# :1683-1684, unet_t2v.py:103-104,208) -- used only for default (no-checkpoint) initialisation.
def unet_zero_init(name: str) -> bool:
    if name.endswith("proj_out.weight") or name.endswith("proj_out.bias"):
        return True
    if ".out_layers.3." in name or ".temopral_conv.conv4.3." in name:
        return True
    if name.startswith(("asim_embedding.2.", "msim_embedding.2.", "img_embedding.")):
        return True  # unet_higen.py:276-289
    return name == "out.2.weight" or name.startswith("fps_embedding.2.")


# ----------------------------------------------------------------------------------------- VAE
@dataclass
class VaePlan:
    ch: int
    ch_mult: Tuple[int, ...]
    num_res_blocks: int
    z_channels: int
    in_channels: int
    out_ch: int
    embed_dim: int
    double_z: bool


def vae_plan(ddconfig, embed_dim) -> VaePlan:
    if ddconfig.get("attn_resolutions"):
        raise NotImplementedError("VAE attn_resolutions must be empty (SD-2.1 VAE)")
    return VaePlan(ddconfig["ch"], tuple(ddconfig["ch_mult"]), ddconfig["num_res_blocks"], ddconfig["z_channels"],
                   ddconfig["in_channels"], ddconfig["out_ch"], embed_dim, bool(ddconfig.get("double_z", True)))


def _resnet(p, cin, cout) -> Spec:
    s = _norm(p + "norm1.", cin) + _conv(p + "conv1.", cout, cin, 3, 3) + _norm(p + "norm2.", cout) + \
        _conv(p + "conv2.", cout, cout, 3, 3)
    if cin != cout:
        s += _conv(p + "nin_shortcut.", cout, cin, 1, 1)
    return s


def _vae_attn(p, c) -> Spec:
    return _norm(p + "norm.", c) + _conv(p + "q.", c, c, 1, 1) + _conv(p + "k.", c, c, 1, 1) + _conv(p + "v.", c, c, 1, 1) + \
        _conv(p + "proj_out.", c, c, 1, 1)


def vae_spec(v: VaePlan) -> Spec:
    """Encoder (autoencoder.py:483-547), Decoder (:581-651), quant convs (:49-50) in registration order."""
    nres = len(v.ch_mult)
    s: Spec = _conv("encoder.conv_in.", v.ch, v.in_channels, 3, 3)
    in_mult = (1,) + v.ch_mult
    block_in = v.ch
    for lvl in range(nres):
        block_in = v.ch * in_mult[lvl]
        block_out = v.ch * v.ch_mult[lvl]
        for j in range(v.num_res_blocks):
            s += _resnet(f"encoder.down.{lvl}.block.{j}.", block_in, block_out)
            block_in = block_out
        if lvl != nres - 1:
            s += _conv(f"encoder.down.{lvl}.downsample.conv.", block_in, block_in, 3, 3)
    s += _resnet("encoder.mid.block_1.", block_in, block_in) + _vae_attn("encoder.mid.attn_1.", block_in) + \
        _resnet("encoder.mid.block_2.", block_in, block_in)
    s += _norm("encoder.norm_out.", block_in)
    s += _conv("encoder.conv_out.", 2 * v.z_channels if v.double_z else v.z_channels, block_in, 3, 3)
    # decoder
    block_in = v.ch * v.ch_mult[-1]
    s += _conv("decoder.conv_in.", block_in, v.z_channels, 3, 3)
    s += _resnet("decoder.mid.block_1.", block_in, block_in) + _vae_attn("decoder.mid.attn_1.", block_in) + \
        _resnet("decoder.mid.block_2.", block_in, block_in)
    ups = {}
    for lvl in reversed(range(nres)):
        block_out = v.ch * v.ch_mult[lvl]
        u: Spec = []
        for j in range(v.num_res_blocks + 1):
            u += _resnet(f"decoder.up.{lvl}.block.{j}.", block_in, block_out)
            block_in = block_out
        if lvl != 0:
            u += _conv(f"decoder.up.{lvl}.upsample.conv.", block_in, block_in, 3, 3)
        ups[lvl] = u
    for lvl in range(nres):  # self.up.insert(0, up): registered in ascending level order
        s += ups[lvl]
    s += _norm("decoder.norm_out.", block_in) + _conv("decoder.conv_out.", v.out_ch, block_in, 3, 3)
    s += _conv("quant_conv.", 2 * v.embed_dim, 2 * v.z_channels, 1, 1) + _conv("post_quant_conv.", v.z_channels, v.embed_dim, 1, 1)
    return s
