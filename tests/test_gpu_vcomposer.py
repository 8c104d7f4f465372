"""VideoComposer path on the B200: the fused adapter stem kernel, forward / DDIM parity of UNetSD_VideoLCM and
UNetSD_TFT2V with conditions against the reference goldens (tools/make_golden_vcomposer.py), the once-per-video memo of
the adapter stage, CFG batching of shared conditions, CUDA-graph replay, and one full-size TF-T2V case.

Gates follow tests/test_gpu_parity.py and tests/test_gpu_fullsize.py: our error against the fp32 truth must not exceed
1.25x the reference's own fp16-autocast error (plus a small absolute term) and an absolute cap."""
import gc
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import vgen_b200
from oracle import synth, vgen_oracle as vo
from vgen_b200 import diffusion, graph, lib, ops
from vcomposer_oracle import (FULL_VCOMPOSER, VCOMPOSER_CASES, cond_kwargs, config, ctor, make_vcomposer_inputs, resolution,
                              unet_vcomposer_forward)

pytestmark = pytest.mark.gpu


def _rel_l2(a, b):
    a, b = a.float(), b.float()
    return float((a - b).norm() / (b.norm() + 1e-12))


# ------------------------------------------------------------------------------------------ vgen_cond_stem
def _stem_inputs(b, cin, f, H, W, cout, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, cin, f, H, W, generator=g).mul_(2).sub_(1).to("cuda", dtype)
    w = torch.randn(cout, cin, 3, 3, generator=g) / (9 * cin) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.05
    return x, w, bias


def _stem_ref32(x, w, bias, oh, ow):
    b, cin, f, H, W = x.shape
    z = x.float().permute(0, 2, 1, 3, 4).reshape(b * f, cin, H, W)
    z = F.adaptive_avg_pool2d(F.silu(F.conv2d(z, w.cuda(), bias.cuda(), padding=1)), (oh, ow))
    return z.permute(0, 2, 3, 1)


def _stem_ref_rounded(x, w, bias, oh, ow):
    """Same rounding points as the kernel: fp16 input / weights, fp32 conv + fp32 bias -> fp16, SiLU -> fp16, fp32 mean -> fp16.
    Also returns, per output, the largest |SiLU| term of its pooling window (the magnitude the fp16 roundings happen at)."""
    b, cin, f, H, W = x.shape
    z = x.half().float().permute(0, 2, 1, 3, 4).reshape(b * f, cin, H, W)
    z = F.conv2d(z, w.half().float().cuda(), bias.cuda(), padding=1).half().float()
    z = F.silu(z).half().float()
    wmax = F.adaptive_max_pool2d(z.abs(), (oh, ow)).permute(0, 2, 3, 1)
    return F.adaptive_avg_pool2d(z, (oh, ow)).half().permute(0, 2, 3, 1), wmax


def _ulp16(v):
    a = v.float().abs().clamp_min(2.0 ** -14)
    return torch.exp2(torch.floor(torch.log2(a)) - 10)


STEM_SHAPES = [(2, 3, 256, 448, 128, 224), (2, 3, 67, 101, 33, 50)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("cin", [1, 2, 3, 4])
@pytest.mark.parametrize("shape", STEM_SHAPES + [(1, 16, 512, 896, 256, 448)])
def test_cond_stem_op(shape, cin, dtype):
    torch.backends.cudnn.allow_tf32 = False
    b, f, H, W, oh, ow = shape
    if H == 512 and (cin, dtype) not in ((4, torch.float32), (1, torch.float16)):
        pytest.skip("full resolution: one fp32 4-channel and one fp16 1-channel case")
    x, w, bias = _stem_inputs(b, cin, f, H, W, 32, dtype, seed=cin * 7 + H)
    out = ops.cond_stem(x, ops.pack_cond_stem_weight(w).half().cuda(), bias.float().cuda(), oh, ow)
    torch.cuda.synchronize()
    assert out.shape == (b * f, oh, ow, 32) and out.dtype == torch.float16
    r32 = _stem_ref32(x, w, bias, oh, ow)
    rr, wmax = _stem_ref_rounded(x, w, bias, oh, ow)
    e = _rel_l2(out, r32)
    d = (out.float() - rr.float()).abs()
    # the fp32 conv sums of the kernel and of cuDNN differ in order, so a conv value near a rounding tie may land one
    # fp16 ulp apart; that ulp is the ulp of the window's terms, so the gate is 2 ulp at max(|output|, largest |term|)
    ulps = float((d / _ulp16(torch.maximum(rr.float().abs(), wmax))).max())
    print(f"cond_stem cin{cin} {dtype} {shape}: rel-L2 vs fp32 {e:.2e}, max {ulps:.2f} fp16 ulp (at the window's term scale) "
          f"vs rounded restatement, {float((d / _ulp16(rr)).max()):.0f} ulp of the output itself, max abs {float(d.max()):.2e}")
    assert e < 1e-3
    assert ulps <= 2.0


@pytest.mark.parametrize("cout", [8, 64])
def test_cond_stem_channel_counts(cout):
    x, w, bias = _stem_inputs(1, 2, 3, 64, 96, cout, torch.float32, seed=cout)
    out = ops.cond_stem(x, ops.pack_cond_stem_weight(w).half().cuda(), bias.float().cuda(), 32, 48)
    assert _rel_l2(out, _stem_ref32(x, w, bias, 32, 48)) < 1e-3


def test_cond_sum_fp32_accumulation():
    g = torch.Generator().manual_seed(3)
    srcs = [(torch.randn(1000, 8, generator=g) * 10 ** i).half().cuda() for i in range(-1, 3)]
    out = ops.cond_sum(srcs)
    ref = srcs[0].float()
    for s in srcs[1:]:
        ref = ref + s.float()
    assert torch.equal(out, ref.half())


# ------------------------------------------------------------------------------------------ model parity
def _setup(golden_dir, name, case=None):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    case = case or VCOMPOSER_CASES[name]
    spec = [(k, tuple(s)) for k, s in json.load(open(os.path.join(golden_dir, f"{name}.spec.json")))]
    sd = synth.state_dict(spec, seed=case["seed"])
    m = getattr(vgen_b200, case["cls"])(config=config(case), **ctor(case))
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    inp = {k: v.cuda() for k, v in make_vcomposer_inputs(case).items()}
    sdg = {k: v.cuda() for k, v in sd.items()}
    return case, m, inp, sdg


@pytest.mark.parametrize("name", sorted(VCOMPOSER_CASES))
def test_forward_parity(golden_dir, name):
    case, m, inp, sdg = _setup(golden_dir, name)
    ck = cond_kwargs(inp)
    with torch.no_grad():
        mine = m(inp["x"], inp["t"], y=inp["y"], **ck)
        o32 = unet_vcomposer_forward(sdg, inp["x"], inp["t"], inp["y"], resolution(case), **ck)
        with torch.autocast("cuda", dtype=torch.float16):
            o16 = unet_vcomposer_forward(sdg, inp["x"], inp["t"], inp["y"], resolution(case), **ck)
    truth = torch.from_numpy(np.load(os.path.join(golden_dir, f"{name}.npz"))["out"]).cuda()
    assert mine.shape == truth.shape and mine.dtype == torch.float16 and torch.isfinite(mine.float()).all()
    assert _rel_l2(o32, truth) < 1e-4
    e_mine, e_ref16 = _rel_l2(mine, truth), _rel_l2(o16, truth)
    print(f"{name}: ours vs fp32 truth {e_mine:.3e}; reference-autocast {e_ref16:.3e}")
    assert e_mine < 5e-3 and e_mine < 1.25 * e_ref16 + 2e-4


def _uncond(inp):
    kw = dict(cond_kwargs(inp), y=inp["y_neg"])
    if "image" in kw:
        kw["image"] = torch.zeros_like(inp["image"])
    return kw


def test_ddim_loop_parity(golden_dir):
    name = "vc_tft2v_all"
    case, m, inp, sdg = _setup(golden_dir, name)
    dd = case["ddim"]
    diff = vgen_b200.DiffusionDDIM(schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                                   mean_type="v", var_type="fixed_small")
    kw = [dict(cond_kwargs(inp), y=inp["y"]), _uncond(inp)]
    runs0 = m.adapter_runs
    lat = diff.ddim_sample_loop(inp["x"], m, kw, guide_scale=dd["guide_scale"], ddim_timesteps=dd["steps"], eta=0.0)
    assert m.adapter_runs - runs0 == 1, "the conditions of one video must go through the adapters once"
    betas = vo.make_betas("cosine", 1000, True, cosine_s=0.008)
    fn = lambda xt, t, **k: unet_vcomposer_forward(sdg, xt, t, res=resolution(case), **k)  # noqa: E731
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        lat16 = vo.ddim_sample_loop(inp["x"].clone(), fn, kw, betas, dd["guide_scale"], dd["steps"], autocast_cfg=True)
    truth = torch.from_numpy(np.load(os.path.join(golden_dir, f"{name}.npz"))["ddim_latent"]).cuda()
    e_mine, e_ref16 = _rel_l2(lat, truth), _rel_l2(lat16, truth)
    print(f"{name} ddim: ours {e_mine:.3e}; reference-autocast {e_ref16:.3e}")
    assert lat.dtype == torch.float32 and torch.isfinite(lat).all()
    assert e_mine < 2.5e-2 and e_mine < 1.25 * e_ref16 + 5e-4


# ------------------------------------------------------------------------------------------ memo, graphs, CFG
def test_memo_hit_and_inplace_edit(golden_dir, monkeypatch):
    monkeypatch.setenv("VGEN_CUDA_GRAPH", "0")
    case, m, inp, sdg = _setup(golden_dir, "vc_videolcm_b2")
    ck = cond_kwargs(inp)
    a = m(inp["x"], inp["t"], y=inp["y"], **ck)
    runs, l0 = m.adapter_runs, lib.launch_count()
    b = m(inp["x"], inp["t"], y=inp["y"], **ck)
    hit_launches = lib.launch_count() - l0
    assert m.adapter_runs == runs and torch.equal(a, b)
    ck2 = {k: v.clone() for k, v in ck.items()}        # fresh tensors: recomputed, same values
    l0 = lib.launch_count()
    c = m(inp["x"], inp["t"], y=inp["y"], **ck2)
    assert m.adapter_runs == runs + 1 and torch.equal(a, c) and lib.launch_count() - l0 > hit_launches
    ck2["depth"].mul_(0.5)                               # in-place edit of one condition
    d = m(inp["x"], inp["t"], y=inp["y"], **ck2)
    assert m.adapter_runs == runs + 2
    with torch.no_grad():
        o32 = unet_vcomposer_forward(sdg, inp["x"], inp["t"], inp["y"], resolution(case), **ck2)
        with torch.autocast("cuda", dtype=torch.float16):
            o16 = unet_vcomposer_forward(sdg, inp["x"], inp["t"], inp["y"], resolution(case), **ck2)
    e_mine, e_ref16 = _rel_l2(d, o32), _rel_l2(o16, o32)
    assert not torch.equal(c, d) and e_mine < 5e-3 and e_mine < 1.25 * e_ref16 + 2e-4
    with torch.inference_mode():                         # no version counter: always recomputed
        ci = {k: v.clone() for k, v in ck.items()}
        m(inp["x"], inp["t"], y=inp["y"], **ci)
        m(inp["x"], inp["t"], y=inp["y"], **ci)
    assert m.adapter_runs == runs + 4


def test_graph_replay_matches_eager(golden_dir):
    case, m, inp, sdg = _setup(golden_dir, "vc_tft2v_all")
    ck = cond_kwargs(inp)
    eager = m._forward_cond.__wrapped_eager__
    outs = [m(inp["x"], inp["t"], y=inp["y"], **ck) for _ in range(3)]
    st = graph.stats(m)
    assert st.get("forward_vcomposer", (0, 0))[0] == 1 and st["forward_vcomposer"][1] >= 1, st
    assert "forward" not in st, "the conditioned path must not use the text-only graph"
    concat = m._packed["__cond_memo__"][1]
    with torch.no_grad():
        ref = eager(m, inp["x"], inp["t"], concat=concat, y=inp["y"], image=inp["image"])
    assert torch.equal(outs[0], ref) and torch.equal(outs[2], ref)
    x2 = inp["x"] * 0.5 + 0.1
    r2 = m(x2, inp["t"], y=inp["y"], **ck)
    with torch.no_grad():
        e2 = eager(m, x2, inp["t"], concat=concat, y=inp["y"], image=inp["image"])
    assert torch.equal(r2, e2) and not torch.equal(r2, ref)


def test_cfg_shared_batch_equals_separate(golden_dir):
    case, m, inp, sdg = _setup(golden_dir, "vc_tft2v_all")
    kc, ku = dict(cond_kwargs(inp), y=inp["y"]), _uncond(inp)
    with torch.no_grad():
        ya, ua = diffusion.cfg_forward(m, inp["x"], inp["t"], [kc, ku])
        yb, ub = m(inp["x"], inp["t"], **kc), m(inp["x"], inp["t"], **ku)
    assert torch.equal(ya, yb) and torch.equal(ua, ub)


def test_text_only_tft2v_ignores_t_w(golden_dir):
    case, m, inp, sdg = _setup(golden_dir, "vc_tft2v_textimg")
    a = m(inp["x"], inp["t"], y=inp["y"])
    b = m(inp["x"], inp["t"], y=inp["y"], t_w=inp["t"])
    assert torch.equal(a, b)
    assert "forward" in graph.stats(m)


def test_condition_errors(golden_dir):
    case, m, inp, sdg = _setup(golden_dir, "vc_videolcm_b2")
    with pytest.raises(ValueError):                      # not built with 'motion'
        m(inp["x"], inp["t"], y=inp["y"], motion=torch.zeros(2, 2, 3, 64, 48, device="cuda"))
    with pytest.raises(ValueError):                      # built without inpainting
        m(inp["x"], inp["t"], y=inp["y"], masked=torch.zeros(2, 4, 3, 64, 48, device="cuda"))
    with pytest.raises(ValueError):                      # latent does not match config.resolution
        m(inp["x"][..., :4], inp["t"], y=inp["y"], depth=inp["depth"])


# ------------------------------------------------------------------------------------------ full size
def test_fullsize_tft2v_all_compositions():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    gc.collect()
    torch.cuda.empty_cache()
    case = FULL_VCOMPOSER
    m = getattr(vgen_b200, case["cls"])(config=config(case), **ctor(case))
    sd = synth.state_dict([(k, tuple(v.shape)) for k, v in m.state_dict().items()], seed=case["seed"])
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    sdg = {k: v.cuda() for k, v in sd.items()}
    del sd
    inp = {k: v.cuda() for k, v in make_vcomposer_inputs(case).items()}
    ck = cond_kwargs(inp)
    with torch.no_grad():
        mine = m(inp["x"], inp["t"], y=inp["y"], **ck)
        o32 = unet_vcomposer_forward(sdg, inp["x"], inp["t"], inp["y"], resolution(case), **ck)
        with torch.autocast("cuda", dtype=torch.float16):
            o16 = unet_vcomposer_forward(sdg, inp["x"], inp["t"], inp["y"], resolution(case), **ck)
    e_mine, e_ref16 = _rel_l2(mine, o32), _rel_l2(o16, o32)
    print(f"[fullsize] tft2v_vcomposer [1,4,16,32,56]: ours {e_mine:.3e}; reference-autocast {e_ref16:.3e}")
    assert torch.isfinite(mine.float()).all()
    assert e_mine < 6e-3 and e_mine <= 1.25 * e_ref16
