#!/usr/bin/env python
"""TF-T2V with VideoComposer conditions on one B200: CFG DDIM steps (guide 9) of UNetSD_TFT2V (the real 1.41 B
architecture of configs/tft2v_vcomposer_infer.yaml, synthetic weights) with all seven spatial compositions plus image.

One JSON line per workload (16 f x 448x256 and 16 f x 896x512), printed and, with --out, appended to that file:
  steps_per_s_memo_hit    the engines' pattern: the same condition tensors every step, so the adapters run once
  steps_per_s_memo_miss   every step gets fresh clones of the conditions: the adapters run every step
  steps_per_s_text_only   UNetSD_TFT2V(['text', 'image']) called without image (the text-only TF-T2V configs)
  adapter_ms_per_video    the adapter stage alone (seven adapters + fp32 sum)
  stem                    vgen_cond_stem against im2col + linear + adaptive_avgpool for the same math, alternated in one
                          process: ms, GB/s (condition read + pooled write), share of the 6 572 GB/s copy rate
  gpu / power_limit_w     read with nvidia-smi in the same run
Step rates are host wall time over K steps ending in a device synchronise; kernel times are CUDA events.

    python tools/bench_vcomposer.py [--steps K] [--warmup W] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import vgen_b200  # noqa: E402
from vgen_b200 import ops, unet  # noqa: E402
from vcomposer_oracle import ALL_COMPS, CONDITIONS  # noqa: E402
from oracle.cases import _FULL_UNET  # noqa: E402

COPY_GBPS = 6572.0   # measured device-to-device copy rate (DESIGN.md)
CTOR = dict(_FULL_UNET, concat_dim=8, num_tokens=4)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def conditions(b, f, H, W, g):
    d = {}
    for name, _, _, _, cin in CONDITIONS:
        d[name] = torch.rand(b, cin, f, H, W, generator=g).cuda()
    return d


class FreshConditions:
    """Calls the model with clones of the condition tensors: every call misses the adapter memo."""

    def __init__(self, m):
        self.module = m

    def __call__(self, x, t, **kw):
        kw = {k: (v.clone() if k in self.module.cfg_shared_kwargs and v is not None else v) for k, v in kw.items()}
        return self.module(x, t, **kw)


def steps_per_s(diff, model, noise, kw, steps, warmup):
    # at least two warm-up steps: the second forward of a signature is the one captured into a CUDA graph
    diff.ddim_sample_loop(noise, model, kw, guide_scale=9.0, ddim_timesteps=max(warmup, 2))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    diff.ddim_sample_loop(noise, model, kw, guide_scale=9.0, ddim_timesteps=steps)
    torch.cuda.synchronize()
    return steps / (time.perf_counter() - t0)


def event_ms(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def stem_vs_chain(cond, w, bias, oh, ow, reps, rounds):
    """vgen_cond_stem against the unfused chain (cp_to_pc -> im2col -> linear -> adaptive_avgpool(silu_in)), alternated."""
    b, cin, f, H, W = cond.shape
    wk = ops.pack_cond_stem_weight(w).half().cuda()
    wc = unet._pack_conv3x3(w, cond.device, cin_pad=8)
    bc = bias.float().cuda()

    def stem():
        return ops.cond_stem(cond, wk, bc, oh, ow)

    def chain():
        xp = ops.cp_to_pc(cond, b, cin, f * H * W, c_pad=8).view(b * f, H, W, 8)
        col = ops.im2col(xp, 3, 3, 1, 1, 1, H, W, wc.shape[1])
        z = ops.linear(col, wc, bias=bc).view(b * f, H, W, wc.shape[0])
        return ops.adaptive_avgpool(z, oh, ow, silu_in=True)

    a, c = stem(), chain()
    torch.cuda.synchronize()
    diff = float((a.float() - c.float()).abs().max())
    ts, tc = [], []
    for _ in range(rounds):
        ts.append(event_ms(stem, reps))
        tc.append(event_ms(chain, reps))
    ms_s, ms_c = min(ts), min(tc)
    nbytes = cond.numel() * cond.element_size() + 2.0 * b * f * oh * ow * w.shape[0]
    gbps = nbytes / (ms_s * 1e-3) / 1e9
    return {"cin": cin, "dtype": str(cond.dtype).replace("torch.", ""), "shape": list(cond.shape), "stem_ms": ms_s,
            "chain_ms": ms_c, "speedup": ms_c / ms_s, "stem_GBps": gbps, "share_of_copy_rate": gbps / COPY_GBPS,
            "stem_ms_all_rounds": ts, "chain_ms_all_rounds": tc, "max_abs_diff_vs_chain": diff}


def workload(f, h, w, steps, warmup, info):
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(1)
    H, W = 8 * h, 8 * w
    cfg_all = dict(video_compositions=ALL_COMPS, resolution=[W, H])
    m = vgen_b200.UNetSD_TFT2V(config=cfg_all, **CTOR).cuda().eval()
    diff = vgen_b200.DiffusionDDIM(schedule="linear_sd", schedule_param=dict(num_timesteps=1000, init_beta=0.00085,
                                   last_beta=0.0120, zero_terminal_snr=True), mean_type="v", var_type="fixed_small")
    noise = torch.randn(1, 4, f, h, w, generator=g).cuda()
    y, yn = torch.randn(1, 77, 1024, generator=g).cuda(), torch.randn(1, 77, 1024, generator=g).cuda()
    image = torch.randn(1, 1, 1024, generator=g).cuda()
    conds = conditions(1, f, H, W, g)
    kw = [dict(conds, y=y, image=image), dict(conds, y=yn, image=torch.zeros_like(image))]
    hit = steps_per_s(diff, m, noise, kw, steps, warmup)
    runs0 = m.adapter_runs
    miss = steps_per_s(diff, FreshConditions(m), noise, kw, steps, warmup)
    assert m.adapter_runs - runs0 == steps + max(warmup, 2)
    # adapter stage alone
    W_ = m._packed
    order = [(k, comp, conds[k]) for k, comp in m.CONDITIONS]

    def adapters():
        W_.pop("__cond_memo__", None)
        m._adapter_concat(order, W_, f, h * w)
    adapters()
    adapter_ms = min(event_ms(adapters, 5) for _ in range(3))
    del m
    torch.cuda.empty_cache()
    mt = vgen_b200.UNetSD_TFT2V(config=dict(video_compositions=["text", "image"], resolution=[W, H]), **CTOR).cuda().eval()
    text = steps_per_s(diff, mt, noise, [{"y": y}, {"y": yn}], steps, warmup)
    del mt
    torch.cuda.empty_cache()
    gs = torch.Generator().manual_seed(2)
    stems = []
    for cin, dtype in ((1, torch.float32), (1, torch.float16), (4, torch.float32)):
        cond = torch.rand(1, cin, f, H, W, generator=gs).to("cuda", dtype)
        wt = torch.randn(32, cin, 3, 3, generator=gs) / (9 * cin) ** 0.5
        stems.append(stem_vs_chain(cond, wt, torch.randn(32, generator=gs) * 0.05, H // 2, W // 2, reps=10, rounds=5))
    return {"workload": f"tft2v_vcomposer_{f}f_{W}x{H}_cfg9", "latent": [1, 4, f, h, w], "steps": steps, "warmup": warmup,
            "steps_per_s_memo_hit": hit, "steps_per_s_memo_miss": miss, "steps_per_s_text_only": text,
            "adapter_ms_per_video": adapter_ms, "stem": stems, **info}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vcomposer needs a CUDA device")
    info = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    for f, h, w in ((16, 32, 56), (16, 64, 112)):
        rec = workload(f, h, w, args.steps, args.warmup, info)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(line + "\n")


if __name__ == "__main__":
    main()
