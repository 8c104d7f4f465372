#!/usr/bin/env python
"""bench.py -- denoise-steps/s (and decoded frames/s, videos/s) of the VGen sampling hot path on B200.

Headline workload (BASELINE.json configs[1], `--workload i2vgen`, the default): i2vgen_xl, 16 frames, 1280x704
(latent [1,4,16,88,160]), DDIM with classifier-free guidance (2 UNet evaluations + 1 fused DDIM update per step),
synthetic image + text conditioning, random-init weights of the real architecture (UNetSD_I2VGen, 1.42 B parameters).
A "step" is one denoising step.  N GPUs run N independent trajectories (weak scaling); the only collective is the
one-time NCCL broadcast of the packed fp16 weight arena.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload i2vgen|videolcm|sr600|higen] [--dump-outputs DIR]

The other workloads are BASELINE configs 3 / 4 / 5 driven the way the reference's engines drive them
(inference_videolcm_entrance.py:171-255, inference_sr600_entrance.py:256-280, inference_higen_entrance.py:197-236):
  videolcm  UNetSD_VideoLCM 16f 448x256, 4 LCM steps (no CFG) + 16-frame decode per prompt, one prompt per GPU
  sr600     UNetSD_SR600 32f 1280x720: 30 DDIM-inversion steps + 30 DPM-Solver++(2M) SDE CFG steps + 32-frame decode
  higen     UNetSD_HiGen 448x256: stage 1 (1 frame, 50 CFG DDIM steps) + stage 2 (32 frames, 50 CFG steps) + decode

Prints ONE JSON line on rank 0 (contract in the task statement): value = whole-job steps/s with inputs resident in
HBM; e2e = the same through the public DIFFUSION/MODEL API with HOST (pinned) buffers, H2D/D2H inside the timed
region; roofline for the dominant kernel family (tapgemm, tensor-bound); cpu_baseline = the oracle (CPU port of the
reference) on a bounded sample; gpu_eager_baseline = the oracle on THIS GPU under fp16 autocast (the reference's
PyTorch-eager path with flash SDPA standing in for xformers -- the "beat this" number of SURVEY.md section 8d).
`--impl reference` times the CPU oracle alone (the reference ships no CPU or Blackwell path of its own; DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

_FULL_UNET = dict(in_dim=4, dim=320, y_dim=1024, context_dim=1024, out_dim=4, dim_mult=[1, 2, 4, 4], num_heads=8,
                  head_dim=64, num_res_blocks=2, attn_scales=[1.0, 0.5, 0.25], dropout=0.1, temporal_attention=True,
                  temporal_attn_times=1, use_checkpoint=True, use_fps_condition=False, use_sim_mask=False)
VAE_KW = dict(ddconfig=dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
                            ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0), embed_dim=4)
DDIM_COSINE = dict(schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                   mean_type="v", var_type="fixed_small", loss_type="mse", noise_strength=0.1)
DDIM_LINEAR_SD = dict(schedule="linear_sd", schedule_param=dict(num_timesteps=1000, init_beta=0.00085, last_beta=0.012,
                                                                 zero_terminal_snr=True),
                      mean_type="v", var_type="fixed_small", loss_type="mse", noise_strength=0.1)

# Algorithmic work per denoise step, SURVEY.md section 8d (reference op count, FLOP = 2 MAC).
WORKLOADS = {
    "i2vgen": dict(name="i2vgen_xl_16f_1280x704_ddim_cfg", kind="i2vgen", cls="UNetSD_I2VGen", ctor=dict(_FULL_UNET, concat_dim=4),
                   latent=(1, 4, 16, 88, 160), step_tflop=176.19, fwd_per_step=2, frame_hw=(704, 1280), decode_frames=16,
                   decode_chunk=2, config="configs/i2vgen_xl_infer.yaml"),
    "videolcm": dict(name="videolcm_t2v_16f_448x256_lcm4", kind="videolcm", cls="UNetSD_VideoLCM",
                     ctor=dict(_FULL_UNET, concat_dim=8, num_tokens=4), latent=(1, 4, 16, 32, 56), step_tflop=8.667,
                     fwd_per_step=1, frame_hw=(256, 448), decode_frames=16, decode_chunk=2,
                     config="configs/videolcm_t2v_infer.yaml"),
    "sr600": dict(name="tft2v_sr600_32f_1280x720_dpmpp2m_sde_cfg", kind="sr600", cls="UNetSD_SR600", ctor=dict(_FULL_UNET),
                  latent=(1, 4, 32, 90, 160), step_tflop=2 * 185.3, fwd_per_step=2, frame_hw=(720, 1280), decode_frames=32,
                  decode_chunk=4, config="configs/tft2v_32frames_sr600_infer.yaml"),
    "higen": dict(name="higen_32f_448x256_stage2_ddim_cfg", kind="higen", cls="UNetSD_HiGen",
                  ctor=dict(_FULL_UNET, context_embedding_depth=2, num_tokens=16), latent=(1, 4, 32, 32, 56),
                  step_tflop=2 * 17.22, fwd_per_step=2, frame_hw=(256, 448), decode_frames=32, decode_chunk=2,
                  config="configs/higen_infer.yaml"),
}
LCM_CONFIG = dict(video_compositions=["text"], resolution=[448, 256])


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs"), "tflops": d.get("bf16_tflops_sustained") or d.get("bf16_tflops"),
                "source": "MEASURED_PEAKS.json (bf16_tflops_sustained: kernel timed inside a long step)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._th = None

    def _loop(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.25)

    def __enter__(self):
        self._th = threading.Thread(target=self._loop, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=6)

    def summary(self):
        sm = sorted(float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for nm, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def synth_conditioning(wl, seed, device):
    """SURVEY.md section 8d synthetic inputs (CPU generator, then moved): unit-scale text tokens etc."""
    b, c, f, h, w = wl["latent"]
    g = torch.Generator().manual_seed(seed)
    host = dict(y=torch.randn(1, 77, 1024, generator=g), y_neg=torch.randn(1, 77, 1024, generator=g))
    if wl["kind"] == "i2vgen":
        host["image"] = torch.randn(1, 1, 1024, generator=g)
        host["local_image"] = (0.18215 * torch.randn(1, 4, 1, h, w, generator=g)).repeat(1, 1, f, 1, 1).contiguous()
        host["fps"] = torch.tensor([16], dtype=torch.long)
    host["noise"] = torch.randn(1, 4, f, h, w, generator=g)
    if wl["kind"] == "higen":   # inference_higen_entrance.py:197-229 (motion_factor 500, appearance_factor 1.0)
        host["spat_noise"] = torch.randn(1, 4, 1, h, w, generator=g)
        sim = torch.cat([torch.linspace(0.0, 1.0, f)[:-1], torch.linspace(1.0, 0.0, f)])
        host["appearance"] = torch.stack([sim[i:i + f] for i in range(len(sim) - f, -1, -1)])[None].contiguous()
        host["motion"] = torch.tensor([[500] * (f - 1)], dtype=torch.long)
    if device is None:
        return host
    return {k: v.to(device) for k, v in host.items()}


def usable_cpus():
    """Cores this process may actually run on: affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the host's cores, and oversubscribed OpenMP threads crawl)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt[0] != "max":
            n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
    except Exception:  # noqa: BLE001
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:  # noqa: BLE001
            pass
    return max(1, min(n, 64))


# ------------------------------------------------------------------------------------------------
# oracle plumbing (cpu_baseline, --impl reference, gpu_eager_baseline): the ONLY places bench.py touches oracle/
def _oracle_forward(kind):
    from oracle import vgen_oracle as vo
    return {"i2vgen": vo.unet_i2vgen_forward, "videolcm": vo.unet_videolcm_forward, "sr600": vo.unet_sr600_forward,
            "higen": vo.unet_higen_forward}[kind]


def _oracle_kwargs(kind, c, f, neg=False):
    """Keyword arguments of one oracle / model call from a conditioning dict (cond or uncond branch)."""
    y = c["y_neg"] if neg else c["y"]
    if kind == "i2vgen":
        return dict(y=y, image=torch.zeros_like(c["image"]) if neg else c["image"], local_image=c["local_image"], fps=c["fps"])
    if kind == "higen":
        return dict(y=y, spat_prior=c["spat_prior"], motion_cond=c["motion"], appearance_cond=c["appearance"])
    return dict(y=y)


_CPU_CACHE = {}
# latents the CPU sample may use, smallest first; the largest whose CFG step fits the budget is taken
_CPU_LADDER = [(2, 16, 16), (4, 32, 32), (4, 48, 80), (8, 48, 80), (8, 88, 160), (16, 88, 160)]


def _cpu_oracle_setup(wl_key, threads):
    """Full-size weights for the CPU oracle (values are irrelevant for timing: a 16M-value random base is tiled with
    per-tensor scales, generated in ~1 s instead of 15 s of randn)."""
    if wl_key in _CPU_CACHE:
        return _CPU_CACHE[wl_key]
    from vgen_b200 import arch
    wl = WORKLOADS[wl_key]
    torch.set_num_threads(threads)
    spec = arch.unet_spec(arch.unet_plan(wl["kind"], **wl["ctor"]))
    base = torch.randn(1 << 24, generator=torch.Generator().manual_seed(0))
    sd = {}
    off = 0
    for name, shape in spec:
        n = 1
        for d in shape:
            n *= d
        fan = n // shape[0] if len(shape) > 1 else 1
        reps = (n + base.numel() - 1) // base.numel()
        if reps > 1:
            flat = base.repeat(reps)[:n]
        else:
            st = (off * 7919) % (base.numel() - n + 1)
            flat = base[st:st + n]
        flat = flat * (fan ** -0.5 if len(shape) > 1 else 0.05)
        if len(shape) == 1 and name.endswith("weight"):
            flat = flat + 1.0
        sd[name] = flat.reshape(shape).contiguous()
        off += n
    _CPU_CACHE[wl_key] = dict(sd=sd, spec=spec, flops={})
    return _CPU_CACHE[wl_key]


def _cpu_inputs(wl, f, h, w, device="cpu"):
    gi = torch.Generator().manual_seed(1)
    c = dict(y=torch.randn(1, 77, 1024, generator=gi), y_neg=torch.randn(1, 77, 1024, generator=gi))
    if wl["kind"] == "i2vgen":
        c.update(image=torch.randn(1, 1, 1024, generator=gi), local_image=torch.randn(1, 4, f, h, w, generator=gi), fps=torch.tensor([16]))
    if wl["kind"] == "higen":
        c.update(spat_prior=torch.randn(1, 4, h, w, generator=gi), appearance=torch.rand(1, f, 32, generator=gi),
                 motion=torch.full((1, max(f - 1, 1)), 500, dtype=torch.long) if f > 1 else torch.zeros(1, dtype=torch.long))
    x = torch.randn(1, 4, f, h, w, generator=gi)
    return x, {k: v.to(device) for k, v in c.items()}


def _forward_flops(wl_key, f, h, w):
    """Algorithmic FLOPs of one oracle forward at this latent, counted on meta tensors."""
    from torch.utils.flop_counter import FlopCounterMode
    c = _cpu_oracle_setup(wl_key, usable_cpus())
    if (f, h, w) in c["flops"]:
        return c["flops"][(f, h, w)]
    wl = WORKLOADS[wl_key]
    fwd = _oracle_forward(wl["kind"])
    msd = {n: torch.empty(s, device="meta") for n, s in c["spec"]}
    x, kw = _cpu_inputs(wl, f, h, w, "meta")
    with torch.no_grad(), FlopCounterMode(display=False) as fc:
        fwd(msd, torch.empty(x.shape, device="meta"), torch.empty(1, device="meta", dtype=torch.long), **_oracle_kwargs(wl["kind"], kw, f))
    c["flops"][(f, h, w)] = float(fc.get_total_flops())
    return c["flops"][(f, h, w)]


def cpu_oracle_sample(wl_key="i2vgen", budget_s=20.0, threads=None, max_reps=4, cpu_tflops_hint=None):
    """Time the oracle (CPU restatement of the reference, fp32, all usable host cores) on a bounded sample of the
    workload: CFG denoise steps of the SAME 1.4 B-parameter architecture at the LARGEST latent of a ladder whose step
    fits the budget, scaled to the metric's unit by algorithmic FLOPs (the ratio to the full config is stated)."""
    threads = threads or usable_cpus()
    wl = WORKLOADS[wl_key]
    c = _cpu_oracle_setup(wl_key, threads)
    fwd = _oracle_forward(wl["kind"])
    nf = wl["fwd_per_step"]
    t = torch.tensor([500])
    full_f = wl["latent"][2]
    # UNetSD_SR600's (2,1)-padded down / row-cropped up-sampling round-trips only for heights 8k+2 (unet_sr600.py:151-153)
    ladder = [(min(f, full_f), h + 2 if wl["kind"] == "sr600" else h, w) for f, h, w in _CPU_LADDER
              if h <= wl["latent"][3] and w <= wl["latent"][4]]
    # probe the smallest latent to learn this host's throughput (counts as the warm-up), then pick the rung
    f0, h0, w0 = ladder[0]
    x, kw = _cpu_inputs(wl, f0, h0, w0)
    with torch.no_grad():
        t0 = time.perf_counter()
        fwd(c["sd"], x, t, **_oracle_kwargs(wl["kind"], kw, f0))
        probe_s = time.perf_counter() - t0
    rate = cpu_tflops_hint or (_forward_flops(wl_key, f0, h0, w0) / probe_s / 1e12)
    pick = ladder[0]
    for rung in ladder:
        if nf * _forward_flops(wl_key, *rung) / 1e12 / max(rate, 1e-3) <= 0.6 * budget_s:
            pick = rung
    f, h, w = pick
    x, kw = _cpu_inputs(wl, f, h, w)
    flops = _forward_flops(wl_key, f, h, w)
    with torch.no_grad():
        t0 = time.perf_counter()
        n = 0
        while True:
            for neg in ([False, True] if nf == 2 else [False]):
                fwd(c["sd"], x, t, **_oracle_kwargs(wl["kind"], kw, f, neg))
            n += 1
            if time.perf_counter() - t0 > budget_s or n >= max_reps:
                break
        dt = time.perf_counter() - t0
    tflops = nf * n * flops / dt / 1e12
    ratio = nf * flops / 1e12 / wl["step_tflop"]
    return {"value": tflops / wl["step_tflop"], "unit": "denoise-steps/s", "cores": threads, "kind": "port",
            "sample": f"{n} denoise step(s) ({nf} forward(s) each) of {wl['cls']}, full 1.4B-param architecture, fp32 oracle, latent "
                      f"[1,4,{f},{h},{w}] ({flops / 1e12:.3f} TFLOP/forward = {ratio:.4f} of the {wl['step_tflop']} TFLOP step of "
                      f"{wl['name']}) in {dt:.1f}s = {tflops:.3f} TFLOP/s; scaled to the full step by algorithmic FLOPs",
            "cpu_tflops": tflops, "sample_latent": [1, 4, f, h, w], "sample_fraction_of_step": ratio}


def cpu_oracle_sample_subprocess(wl_key, budget_s=20.0, timeout_s=300):
    """Run the CPU baseline in a child process with a hard timeout so it can never stall the bench."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-sample", str(budget_s), "--workload", wl_key],
                           capture_output=True, text=True, timeout=timeout_s)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"error": "no output", "stderr": r.stderr[-400:]}
    except subprocess.TimeoutExpired:
        return {"error": f"timeout after {timeout_s}s"}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    total_budget = 170.0
    per = max(4.0, min(30.0, total_budget / max(1, args.steps + args.warmup)))
    hint = None
    for _ in range(max(1, min(args.warmup, 2))):
        hint = cpu_oracle_sample(args.workload, budget_s=per / 2, max_reps=1)["cpu_tflops"]
    vals = []
    t0 = time.perf_counter()
    last = None
    for _ in range(args.steps):
        last = cpu_oracle_sample(args.workload, budget_s=per, max_reps=2, cpu_tflops_hint=hint)
        vals.append(last["value"])
    dt = time.perf_counter() - t0
    v = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": "denoise_steps_per_s", "value": v, "unit": "denoise-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v if v > 0 else None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "note": "CPU oracle (port of the reference's PyTorch path; the reference has no "
                       "CPU/Blackwell path of its own); each step = a bounded sample at a reduced latent, FLOP-scaled",
                       "sample_latent": last["sample_latent"], "sample_fraction_of_step": last["sample_fraction_of_step"]},
            "cpu_baseline": dict(last, value=v), "e2e": {"value": v, "unit": "denoise-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": dt}
    print(json.dumps(line), flush=True)
    return 0


def gpu_eager_baseline(wl_key, model, cond, dev, steps=2):
    """The reference's PyTorch-eager GPU path on THIS GPU: the oracle (pinned to the reference) under
    torch.autocast(fp16) -- cuBLAS / cuDNN / flash SDPA, fp32 master weights cast per op as autocast does -- for
    `steps` denoise steps of the workload (same shapes, same weights).  An extra key, not the reference arm."""
    wl = WORKLOADS[wl_key]
    fwd = _oracle_forward(wl["kind"])
    sd = {k: v for k, v in model.state_dict().items()}        # the module's own device-resident fp32 masters (no copy)
    nf = wl["fwd_per_step"]
    f = wl["latent"][2]
    x = cond["noise"].clone()
    t = torch.full((1,), 481, dtype=torch.long, device=dev)

    def step():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            outs = [fwd(sd, x, t, **_oracle_kwargs(wl["kind"], cond, f, neg)) for neg in ([False, True] if nf == 2 else [False])]
        return outs
    try:
        step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            o = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {"value": 1000.0 / ms, "unit": "denoise-steps/s", "ms_per_step": ms, "steps": steps, "finite": bool(torch.isfinite(o[0]).all()),
                "what": f"oracle (reference restatement) on cuda under torch.autocast(fp16), {nf} forward(s)/step, flash SDPA, "
                        f"torch {torch.__version__}; UNet forwards only (no sampler update)"}
    except Exception as e:  # noqa: BLE001 - a comparator must never take the bench down
        return {"error": repr(e)[:300]}
    finally:
        del sd
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------
def ncu_traffic(kernels):
    """DRAM bytes per launch of a kernel family, from the committed ncu launch list of this same command
    (profiles/<tag>_traffic.json, written by tools/ncu_summary.py); None when no capture is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None
    try:
        d = json.load(open(files[-1]))
        hit = [k for k in d if k.startswith(tuple(kernels))]       # template instantiations share the prefix
        n = sum(d[k]["launches"] for k in hit)
        b = sum(d[k]["launches"] * (d[k]["dram_read_bytes_per_launch"] + d[k]["dram_write_bytes_per_launch"]) for k in hit)
        if n == 0 or b == 0:
            return None
        return {"bytes_per_launch": b / n, "source": "profiles/" + os.path.basename(files[-1])}
    except Exception:  # noqa: BLE001
        return None


def build_model(wl, registry, rank, dev):
    """Random-init weights of the real architecture; every zero-initialised tensor (proj_out, ...) is randomised on
    rank 0 so no branch multiplies by zero; the other ranks receive the packed arena over NCCL."""
    torch.manual_seed(1234)
    cfg = dict(type=wl["cls"], **wl["ctor"])
    if wl["kind"] == "videolcm":
        cfg["config"] = dict(LCM_CONFIG)
    model = registry.build(cfg)
    if rank == 0:
        g = torch.Generator().manual_seed(4321)
        for _, p in model.named_parameters():
            if float(p.detach().abs().sum()) == 0.0:
                p.data.normal_(0, 0.02, generator=g)
    return model.to(dev).eval()


def build_vae(registry, dev):
    vae = registry.build(dict(type="AutoencoderKL", **VAE_KW))
    gv = torch.Generator().manual_seed(99)
    for p in vae.parameters():
        if p.dim() > 1:
            p.data.normal_(0, (p[0].numel()) ** -0.5, generator=gv)
    return vae.to(dev).eval()


def timed(fn, dev, parallel):
    """CUDA-event time of fn() on the current stream (ms), max over ranks."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    parallel.barrier()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return parallel.max_over_ranks(e0.elapsed_time(e1), dev), r


def decode_video(vae, lat, chunk, keep=False):
    """video_data = latents / scale_factor; chunks of decoder_bs frames through AutoencoderKL.decode
    (inference_i2vgen_entrance.py:222-230).  keep: return all frames as [1, 3, f, H, W] (the tensor the engines hand to
    save_i2vgen_video_safe) instead of the last chunk."""
    z = (lat / 0.18215)[0].permute(1, 0, 2, 3).contiguous()
    z = torch.nan_to_num(z).clamp(-10, 10)         # random-weight latents may blow up; values are irrelevant for timing
    out, frames = None, []
    for i in range(0, z.shape[0], chunk):
        out = vae.decode(z[i:i + chunk])
        if keep:
            frames.append(out)
    if keep:
        return torch.cat(frames, dim=0).permute(1, 0, 2, 3).unsqueeze(0).contiguous()
    return out


def write_out_video(frames):
    """Frames to bytes to file through the drop-in writer (vgen_b200.video_io, utils/video_op.py:167-213): device kernel +
    pinned D2H timed with CUDA events, the encoder (ffmpeg pipe or OpenCV) with the host clock."""
    import tempfile

    from vgen_b200 import video_io
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    host, band, ev = video_io.frames_to_host(frames, [0.5] * 3, [0.5] * 3)
    e1.record()
    ev.synchronize()
    torch.cuda.synchronize()
    n = video_io.select_frames(host, band)
    res = {"frames": int(n), "bytes_d2h": int(host.numel()), "ms_kernel_plus_d2h": e0.elapsed_time(e1)}
    t0 = time.perf_counter()
    try:
        with tempfile.TemporaryDirectory() as td:
            path = video_io._encode(os.path.join(td, "bench.mp4"), host[:n].numpy(), 8)
            res["file_bytes"] = os.path.getsize(path)
        res["ms_encode_host"] = (time.perf_counter() - t0) * 1e3
    except Exception as e:  # noqa: BLE001 - no encoder on the box: the bytes still left the GPU
        res["encode_error"] = repr(e)[:160]
    return res


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32.  Weights and inputs are seeded, so the same arguments give the
    same inputs on every run and two builds can be compared output for output.  The largest latent (sr600,
    [1,4,32,90,160]) is 7.4 MB, well under the 64 MB a dump may take."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def ops_lincomb(terms):
    from vgen_b200 import ops
    return ops.lincomb_f32(terms)


class Stepper:
    """One denoise step of a workload through the public sampler classes, the way its engine calls them."""

    def __init__(self, wl_key, model, dev, cond, DIFFUSION):
        import vgen_b200
        self.wl, self.k, self.model, self.dev, self.c = WORKLOADS[wl_key], wl_key, model, dev, cond
        kind = self.wl["kind"]
        f = self.wl["latent"][2]
        if kind == "i2vgen":
            self.diff = DIFFUSION.build(dict(type="DiffusionDDIM", **DDIM_COSINE))
            self.kw = [_oracle_kwargs(kind, cond, f), _oracle_kwargs(kind, cond, f, True)]
            self.steps = [int(s) for s in self.diff.ddim_steps(50)]
        elif kind == "higen":
            self.diff = DIFFUSION.build(dict(type="DiffusionDDIM", **DDIM_LINEAR_SD))
            cond["spat_prior"] = torch.zeros(1, 4, *self.wl["latent"][3:], device=dev)
            self.kw = [_oracle_kwargs(kind, cond, f), _oracle_kwargs(kind, cond, f, True)]
            self.steps = [int(s) for s in self.diff.ddim_steps(50)]
        elif kind == "videolcm":
            self.sched = vgen_b200.LCMScheduler(prediction_type="v_prediction", beta_schedule="scaled_linear", clip_sample=False,
                                                timestep_spacing="linspace", rescale_betas_zero_snr=True)
            self.sched.set_timesteps(4, device=dev)
            self.kw = _oracle_kwargs(kind, cond, f)
        elif kind == "sr600":
            self.diff = DIFFUSION.build(dict(
                type="DiffusionDDIMSR",
                reverse_diffusion=dict(schedule="cosine", mean_type="v", schedule_param=dict(num_timesteps=1000, zero_terminal_snr=True)),
                forward_diffusion=dict(schedule="logsnr_cosine_interp", mean_type="v",
                                       schedule_param=dict(num_timesteps=1000, zero_terminal_snr=True, scale_min=2.0, scale_max=4.0))))
            self.kw = [_oracle_kwargs(kind, cond, f), _oracle_kwargs(kind, cond, f, True)]

    def step(self, xt, i):
        kind = self.wl["kind"]
        if kind in ("i2vgen", "higen"):
            s = self.steps[i % len(self.steps)]
            t = torch.full((1,), s, dtype=torch.long, device=self.dev)
            return self.diff._ddim_step(xt, s, t, self.model, self.kw, 9.0 if kind == "i2vgen" else 12.0, 50, 0.0)[0]
        if kind == "videolcm":
            if i % 4 == 0:
                self.sched._step_index = None
            t = self.sched.timesteps[i % 4]
            out = self.model(self.sched.scale_model_input(xt, t), t.repeat(xt.size(0)).to(xt.dtype), t_w=None, **self.kw)
            return self.sched.step(out, t, xt, return_dict=False)[0]
        # sr600: one CFG denoise of the DPM-Solver++ loop (GaussianDiffusion.denoise at a fixed noise level, :163-247)
        fd = self.diff.forward_diffusion
        t = torch.full((1,), 400, dtype=torch.long, device=self.dev)
        x0 = fd.denoise(xt, t, None, self.model, self.kw, guide_scale=9.0, guide_rescale=0.3)[-2]
        return ops_lincomb([(0.9, xt), (0.1, x0)])       # a solver-update-sized kernel that keeps the latent's scale

    def full_video(self, vae):
        """One whole prompt the way the engine runs it (sampling + decode); returns (latent, frames)."""
        kind, c, wl = self.wl["kind"], self.c, self.wl
        if kind == "i2vgen":
            lat = self.diff.ddim_sample_loop(c["noise"].clone(), self.model, self.kw, guide_scale=9.0, ddim_timesteps=50, eta=0.0)
        elif kind == "videolcm":
            self.sched.set_timesteps(4, device=self.dev)
            lat = c["noise"].clone()
            for t in self.sched.timesteps:
                out = self.model(self.sched.scale_model_input(lat, t), t.repeat(1).to(lat.dtype), t_w=None, **self.kw)
                lat = self.sched.step(out, t, lat, return_dict=False)[0]
        elif kind == "sr600":
            rev = self.diff.reverse_diffusion.ddim_reverse_sample_loop(x0=c["noise"] * 0.18215, model=self.model,
                                                                      model_kwargs={"y": c["y_neg"]}, ddim_timesteps=30, reverse_steps=700)
            lat = self.diff.forward_diffusion.sample(noise=rev, model=self.model, model_kwargs=self.kw, guide_scale=9.0,
                                                     guide_rescale=0.3, solver="dpmpp_2m_sde", steps=30, t_max=699, t_min=0,
                                                     discretization="trailing")
        else:  # higen: spatial stage (1 frame) then temporal stage (32 frames)
            f = wl["latent"][2]
            spat_kw = [dict(y=c["y"], spat_prior=c["spat_prior"], motion_cond=torch.zeros(1, dtype=torch.long, device=self.dev),
                            appearance_cond=torch.ones(1, 1, f, device=self.dev)),
                       dict(y=c["y_neg"], spat_prior=c["spat_prior"], motion_cond=torch.zeros(1, dtype=torch.long, device=self.dev),
                            appearance_cond=torch.ones(1, 1, f, device=self.dev))]
            spat = self.diff.ddim_sample_loop(c["spat_noise"].clone(), self.model, spat_kw, guide_scale=12.0, ddim_timesteps=50, eta=0.0)
            vae.decode((spat.squeeze(2) / 0.18215).clamp(-10, 10))
            kw = [dict(k, spat_prior=torch.nan_to_num(spat.squeeze(2)).clamp(-10, 10)) for k in self.kw]
            lat = self.diff.ddim_sample_loop(c["noise"].clone(), self.model, kw, guide_scale=12.0, ddim_timesteps=50, eta=0.0)
        return lat, decode_video(vae, lat, wl["decode_chunk"], keep=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="i2vgen", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=float, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg (profiling runs only: the line then has no e2e value)")
    ap.add_argument("--full-video", type=int, default=None, help="time one whole prompt (sampling + decode); default: on except i2vgen")
    ap.add_argument("--profile-pass", type=int, default=1, help="run one instrumented step for the roofline line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the latent the last timed step returned (rank 0) as DIR/latent.npy, float32")
    args = ap.parse_args()

    if args.cpu_sample is not None:
        print(json.dumps(cpu_oracle_sample(args.workload, budget_s=args.cpu_sample)), flush=True)
        return 0
    from vgen_b200 import parallel
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        return run_reference_arm(args, rank, int(os.environ.get("WORLD_SIZE", "1")))

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: vgen_b200 has no CPU path"}))
        return 1
    wl = WORKLOADS[args.workload]
    rank, world, local_rank = parallel.init_from_env("nccl")
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    import vgen_b200
    from vgen_b200 import graph, lib, ops
    MODEL, DIFFUSION, AUTO_ENCODER = vgen_b200.register(force_local=True)
    model = build_model(wl, MODEL, rank, dev)
    # one-time weight distribution: the packed fp16 arena over NCCL / NVLink (timed on the device, untimed for the metric)
    model.packed_tensors()
    bc_ms, bcast_bytes = timed(lambda: parallel.broadcast_packed(model, src=0), dev, parallel)
    c = synth_conditioning(wl, 8888 + rank, dev)
    stepper = Stepper(args.workload, model, dev, c, DIFFUSION)

    xt = c["noise"].clone()
    for i in range(args.warmup):
        xt = stepper.step(xt, i)
    torch.cuda.synchronize()
    parallel.barrier()

    # ---- timed: K steps, inputs resident in HBM, CUDA events on the launching stream
    l0 = lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        torch.cuda.synchronize()
        ev0.record()
        for i in range(args.steps):
            xt = stepper.step(xt, args.warmup + i)
        ev1.record()
        torch.cuda.synchronize()
    launches_eager = lib.launch_count() - l0
    gstats = graph.stats(model)
    ms = ev0.elapsed_time(ev1)
    parallel.barrier()
    ms_max = parallel.max_over_ranks(ms, dev)
    finite = bool(torch.isfinite(xt).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"latent": xt})

    # ---- e2e: same step through the public API from HOST (pinned) buffers, H2D + D2H inside the timed region
    host = synth_conditioning(wl, 8888 + rank, None)
    cond_keys = [k for k in host if k not in ("noise", "spat_noise")]
    pinned = {k: v.pin_memory() for k, v in host.items()}
    xt_host = pinned["noise"].clone().pin_memory()
    out_host = torch.empty_like(xt_host).pin_memory()
    h2d = sum(pinned[k].numel() * pinned[k].element_size() for k in cond_keys) + xt_host.numel() * 4
    d2h = out_host.numel() * 4

    def e2e_step(i):
        d = {k: pinned[k].to(dev, non_blocking=True) for k in cond_keys}
        for k in c:
            if k not in d:
                d[k] = c[k]
        x = xt_host.to(dev, non_blocking=True)
        st = Stepper.__new__(Stepper)
        st.__dict__.update(stepper.__dict__)
        f = wl["latent"][2]
        if isinstance(stepper.kw, list):
            st.kw = [_oracle_kwargs(wl["kind"], d, f), _oracle_kwargs(wl["kind"], d, f, True)]
        else:
            st.kw = _oracle_kwargs(wl["kind"], d, f)
        x = st.step(x, i)
        out_host.copy_(x, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        xt_host.copy_(torch.nan_to_num(out_host).clamp_(-1e4, 1e4))

    n_e2e = max(2, min(args.steps, 4))
    e2e_ms = None
    if not args.no_e2e:
        e2e_step(0)
        e2e_ms, _ = timed(lambda: [e2e_step(1 + i) for i in range(n_e2e)], dev, parallel)

    # ---- decode: AutoencoderKL.decode in chunks of decoder_bs frames
    decode = None
    vae = None
    if not args.no_decode:
        vae = build_vae(AUTO_ENCODER, dev)
        decode_video(vae, xt[:, :, :3 * wl["decode_chunk"]], wl["decode_chunk"])     # warm-up: pack, sighting, graph capture
        nfr = min(wl["decode_frames"], xt.shape[2])
        dms, img = timed(lambda: decode_video(vae, xt[:, :, :nfr], wl["decode_chunk"]), dev, parallel)
        decode = {"frames_per_s": world * nfr / (dms / 1e3), "ms": dms, "frames": nfr, "frame_hw": list(wl["frame_hw"]),
                  "chunk": wl["decode_chunk"], "dtype": "f16 activations / f32 accumulate", "finite": bool(torch.isfinite(img).all())}
        del img

    # ---- whole prompt (sampling + decode), the engines' end-to-end unit
    full = None
    want_full = args.full_video if args.full_video is not None else int(args.workload != "i2vgen")
    if want_full and vae is not None:
        if args.workload in ("videolcm",):
            stepper.full_video(vae)                  # cheap: warm once so the timed prompt replays graphs
        fms, (lat, frames) = timed(lambda: stepper.full_video(vae), dev, parallel)
        nfr = wl["decode_frames"] + (1 if args.workload == "higen" else 0)
        wo = write_out_video(frames)
        full = {"videos_per_s": world / (fms / 1e3), "s_per_video": fms / 1e3, "frames_per_s_e2e": world * nfr / (fms / 1e3),
                "write_out": wo,
                "prompts": world, "finite": bool(torch.isfinite(lat).all()),
                "what": {"i2vgen": "50 CFG DDIM steps + 16-frame decode", "videolcm": "4 LCM steps + 16-frame decode (8 chunks x 2)",
                         "sr600": "30 DDIM-inversion steps + 30 DPM-Solver++(2M) SDE CFG steps + 32-frame decode",
                         "higen": "stage 1: 50 CFG steps @1 frame + key-frame decode; stage 2: 50 CFG steps @32 frames + 32-frame decode"}[args.workload]}
        del lat, frames
    del vae
    torch.cuda.empty_cache()

    # ---- instrumented pass: per-kernel-family device time (CUDA events around every launch; graphs bypassed)
    roofline = None
    families = None
    launches_step = None
    if args.profile_pass and rank == 0:
        ops.PROF = ops.KernelProfile()
        l1 = lib.launch_count()
        xt2 = stepper.step(xt, 0)
        launches_step = lib.launch_count() - l1
        summ = ops.PROF.summary()
        ops.PROF = None
        del xt2
        families = {k: {"launches": v["launches"], "ms": round(v["ms"], 3), "tflops": round(v["flops"] / 1e9 / max(v["ms"], 1e-9), 1) if v["flops"] else None,
                        "gbs": round(v["bytes"] / 1e6 / max(v["ms"], 1e-9), 1)} for k, v in summ.items()}
        tg = summ.get("tapgemm")
        pk = measured_peaks()
        if tg:
            ach = tg["flops"] / (tg["ms"] / 1e3) / 1e12
            roofline = {"kernel": "tapgemm_sm100_kernel (conv3x3 / temporal conv / linear, tcgen05)", "bound": "tensor",
                        "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"], "traffic": None,
                        "launches_per_step": tg["launches"], "avg_launch_ms": tg["ms"] / tg["launches"],
                        "algorithmic_tflop_per_step": tg["flops"] / 1e12, "peak_source": pk["source"]}
            tr = ncu_traffic(("tapgemm_sm100_2cta_kernel", "tapgemm_sm100_kernel")) if args.workload == "i2vgen" else None
            if tr:
                roofline["traffic"] = tr["bytes_per_launch"]
                roofline["traffic_unit"] = "DRAM bytes / launch (dram__bytes_read.sum + dram__bytes_write.sum)"
                roofline["traffic_source"] = tr["source"]
                roofline["algorithmic_bytes_per_launch"] = tg["bytes"] / tg["launches"]

    # kernels of OUR library executed inside the timed region: launches issued directly + graph replays x kernels per graph
    replays = sum(v[1] for v in gstats.values())
    launches = launches_eager
    if launches_step is not None and replays:
        launches = launches_step * args.steps       # every step replays the captured forward(s): same kernels as the eager step
    value = world * args.steps / (ms_max / 1e3)
    line = {"metric": "denoise_steps_per_s", "value": value, "unit": "denoise-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": wl["name"], "reference_config": wl["config"], "latent": list(wl["latent"]),
                       "forwards_per_step": wl["fwd_per_step"], "cfg_batched": wl["fwd_per_step"] == 2,
                       "l2": "inputs larger than L2 (2.8 GB of weights stream from HBM every forward)",
                       "parallelism": f"{world} independent trajectories (no data-path collective)",
                       "cuda_graph": {"enabled": graph.enabled(), "captures_replays": gstats,
                                      "launches_issued_from_python_in_timed_region": launches_eager},
                       "weight_broadcast": {"bytes": bcast_bytes, "ms": bc_ms, "what": "packed fp16 arena, NCCL, flat 256 MB buckets"}},
            "e2e": {"value": world * n_e2e / (e2e_ms / 1e3) if e2e_ms else None, "unit": "denoise-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clk.summary(), "finite": finite,
            "tflops_effective": value * wl["step_tflop"] / world, "decode": decode, "full_video": full, "roofline": roofline,
            "kernel_families": families}
    if rank == 0 and not args.no_eager_baseline:
        line["gpu_eager_baseline"] = gpu_eager_baseline(args.workload, model, c, dev)
    if rank == 0 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_oracle_sample_subprocess(args.workload, budget_s=20.0)
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    parallel.barrier()
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
