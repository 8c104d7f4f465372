"""Host-side logic that needs no GPU: parameter specs, strict state_dict compatibility, registry
contract, DDIM host math (bit-exact), C-ABI surface, multi-process sharding/broadcast over gloo."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import vgen_b200
from oracle import synth, vgen_oracle as vo
from oracle.cases import CASES, FULL_CTORS
from _helpers import build_product
from vgen_b200 import arch, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gold_spec(golden_dir, name):
    return [(k, tuple(s)) for k, s in json.load(open(os.path.join(golden_dir, f"{name}.spec.json")))]


@pytest.mark.parametrize("name", list(CASES) + list(FULL_CTORS))
def test_param_spec_equals_reference(golden_dir, name):
    kind, ctor = (CASES[name]["kind"], CASES[name]["ctor"]) if name in CASES else FULL_CTORS[name]
    if kind == "vae":
        mine = arch.vae_spec(arch.vae_plan(ctor["ddconfig"], ctor["embed_dim"]))
    else:
        mine = arch.unet_spec(arch.unet_plan(kind, **ctor))
    assert mine == _gold_spec(golden_dir, name)       # names, shapes AND registration order


def test_full_size_tensor_counts(golden_dir):
    assert len(_gold_spec(golden_dir, "full_t2v")) == 1480
    assert len(_gold_spec(golden_dir, "full_i2vgen")) == 1509      # SURVEY.md section 8b
    assert len(_gold_spec(golden_dir, "full_vae")) == 248
    assert len(_gold_spec(golden_dir, "full_videolcm")) == 1480 and len(_gold_spec(golden_dir, "full_sr600")) == 1480
    assert len(_gold_spec(golden_dir, "full_higen")) == 1535


@pytest.mark.parametrize("name", list(CASES))
def test_strict_state_dict_roundtrip(golden_dir, name):
    case = CASES[name]
    m = build_product(case)
    spec = _gold_spec(golden_dir, name)
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == spec
    sd = synth.state_dict(spec, seed=case["seed"])
    m.load_state_dict(sd, strict=True)
    assert torch.equal(m.state_dict()[spec[5][0]], sd[spec[5][0]])
    assert any(p.requires_grad for p in m.parameters())          # DistributedDataParallel needs one
    bad = dict(sd)
    bad.pop(spec[0][0])
    with pytest.raises(RuntimeError):
        m.load_state_dict(bad, strict=True)


def test_registry_contract():
    M, D, A = vgen_b200.register(force_local=True)
    case = CASES["t2v_tiny"]
    # YAML dicts carry extra keys (upper_len, default_fps, misc_dropout ...): constructors must swallow them
    m = M.build(dict(type="UNetSD_T2VBase", **case["ctor"], upper_len=128, default_fps=8, misc_dropout=0.4))
    assert type(m).__name__ == "UNetSD_T2VBase" and m.device.type == "cpu"
    with pytest.raises(KeyError):
        M.build(dict(type="NoSuchModel"))
    with pytest.raises(Exception, match="Failed to init class"):
        M.build(dict(type="UNetSD_T2VBase", **dict(case["ctor"], head_dim=32)))
    d = D.build(dict(type="DiffusionDDIM", schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                     mean_type="v", var_type="fixed_small", loss_type="mse", noise_strength=0.1))
    assert d.num_timesteps == 1000
    a = A.build(dict(type="AutoencoderKL", **CASES["vae_tiny"]["ctor"]))
    assert hasattr(a, "decode") and hasattr(a, "encode_firsr_stage")


def test_registers_into_reference_registry_when_available(monkeypatch):
    """With the reference's `utils.registry_class` importable (a stand-in module holding its four singletons here),
    register() fills those registries instead of the local mirror."""
    import types
    from vgen_b200 import registry
    host = types.ModuleType("utils.registry_class")
    for name in ("MODEL", "DIFFUSION", "AUTO_ENCODER", "EMBEDDER"):
        setattr(host, name, registry.Registry(name))
    monkeypatch.setitem(sys.modules, "utils", types.ModuleType("utils"))
    monkeypatch.setitem(sys.modules, "utils.registry_class", host)
    for name in ("MODEL", "DIFFUSION", "AUTO_ENCODER", "EMBEDDER", "USING_REFERENCE_REGISTRY"):
        monkeypatch.setattr(registry, name, getattr(registry, name))   # restored for the other tests in this process
    M, D, A = vgen_b200.register()
    assert M is host.MODEL and D is host.DIFFUSION and A is host.AUTO_ENCODER and registry.USING_REFERENCE_REGISTRY
    assert M.get("UNetSD_I2VGen") is vgen_b200.UNetSD_I2VGen and D.get("DiffusionDDIM") is vgen_b200.DiffusionDDIM
    assert A.get("AutoencoderKL") is vgen_b200.AutoencoderKL
    assert host.EMBEDDER.get("FrozenOpenCLIPEmbedder") is vgen_b200.clip.FrozenOpenCLIPEmbedder


def test_no_cpu_fallback():
    case = CASES["t2v_tiny"]
    m = vgen_b200.UNetSD_T2VBase(**case["ctor"])
    with pytest.raises(Exception, match="CUDA"):
        m(torch.zeros(1, 4, 2, 8, 8), torch.zeros(1, dtype=torch.long), y=torch.zeros(1, 5, 1024))
    v = vgen_b200.AutoencoderKL(**CASES["vae_tiny"]["ctor"])
    with pytest.raises(Exception, match="CUDA"):
        v.decode(torch.zeros(1, 4, 8, 8))


def test_product_never_imports_oracle():
    for fn in os.listdir(os.path.join(ROOT, "vgen_b200")):
        if fn.endswith(".py"):
            src = open(os.path.join(ROOT, "vgen_b200", fn)).read()
            assert "oracle" not in re.sub(r'""".*?"""', "", src, flags=re.S), fn


# ------------------------------------------------------------------------------------ DDIM host math
def test_ddim_tables_and_steps_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "schedules.npz"))
    d = vgen_b200.DiffusionDDIM(schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                                mean_type="v", var_type="fixed_small")
    assert np.array_equal(d.betas.numpy(), g["cosine_zsnr.betas"])
    assert np.array_equal(d.alphas_cumprod.numpy(), g["cosine_zsnr.alphas_cumprod"])
    d2 = vgen_b200.DiffusionDDIM(schedule="linear_sd", schedule_param=dict(num_timesteps=1000, init_beta=0.00085, last_beta=0.012, zero_terminal_snr=True),
                                 mean_type="v", var_type="fixed_small")
    assert np.array_equal(d2.alphas_cumprod.numpy(), g["linear_sd_zsnr.alphas_cumprod"])
    for S in (50, 4, 20):
        assert np.array_equal(d.ddim_steps(S).numpy(), g[f"steps_{S}"])


def test_ddim_step_coefficients_match_reference_formulas():
    d = vgen_b200.DiffusionDDIM(schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                                mean_type="v", var_type="fixed_small")
    tab = vo.ddim_tables(vo.make_betas("cosine", 1000, True, cosine_s=0.008))
    for S in (50, 4):
        stride = 1000 // S
        for step in d.ddim_steps(S).tolist():
            c = d.step_coefficients(step, S, 0.0)
            f32 = torch.float32
            a_prev = tab["alphas_cumprod"][max(step - stride, 0)].to(f32)
            want = [tab["sqrt_alphas_cumprod"][step].to(f32), tab["sqrt_one_minus_alphas_cumprod"][step].to(f32),
                    tab["sqrt_recip_alphas_cumprod"][step].to(f32), tab["sqrt_recipm1_alphas_cumprod"][step].to(f32),
                    torch.sqrt(a_prev), torch.sqrt(1 - a_prev), torch.tensor(0.0)]
            assert c == [float(w) for w in want]
    # last step uses alphas_cumprod[0], not 1 (diffusion_ddim.py:233)
    assert d.step_coefficients(1, 50, 0.0)[4] == float(torch.sqrt(tab["alphas_cumprod"][0].to(torch.float32)))
    with pytest.raises(NotImplementedError):
        d.ddim_sample(torch.zeros(1, 4, 1, 2, 2), torch.tensor([1]), lambda *a, **k: None, {}, clamp=1.0)


# ------------------------------------------------------------------------------------ C ABI surface
def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "vgen_b200.h")).read()
    declared = set(re.findall(r"\b(vgen_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(lib.declared_symbols()), declared ^ set(lib.declared_symbols())
    dll = ctypes.CDLL(str(lib.LIB_PATH))
    for name in declared:
        assert hasattr(dll, name), name
    l = lib.load()
    assert l.vgen_abi_version() == 2
    # the launch counter is per process and GPU tests that ran earlier in this process have launched kernels: read it in a fresh one
    code = f"import sys; sys.path.insert(0, {ROOT!r}); from vgen_b200 import lib; print(lib.load().vgen_launch_count())"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == "0", r.stdout + r.stderr[-2000:]
    assert l.vgen_set_tapgemm_impl(7) != 0 and b"impl" in l.vgen_last_error()
    assert l.vgen_set_tapgemm_impl(0) == 0
    assert l.vgen_group_norm_workspace_bytes(2) > 0
    assert ctypes.sizeof(lib.Epilogue) == 80       # struct vgen_epilogue layout (x86-64 SysV; ABI 2 added row_stats, col_sum)


# ------------------------------------------------------------------------------------ multi-process (gloo)
_WORKER = r'''
import os, sys, torch
sys.path.insert(0, %r)
import torch.distributed as dist
from vgen_b200 import parallel
import vgen_b200
from oracle.cases import CASES
rank, world, _ = parallel.init_from_env("gloo")
torch.manual_seed(100 + rank)                       # every rank starts from DIFFERENT weights
m = vgen_b200.AutoencoderKL(**CASES["vae_tiny"]["ctor"])
for p in m.parameters():
    p.data.normal_()
nbytes = parallel.broadcast_parameters(m, src=0, bucket_bytes=1 << 20)
chk = torch.cat([p.data.reshape(-1) for p in m.parameters()]).double().sum()
allc = [torch.zeros_like(chk) for _ in range(world)]
dist.all_gather(allc, chk)
assert all(float(c) == float(allc[0]) for c in allc), allc
assert nbytes == sum(p.numel() * 4 for p in m.parameters())
# packed-arena broadcast (what the GPU path ships: fp16 GEMM matrices + fp32 vectors), here on a stand-in module whose
# "packed" tensors live on the CPU (the real _pack() needs a CUDA device): mixed dtypes, several buckets
class _Packed:
    def __init__(self, seed):
        g = torch.Generator().manual_seed(seed)
        self.t = [("a.w", torch.randn(300, 70, generator=g).half()), ("a.b", torch.randn(300, generator=g)),
                  ("b.w", torch.randn(1000, 129, generator=g).half()), ("c.b", torch.randn(7, generator=g))]
        self.offloaded = False
    def packed_tensors(self):
        return self.t
    def offload_masters(self):
        self.offloaded = True
pm = _Packed(500 + rank)
nb2 = parallel.broadcast_packed(pm, src=0, bucket_bytes=64 << 10, offload_masters=True)
ref = _Packed(500)
assert all(torch.equal(a[1], b[1]) for a, b in zip(pm.t, ref.t)), "every rank must hold rank 0's packed weights"
assert nb2 == sum(t.numel() * t.element_size() for _, t in ref.t) and pm.offloaded
prompts = [f"p{i}" for i in range(8)]
mine = parallel.shard_items(prompts, rank, world)
got = [None] * world
dist.all_gather_object(got, mine)
assert sorted(sum(got, [])) == sorted(prompts) and all(len(g) == 4 for g in got)
assert parallel.shard_items(prompts, rank, world, "replicate") == prompts
assert parallel.max_over_ranks(float(rank)) == float(world - 1)
parallel.barrier()
import os
os.write(1, f"RANK_OK_{rank}\n".encode())   # one write(2) per rank: lines of concurrent ranks cannot interleave
'''


def test_gloo_world2_broadcast_and_sharding(tmp_path):
    import socket
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % ROOT)
    with socket.socket() as sk:                      # a free port: back-to-back runs must not collide
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "RANK_OK_0" in r.stdout and "RANK_OK_1" in r.stdout


def test_gauss_host_math_is_bit_exact(golden_dir):
    """GaussianDiffusion host side (sigma tables, ladder, sigma<->t) against the oracle / the reference golden."""
    from oracle import gauss_oracle as go
    from oracle.cases import GAUSS_CASE as gc
    from vgen_b200 import diffusion_gauss as dg
    g = np.load(os.path.join(golden_dir, "gauss.npz"))
    d = dg.DiffusionDDIMSR(gc["schedules"]["reverse"], gc["schedules"]["forward"])
    assert np.array_equal(d.reverse_diffusion.sigmas.numpy(), g["sigmas.reverse"].astype(np.float32))
    assert np.array_equal(d.forward_diffusion.sigmas.numpy(), g["sigmas.forward"].astype(np.float32))
    assert d.reverse_diffusion.prediction_type == "v" and d.forward_diffusion.num_timesteps == 1000
    fwd, o = d.forward_diffusion, go.GaussOracle(torch.from_numpy(g["sigmas.forward"]), "v")
    for steps, disc in ((4, "trailing"), (30, "trailing"), (7, "linspace"), (5, "leading")):
        mine = fwd._sigma_ladder(steps, 599, 0, disc, True)
        ref = o.sample_sigmas(steps, 599, 0, disc, True)
        assert torch.equal(mine, ref), (steps, disc)
        for s in mine[:-1]:
            assert torch.equal(fwd._sigma_to_t(s), o.sigma_to_t(s))
    assert np.array_equal(fwd._sigma_ladder(4, 599, 0, "trailing", True)[:-1].numpy(), g["ladder"][:4])
    with pytest.raises(NotImplementedError):
        fwd.sample(torch.zeros(1, 4, 2, 4, 4), None, solver="heun")
    M, D, A = vgen_b200.register(force_local=True)
    assert D.get("DiffusionDDIMSR") is vgen_b200.DiffusionDDIMSR


def test_brownian_tree_increments_are_consistent():
    from vgen_b200.brownian import BrownianTree
    w0 = torch.zeros(4000)
    tr = BrownianTree(0.1, w0, 2.1, entropy=7)
    a, b, c = tr(0.5, 1.0), tr(1.0, 1.7), tr(0.5, 1.7)
    assert torch.allclose(a + b, c, atol=1e-6)
    tr2 = BrownianTree(0.1, w0, 2.1, entropy=7)                                 # same seed + same query order -> same path
    assert torch.equal(tr2(0.5, 1.0), a) and torch.equal(tr2(1.0, 1.7), b)
    assert abs(float(a.var()) - 0.5) < 0.05 and abs(float(b.var()) - 0.7) < 0.07 and abs(float((a * b).mean())) < 0.05


def test_lcm_scheduler_host_math():
    """LCMScheduler stand-in (diffusers is absent: parity unpinned): host tables and timestep selection
    against the oracle restatement and the documented properties of the algorithm."""
    from oracle import lcm_oracle as lo
    from vgen_b200.lcm import LCMScheduler
    s = LCMScheduler(prediction_type="v_prediction", beta_schedule="scaled_linear", clip_sample=False,
                     timestep_spacing="linspace", rescale_betas_zero_snr=True)
    s.set_timesteps(4, device="cpu")
    assert s.timesteps.tolist() == [999, 759, 499, 259] == lo.lcm_timesteps(4)
    assert torch.equal(s.alphas_cumprod, lo.alphas_cumprod(True))
    assert float(s.alphas_cumprod[999]) == 0.0 and 0.99 < float(s.alphas_cumprod[0]) < 1.0
    for t in (999, 259, 19):
        assert s.boundary_scalings(t) == pytest.approx(lo.boundary_scalings(float(t)), rel=1e-12)
    cs, co = s.boundary_scalings(0)
    assert cs == 1.0 and co == 0.0                      # consistency boundary condition f(x, 0) = x
    s.set_timesteps(8)
    assert s.timesteps.tolist() == lo.lcm_timesteps(8) and len(set(s.timesteps.tolist())) == 8
    assert torch.equal(s.scale_model_input(torch.ones(2)), torch.ones(2))


def test_cfg_forward_batches_only_when_safe(monkeypatch):
    """diffusion.cfg_forward (host logic): one batch-2b call for models that opt in and kwargs that can be stacked,
    otherwise the reference's two calls; outputs are split back in (cond, uncond) order."""
    from vgen_b200.diffusion import cfg_forward

    class Fake:
        cfg_batch = True

        def __init__(self):
            self.calls = []

        def __call__(self, x, t=None, **kw):
            self.calls.append((x.shape[0], sorted(kw), t.shape[0]))
            return x * 2 + kw["y"].sum(dim=(1, 2)).view(-1, 1, 1, 1, 1)

    x, t = torch.randn(1, 4, 2, 3, 3), torch.tensor([7])
    kc, ku = {"y": torch.ones(1, 5, 8), "fps": torch.tensor([8])}, {"y": torch.zeros(1, 5, 8), "fps": torch.tensor([8])}
    monkeypatch.setenv("VGEN_CFG_BATCH", "1")
    m = Fake()
    yo, uo = cfg_forward(m, x, t, [kc, ku])
    assert m.calls == [(2, ["fps", "y"], 2)]
    assert torch.equal(yo, x * 2 + 40) and torch.equal(uo, x * 2)
    m = Fake()
    cfg_forward(m, x, t, [kc, ku], by_keyword=True)            # GaussianDiffusion calls model(xt, t=t, **kw)
    assert m.calls == [(2, ["fps", "y"], 2)]
    m = Fake()
    cfg_forward(m, x, t, [kc, dict(ku, extra=torch.zeros(1))])  # different key sets -> the reference's two calls
    assert [c[0] for c in m.calls] == [1, 1]
    m = Fake()
    cfg_forward(m, x, t, [dict(kc, y=torch.ones(1, 6, 8)), ku])  # shapes that cannot be stacked
    assert [c[0] for c in m.calls] == [1, 1]
    monkeypatch.setenv("VGEN_CFG_BATCH", "0")
    m = Fake()
    cfg_forward(m, x, t, [kc, ku])
    assert [c[0] for c in m.calls] == [1, 1]
    m = Fake()
    m.cfg_batch = False                                          # e.g. a reference model passed to our sampler
    monkeypatch.setenv("VGEN_CFG_BATCH", "1")
    cfg_forward(m, x, t, [kc, ku])
    assert [c[0] for c in m.calls] == [1, 1]


def test_fastdiv_multiply_shift_is_exact():
    """Mirror of make_fastdiv / fd_div (vgen_b200/csrc/tapgemm.h): the tile-index decomposition of the persistent
    kernels must be exact for every divisor and every 31-bit numerator it can meet."""
    rng = np.random.default_rng(0)

    def make(d):
        if d == 1:
            return 0, 0
        lg = int(np.ceil(np.log2(d)))
        while (1 << lg) < d:
            lg += 1
        while lg > 0 and (1 << (lg - 1)) >= d:
            lg -= 1
        p = 31 + lg
        return ((1 << p) + d - 1) // d, p - 32

    ds = list(range(1, 2000)) + [int(v) for v in rng.integers(2000, 1 << 20, 300)]
    xs = np.concatenate([np.arange(0, 5000), rng.integers(0, 1 << 31, 4000), np.array([(1 << 31) - 1])]).astype(np.uint64)
    for d in ds:
        mul, shr = make(d)
        assert mul < (1 << 32)
        q = xs if d == 1 else ((xs * np.uint64(mul)) >> np.uint64(32)) >> np.uint64(shr)
        assert np.array_equal(q, xs // np.uint64(d)), d


def test_clip_spec_and_tokenizer(golden_dir, monkeypatch):
    """CLIP conditioning host side: parameter spec == open_clip's CLIP.state_dict() (names, shapes, order), embedders are
    registered, and -- index work, bit-exact -- tokenizer ids == the ids the reference's vendored tokenizer produced
    (tests/golden/clip_tiny.npz, oracle_pin.npz), with the merge list cut down to the merges those strings meet."""
    from oracle.make_golden_clip import PROMPTS, TINY
    from oracle.make_golden_pin import TOKENIZER_EXTRA
    from vgen_b200 import clip, clip_tokenizer as ct, registry
    spec = [(k, tuple(s)) for k, s in json.load(open(os.path.join(golden_dir, "clip_tiny.spec.json")))]
    assert clip.clip_spec(TINY) == spec
    full = clip.clip_spec(clip.ARCHS["ViT-H-14"])
    assert len(full) == 686 and sum(int(np.prod(s)) for _, s in full) == 986109441      # open_clip ViT-H-14
    vgen_b200.register(force_local=True)
    assert {"FrozenOpenCLIPEmbedder", "FrozenOpenCLIPVisualEmbedder", "FrozenOpenCLIPTextVisualEmbedder"} <= set(registry.EMBEDDER.class_map)
    e = clip.FrozenOpenCLIPTextVisualEmbedder(None, arch=TINY, layer="penultimate")
    assert e.layer_idx == 1 and all(k.startswith("model.") for k in e.state_dict()) and len(e.state_dict()) == len(spec)
    assert not any(p.requires_grad for p in e.parameters())
    with pytest.raises(lib.VgenError):
        e.model.text_tokens(torch.zeros(1, 77, dtype=torch.long))              # CPU: no fallback
    bpe = os.path.join(golden_dir, "clip_bpe_subset.txt.gz")
    monkeypatch.setenv("VGEN_CLIP_BPE", bpe)
    monkeypatch.setattr(ct, "_DEFAULT", None)
    assert ct.find_bpe_file() == bpe
    g = np.load(os.path.join(golden_dir, "clip_tiny.npz"))
    assert np.array_equal(ct.tokenize(PROMPTS).numpy(), g["tokens"])
    assert np.array_equal(ct.tokenize(TOKENIZER_EXTRA).numpy(), np.load(os.path.join(golden_dir, "oracle_pin.npz"))["clip.extra_tokens"])


def test_layer_norm_fold_algebra():
    """ops.fold_layer_norm (host side of vgen_epilogue.row_stats / col_sum): rstd (x w'^T) - mean rstd col_sum + bias' equals
    LayerNorm -> Linear, including rows whose mean dwarfs their spread (the constant part cancels exactly because col_sum is
    taken from the ROUNDED weights), and survives the GEGLU row interleave."""
    import torch
    from vgen_b200 import ops
    g = torch.Generator().manual_seed(11)
    m, k, n = 64, 320, 96
    x = (torch.randn(m, k, generator=g) * 1.5 + 6.0 * torch.randn(m, 1, generator=g)).half()
    w, b = torch.randn(n, k, generator=g) * k ** -0.5, torch.randn(n, generator=g)
    gam, bet = 1.0 + 0.3 * torch.randn(k, generator=g), 0.2 * torch.randn(k, generator=g)
    ref = torch.nn.functional.layer_norm(x.double(), (k,), gam.double(), bet.double(), 1e-5) @ w.double().t() + b.double()
    wf, cs, lb = ops.fold_layer_norm(w, b, gam, bet)
    assert wf.dtype == torch.float16 and cs.dtype == torch.float32 and lb.dtype == torch.float32
    xd = x.double()
    mean = xd.mean(1, keepdim=True)
    rstd = (xd.var(1, unbiased=False, keepdim=True) + 1e-5).rsqrt()
    got = rstd * (xd @ wf.double().t()) + (-mean * rstd) * cs.double()[None, :] + lb.double()[None, :]
    assert float((got - ref).abs().max() / ref.abs().max()) < 1e-3
    # a constant row is mapped to bias' exactly
    const = torch.full((1, k), 3.0, dtype=torch.float64)
    got_c = (1e-5 ** -0.5) * (const @ wf.double().t()) + (-3.0 * 1e-5 ** -0.5) * cs.double()[None, :] + lb.double()[None, :]
    assert float((got_c - lb.double()[None, :]).abs().max()) < 1e-2       # 316 * fp32 rounding of col_sum
    # GEGLU: fold first, then interleave rows; col_sum of the packed rows follows the same permutation as the bias
    wp, bp = ops.pack_geglu_weight(w * gam[None, :], b + w @ bet, 32)
    wp16 = wp.half()
    perm_cs = wp16.double().sum(1)
    wp_ref, cs_ref = ops.pack_geglu_weight(wf.float(), cs, 32)
    assert torch.equal(wp_ref.half(), wp16) and torch.allclose(perm_cs.float(), cs_ref, rtol=0, atol=1e-6)
