"""Direct pin of the oracle against the real reference classes, on cases the other golden files do not cover (weight
seeds the golden files do not use, the fps-condition and per-frame-motion branches, the default initialisation, the DDIM
tables).  The reference's outputs are stored in tests/golden/oracle_pin.npz (oracle/make_golden_pin.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import synth, vgen_oracle as vo
from oracle.cases import CASES, make_inputs
from oracle.make_golden_pin import higen_per_frame_motion


@pytest.fixture(scope="module")
def pin(golden_dir):
    return np.load(os.path.join(golden_dir, "oracle_pin.npz"))


def _spec(golden_dir, name):
    return [(k, tuple(s)) for k, s in json.load(open(os.path.join(golden_dir, f"{name}.spec.json")))]


def _maxrel(a, b):
    b = torch.from_numpy(b)
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def test_unet_t2v_against_reference_class(golden_dir, pin):
    torch.set_grad_enabled(False)
    case = CASES["t2v_tiny_b2"]
    sd = synth.state_dict(_spec(golden_dir, "t2v_tiny_b2"), seed=77)          # a seed the golden files do not use
    inp = make_inputs(case)
    assert _maxrel(vo.unet_t2v_forward(sd, inp["x"], inp["t"], inp["y"]), pin["t2v_tiny_b2.seed77"]) < 2e-5


@pytest.mark.parametrize("name", ["videolcm_tiny", "sr600_tiny", "higen_tiny", "higen_tiny_f1"])
def test_unet_variants_against_reference_classes(golden_dir, pin, name):
    """a21 variants, with weights from a seed the golden files do not use."""
    from _helpers import oracle_call
    torch.set_grad_enabled(False)
    case = CASES[name]
    sd = synth.state_dict(_spec(golden_dir, name), seed=78)
    inp = make_inputs(case)
    assert _maxrel(oracle_call(case, sd, inp), pin[f"{name}.seed78"]) < 2e-5


def test_default_init_is_degenerate_and_synth_is_not(golden_dir, pin):
    """SURVEY.md section 8c hygiene: with the reference's default init the output is a per-channel constant."""
    torch.set_grad_enabled(False)
    out = torch.from_numpy(pin["t2v_tiny.default_init"])
    assert float(out.std(dim=(2, 3, 4)).max()) < 1e-6
    case = CASES["t2v_tiny"]
    inp = make_inputs(case)
    sd = synth.state_dict(_spec(golden_dir, "t2v_tiny"), seed=case["seed"])
    assert float(vo.unet_t2v_forward(sd, inp["x"], inp["t"], inp["y"]).std()) > 0.1


def test_ddim_tables_against_reference_class(pin):
    tab = vo.ddim_tables(vo.make_betas("cosine", 1000, True, cosine_s=0.008))
    for k, v in tab.items():
        assert torch.equal(v, torch.from_numpy(pin[f"ddim.{k}"])), k


def test_higen_motion_cond_per_frame_branch(golden_dir, pin):
    """get_motion_embedding with motion_cond.size(1) == f (no interpolation), unet_higen.py:393-394."""
    torch.set_grad_enabled(False)
    case = CASES["higen_tiny"]
    sd = synth.state_dict(_spec(golden_dir, "higen_tiny"), seed=79)
    inp = make_inputs(case)
    mc = higen_per_frame_motion(inp["x"].shape[0], inp["x"].shape[2])
    kw = dict(spat_prior=inp["spat_prior"], motion_cond=mc, appearance_cond=inp["appearance_cond"])
    assert _maxrel(vo.unet_higen_forward(sd, inp["x"], inp["t"], inp["y"], **kw), pin["higen_tiny.motion_per_frame"]) < 2e-5


@pytest.mark.parametrize("kind", ["t2v", "videolcm"])
def test_fps_condition_branch(golden_dir, pin, kind):
    """use_fps_condition=True adds fps_embedding(sinusoidal(fps)) to the time embedding (unet_t2v.py:246-249)."""
    torch.set_grad_enabled(False)
    case = CASES["t2v_tiny" if kind == "t2v" else "videolcm_tiny"]
    ctor = dict(case["ctor"], use_fps_condition=True)
    spec = _spec(golden_dir, f"{kind}_tiny_fps")
    sd = synth.state_dict(spec, seed=80)
    inp = make_inputs(case)
    fps = torch.tensor([8] * inp["x"].shape[0], dtype=torch.long)
    fn = vo.unet_t2v_forward if kind == "t2v" else vo.unet_videolcm_forward
    assert _maxrel(fn(sd, inp["x"], inp["t"], inp["y"], fps=fps, use_fps_condition=True), pin[f"{kind}_tiny.fps"]) < 2e-5
    # and the product's parameter spec follows the flag
    from vgen_b200 import arch
    kk = dict(ctor, dim_mult=tuple(ctor["dim_mult"]), attn_scales=tuple(ctor["attn_scales"]))
    assert arch.unet_spec(arch.unet_plan(kind, **kk)) == spec
