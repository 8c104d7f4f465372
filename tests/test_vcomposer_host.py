"""Host-side checks of the VideoComposer path (UNetSD_VideoLCM / UNetSD_TFT2V with condition adapters): the oracle
against the reference goldens, parameter specs and strict checkpoint loading, registration, constructor limits, and the
CFG batching of shared condition tensors."""
import json
import os

import numpy as np
import pytest
import torch

import vgen_b200
from oracle import synth
from vgen_b200 import diffusion
from vcomposer_oracle import VCOMPOSER_CASES, cond_kwargs, config, ctor, make_vcomposer_inputs, resolution, unet_vcomposer_forward


def _spec(golden_dir, name):
    return [(k, tuple(s)) for k, s in json.load(open(os.path.join(golden_dir, f"{name}.spec.json")))]


def _build(case):
    return getattr(vgen_b200, case["cls"])(config=config(case), **ctor(case))


@pytest.mark.parametrize("name", sorted(VCOMPOSER_CASES))
def test_oracle_matches_reference_golden(golden_dir, name):
    case = VCOMPOSER_CASES[name]
    sd = synth.state_dict(_spec(golden_dir, name), seed=case["seed"])
    inp = make_vcomposer_inputs(case)
    with torch.no_grad():
        out = unet_vcomposer_forward(sd, inp["x"], inp["t"], inp["y"], resolution(case), **cond_kwargs(inp))
    gold = torch.from_numpy(np.load(os.path.join(golden_dir, f"{name}.npz"))["out"])
    assert float((out - gold).abs().max() / gold.abs().max()) <= 1e-5


@pytest.mark.parametrize("name", sorted(VCOMPOSER_CASES))
def test_param_spec_and_strict_load(golden_dir, name):
    case = VCOMPOSER_CASES[name]
    gold = _spec(golden_dir, name)
    m = _build(case)
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == gold
    sd = synth.state_dict(gold, seed=case["seed"])
    m.load_state_dict(sd, strict=True)
    back = m.state_dict()
    assert all(torch.equal(back[k], sd[k]) for k in sd)
    missing = dict(sd)
    missing.pop(next(k for k in sd if "_embedding_after." in k or k.startswith("pre_image_condition.")))
    with pytest.raises(RuntimeError):
        m.load_state_dict(missing, strict=True)


def test_inpainting_false_keeps_only_the_mask_transformer():
    case = dict(VCOMPOSER_CASES["vc_tft2v_all"], inpainting=False)
    keys = _build(case).state_dict().keys()
    assert not any(k.startswith("masked_embedding.") for k in keys)
    assert any(k.startswith("mask_embedding_after.") for k in keys)


def test_text_only_spec_unchanged(golden_dir):
    """video_compositions == ['text'] builds exactly the parameters the text-to-video VideoLCM always had."""
    case = VCOMPOSER_CASES["vc_tft2v_textimg"]
    m = vgen_b200.UNetSD_VideoLCM(config=dict(video_compositions=["text"], resolution=[448, 256]), **ctor(case))
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == _spec(golden_dir, "videolcm_tiny")


def test_register_maps_tft2v():
    from vgen_b200 import registry
    M, _, _ = registry.register(force_local=True)
    assert M.get("UNetSD_TFT2V") is vgen_b200.UNetSD_TFT2V
    assert M.get("UNetSD_VideoLCM") is vgen_b200.UNetSD_VideoLCM
    assert issubclass(vgen_b200.UNetSD_TFT2V, vgen_b200.UNetSD_VideoLCM)


@pytest.mark.parametrize("cls", ["UNetSD_VideoLCM", "UNetSD_TFT2V"])
def test_constructor_rejects_unsupported(cls):
    kw = ctor(VCOMPOSER_CASES["vc_tft2v_all"])
    with pytest.raises(NotImplementedError):
        getattr(vgen_b200, cls)(config=dict(video_compositions=["text", "histogram"], resolution=[96, 64]), **kw)
    with pytest.raises(NotImplementedError):
        getattr(vgen_b200, cls)(config=dict(video_compositions=["text"], resolution=[96, 64], use_text_clip_vip_model=True), **kw)


class _FakeModel:
    """Records the calls cfg_forward makes; returns x + 0 so the halves can be told apart."""
    cfg_batch = True

    def __init__(self, shared):
        if shared is not None:
            self.cfg_shared_kwargs = shared
        self.calls = []

    def __call__(self, x, t, **kw):
        self.calls.append((x.shape[0], {k: (v.shape[0] if torch.is_tensor(v) else v) for k, v in kw.items()}))
        return x.clone()


def test_cfg_forward_shared_kwargs():
    x, t = torch.randn(1, 4, 2, 3, 3), torch.tensor([5])
    depth = torch.rand(1, 1, 2, 24, 24)
    same_value = depth.clone()
    kc = {"y": torch.randn(1, 3, 8), "depth": depth, "sketch": same_value}
    ku = {"y": torch.randn(1, 3, 8), "depth": depth, "sketch": same_value.clone()}
    m = _FakeModel(frozenset({"depth", "sketch"}))
    a, b = diffusion.cfg_forward(m, x, t, [kc, ku])
    assert m.calls == [(2, {"y": 2, "depth": 1, "sketch": 2})]   # shared object passed once; equal values still concatenated
    assert torch.equal(a, x) and torch.equal(b, x)


def test_cfg_forward_without_shared_kwargs_is_unchanged():
    x, t = torch.randn(1, 4, 2, 3, 3), torch.tensor([5])
    depth = torch.rand(1, 1, 2, 24, 24)
    kc, ku = {"y": torch.randn(1, 3, 8), "depth": depth}, {"y": torch.randn(1, 3, 8), "depth": depth}
    m = _FakeModel(None)
    diffusion.cfg_forward(m, x, t, [kc, ku])
    assert m.calls == [(2, {"y": 2, "depth": 2})]
