"""TEST INFRASTRUCTURE ONLY -- freeze outputs of the REAL reference UNetSD_VideoLCM / UNetSD_TFT2V with condition
adapters into tests/golden/ (the cases of tests/vcomposer_oracle.py).

Run where the reference is mounted (it never reaches the GPU machines):

    python tools/make_golden_vcomposer.py

For every case it builds the reference class on CPU with the case's video_compositions, loads a synthetic state_dict
made by oracle/synth.py from the reference's own (name, shape) list, runs the reference forward in fp32, checks the
restatement tests/vcomposer_oracle.py:unet_vcomposer_forward against it and stores the parameter spec and the output.
A case with `ddim` also runs the reference's DiffusionDDIM.ddim_sample_loop with CFG, the unconditional branch reusing
the same condition tensors and passing zeros_like(image), like inference_tft2v_vcomposer_entrance.py:457-501.
"""
from __future__ import annotations

import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import refload, synth, vgen_oracle as vo  # noqa: E402
from vcomposer_oracle import (VCOMPOSER_CASES, cond_kwargs, config, ctor, make_vcomposer_inputs, resolution,  # noqa: E402
                              unet_vcomposer_forward)

GOLD = os.path.join(ROOT, "tests", "golden")


def _maxrel(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def reference_class(ref, name):
    if name == "UNetSD_TFT2V":
        return importlib.import_module("tools.modules.unet.unet_tf2tv").UNetSD_TFT2V
    return ref.UNetSD_VideoLCM


def uncond_kwargs(inp):
    kw = dict(cond_kwargs(inp), y=inp["y_neg"])
    if "image" in kw:
        kw["image"] = torch.zeros_like(inp["image"])
    return kw


def main():
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    ref = refload.load()
    from easydict import EasyDict
    report = {}
    for cname, case in VCOMPOSER_CASES.items():
        m = reference_class(ref, case["cls"])(config=EasyDict(**config(case)), **ctor(case)).eval()
        spec = synth.spec_of(m)
        sd = synth.state_dict(spec, seed=case["seed"])
        m.load_state_dict(sd, strict=True)
        inp = make_vcomposer_inputs(case)
        res = resolution(case)
        ck = cond_kwargs(inp)
        out = m(inp["x"], inp["t"], y=inp["y"], **ck)
        mine = unet_vcomposer_forward(sd, inp["x"], inp["t"], inp["y"], res, **ck)
        err = _maxrel(mine, out)
        assert err < 1e-5, (cname, err)
        arrays, extra = {"out": out.numpy()}, {}
        if case.get("ddim"):
            dd = case["ddim"]
            diff = ref.DiffusionDDIM(schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                                     mean_type="v", var_type="fixed_small")
            kw = [dict(ck, y=inp["y"]), uncond_kwargs(inp)]
            torch.manual_seed(123)
            lat = diff.ddim_sample_loop(inp["x"].clone(), m, kw, guide_scale=dd["guide_scale"], ddim_timesteps=dd["steps"], eta=0.0)
            betas = vo.make_betas("cosine", 1000, True, cosine_s=0.008)
            fn = lambda xt, t, **k: unet_vcomposer_forward(sd, xt, t, res=res, **k)  # noqa: E731
            torch.manual_seed(123)
            mine_lat = vo.ddim_sample_loop(inp["x"].clone(), fn, kw, betas, dd["guide_scale"], dd["steps"])
            e2 = _maxrel(mine_lat, lat)
            assert e2 < 1e-5, (cname, "ddim", e2)
            arrays["ddim_latent"] = lat.numpy()
            extra["ddim_err"] = e2
        np.savez_compressed(os.path.join(GOLD, f"{cname}.npz"), **arrays)
        with open(os.path.join(GOLD, f"{cname}.spec.json"), "w") as fh:
            json.dump([[k, list(s)] for k, s in spec], fh)
        report[cname] = {"oracle_vs_reference_maxrel": err, "tensors": len(spec), **extra}
        print(cname, report[cname], flush=True)
    with open(os.path.join(GOLD, "vc_REPORT.json"), "w") as fh:
        json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
