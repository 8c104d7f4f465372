"""TEST INFRASTRUCTURE ONLY -- freeze what tests/test_oracle_pin.py and the tokenizer check compare against.

Those tests pin the oracle to the reference classes on cases the other golden files do not cover (weight seeds
77-80, the fps-condition branch, HiGen's per-frame motion branch, the default initialisation, the DDIM tables) and
the CLIP tokenizer to the reference's vendored tokenizer.  This script runs the reference once (it needs the
reference tree, see oracle/refload.py) and stores its outputs, so the tests run without it:

    python -m oracle.make_golden_pin

  * oracle_pin.npz           reference outputs / tables, keyed as the tests read them
  * {t2v,videolcm}_tiny_fps.spec.json   parameter specs of the use_fps_condition=True models
  * clip_bpe_subset.txt.gz   the CLIP merge list (1.3 MB) cut down to the merges the tokenizer meets on the test
                             strings; every other line is a placeholder pair that no text can produce, so line
                             numbers -- and hence token ids -- are those of the full list.  Greedy BPE only ever
                             merges the lowest-ranked pair present, so keeping every merge that was looked up and
                             found gives the same pieces as the full list; checked below with the reference
                             tokenizer itself.
"""
from __future__ import annotations

import gzip
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import refload, synth, vgen_oracle as vo  # noqa: E402
from oracle.cases import CASES, make_inputs  # noqa: E402
from oracle.make_golden import GOLD, _maxrel, build_variant  # noqa: E402

VARIANTS = ["videolcm_tiny", "sr600_tiny", "higen_tiny", "higen_tiny_f1"]
TOKENIZER_EXTRA = ["", "naive cafe 42", "a " * 200, "UPPER lower MiXeD", "tab\tand\nnewline",
                   "emoji \U0001F680 日本語"]
BPE_PLACEHOLDER = "<unused> <unused>"


def _gold_spec(name):
    return [(k, tuple(s)) for k, s in json.load(open(os.path.join(GOLD, f"{name}.spec.json")))]


def higen_per_frame_motion(b, f):
    """motion_cond with one factor per frame (size(1) == f), the branch unet_higen.py:393-394 takes."""
    return torch.tensor([[100 + 37 * i + 11 * j for j in range(f)] for i in range(b)], dtype=torch.long)


def _reference_outputs(ref):
    from _helpers import oracle_call, product_call       # tests/_helpers.py: the reference call of each case
    out, specs = {}, {}
    case = CASES["t2v_tiny_b2"]
    m = ref.UNetSD_T2VBase(**case["ctor"]).eval()
    assert synth.spec_of(m) == _gold_spec("t2v_tiny_b2")
    sd = synth.state_dict(synth.spec_of(m), seed=77)
    m.load_state_dict(sd, strict=True)
    inp = make_inputs(case)
    out["t2v_tiny_b2.seed77"] = m(inp["x"], inp["t"], y=inp["y"])
    assert _maxrel(vo.unet_t2v_forward(sd, inp["x"], inp["t"], inp["y"]), out["t2v_tiny_b2.seed77"]) < 2e-5

    for name in VARIANTS:
        case = CASES[name]
        m = build_variant(ref, case["kind"], case["ctor"]).eval()
        assert synth.spec_of(m) == _gold_spec(name), name
        sd = synth.state_dict(synth.spec_of(m), seed=78)
        m.load_state_dict(sd, strict=True)
        inp = make_inputs(case)
        out[f"{name}.seed78"] = product_call(case, m, inp)
        assert _maxrel(oracle_call(case, sd, inp), out[f"{name}.seed78"]) < 2e-5, name

    case = CASES["t2v_tiny"]
    torch.manual_seed(0)
    m = ref.UNetSD_T2VBase(**case["ctor"]).eval()
    inp = make_inputs(case)
    out["t2v_tiny.default_init"] = m(inp["x"], inp["t"], y=inp["y"])

    case = CASES["higen_tiny"]
    m = build_variant(ref, "higen", case["ctor"]).eval()
    sd = synth.state_dict(synth.spec_of(m), seed=79)
    m.load_state_dict(sd, strict=True)
    inp = make_inputs(case)
    kw = dict(spat_prior=inp["spat_prior"], motion_cond=higen_per_frame_motion(inp["x"].shape[0], inp["x"].shape[2]),
              appearance_cond=inp["appearance_cond"])
    out["higen_tiny.motion_per_frame"] = m(inp["x"], inp["t"], y=inp["y"], **kw)
    assert _maxrel(vo.unet_higen_forward(sd, inp["x"], inp["t"], inp["y"], **kw), out["higen_tiny.motion_per_frame"]) < 2e-5

    for kind in ("t2v", "videolcm"):
        case = CASES[f"{kind}_tiny"]
        ctor = dict(case["ctor"], use_fps_condition=True)
        m = (ref.UNetSD_T2VBase(**ctor) if kind == "t2v" else build_variant(ref, "videolcm", ctor)).eval()
        specs[f"{kind}_tiny_fps"] = synth.spec_of(m)
        sd = synth.state_dict(synth.spec_of(m), seed=80)
        m.load_state_dict(sd, strict=True)
        inp = make_inputs(case)
        fps = torch.tensor([8] * inp["x"].shape[0], dtype=torch.long)
        out[f"{kind}_tiny.fps"] = m(inp["x"], inp["t"], y=inp["y"], fps=fps)

    d = ref.DiffusionDDIM(schedule="cosine", schedule_param=dict(num_timesteps=1000, cosine_s=0.008, zero_terminal_snr=True),
                          mean_type="v", var_type="fixed_small")
    for k in vo.ddim_tables(d.betas):
        out[f"ddim.{k}"] = getattr(d, k)
    return {k: v.numpy() for k, v in out.items()}, specs


def _tokenizer_golden():
    from oracle.make_golden_clip import PROMPTS, load_reference_open_clip
    from vgen_b200 import clip_tokenizer as ct
    _, tok_mod = load_reference_open_clip()
    full = tok_mod.default_bpe()
    texts = PROMPTS + TOKENIZER_EXTRA

    class _Found(dict):
        def get(self, key, default=None):
            r = dict.get(self, key, default)
            if r is not None:
                found.add(key)
            return r

    found = set()
    tok = ct.ClipTokenizer(full)
    tok.rank = _Found(tok.rank)
    want = tok(texts)
    lines = gzip.open(full).read().decode("utf-8").split("\n")[:1 + ct._N_MERGES]
    keep = [lines[0]] + [ln if tuple(ln.split()) in found else BPE_PLACEHOLDER for ln in lines[1:]]
    path = os.path.join(GOLD, "clip_bpe_subset.txt.gz")
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write("\n".join(keep).encode("utf-8"))
    ref_ids = tok_mod.tokenize(texts)
    assert torch.equal(want, ref_ids)
    full_tok, tok_mod._tokenizer = tok_mod._tokenizer, tok_mod.SimpleTokenizer(path)
    try:
        assert torch.equal(tok_mod.tokenize(texts), ref_ids), "the cut-down merge list changes the reference's ids"
    finally:
        tok_mod._tokenizer = full_tok
    assert torch.equal(ct.ClipTokenizer(path)(texts), ref_ids)
    print(f"clip_bpe_subset.txt.gz: {len(found)} merges kept, {os.path.getsize(path)} bytes", flush=True)
    return ref_ids[len(PROMPTS):].numpy()


def main():
    torch.set_grad_enabled(False)
    sys.path.insert(0, os.path.dirname(GOLD))
    ref = refload.load()
    arrays, specs = _reference_outputs(ref)
    arrays["clip.extra_tokens"] = _tokenizer_golden()
    np.savez_compressed(os.path.join(GOLD, "oracle_pin.npz"), **arrays)
    for name, spec in specs.items():
        with open(os.path.join(GOLD, f"{name}.spec.json"), "w") as fh:
            json.dump([[k, list(s)] for k, s in spec], fh)
    print("oracle_pin.npz:", {k: list(v.shape) for k, v in arrays.items()}, flush=True)


if __name__ == "__main__":
    main()
