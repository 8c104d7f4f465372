"""Tensor-level wrappers over the C ABI: they check shapes/dtypes, allocate outputs with torch
(device memory plumbing only) and pass raw pointers + the current CUDA stream to libvgen_b200.so.

Layout convention: activations fp16 channels-last ("rows x channels"); weights fp16 [out][taps*in];
bias / affine parameters fp32.
"""
from __future__ import annotations

import ctypes

import torch

from . import lib as _l
from .lib import Epilogue


class KernelProfile:
    """Optional per-kernel-family device timing (CUDA events on the launching stream) + algorithmic
    work counters.  Used by bench.py for the roofline line; off by default (PROF is None)."""

    def __init__(self):
        self.records = []  # (family, flops, bytes, start_event, stop_event)

    def run(self, family, flops, nbytes, fn, tag=None):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = fn()
        e.record()
        self.records.append((family, float(flops), float(nbytes), s, e, tag))
        return rc

    def by_shape(self):
        torch.cuda.synchronize()
        out = {}
        for fam, fl, nb, s, e, tag in self.records:
            d = out.setdefault(f"{fam}:{tag}", {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            d["launches"] += 1
            d["ms"] += s.elapsed_time(e)
            d["flops"] += fl
            d["bytes"] += nb
        return out

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for fam, fl, nb, s, e, _tag in self.records:
            d = out.setdefault(fam, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            d["launches"] += 1
            d["ms"] += s.elapsed_time(e)
            d["flops"] += fl
            d["bytes"] += nb
        return out


PROF = None  # set to a KernelProfile() to instrument calls


def _run(family, flops, nbytes, fn, tag=None):
    if PROF is None:
        return fn()
    return PROF.run(family, flops, nbytes, fn, tag)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk16(t, name):
    if t.dtype != torch.float16 or not t.is_cuda:
        raise _l.VgenError(f"{name}: expected a CUDA fp16 tensor, got {t.dtype} on {t.device}")


def _rows_view(t, name):
    """(rows, ld) of a tensor whose last dim is contiguous and whose leading dims are row-dense."""
    if t.stride(-1) != 1:
        raise _l.VgenError(f"{name}: innermost dimension must be contiguous")
    t2 = t.reshape(-1, t.shape[-1]) if t.is_contiguous() else t
    if t2.dim() != 2:
        raise _l.VgenError(f"{name}: non-contiguous tensors must be 2-D row views")
    return t2, t2.stride(0)


def _epilogue(n_out, bias=None, group_bias=None, residual=None, alpha=1.0, geglu=False, bn=0, group_div=1, ln=None):
    e = Epilogue()
    e.alpha = float(alpha)
    keep = []
    if ln is not None:   # (row_stats [rows, 2] fp32, col_sum [n] fp32): LayerNorm folded into the GEMM
        stats, col_sum = ln
        if stats.dtype != torch.float32 or col_sum.dtype != torch.float32 or not stats.is_contiguous() or not col_sum.is_contiguous():
            raise _l.VgenError("ln: row_stats and col_sum must be contiguous fp32 tensors")
        if residual is not None or group_bias is not None:
            raise _l.VgenError("ln: a folded LayerNorm cannot be combined with residual / group_bias")
        e.row_stats = stats.data_ptr()
        e.col_sum = col_sum.data_ptr()
        keep += [stats, col_sum]
    if bias is not None:
        if bias.dtype != torch.float32:
            raise _l.VgenError("bias must be fp32")
        e.bias = bias.data_ptr()
        keep.append(bias)
    if group_bias is not None:
        _chk16(group_bias, "group_bias")
        e.group_bias = group_bias.data_ptr()
        e.group_bias_ld = group_bias.stride(0)
        e.group_bias_div = int(group_div)
        keep.append(group_bias)
    if residual is not None:
        _chk16(residual, "residual")
        r2, ldr = _rows_view(residual, "residual")
        if r2.shape[-1] != n_out:
            raise _l.VgenError(f"residual has {r2.shape[-1]} columns, expected {n_out}")
        e.residual = r2.data_ptr()
        e.residual_ld = ldr
        keep.append(r2)
    e.geglu = 1 if geglu else 0
    e.bn = int(bn)
    return e, keep


def linear(a, w, bias=None, residual=None, alpha=1.0, geglu=False, out=None, bn=0, ln=None):
    """out[m, n] = epi(a[m, k] @ w[n, k]^T).  `a` may be a row-strided 2-D view.

    ln = (row_stats(a), col_sum): `a` is the INPUT of a LayerNorm whose affine part was folded into w / bias
    (fold_layer_norm); the epilogue applies the per-row statistics, so LN(a) is never materialised."""
    _chk16(a, "a"), _chk16(w, "w")
    lead = a.shape[:-1]
    a2, lda = _rows_view(a, "a")
    m, k = a2.shape
    n = w.shape[0]
    if w.shape[1] != k or not w.is_contiguous():
        raise _l.VgenError(f"linear: weight {tuple(w.shape)} does not match k={k}")
    n_out = n // 2 if geglu else n
    if out is None:
        out = torch.empty(*lead, n_out, device=a.device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    if ln is not None and (ln[0].shape != (m, 2) or ln[1].numel() != n):
        raise _l.VgenError(f"linear: ln shapes {tuple(ln[0].shape)} / {tuple(ln[1].shape)} do not match m={m}, n={n}")
    e, keep = _epilogue(n_out, bias, None, residual, alpha, geglu, bn, ln=ln)
    rc = _run("tapgemm", 2.0 * m * n * k, 2.0 * (m * k + n * k + m * n_out),
              lambda: _l.load().vgen_linear(_p(a2), m, k, lda, _p(w), n, _p(o2), ldo, ctypes.byref(e), _stream()),
              tag=f"linear m{m} k{k} n{n}{' geglu' if geglu else ''}{' res' if residual is not None else ''}{' ln' if ln is not None else ''}")
    _l.check(rc, "vgen_linear")
    return out


def conv2d_3x3(x, w, bias=None, group_bias=None, residual=None, out=None, bn=0, group_div=1):
    """x [nimg, h, w, c] fp16 -> [nimg, h, w, n]; w [n, 9*c] with k = (ky*3+kx)*c + ci."""
    _chk16(x, "x"), _chk16(w, "w")
    if not x.is_contiguous() or x.dim() != 4:
        raise _l.VgenError("conv2d_3x3: x must be contiguous [nimg,h,w,c]")
    nimg, h, wd, c = x.shape
    n = w.shape[0]
    if w.shape[1] != 9 * c or not w.is_contiguous():
        raise _l.VgenError(f"conv2d_3x3: weight {tuple(w.shape)} does not match c={c}")
    if out is None:
        out = torch.empty(nimg, h, wd, n, device=x.device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    e, keep = _epilogue(n, bias, group_bias, residual, 1.0, False, bn, group_div)
    rows = nimg * h * wd
    rc = _run("tapgemm", 2.0 * rows * n * 9 * c, 2.0 * (rows * c + 9 * c * n + rows * n),
              lambda: _l.load().vgen_conv2d_3x3(_p(x), nimg, h, wd, c, _p(w), n, _p(o2), ldo, ctypes.byref(e), _stream()),
              tag=f"conv3x3 {nimg}x{h}x{wd} c{c} n{n}")
    _l.check(rc, "vgen_conv2d_3x3")
    return out


def tconv3(x, w, bias=None, residual=None, out=None, bn=0):
    """x [f, hw, c] (one video) or [b, f, hw, c] (videos back to back) fp16 -> same with n channels; temporal 3-tap
    conv, zero padded at every video's first / last frame; w [n, 3*c], k = kt*c + ci."""
    _chk16(x, "x"), _chk16(w, "w")
    if not x.is_contiguous() or x.dim() not in (3, 4):
        raise _l.VgenError("tconv3: x must be contiguous [f,hw,c] or [b,f,hw,c]")
    b = 1 if x.dim() == 3 else x.shape[0]
    f, hw, c = x.shape[-3:]
    n = w.shape[0]
    if w.shape[1] != 3 * c or not w.is_contiguous():
        raise _l.VgenError(f"tconv3: weight {tuple(w.shape)} does not match c={c}")
    if out is None:
        out = torch.empty(*x.shape[:-1], n, device=x.device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    e, keep = _epilogue(n, bias, None, residual, 1.0, False, bn)
    rc = _run("tapgemm", 2.0 * b * f * hw * n * 3 * c, 2.0 * (b * f * hw * c + 3 * c * n + b * f * hw * n),
              lambda: _l.load().vgen_tconv3_batch(_p(x), b, f, hw, c, _p(w), n, _p(o2), ldo, ctypes.byref(e), _stream()),
              tag=f"tconv3 b{b} f{f} hw{hw} c{c} n{n}")
    _l.check(rc, "vgen_tconv3")
    return out


def set_tapgemm_impl(impl: str):
    _l.check(_l.load().vgen_set_tapgemm_impl({"auto": 0, "sm100": 0, "simt": 1, "1cta": 2, "2cta": 3}[impl]), "vgen_set_tapgemm_impl")


def pack_geglu_weight(w, bias, bn):
    """Interleave GEGLU.proj rows so every bn-block holds bn/2 value rows then their bn/2 gate rows.

    w: [2*inner, k] (first half = value, second half = gate, reference util.py:711-714).
    """
    two_inner, k = w.shape
    inner = two_inner // 2
    hb = bn // 2
    assert inner % hb == 0
    v = w[:inner].reshape(inner // hb, hb, k)
    g = w[inner:].reshape(inner // hb, hb, k)
    wp = torch.cat([v, g], dim=1).reshape(two_inner, k).contiguous()
    bp = None
    if bias is not None:
        bv = bias[:inner].reshape(inner // hb, hb)
        bg = bias[inner:].reshape(inner // hb, hb)
        bp = torch.cat([bv, bg], dim=1).reshape(two_inner).contiguous()
    return wp, bp


# ------------------------------------------------------------------------------------------------
# normalisation
_gn_ws = {}


def _gn_workspace(device, n):
    """Partial-statistics scratch of vgen_group_norm, one per (device, stream): two streams of one device must not
    share it (the stats -> finalize -> apply launches of different calls would interleave)."""
    need = int(_l.load().vgen_group_norm_workspace_bytes(n))
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ws = _gn_ws.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, device=device, dtype=torch.uint8)
        _gn_ws[key] = ws
    return ws


def group_norm(x, gamma, beta, eps, silu, n=None, out=None):
    """x [..., c] fp16 channels-last; statistics per sample over everything but the leading `n` dim.
    x is viewed as [n, p, c]: pass n explicitly when the leading dims are not (n, ...)."""
    _chk16(x, "x")
    if not x.is_contiguous():
        raise _l.VgenError("group_norm: x must be contiguous")
    c = x.shape[-1]
    n = x.shape[0] if n is None else n
    p = x.numel() // (n * c)
    if out is None:
        out = torch.empty_like(x)
    ws = _gn_workspace(x.device, n)
    rc = _run("group_norm", 0.0, 4.0 * x.numel(),
              lambda: _l.load().vgen_group_norm(_p(x), _p(out), n, p, c, _p(gamma), _p(beta), float(eps), 1 if silu else 0,
                                                _p(ws), _stream()),
              tag=f"n{n} p{p} c{c}")
    _l.check(rc, "vgen_group_norm")
    return out


def layer_norm(x, gamma, beta, eps=1e-5, out=None):
    _chk16(x, "x")
    x2, ldx = _rows_view(x, "x")
    rows, c = x2.shape
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    rc = _run("layer_norm", 0.0, 4.0 * rows * c,
              lambda: _l.load().vgen_layer_norm(_p(x2), _p(o2), rows, c, ldx, ldo, _p(gamma), _p(beta), float(eps), _stream()),
              tag=f"rows{rows} c{c}")
    _l.check(rc, "vgen_layer_norm")
    return out


def row_stats(x, eps=1e-5):
    """LayerNorm statistics of the rows of x [rows, c] -> fp32 [rows, 2] = {rstd, -mean * rstd} (for linear(..., ln=...))."""
    _chk16(x, "x")
    x2, ldx = _rows_view(x, "x")
    rows, c = x2.shape
    out = torch.empty(rows, 2, device=x.device, dtype=torch.float32)
    rc = _run("layer_norm", 0.0, 2.0 * rows * c + 8.0 * rows,
              lambda: _l.load().vgen_row_stats(_p(x2), rows, c, ldx, float(eps), _p(out), _stream()), tag=f"stats rows{rows} c{c}")
    _l.check(rc, "vgen_row_stats")
    return out


def fold_layer_norm(w, bias, gamma, beta):
    """Fold a LayerNorm's affine part into the linear that follows it (host-side, once per weight load).

    w [n, k] / bias [n] or None (fp32 masters), gamma / beta [k].  Returns (w' fp16 [n, k] = w * gamma, col_sum fp32 [n] of the
    ROUNDED w', bias' fp32 [n] = bias + w @ beta):  LN(x) w^T + bias = rstd (x w'^T) - mean rstd col_sum + bias'."""
    w32, g, be = w.detach().float(), gamma.detach().float(), beta.detach().float()
    wf = (w32 * g[None, :]).to(torch.float16)
    lb = w32.double() @ be.double()
    if bias is not None:
        lb = lb + bias.detach().double()
    return wf, wf.double().sum(1).float(), lb.float()


# ------------------------------------------------------------------------------------------------
# attention
def attention_d64(q, k, v, heads, kv_batch_div=1, out=None):
    """q [b, lq, heads*64] (last-dim-contiguous views allowed, e.g. slices of a fused qkv buffer),
    k/v [b // kv_batch_div, lk, heads*64] -> out [b, lq, heads*64]."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        _chk16(t, nm)
        if t.dim() != 3 or t.stride(2) != 1 or t.stride(0) != t.shape[1] * t.stride(1):
            raise _l.VgenError(f"attention_d64: {nm} must be [b, l, h*64] with dense batch stride")
    b, lq, inner = q.shape
    lk = k.shape[1]
    if inner != heads * 64 or k.shape[2] != inner or v.shape != k.shape or k.shape[0] * kv_batch_div != b:
        raise _l.VgenError("attention_d64: shape mismatch")
    if out is None:
        out = torch.empty(b, lq, inner, device=q.device, dtype=torch.float16)
    rc = _run("attention_d64", 4.0 * b * heads * lq * lk * 64, 2.0 * (2 * b * lq * inner + 2 * k.shape[0] * lk * inner),
              lambda: _l.load().vgen_attention_d64(_p(q), _p(k), _p(v), _p(out), b, heads, lq, lk, q.stride(1), k.stride(1),
                                                   v.stride(1), out.stride(1), kv_batch_div, 64 ** -0.5, _stream()),
              tag=f"b{b} h{heads} lq{lq} lk{lk}")
    _l.check(rc, "vgen_attention_d64")
    return out


def attention_d512(q, k, v, out=None):
    """Single-head flash attention, head_dim 512: q [b, lq, 512], k/v [b, lk, 512] (last-dim-contiguous views allowed,
    e.g. slices of a fused qkv buffer) -> [b, lq, 512]."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        _chk16(t, nm)
        if t.dim() != 3 or t.shape[2] != 512 or t.stride(2) != 1 or t.stride(0) != t.shape[1] * t.stride(1):
            raise _l.VgenError(f"attention_d512: {nm} must be [b, l, 512] with dense batch stride")
    b, lq, _ = q.shape
    lk = k.shape[1]
    if k.shape[0] != b or v.shape != k.shape:
        raise _l.VgenError("attention_d512: shape mismatch")
    if out is None:
        out = torch.empty(b, lq, 512, device=q.device, dtype=torch.float16)
    rc = _run("attention_d512", 4.0 * b * lq * lk * 512, 2.0 * (2 * b * lq * 512 + 2 * b * lk * 512),
              lambda: _l.load().vgen_attention_d512(_p(q), _p(k), _p(v), _p(out), b, lq, lk, q.stride(1), k.stride(1), v.stride(1),
                                                    out.stride(1), 512 ** -0.5, _stream()),
              tag=f"b{b} lq{lq} lk{lk}")
    _l.check(rc, "vgen_attention_d512")
    return out


def attention_temporal(q, k, v, heads, head_dim, out=None):
    """q/k/v [f, npix, heads*head_dim] views (frame-major) of one video, or [b, f, npix, heads*head_dim] for b videos back
    to back (one launch): attention over the f tokens of each pixel."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        _chk16(t, nm)
        if t.dim() not in (3, 4) or t.stride(-1) != 1:
            raise _l.VgenError(f"attention_temporal: {nm} must be [(b,) f, npix, c] with contiguous channels")
    if q.dim() == 3:
        q, k, v = q.unsqueeze(0), k.unsqueeze(0), v.unsqueeze(0)
        out4 = None if out is None else out.unsqueeze(0)
        squeeze = True
    else:
        out4, squeeze = out, False
    b, f, npix, inner = q.shape
    if inner != heads * head_dim or k.shape != q.shape or v.shape != q.shape:
        raise _l.VgenError("attention_temporal: shape mismatch")
    if k.stride() != q.stride() or v.stride() != q.stride():
        raise _l.VgenError("attention_temporal: q/k/v must share strides")
    if out4 is None:
        out4 = torch.empty(b, f, npix, inner, device=q.device, dtype=torch.float16)
    elif out4.shape != q.shape or out4.stride(-1) != 1:
        raise _l.VgenError("attention_temporal: out must be shaped like q with contiguous channels")
    rc = _run("attention_temporal", 4.0 * b * npix * heads * f * f * head_dim, 2.0 * 4 * b * f * npix * inner,
              lambda: _l.load().vgen_attention_temporal(_p(q), _p(k), _p(v), _p(out4), b * npix, heads, f, head_dim, q.stride(1),
                                                        q.stride(2), out4.stride(1), out4.stride(2), npix, q.stride(0),
                                                        out4.stride(0), head_dim ** -0.5, _stream()))
    _l.check(rc, "vgen_attention_temporal")
    return out4[0] if squeeze else out4


def attention_cross_small(q, k, v, heads, kv_batch_div=1, out=None, causal=False):
    """q [b, lq, heads*d], k/v [b // kv_batch_div, lk, heads*d] for any d <= 256 (tiny problems only); causal: query i
    attends keys 0 .. i + (lk - lq) (the CLIP text tower's mask)."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        _chk16(t, nm)
        if t.dim() != 3 or t.stride(2) != 1 or t.stride(0) != t.shape[1] * t.stride(1):
            raise _l.VgenError(f"attention_cross_small: {nm} must be [b, l, h*d] with dense batch stride")
    b, lq, inner = q.shape
    lk = k.shape[1]
    d = inner // heads
    if inner != heads * d or k.shape[2] != inner or v.shape != k.shape or k.shape[0] * kv_batch_div != b:
        raise _l.VgenError("attention_cross_small: shape mismatch")
    if out is None:
        out = torch.empty(b, lq, inner, device=q.device, dtype=torch.float16)
    rc = _l.load().vgen_attention_cross_small(_p(q), _p(k), _p(v), _p(out), b, heads, lq, lk, d, q.stride(1), k.stride(1),
                                              v.stride(1), out.stride(1), kv_batch_div, 1 if causal else 0, d ** -0.5, _stream())
    _l.check(rc, "vgen_attention_cross_small")
    return out


def interp_linear_rows(x, lout):
    """x [nseq, lin, c] fp16 -> [nseq, lout, c] (F.interpolate mode='linear' over the middle axis)."""
    _chk16(x, "x")
    if x.dim() != 3 or not x.is_contiguous():
        raise _l.VgenError("interp_linear_rows: x must be contiguous [nseq, lin, c]")
    nseq, lin, c = x.shape
    y = torch.empty(nseq, lout, c, device=x.device, dtype=torch.float16)
    rc = _l.load().vgen_interp_linear_rows(_p(x), _p(y), nseq, lin, lout, c, _stream())
    _l.check(rc, "vgen_interp_linear_rows")
    return y


def fourier_lowfreq_filter(x, scale, out=None):
    """Fourier_filter(threshold=1) on channels-last x [nimg, h, w, c]; `out` may be a channel slice of a
    wider channels-last buffer."""
    _chk16(x, "x")
    nimg, h, w, c = x.shape
    x2, ldx = _rows_view(x, "x")
    if out is None:
        out = torch.empty(nimg, h, w, c, device=x.device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    if o2.shape != x2.shape:
        raise _l.VgenError("fourier_lowfreq_filter: shape mismatch")
    rc = _l.load().vgen_fourier_lowfreq_filter(_p(x2), ldx, _p(o2), ldo, nimg, h, w, c, float(scale), _stream())
    _l.check(rc, "vgen_fourier_lowfreq_filter")
    return out


def scale_copy2d(src, dst, s):
    s2, lds = _rows_view(src, "src")
    d2, ldd = _rows_view(dst, "dst")
    if s2.shape != d2.shape:
        raise _l.VgenError("scale_copy2d: shape mismatch")
    rc = _l.load().vgen_scale_copy2d(_p(s2), lds, _p(d2), ldd, s2.shape[0], s2.shape[1], float(s), _stream())
    _l.check(rc, "vgen_scale_copy2d")
    return dst


def softmax_rows_(x, scale=1.0):
    _chk16(x, "x")
    x2, ld = _rows_view(x, "x")
    rc = _l.load().vgen_softmax_rows(_p(x2), x2.shape[0], x2.shape[1], ld, float(scale), _stream())
    _l.check(rc, "vgen_softmax_rows")
    return x


# ------------------------------------------------------------------------------------------------
# data movement / pointwise
def cp_to_pc(x, n, c, p, c_pad=None):
    """x viewed as [n, c, p] (fp32 or fp16, contiguous) -> [n, p, c_pad] fp16."""
    c_pad = c if c_pad is None else c_pad
    if not x.is_contiguous() or x.dtype not in (torch.float32, torch.float16):
        raise _l.VgenError("cp_to_pc: x must be contiguous fp32/fp16")
    y = torch.empty(n, p, c_pad, device=x.device, dtype=torch.float16)
    rc = _l.load().vgen_cp_to_pc(_p(x), 1 if x.dtype == torch.float32 else 0, _p(y), n, c, p, c_pad, _stream())
    _l.check(rc, "vgen_cp_to_pc")
    return y


def pc_to_cp(x, n, c, p, out_dtype=torch.float16):
    """x [n, p, ld>=c] fp16 -> [n, c, p]."""
    _chk16(x, "x")
    ldx = x.shape[-1]
    y = torch.empty(n, c, p, device=x.device, dtype=out_dtype)
    rc = _l.load().vgen_pc_to_cp(_p(x), ldx, _p(y), 1 if out_dtype == torch.float32 else 0, n, c, p, _stream())
    _l.check(rc, "vgen_pc_to_cp")
    return y


def im2col(x, kh, kw, stride, pad_t, pad_l, ho, wo, kpad, act_silu=False):
    _chk16(x, "x")
    nimg, h, w, c = x.shape
    out = torch.empty(nimg * ho * wo, kpad, device=x.device, dtype=torch.float16)
    rc = _l.load().vgen_im2col(_p(x), _p(out), nimg, h, w, c, kh, kw, stride, pad_t, pad_l, ho, wo, kpad,
                               1 if act_silu else 0, _stream())
    _l.check(rc, "vgen_im2col")
    return out


def upsample_nearest2x(x):
    _chk16(x, "x")
    nimg, h, w, c = x.shape
    y = torch.empty(nimg, 2 * h, 2 * w, c, device=x.device, dtype=torch.float16)
    rc = _l.load().vgen_upsample_nearest2x(_p(x), _p(y), nimg, h, w, c, _stream())
    _l.check(rc, "vgen_upsample_nearest2x")
    return y


def upsample_nearest2x_rows(x, row0, rows_out):
    """nearest x2 upsampling keeping rows [row0, row0+rows_out) (UpsampleSR600 crops one row each side)."""
    _chk16(x, "x")
    nimg, h, w, c = x.shape
    y = torch.empty(nimg, rows_out, 2 * w, c, device=x.device, dtype=torch.float16)
    rc = _l.load().vgen_upsample_nearest2x_rows(_p(x), _p(y), nimg, h, w, c, row0, rows_out, _stream())
    _l.check(rc, "vgen_upsample_nearest2x_rows")
    return y


def copy2d(src, dst):
    """dst[r, :cols] = src[r, :cols] for 2-D row views."""
    s2, lds = _rows_view(src, "src")
    d2, ldd = _rows_view(dst, "dst")
    if s2.shape != d2.shape:
        raise _l.VgenError("copy2d: shape mismatch")
    rc = _l.load().vgen_copy2d(_p(s2), lds, _p(d2), ldd, s2.shape[0], s2.shape[1], _stream())
    _l.check(rc, "vgen_copy2d")
    return dst


def concat_channels(a, b):
    """torch.cat([a, b], dim=-1) for channels-last tensors with equal leading dims."""
    ca, cb = a.shape[-1], b.shape[-1]
    out = torch.empty(*a.shape[:-1], ca + cb, device=a.device, dtype=torch.float16)
    o2 = out.reshape(-1, ca + cb)
    copy2d(a.reshape(-1, ca), o2[:, :ca])
    copy2d(b.reshape(-1, cb), o2[:, ca:])
    return out


_ELT = {"silu": 0, "add": 1, "gelu": 2, "scale": 3, "axpy": 4}


def eltwise(op, a, b=None, s=1.0, out=None):
    _chk16(a, "a")
    if out is None:
        out = torch.empty_like(a)
    rc = _l.load().vgen_eltwise(_ELT[op], _p(a), _p(b), _p(out), a.numel(), float(s), _stream())
    _l.check(rc, "vgen_eltwise")
    return out


def linear_small(a, w, bias=None, residual=None, silu_in=False, gelu_out=False, out=None):
    _chk16(a, "a"), _chk16(w, "w")
    lead = a.shape[:-1]
    a2, lda = _rows_view(a, "a")
    m, k = a2.shape
    n = w.shape[0]
    if out is None:
        out = torch.empty(*lead, n, device=a.device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    r2, ldr = (None, 0) if residual is None else _rows_view(residual, "residual")
    rc = _l.load().vgen_linear_small(_p(a2), m, k, lda, _p(w), _p(bias), n, _p(r2), ldr, _p(o2), ldo,
                                     1 if silu_in else 0, 1 if gelu_out else 0, _stream())
    _l.check(rc, "vgen_linear_small")
    return out


def sinusoidal_embedding(t, dim):
    t32 = t.to(torch.float32).contiguous()
    out = torch.empty(t32.numel(), dim, device=t.device, dtype=torch.float16)
    rc = _l.load().vgen_sinusoidal_embedding(_p(t32), _p(out), t32.numel(), dim, _stream())
    _l.check(rc, "vgen_sinusoidal_embedding")
    return out


def adaptive_avgpool(x, oh, ow, silu_in=False):
    _chk16(x, "x")
    nimg, h, w, c = x.shape
    y = torch.empty(nimg, oh, ow, c, device=x.device, dtype=torch.float16)
    rc = _l.load().vgen_adaptive_avgpool(_p(x), _p(y), nimg, h, w, c, oh, ow, 1 if silu_in else 0, _stream())
    _l.check(rc, "vgen_adaptive_avgpool")
    return y


def cond_stem_k(cin):
    """K (row length) of the vgen_cond_stem weight matrix: 9*cin padded to a multiple of 16."""
    return (9 * cin + 15) // 16 * 16


def pack_cond_stem_weight(w):
    """Conv2d weight [cout, cin, 3, 3] -> fp32 [cout, cond_stem_k(cin)] with k = (ky*3+kx)*cin + ci, padding zero."""
    cout, cin = w.shape[0], w.shape[1]
    wp = torch.zeros(cout, cond_stem_k(cin), dtype=torch.float32)
    wp[:, :9 * cin] = w.detach().float().cpu().permute(0, 2, 3, 1).reshape(cout, 9 * cin)
    return wp


def cond_stem(x, w, bias, oh, ow):
    """Conv2d(3x3, pad 1) + bias -> SiLU -> AdaptiveAvgPool2d((oh, ow)) of every frame of a condition, one kernel.

    x [b, cin, f, H, W] contiguous CUDA fp32 or fp16 (the reference layout), cin 1..4; w fp16 [cout, cond_stem_k(cin)]
    (pack_cond_stem_weight), bias fp32 [cout], cout 8..64 in steps of 8 -> fp16 channels-last [(b f), oh, ow, cout]."""
    if not x.is_cuda or x.dim() != 5 or not x.is_contiguous() or x.dtype not in (torch.float32, torch.float16):
        raise _l.VgenError("cond_stem: x must be a contiguous CUDA fp32/fp16 tensor [b, cin, f, H, W]")
    b, cin, f, h, wd = x.shape
    _chk16(w, "w")
    cout = w.shape[0]
    if w.dim() != 2 or w.shape[1] != cond_stem_k(cin) or not w.is_contiguous():
        raise _l.VgenError(f"cond_stem: weight {tuple(w.shape)} must be contiguous [cout, {cond_stem_k(cin)}] for cin={cin}")
    if bias.dtype != torch.float32 or not bias.is_contiguous() or bias.numel() != cout or not bias.is_cuda:
        raise _l.VgenError("cond_stem: bias must be a contiguous CUDA fp32 tensor [cout]")
    out = torch.empty(b * f, oh, ow, cout, device=x.device, dtype=torch.float16)
    n = b * f
    rc = _run("cond_stem", 2.0 * n * h * wd * 9 * cin * cout, x.element_size() * x.numel() + 2.0 * out.numel() + 2.0 * w.numel(),
              lambda: _l.load().vgen_cond_stem(_p(x), 1 if x.dtype == torch.float32 else 0, b, cin, f, h, wd, _p(w), _p(bias),
                                               cout, oh, ow, _p(out), _stream()),
              tag=f"cin{cin} {n}x{h}x{wd} -> {oh}x{ow}x{cout}")
    _l.check(rc, "vgen_cond_stem")
    return out


def cond_sum(srcs, out=None):
    """fp16(sum of the fp16 [rows, cols] tensors `srcs`, accumulated in fp32 in list order), 1..8 sources."""
    if not 1 <= len(srcs) <= 8:
        raise _l.VgenError("cond_sum: 1..8 sources")
    views = []
    for i, s in enumerate(srcs):
        _chk16(s, f"srcs[{i}]")
        views.append(_rows_view(s, f"srcs[{i}]"))
    rows, cols = views[0][0].shape
    ld = views[0][1]
    if any(v.shape != (rows, cols) or l != ld for v, l in views):
        raise _l.VgenError("cond_sum: sources must share shape and row stride")
    if out is None:
        out = torch.empty(rows, cols, device=srcs[0].device, dtype=torch.float16)
    o2, ldo = _rows_view(out, "out")
    if o2.shape != (rows, cols):
        raise _l.VgenError("cond_sum: out shape mismatch")
    ptrs = (ctypes.c_void_p * len(srcs))(*[v.data_ptr() for v, _ in views])
    rc = _l.load().vgen_cond_sum(ptrs, len(srcs), rows, cols, ld, _p(o2), ldo, _stream())
    _l.check(rc, "vgen_cond_sum")
    return out


def ddim_step_(xt, y, u, coef7, guide_scale, mean_type_v=True, noise=None, x0_out=None):
    """In-place fused CFG + DDIM update of the fp32 latent xt; y/u fp16 model outputs (same layout).
    x0_out (optional, fp32 like xt) receives the predicted x0 (diffusion_ddim.py:241 returns it)."""
    if xt.dtype != torch.float32 or not xt.is_contiguous() or not xt.is_cuda:
        raise _l.VgenError("ddim_step_: xt must be a contiguous CUDA fp32 tensor")
    _chk16(y, "y")
    if not y.is_contiguous() or y.numel() != xt.numel():
        raise _l.VgenError("ddim_step_: y must be contiguous with xt's element count")
    if u is not None:
        _chk16(u, "u")
        if not u.is_contiguous() or u.numel() != xt.numel():
            raise _l.VgenError("ddim_step_: u must be contiguous with xt's element count")
    if noise is not None and (noise.dtype != torch.float32 or not noise.is_contiguous() or not noise.is_cuda
                              or noise.numel() != xt.numel()):
        raise _l.VgenError("ddim_step_: noise must be a contiguous CUDA fp32 tensor with xt's element count")
    if x0_out is not None and (x0_out.dtype != torch.float32 or not x0_out.is_contiguous() or x0_out.numel() != xt.numel()):
        raise _l.VgenError("ddim_step_: x0_out must be a contiguous fp32 tensor with xt's element count")
    c = (ctypes.c_float * 7)(*[float(v) for v in coef7])
    rc = _l.load().vgen_ddim_step(_p(xt), _p(y), _p(u), _p(noise), xt.numel(), float(guide_scale or 0.0), c,
                                  1 if mean_type_v else 0, _p(x0_out), _stream())
    _l.check(rc, "vgen_ddim_step")
    return xt


def cfg_combine(y, u, guide_scale):
    """out = u + g*(y-u) (fp16) and the fp64 per-sample sums needed by the std-ratio guidance rescale."""
    _chk16(y, "y"), _chk16(u, "u")
    if y.shape != u.shape or not y.is_contiguous() or not u.is_contiguous():
        raise _l.VgenError("cfg_combine: y/u must be contiguous and equally shaped")
    b = y.shape[0]
    out = torch.empty_like(y)
    stats = torch.empty(b, 4, device=y.device, dtype=torch.float64)
    rc = _l.load().vgen_cfg_combine(_p(y), _p(u), _p(out), b, y.numel() // b, float(guide_scale), _p(stats), _stream())
    _l.check(rc, "vgen_cfg_combine")
    return out, stats


def gauss_x0(xt, out, alpha, sigma, prediction_type, stats=None, guide_rescale=0.0):
    """x0 prediction of GaussianDiffusion.denoise from the fp32 latent and the fp16 model output."""
    _chk16(out, "out")
    if xt.dtype != torch.float32 or not xt.is_contiguous() or not out.is_contiguous() or xt.shape != out.shape:
        raise _l.VgenError("gauss_x0: xt must be contiguous fp32 and shaped like out")
    b = xt.shape[0]
    x0 = torch.empty_like(xt)
    rc = _l.load().vgen_gauss_x0(_p(xt), _p(out), _p(stats), float(guide_rescale), float(alpha), float(sigma),
                                 {"x0": 0, "eps": 1, "v": 2}[prediction_type], _p(x0), b, xt.numel() // b, _stream())
    _l.check(rc, "vgen_gauss_x0")
    return x0


def lincomb_f32(terms, out=None):
    """out = sum_i a_i * x_i over up to four (a_i, x_i) fp32 terms."""
    if not 1 <= len(terms) <= 4:
        raise _l.VgenError("lincomb_f32: 1..4 terms")
    x0 = terms[0][1]
    for a, x in terms:
        if x.dtype != torch.float32 or not x.is_contiguous() or x.shape != x0.shape or not x.is_cuda:
            raise _l.VgenError("lincomb_f32: terms must be contiguous CUDA fp32 tensors of one shape")
    if out is None:
        out = torch.empty_like(x0)
    args = []
    for i in range(4):
        a, x = terms[i] if i < len(terms) else (0.0, None)
        args += [_p(x), float(a)]
    rc = _l.load().vgen_lincomb_f32(_p(out), x0.numel(), *args, _stream())
    _l.check(rc, "vgen_lincomb_f32")
    return out


def vae_sample(moments, noise, scale):
    """moments fp16 [n, p, 2*zc] (mean | logvar), noise fp32 [n, zc, p] -> fp32 z [n, zc, p]."""
    _chk16(moments, "moments")
    n, p, c2 = moments.shape
    zc = c2 // 2
    if noise.dtype != torch.float32 or not noise.is_contiguous() or noise.numel() != n * zc * p:
        raise _l.VgenError("vae_sample: noise must be contiguous fp32 [n, zc, p]")
    z = torch.empty(n, zc, p, device=moments.device, dtype=torch.float32)
    rc = _l.load().vgen_vae_sample(_p(moments), _p(noise), _p(z), n, zc, p, float(scale), _stream())
    _l.check(rc, "vgen_vae_sample")
    return z


def video_to_rgb8(video, mean, std, want_band=True):
    """video fp32 [3, f, h, w] (one batch entry, contiguous, CUDA) -> (uint8 [f, h, w, 3], per-frame count of bytes in
    [117, 137] or None).  mean / std: 3 floats each (cfg.mean / cfg.std)."""
    if video.dtype != torch.float32 or not video.is_cuda or not video.is_contiguous() or video.dim() != 4 or video.shape[0] != 3:
        raise _l.VgenError("video_to_rgb8: video must be a contiguous CUDA fp32 tensor [3, f, h, w]")
    c, f, h, w = video.shape
    out = torch.empty(f, h, w, 3, device=video.device, dtype=torch.uint8)
    band = torch.empty(f, device=video.device, dtype=torch.int64) if want_band else None
    m3 = (ctypes.c_float * 3)(*[float(v) for v in mean])
    s3 = (ctypes.c_float * 3)(*[float(v) for v in std])
    rc = _run("video_out", 0.0, 5.0 * video.numel(),
              lambda: _l.load().vgen_video_to_rgb8(_p(video), c, f, h, w, m3, s3, _p(out), _p(band), _stream()))
    _l.check(rc, "vgen_video_to_rgb8")
    return out, band


def embed_tokens(ids, table, pos):
    """ids int64 [b, L] (CUDA), table fp32 [vocab, W], pos fp32 [L, W] -> fp16 [b, L, W] = table[ids] + pos."""
    if ids.dtype != torch.int64 or not ids.is_cuda or not ids.is_contiguous() or ids.dim() != 2:
        raise _l.VgenError("embed_tokens: ids must be a contiguous CUDA int64 tensor [b, L]")
    for t, nm in ((table, "table"), (pos, "pos")):
        if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
            raise _l.VgenError(f"embed_tokens: {nm} must be a contiguous CUDA fp32 tensor")
    b, L = ids.shape
    vocab, W = table.shape
    if pos.shape != (L, W):
        raise _l.VgenError("embed_tokens: pos must be [L, W]")
    out = torch.empty(b, L, W, device=ids.device, dtype=torch.float16)
    rc = _l.load().vgen_embed_tokens(_p(ids), _p(table), _p(pos), _p(out), b * L, L, W, vocab, _stream())
    _l.check(rc, "vgen_embed_tokens")
    return out


def add_rows_f32_(x, add):
    """x fp16 [b, ...] += add fp32 [...] broadcast over the leading dim, in place."""
    _chk16(x, "x")
    if not x.is_contiguous() or add.dtype != torch.float32 or not add.is_contiguous() or add.numel() * x.shape[0] != x.numel():
        raise _l.VgenError("add_rows_f32_: x must be contiguous fp16 [b, n...] and add contiguous fp32 [n...]")
    rc = _l.load().vgen_add_rows_f32(_p(x), _p(add), x.shape[0], add.numel(), _stream())
    _l.check(rc, "vgen_add_rows_f32")
    return x
