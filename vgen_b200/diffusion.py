"""B200-native DiffusionDDIM: the reference's DDIM sampler interface
(tools/modules/diffusions/diffusion_ddim.py:27-254) with the per-step tensor arithmetic fused into one
kernel (vgen_ddim_step: CFG mix + v->x0 + eps + x_{t-1}).

Host side (kept in fp64 torch / Python exactly like the reference, so it is bit-exact):
  * beta schedules `cosine`, `linear_sd` (+ zero-terminal-SNR rescale)     schedules.py:5-21,62-63,72-79,143-165
  * cumulative-product tables                                             diffusion_ddim.py:46-78
  * the timestep list  (1 + arange(0, T, T // S)).clamp(0, T-1).flip(0)   diffusion_ddim.py:250
Only the sampling entry points used by the inference engines are provided: ddim_sample_loop and ddim_sample for
var_type fixed_small / mean_type v|eps.  The arithmetic of the reference's p_mean_variance (:147-206: two model calls,
CFG mix, v -> x0) has no method of its own here -- it lives inside the fused step kernel; the training losses, PLMS and
reward variants are out of scope and absent (calling them raises AttributeError, not a fallback).
"""
from __future__ import annotations

import math
import os

import torch

from . import ops


def _cosine_betas(num_timesteps, cosine_s=0.008, **kw):
    def abar(u):
        return math.cos((u + cosine_s) / (1 + cosine_s) * math.pi / 2) ** 2
    out = []
    for step in range(num_timesteps):
        out.append(min(1.0 - abar((step + 1) / num_timesteps) / abar(step / num_timesteps), 0.999))
    return torch.tensor(out, dtype=torch.float64)


def _linear_sd_betas(num_timesteps, init_beta, last_beta, **kw):
    return torch.linspace(init_beta ** 0.5, last_beta ** 0.5, num_timesteps, dtype=torch.float64) ** 2


def _rescale_zero_terminal_snr(betas):
    abs_ = (1 - betas).cumprod(0).sqrt()
    a0, aT = abs_[0].clone(), abs_[-1].clone()
    abs_ = abs_ - aT
    abs_ = abs_ * (a0 / (a0 - aT))
    ab = abs_ ** 2
    alphas = torch.cat([ab[0:1], ab[1:] / ab[:-1]])
    return 1 - alphas


def beta_schedule(schedule="cosine", num_timesteps=1000, zero_terminal_snr=False, **kwargs):
    fn = {"cosine": _cosine_betas, "linear_sd": _linear_sd_betas}.get(schedule)
    if fn is None:
        raise NotImplementedError(f"vgen_b200: beta schedule '{schedule}' is not used by the supported configs")
    betas = fn(num_timesteps, **kwargs)
    if zero_terminal_snr and abs(betas.max() - 1.0) > 0.0001:
        betas = _rescale_zero_terminal_snr(betas)
    return betas


def _unwrap(model):
    return getattr(model, "module", model)


def cfg_forward(model, xt, ts, model_kwargs, by_keyword=False):
    """The two classifier-free-guidance evaluations of one step (diffusion_ddim.py:157-158, diffusion_gauss.py:204-208).

    A vgen_b200 UNet (`cfg_batch = True`) evaluates both branches as ONE forward of batch 2b -- the same arithmetic
    per sample (batch entries never interact), half the launches, and two tiles per CTA pair on the low-resolution
    layers so their epilogue overlaps a main loop.  Any other callable (e.g. a reference model) gets the reference's
    two separate calls.  VGEN_CFG_BATCH=0 disables the batching.

    A model may declare `cfg_shared_kwargs`: a keyword in that set whose two branches hold the SAME tensor object (the
    VideoComposer engines pass one condition tensor to both branches) is passed once, at batch b, and the model applies
    it to both halves of the batch-2b forward.  Equal values in distinct tensors are concatenated like any other input."""
    kc, ku = model_kwargs
    m = _unwrap(model)
    call = (lambda x, t, kw: model(x, t=t, **kw)) if by_keyword else (lambda x, t, kw: model(x, t, **kw))
    if getattr(m, "cfg_batch", False) and os.environ.get("VGEN_CFG_BATCH", "1") != "0" and kc.keys() == ku.keys():
        shared = getattr(m, "cfg_shared_kwargs", ())
        merged = {}
        for k in kc:
            a, b = kc[k], ku[k]
            if k in shared and a is b and torch.is_tensor(a):
                merged[k] = a
            elif torch.is_tensor(a) and torch.is_tensor(b) and a.shape == b.shape and a.dtype == b.dtype and a.dim() >= 1 \
                    and a.size(0) == xt.size(0):
                merged[k] = torch.cat([a, b], dim=0)
            elif a is None and b is None:
                merged[k] = None
            else:
                merged = None
                break
        if merged is not None:
            out = call(torch.cat([xt, xt], dim=0), torch.cat([ts, ts], dim=0), merged)
            n = xt.size(0)
            return out[:n], out[n:]
    return call(xt, ts, kc), call(xt, ts, ku)


class DiffusionDDIM(object):
    def __init__(self, schedule="linear_sd", schedule_param={}, mean_type="eps", var_type="learned_range", loss_type="mse",
                 epsilon=1e-12, rescale_timesteps=False, noise_strength=0.0, **kwargs):
        assert mean_type in ["x0", "x_{t-1}", "eps", "v"]
        assert var_type in ["learned", "learned_range", "fixed_large", "fixed_small"]
        betas = beta_schedule(schedule, **schedule_param)
        assert min(betas) > 0 and max(betas) <= 1
        self.betas = betas
        self.num_timesteps = len(betas)
        self.mean_type, self.var_type, self.loss_type = mean_type, var_type, loss_type
        self.epsilon, self.rescale_timesteps, self.noise_strength = epsilon, rescale_timesteps, noise_strength
        alphas = 1 - self.betas
        self.alphas_cumprod = torch.cumprod(alphas, dim=0)
        self.alphas_cumprod_prev = torch.cat([alphas.new_ones([1]), self.alphas_cumprod[:-1]])
        self.alphas_cumprod_next = torch.cat([self.alphas_cumprod[1:], alphas.new_zeros([1])])
        self.sqrt_alphas_cumprod = torch.sqrt(self.alphas_cumprod)
        self.sqrt_one_minus_alphas_cumprod = torch.sqrt(1.0 - self.alphas_cumprod)
        self.log_one_minus_alphas_cumprod = torch.log(1.0 - self.alphas_cumprod)
        self.sqrt_recip_alphas_cumprod = torch.sqrt(1.0 / self.alphas_cumprod)
        self.sqrt_recipm1_alphas_cumprod = torch.sqrt(1.0 / self.alphas_cumprod - 1)
        self.posterior_variance = betas * (1.0 - self.alphas_cumprod_prev) / (1.0 - self.alphas_cumprod)
        self.posterior_log_variance_clipped = torch.log(self.posterior_variance.clamp(1e-20))
        self.posterior_mean_coef1 = betas * torch.sqrt(self.alphas_cumprod_prev) / (1.0 - self.alphas_cumprod)
        self.posterior_mean_coef2 = (1.0 - self.alphas_cumprod_prev) * torch.sqrt(alphas) / (1.0 - self.alphas_cumprod)

    # ---- timestep / index math (host, integer-exact) --------------------------------------------
    def ddim_steps(self, ddim_timesteps):
        T = self.num_timesteps
        return (1 + torch.arange(0, T, T // ddim_timesteps)).clamp(0, T - 1).flip(0)

    def _scale_timesteps(self, t):
        if self.rescale_timesteps:
            return t.float() * 1000.0 / self.num_timesteps
        return t

    def step_coefficients(self, step, ddim_timesteps, eta=0.0):
        """The seven fp32 scalars of one DDIM update, computed like the reference does: fp64 table
        entries cast to fp32 by _i() (:10-16), then fp32 arithmetic (:230-240)."""
        T = self.num_timesteps
        stride = T // ddim_timesteps
        t = int(step)
        tp = max(t - stride, 0)
        f32 = torch.float32
        a_t = self.alphas_cumprod[t].to(f32)
        a_prev = self.alphas_cumprod[tp].to(f32)
        sigma = eta * torch.sqrt((1 - a_prev) / (1 - a_t) * (1 - a_t / a_prev))
        coef = [self.sqrt_alphas_cumprod[t].to(f32), self.sqrt_one_minus_alphas_cumprod[t].to(f32),
                self.sqrt_recip_alphas_cumprod[t].to(f32), self.sqrt_recipm1_alphas_cumprod[t].to(f32),
                torch.sqrt(a_prev), torch.sqrt(1 - a_prev - sigma ** 2), sigma * (1.0 if t != 0 else 0.0)]
        return [float(c) for c in coef]

    # ---- sampling ----------------------------------------------------------------------------------
    @torch.no_grad()
    def ddim_sample(self, xt, t, model, model_kwargs={}, clamp=None, percentile=None, condition_fn=None, guide_scale=None,
                    ddim_timesteps=20, eta=0.0):
        """One DDIM step (diffusion_ddim.py:209-241); returns (x_{t-1}, x0) like the reference.  All batch entries
        share the timestep (true for every caller on the sampling path)."""
        if clamp is not None or percentile is not None or condition_fn is not None:
            raise NotImplementedError("vgen_b200 DiffusionDDIM: clamp / percentile / condition_fn are not used by the "
                                      "supported inference configs")
        if self.var_type != "fixed_small" or self.mean_type not in ("v", "eps"):
            raise NotImplementedError("vgen_b200 DiffusionDDIM: only var_type fixed_small with mean_type v|eps")
        return self._ddim_step(xt, int(t.flatten()[0]), t, model, model_kwargs, guide_scale, ddim_timesteps, eta, want_x0=True)

    def _ddim_step(self, xt, step, t, model, model_kwargs, guide_scale, ddim_timesteps, eta, want_x0=False):
        if self.var_type != "fixed_small" or self.mean_type not in ("v", "eps"):
            raise NotImplementedError("vgen_b200 DiffusionDDIM: only var_type fixed_small with mean_type v|eps")
        ts = self._scale_timesteps(t)
        if guide_scale is None:
            y_out = model(xt, ts, **model_kwargs)
            u_out = None
        else:
            assert isinstance(model_kwargs, list) and len(model_kwargs) == 2
            y_out, u_out = cfg_forward(model, xt, ts, model_kwargs)
        coef = self.step_coefficients(step, ddim_timesteps, eta)
        # the reference draws the noise in xt's dtype even when eta == 0 (:237) -- keeps the device RNG stream aligned;
        # the kernel reads fp32, so a non-fp32 draw is converted (never reinterpreted)
        noise = torch.randn_like(xt)
        y16 = y_out if y_out.dtype == torch.float16 else y_out.to(torch.float16)
        u16 = None if u_out is None else (u_out if u_out.dtype == torch.float16 else u_out.to(torch.float16))
        xt = xt if (xt.dtype == torch.float32 and xt.is_contiguous()) else xt.float().contiguous()
        xt = xt.clone()
        x0 = torch.empty_like(xt) if want_x0 else None
        ops.ddim_step_(xt, y16.contiguous(), None if u16 is None else u16.contiguous(), coef, guide_scale,
                       mean_type_v=(self.mean_type == "v"),
                       noise=noise.float().contiguous() if coef[6] != 0.0 else None, x0_out=x0)
        return xt, x0

    @torch.no_grad()
    def ddim_sample_loop(self, noise, model, model_kwargs={}, clamp=None, percentile=None, condition_fn=None,
                         guide_scale=None, ddim_timesteps=20, eta=0.0):
        """diffusion_ddim.py:244-254."""
        b = noise.size(0)
        xt = noise
        for step in self.ddim_steps(ddim_timesteps):
            t = torch.full((b,), int(step), dtype=torch.long, device=xt.device)
            if clamp is not None or percentile is not None or condition_fn is not None:
                raise NotImplementedError("vgen_b200 DiffusionDDIM: clamp / percentile / condition_fn are not supported")
            # the step index is known on the host: no device->host read of t inside the loop
            xt, _ = self._ddim_step(xt, int(step), t, model, model_kwargs, guide_scale, ddim_timesteps, eta)
        return xt
