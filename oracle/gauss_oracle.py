"""TEST INFRASTRUCTURE ONLY -- oracle for SURVEY.md section 8 row a22: the SR600 sampler pair
(`DiffusionDDIMSR`, tools/modules/diffusions/diffusion_ddim.py:19-25) built on `GaussianDiffusion`
(tools/modules/diffusions/diffusion_gauss.py:145-499):

    reverse_diffusion.ddim_reverse_sample_loop   (:376-434)  deterministic DDIM inversion of the low-res latent
    forward_diffusion.sample(solver='dpmpp_2m_sde')  (:250-373, :86-142)  DPM-Solver++(2M) SDE with CFG + guide_rescale

A functional restatement in plain torch (CPU, fp32 like the reference's tables).  The stochastic term of
the SDE solver comes from torchsde.BrownianTree upstream -- a pip dependency that is absent here; both
this oracle and the reference (through oracle/refload.py) use oracle/brownian.py, see its header.

Pinning: oracle/make_golden.py runs this file against the real GaussianDiffusion / sigma_schedule
classes and freezes the sigma tables and one sampled latent into tests/golden/gauss.npz.
"""
from __future__ import annotations

import math

import torch

from . import brownian
from . import vgen_oracle as vo


# ------------------------------------------------------------------------------------ sigma schedules
def _logsnr_cosine(n, logsnr_min, logsnr_max):
    """schedules.py:106-111 (fp32 linspace)."""
    t_min = math.atan(math.exp(-0.5 * logsnr_min))
    t_max = math.atan(math.exp(-0.5 * logsnr_max))
    t = torch.linspace(1, 0, n)
    return -2 * torch.log(torch.tan(t_min + t * (t_max - t_min)))


def logsnr_cosine_interp_sigmas(n, scale_min=2, scale_max=4, logsnr_min=-15, logsnr_max=15):
    """schedules.py:52-60,114-140: interpolate two shifted cosine log-SNR curves, sigma = sqrt(sigmoid(-logsnr))."""
    t = torch.linspace(1, 0, n)
    lo = _logsnr_cosine(n, logsnr_min, logsnr_max) + 2 * math.log(1 / scale_min)
    hi = _logsnr_cosine(n, logsnr_min, logsnr_max) + 2 * math.log(1 / scale_max)
    return torch.sqrt(torch.sigmoid(-(t * lo + (1 - t) * hi)))


def sigma_schedule(schedule="cosine", num_timesteps=1000, zero_terminal_snr=False, **kw):
    """schedules.py:24-43.  NOTE (reproduced): the zero-terminal-SNR rescale written for betas is applied
    to the *sigma* table when max(sigma) is not within 1e-4 of 1."""
    if schedule == "logsnr_cosine_interp":
        keys = ("scale_min", "scale_max", "logsnr_min", "logsnr_max")
        sigma = logsnr_cosine_interp_sigmas(num_timesteps, **{k: kw[k] for k in keys if k in kw})
    elif schedule == "cosine":
        sigma = torch.sqrt(1 - torch.cumprod(1 - vo.cosine_betas(num_timesteps, kw.get("cosine_s", 0.008)), dim=0))
    elif schedule == "linear_sd":
        sigma = torch.sqrt(1 - torch.cumprod(1 - vo.linear_sd_betas(num_timesteps, kw["init_beta"], kw["last_beta"]), dim=0))
    else:
        raise NotImplementedError(schedule)
    if zero_terminal_snr and abs(sigma.max() - 1.0) > 0.0001:
        sigma = vo.zero_terminal_snr(sigma)
    return sigma


# ------------------------------------------------------------------------------------ GaussianDiffusion
def _bcast(table, t, x):
    """_i(), diffusion_gauss.py:14-19."""
    return table[t.to(table.device)].view((x.size(0),) + (1,) * (x.ndim - 1)).to(x.device)


class GaussOracle:
    def __init__(self, sigmas, prediction_type="eps"):
        """diffusion_gauss.py:147-152: fp32 tables; alphas from the table at its ORIGINAL precision."""
        self.sigmas = sigmas.float()
        self.alphas = torch.sqrt(1 - sigmas ** 2).float()
        self.num_timesteps = len(sigmas)
        self.prediction_type = prediction_type

    def log_sigmas(self):
        return torch.sqrt(self.sigmas ** 2 / (1 - self.sigmas ** 2)).log()

    def sigma_to_t(self, sigma):
        """:436-456: fractional timestep by linear interpolation in log k-sigma space."""
        if sigma == float("inf"):
            t = torch.full_like(sigma, len(self.sigmas) - 1)
        else:
            ls = self.log_sigmas().to(sigma)
            d = sigma.log() - ls[:, None]
            lo = d.ge(0).cumsum(dim=0).argmax(dim=0).clamp(max=ls.shape[0] - 2)
            hi = lo + 1
            w = ((ls[lo] - sigma.log()) / (ls[lo] - ls[hi])).clamp(0, 1)
            t = ((1 - w) * lo + w * hi).view(sigma.shape)
        return t.unsqueeze(0) if t.ndim == 0 else t

    def t_to_sigma(self, t):
        """:458-464."""
        t = t.float()
        lo, hi, w = t.floor().long(), t.ceil().long(), t.frac()
        ls = self.log_sigmas().to(t)
        v = (1 - w) * ls[lo] + w * ls[hi]
        v[torch.isnan(v) | torch.isinf(v)] = float("inf")
        return v.exp()

    def predict(self, xt, t, model, model_kwargs, guide_scale=None, guide_rescale=None):
        """The model call + CFG + std-ratio rescale (arXiv:2305.08891) of denoise(), :196-218."""
        if guide_scale is None:
            return model(xt, t=t, **model_kwargs)
        y_out = model(xt, t=t, **model_kwargs[0])
        if guide_scale == 1.0:
            return y_out
        u_out = model(xt, t=t, **model_kwargs[1])
        out = u_out + guide_scale * (y_out - u_out)
        if guide_rescale is not None:
            ratio = (y_out.flatten(1).std(dim=1) / (out.flatten(1).std(dim=1) + 1e-12)).view((-1,) + (1,) * (y_out.ndim - 1))
            out = out * (guide_rescale * ratio + (1 - guide_rescale) * 1.0)
        return out

    def x0_eps(self, xt, t, model, model_kwargs, guide_scale=None, guide_rescale=None):
        """x0 / eps of denoise(), :220-247 (no clamp / percentile on the sampling path)."""
        sig, alp = _bcast(self.sigmas, t, xt), _bcast(self.alphas, t, xt)
        out = self.predict(xt, t, model, model_kwargs, guide_scale, guide_rescale)
        if self.prediction_type == "x0":
            x0 = out
        elif self.prediction_type == "eps":
            x0 = (xt - sig * out) / alp
        else:
            x0 = alp * xt - sig * out
        return x0, (xt - alp * x0) / sig

    def ddim_reverse_sample_loop(self, x0, model, model_kwargs, guide_scale=None, guide_rescale=None, ddim_timesteps=20,
                                 reverse_steps=600):
        """:376-434: x_{t+stride} = alpha_s * x0_hat + sigma_s * eps_hat, s = min(t + stride, reverse_steps - 1)."""
        xt = x0
        stride = reverse_steps // ddim_timesteps
        for step in torch.arange(0, reverse_steps, stride):
            t = torch.full((x0.size(0),), int(step), dtype=torch.long, device=xt.device)
            x0h, eps = self.x0_eps(xt, t, model, model_kwargs, guide_scale, guide_rescale)
            s = (t + stride).clamp(0, reverse_steps - 1)
            a_s = _bcast(self.alphas, s, xt)
            xt = a_s * x0h + torch.sqrt(1 - a_s ** 2) * eps
        return xt

    def sample_sigmas(self, steps, t_max=None, t_min=None, discretization="linspace", discard_penultimate_step=True):
        """The sigma ladder of sample(), :318-357 (non-karras solvers)."""
        steps += 1 if discard_penultimate_step else 0
        t_max = self.num_timesteps - 1 if t_max is None else t_max
        t_min = 0 if t_min is None else t_min
        if discretization == "leading":
            ts = torch.arange(t_min, t_max + 1, (t_max - t_min + 1) / steps).flip(0)
        elif discretization == "linspace":
            ts = torch.linspace(t_max, t_min, steps)
        elif discretization == "trailing":
            ts = torch.arange(t_max, t_min - 1, -((t_max - t_min + 1) / steps))
        else:
            raise NotImplementedError(discretization)
        ts = torch.as_tensor(ts.clamp_(t_min, t_max), dtype=torch.float32)
        sig = self.t_to_sigma(ts)
        sig = torch.cat([sig, sig.new_zeros([1])])
        if discard_penultimate_step:
            sig = torch.cat([sig[:-2], sig[-1:]])
        return sig

    def sample_dpmpp_2m_sde(self, noise, model, model_kwargs, guide_scale=None, guide_rescale=None, steps=20, t_max=None,
                            t_min=None, discretization="linspace", eta=1.0, s_noise=1.0, solver_type="midpoint"):
        """sample(solver='dpmpp_2m_sde') :250-373 -> sample_dpmpp_2m_sde :86-142."""
        sigmas = self.sample_sigmas(steps, t_max, t_min, discretization, True).to(noise.device)

        def denoised_fn(xt, sigma):
            t = self.sigma_to_t(sigma).repeat(len(xt)).round().long()
            return self.x0_eps(xt, t, model, model_kwargs, guide_scale, guide_rescale)[0]

        x = noise * sigmas[0]
        s_min, s_max = sigmas[sigmas > 0].min(), sigmas[sigmas < float("inf")].max()
        # BrownianTreeNoiseSampler(x, sigma_min, sigma_max): seed drawn from the global RNG (:29-30)
        seed = torch.randint(0, 2 ** 63 - 1, []).item()
        tree = brownian.BrownianTree(s_min, torch.zeros_like(x), s_max, entropy=seed)

        def noise_sampler(s0, s1):
            a, b, sign = (s0, s1, 1) if s0 < s1 else (s1, s0, -1)
            return tree(a, b) * sign / (s1 - s0).abs().sqrt()

        old, h_last = None, None
        for i in range(len(sigmas) - 1):
            if sigmas[i] == float("inf"):
                den = denoised_fn(noise, sigmas[i])
                x = den + sigmas[i + 1] * noise
                h = None
            else:
                c_in = 1 / (sigmas[i] ** 2 + 1.0) ** 0.5
                den = denoised_fn(x * c_in, sigmas[i])
                if sigmas[i + 1] == 0:
                    x = den
                    h = None
                else:
                    t, s = -sigmas[i].log(), -sigmas[i + 1].log()
                    h = s - t
                    eh = eta * h
                    x = sigmas[i + 1] / sigmas[i] * (-eh).exp() * x + (-h - eh).expm1().neg() * den
                    if old is not None:
                        r = h_last / h
                        if solver_type == "heun":
                            x = x + ((-h - eh).expm1().neg() / (-h - eh) + 1) * (1 / r) * (den - old)
                        else:
                            x = x + 0.5 * (-h - eh).expm1().neg() * (1 / r) * (den - old)
                    x = x + noise_sampler(sigmas[i], sigmas[i + 1]) * sigmas[i + 1] * (-2 * eh).expm1().neg().sqrt() * s_noise
            old = den
            if h is not None:
                h_last = h
        return x
