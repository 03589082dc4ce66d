"""TEST INFRASTRUCTURE — CPU oracle for the sampler loop: fp32 restatement of the reference's
EulerEDMSampler + VanillaCFG + DiscreteDenoiser(EpsScaling, LegacyDDPMDiscretization)
(configs/inference_nuscenes.yaml:18-28,115-126). Pinned by tests/test_oracle_golden.py against known-answer
values and sampler loops computed from the reference in the build container (SURVEY.md section 8c).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this module.
"""
from __future__ import annotations

import numpy as np
import torch


def ddpm_alphas_cumprod(num_timesteps: int = 1000, linear_start: float = 0.00085, linear_end: float = 0.0120):
    """discretizer.py:42-56 + util.py:19-31: betas linear in sqrt-space (float64), cumulative product of 1-beta."""
    betas = torch.linspace(linear_start ** 0.5, linear_end ** 0.5, num_timesteps, dtype=torch.float64) ** 2
    return np.cumprod(1.0 - betas.numpy(), axis=0)


def legacy_ddpm_sigmas(n: int, num_timesteps: int = 1000, append_zero: bool = True) -> torch.Tensor:
    """discretizer.py:11-14,58-69,18-21: descending sigmas at steps linspace(999, 0, n, endpoint=False)[::-1]."""
    ac = ddpm_alphas_cumprod(num_timesteps)
    if n < num_timesteps:
        steps = np.linspace(num_timesteps - 1, 0, n, endpoint=False).astype(int)[::-1]
        ac = ac[steps]
    elif n != num_timesteps:
        raise ValueError(n)
    sig = torch.tensor((1 - ac) / ac, dtype=torch.float32) ** 0.5
    sig = torch.flip(sig, (0,))
    if append_zero:
        sig = torch.cat([sig, sig.new_zeros([1])])
    return sig


class DiscreteDenoiserPort:
    """denoiser.py:31-63 with EpsScaling (denoiser_scaling.py:16-22): ascending table of 1000 sigmas; sigma and
    c_noise are snapped to the nearest table entry; the network sees the int64 index."""

    def __init__(self, num_idx: int = 1000):
        self.sigmas = torch.flip(legacy_ddpm_sigmas(num_idx, append_zero=False), (0,))   # flip=True -> ascending

    def sigma_to_idx(self, sigma: torch.Tensor) -> torch.Tensor:
        return (sigma - self.sigmas[:, None]).abs().argmin(dim=0).view(sigma.shape)

    def __call__(self, network, x, sigma, cond):
        sigma = self.sigmas[self.sigma_to_idx(sigma)]
        shape = sigma.shape
        s = sigma.reshape(-1, *([1] * (x.ndim - 1)))
        c_skip = torch.ones_like(s)
        c_out = -s
        c_in = 1 / (s ** 2 + 1.0) ** 0.5
        c_noise = self.sigma_to_idx(s.clone().reshape(shape))
        return network(x * c_in, c_noise, cond) * c_out + x * c_skip


CFG_KEYS = ("vector", "crossattn", "concat", "cond_feat", "cond_bev_feat")


def cfg_prepare(x, s, c: dict, uc: dict):
    """guiders.py:31-40 VanillaCFG.prepare_inputs: unconditional half FIRST."""
    out = {}
    for k in c:
        if k in CFG_KEYS:
            out[k] = torch.cat((uc[k], c[k]), 0)
        else:
            out[k] = c[k]
    return torch.cat([x] * 2), torch.cat([s] * 2), out


@torch.no_grad()
def euler_edm_sample(network, x, cond: dict, uc: dict, num_steps: int, scale: float = 5.0, denoiser=None, max_steps=None):
    """sampling.py:44-60,96-133,214-218 with s_churn=0 (gamma=0): deterministic Euler steps in sigma space.
    `network(x_in, idx, cond_dict) -> eps`."""
    den = DiscreteDenoiserPort() if denoiser is None else denoiser
    sigmas = legacy_ddpm_sigmas(num_steps)
    x = x * torch.sqrt(1.0 + sigmas[0] ** 2.0)
    s_in = x.new_ones([x.shape[0]])
    for i in range(len(sigmas) - 1 if max_steps is None else min(max_steps, len(sigmas) - 1)):
        sigma, nxt = s_in * sigmas[i], s_in * sigmas[i + 1]
        xx, ss, cc = cfg_prepare(x, sigma, cond, uc)
        d2 = den(network, xx, ss, cc)
        x_u, x_c = d2.chunk(2)
        denoised = x_u + scale * (x_c - x_u)                     # sampling_utils.py:7-9
        d = (x - denoised) / sigma.reshape(-1, *([1] * (x.ndim - 1)))   # sampling_utils.py:39-40
        dt = (nxt - sigma).reshape(-1, *([1] * (x.ndim - 1)))
        x = x + dt * d
    return x
