"""discretizer.py:11-69 LegacyDDPMDiscretization (numpy on the host: float64 schedule, fp32 sigmas) and EDMDiscretization."""
from __future__ import annotations

import numpy as np
import torch


def generate_roughly_equally_spaced_steps(num_substeps: int, max_step: int) -> np.ndarray:
    return np.linspace(max_step - 1, 0, num_substeps, endpoint=False).astype(int)[::-1]


class LegacyDDPMDiscretization:
    def __init__(self, linear_start=0.00085, linear_end=0.0120, num_timesteps=1000):
        self.num_timesteps = num_timesteps
        betas = np.linspace(linear_start ** 0.5, linear_end ** 0.5, num_timesteps, dtype=np.float64) ** 2
        self.alphas_cumprod = np.cumprod(1.0 - betas, axis=0)

    def get_sigmas(self, n, device="cpu"):
        if n < self.num_timesteps:
            ac = self.alphas_cumprod[generate_roughly_equally_spaced_steps(n, self.num_timesteps)]
        elif n == self.num_timesteps:
            ac = self.alphas_cumprod
        else:
            raise ValueError(n)
        sig = torch.tensor((1 - ac) / ac, dtype=torch.float32, device=device) ** 0.5
        return torch.flip(sig, (0,))

    def __call__(self, n, do_append_zero=True, device="cpu", flip=False):
        sig = self.get_sigmas(n, device=device)
        if do_append_zero:
            sig = torch.cat([sig, sig.new_zeros([1])])
        return sig if not flip else torch.flip(sig, (0,))


class EDMDiscretization:
    """discretizer.py:28-39: Karras et al. sigmas, rho-th root spaced between sigma_max and sigma_min (float32 ramp).
    They are not entries of the denoiser's table: the denoiser snaps them (denoiser.py:49-63)."""

    def __init__(self, sigma_min=0.02, sigma_max=80.0, rho=7.0):
        self.sigma_min = sigma_min
        self.sigma_max = sigma_max
        self.rho = rho

    def get_sigmas(self, n, device="cpu"):
        ramp = torch.linspace(0, 1, n, device=device)
        lo, hi = self.sigma_min ** (1 / self.rho), self.sigma_max ** (1 / self.rho)
        return (hi + ramp * (lo - hi)) ** self.rho

    def __call__(self, n, do_append_zero=True, device="cpu", flip=False):
        sig = self.get_sigmas(n, device=device)
        if do_append_zero:
            sig = torch.cat([sig, sig.new_zeros([1])])
        return sig if not flip else torch.flip(sig, (0,))
