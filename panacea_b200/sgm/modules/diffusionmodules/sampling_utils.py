"""sampling_utils.py:7-48 helpers, and the host scalars of the samplers (sampling.py:96-365).

The reference computes every sigma-dependent scalar of its samplers on float32 torch tensors. The functions below take
the same float32 values and evaluate the same expressions on one-element float32 tensors, so the scalars handed to the
update kernel (pn_sampler_step) are the reference's values bit for bit. The LMS coefficients are integrated exactly
(polynomial algebra in float64) instead of with scipy's `quad`."""
from __future__ import annotations

import numpy as np
import torch


class NoDynamicThresholding:
    def __call__(self, uncond, cond, scale):
        return uncond + scale * (cond - uncond)


def append_dims(x, target_dims):
    return x[(...,) + (None,) * (target_dims - x.ndim)]


def to_d(x, sigma, denoised):
    return (x - denoised) / append_dims(sigma, x.ndim)


def to_neg_log_sigma(sigma):
    return sigma.log().neg()


def to_sigma(neg_log_sigma):
    return neg_log_sigma.neg().exp()


def _t(v) -> torch.Tensor:
    return torch.tensor([float(v)], dtype=torch.float32)


def get_ancestral_step(sigma_from, sigma_to, eta=1.0):
    """(sigma_down, sigma_up) of an ancestral step from sigma_from to sigma_to (float32 tensors). eta = 0 returns
    (sigma_to, 0.0): the deterministic limit."""
    if not eta:
        return sigma_to, 0.0
    sigma_up = torch.minimum(sigma_to, eta * (sigma_to ** 2 * (sigma_from ** 2 - sigma_to ** 2) / sigma_from ** 2) ** 0.5)
    sigma_down = (sigma_to ** 2 - sigma_up ** 2) ** 0.5
    return sigma_down, sigma_up


def ancestral_scalars(sigma: float, sigma_next: float, eta: float) -> tuple[float, float]:
    """Host (sigma_down, sigma_up) for float32 sigmas."""
    down, up = get_ancestral_step(_t(sigma), _t(sigma_next), eta)
    return float(down), float(up)


def edm_churn_scalars(sigma: float, gamma: float) -> tuple[float, float]:
    """EDMSampler.sampler_step (sampling.py:96-100): (sigma_hat, amplitude of the churn noise sqrt(sigma_hat^2 - sigma^2))."""
    s = _t(sigma)
    hat = s * (gamma + 1.0)
    return float(hat), float((hat ** 2 - s ** 2) ** 0.5)


def edm_gamma(sigma: float, s_churn: float, s_tmin: float, s_tmax: float, num_sigmas: int) -> float:
    """EDMSampler.__call__ (sampling.py:118-122); the window test compares the float32 sigma like the reference."""
    s = _t(sigma)
    return min(s_churn / (num_sigmas - 1), 2 ** 0.5 - 1) if bool(s_tmin <= s) and bool(s <= s_tmax) else 0.0


def sub32(a: float, b: float) -> float:
    """a - b of two float32 values, rounded to float32 (the reference's dt = next_sigma - sigma on tensors)."""
    return float(_t(a) - _t(b))


def dpmpp2s_scalars(sigma: float, sigma_down: float) -> tuple[float, tuple[float, float, float, float]]:
    """DPMPP2SAncestralSampler.get_variables / get_mult (sampling.py:251-263) for sigma_down > 0:
    (sigma of the midpoint evaluation to_sigma(s), (mult1, mult2, mult3, mult4))."""
    t, t_next = to_neg_log_sigma(_t(sigma)), to_neg_log_sigma(_t(sigma_down))
    h = t_next - t
    s = t + 0.5 * h
    m = (to_sigma(s) / to_sigma(t), (-0.5 * h).expm1(), to_sigma(t_next) / to_sigma(t), (-h).expm1())
    return float(to_sigma(s)), tuple(float(v) for v in m)


def dpmpp2m_scalars(sigma_prev, sigma: float, sigma_next: float):
    """DPMPP2MSampler.get_variables / get_mult (sampling.py:291-311): (mult1, mult2) and (mult3, mult4), the latter None
    on the first step (sigma_prev None) and at sigma_next = 0, where the reference takes x_standard. At sigma_next = 0,
    t_next = inf gives mult1 = 0 and mult2 = -1 exactly as on the reference's tensors; the second pair would be inf
    there and is never formed."""
    t, t_next = to_neg_log_sigma(_t(sigma)), to_neg_log_sigma(_t(sigma_next))
    h = t_next - t
    m12 = (float(to_sigma(t_next) / to_sigma(t)), float((-h).expm1()))
    if sigma_prev is None or sigma_next < 1e-14:
        return m12, None
    r = (t - to_neg_log_sigma(_t(sigma_prev))) / h
    return m12, (float(1 + 1 / (2 * r)), float(1 / (2 * r)))


def linear_multistep_coeff(order, t, i, j, epsrel=1e-4):
    """Integral over [t[i], t[i+1]] of the Lagrange basis polynomial of node t[i-j] on the nodes t[i], ..., t[i-order+1]
    (sampling_utils.py:12-24), computed exactly: the polynomial is formed and integrated in float64 (numpy). `epsrel`
    is accepted for signature compatibility; the result is exact up to float64 rounding."""
    if order - 1 > i:
        raise ValueError(f"Order {order} too high for step {i}")
    nodes = np.asarray(t, dtype=np.float64)
    poly = np.polynomial.Polynomial([1.0])
    for k in range(order):
        if k != j:
            poly = poly * np.polynomial.Polynomial([-nodes[i - k], 1.0]) / (nodes[i - j] - nodes[i - k])
    prim = poly.integ()
    return float(prim(nodes[i + 1]) - prim(nodes[i]))
