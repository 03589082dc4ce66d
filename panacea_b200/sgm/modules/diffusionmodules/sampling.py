"""sampling.py:24-365: the reference's samplers around one fused update kernel per network evaluation.

Every sampler — EulerEDMSampler (with s_churn = 0 the "DDIM (eta=0)" of the reference config,
configs/inference_nuscenes.yaml:115-126, or with churn), Heun, Euler-ancestral, DPM++ 2S a, DPM++ 2M, LMS — runs
through the one host loop of `_Sampler`: the sigma-dependent scalars are computed on the host once per sample
(sampling_utils.py, the reference's float32 expressions), and every eps evaluation of the CFG-doubled batch (ControlNet
+ UNet, optionally one CUDA graph replay) is followed by exactly one pn_sampler_step that applies the denoiser
scalings, the guidance, the sampler's update, its noise and writes the next network input (scaled and batch-doubled).
The reference's per-step torch.cat / dict rebuild (guiders.py:31-40) happens once per sample here. State that a
sampler keeps between evaluations (Heun's d, the evaluation point of Heun / DPM++ 2S, DPM++ 2M's old denoised, LMS's
derivatives) lives in latent-sized fp32 buffers the sampler owns, never in the network's output buffer.

Noise: `noise_sampler` (the reference's attribute) is None by default, and the noise is then drawn inside the kernel
(Philox4x32-10, seed `noise_seed`, or one draw of torch's generator on the latent's device per sample when that is None,
so torch.manual_seed makes a run reproducible). A user-set `noise_sampler(x)` is called exactly where the reference
calls its noise source: once per step on the ancestral samplers (also on the last step, whose draw torch.where
discards), and before every EDM step with gamma > 0 (the reference's torch.randn_like). It receives the latent tensor
and must return N(0,1) draws of its shape."""
from __future__ import annotations

from dataclasses import dataclass, field

import torch

from ...util import default, instantiate_from_config
from . import sampling_utils as U

DEFAULT_GUIDER = {"target": "sgm.modules.diffusionmodules.guiders.IdentityGuider"}


class BoundDenoiser:
    """What `DiffusionEngine3D.sample` passes to the sampler in the reference is a lambda closing over
    (denoiser, model) (diffusion.py:251-254); this object is the same callable with the two parts visible, so the
    sampler can fuse the denoiser scalings, the guidance and its update into one kernel per evaluation."""

    def __init__(self, denoiser, network):
        self.denoiser = denoiser
        self.network = network

    def __call__(self, x, sigma, cond):
        return self.denoiser(self.network, x, sigma, cond)


@dataclass
class _Noise:
    """Noise of one kernel: x += (z * mul) * amp. `call`: a user noise_sampler is called here; `apply`: the draw is added
    (the ancestral samplers call the user's source on the last step too and discard the draw)."""
    mul: float
    amp: float
    draw: int
    call: bool = True
    apply: bool = True


@dataclass
class _Eval:
    """One network evaluation and the pn_sampler_step that follows it."""
    sigma: float                  # sigma handed to the guider / denoiser (snapped by the denoiser for c_in, c_out, t)
    mode: str                     # ops.SAMPLER_MODES key
    at_eval: bool = False         # the network input is the sampler's x_eval buffer, not x
    step: int | None = None       # the sampler step this evaluation completes
    kw: dict = field(default_factory=dict)      # kernel scalars (sigma for to_d, dt, m, lms_*)
    noise: _Noise | None = None


class _Sampler:
    """Shared host loop of the samplers. Subclasses return the evaluation plan of one sample from `_plan(sigmas)`:
    (noise applied before the first evaluation or None, [_Eval, ...])."""

    state_buffers = ()            # which of x_eval / d / old_denoised the sampler keeps

    def __init__(self, discretization_config, num_steps=None, guider_config=None, verbose=False, device="cuda"):
        self.num_steps = num_steps
        self.discretization = instantiate_from_config(discretization_config)
        self.guider = instantiate_from_config(default(guider_config, DEFAULT_GUIDER))
        self.verbose = verbose
        self.device = device
        self.last_timestep_indices = []
        self.step_callback = None           # optional: called as step_callback(i, x) after every sampler step
        self.noise_sampler = None
        self.noise_seed = None
        self._ops = None

    @property
    def ops(self):
        """Op set of the update kernels (panacea_b200.ops.NativeOps unless replaced)."""
        if self._ops is None:
            from ....ops import NativeOps
            self._ops = NativeOps()
        return self._ops

    @ops.setter
    def ops(self, value):
        self._ops = value

    def sigmas(self, num_steps=None):
        return self.discretization(self.num_steps if num_steps is None else num_steps, device="cpu")

    def _plan(self, sig):
        raise NotImplementedError

    def _check_guider(self):
        if not (hasattr(self.guider, "scale") and not type(self.guider).__name__.startswith("Identity")):
            raise NotImplementedError("this sampler implements VanillaCFG (the reference config)")

    @torch.no_grad()
    def __call__(self, denoiser, x, cond, uc=None, num_steps=None):
        """x [N,4,H,W] initial noise (unit variance); cond / uc dicts as produced by the conditioner. `denoiser` is any
        callable (x, sigma, cond) -> denoised, like the reference's lambda (diffusion.py:251-254); a `BoundDenoiser`
        takes the fused path. Returns the final latent, like the reference."""
        self._check_guider()
        ops = self.ops
        uc = default(uc, cond)
        sig_t = self.sigmas(num_steps)
        sig = [float(s) for s in sig_t]
        first_noise, plan = self._plan(sig)
        # prepare_sampling_loop (sampling.py:44-55): x *= sqrt(1 + sigma_0^2), on float32 values
        x = ops.scale_dup(x.float().contiguous(), float(torch.sqrt(1.0 + sig_t[0] ** 2.0)), 1)
        ring = getattr(self, "lms_ring", 1)
        bufs = {name: torch.empty(((ring if name == "d" else 1) * x.shape[0], *x.shape[1:]), device=x.device,
                                  dtype=torch.float32) for name in self.state_buffers}     # never the network's output buffer
        seed = None
        if self.noise_sampler is None and any(nz is not None and nz.apply for nz in [first_noise] + [e.noise for e in plan]):
            seed = self.noise_seed
            if seed is None:        # one draw of torch's generator on the latent's device per sample
                seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64, device=x.device).item())

        def noise_kw(nz):
            if nz is None:
                return {}
            z = self.noise_sampler(x) if self.noise_sampler is not None and nz.call else None
            if not nz.apply:
                return {}
            kw = {"noise_mul": nz.mul, "noise_amp": nz.amp}
            if self.noise_sampler is not None:
                kw["noise"] = z.to(device=x.device, dtype=torch.float32).contiguous()
            else:
                kw.update(seed=seed, draw=nz.draw)
            return kw

        scale = self.guider.scale
        if not isinstance(denoiser, BoundDenoiser):
            return self._generic_loop(ops, denoiser, x, cond, uc, plan, first_noise, bufs, noise_kw, scale)
        den, net = denoiser.denoiser, denoiser.network
        cc = self.guider.prepare_cond(cond, uc)                   # once per sample
        if hasattr(net, "prepare"):
            net.prepare(cc)                                       # step-invariant conditioning work, once per sample
        n = x.shape[0]
        scal = [den.step_scalars(e.sigma) for e in plan]
        self.last_timestep_indices = [s[0] for s in scal]
        t_all = torch.tensor([[s[0]] * (2 * n) for s in scal], dtype=torch.int64, device=x.device)
        x_in = torch.empty((2 * n, *x.shape[1:]), device=x.device, dtype=torch.float32)
        ops.sampler_step("input", x, None, x_in, c_in_next=scal[0][2], **noise_kw(first_noise))
        for k, e in enumerate(plan):
            eps = net(x_in, t_all[k], cc, return_static=True) if hasattr(net, "static_io") else net(x_in, t_all[k], cc)
            last = k + 1 == len(plan)
            ops.sampler_step(e.mode, x, eps.float().contiguous(), None if last else x_in, sigma_q=scal[k][1], scale=scale,
                             c_in_next=0.0 if last else scal[k + 1][2], **bufs, **e.kw, **noise_kw(e.noise))
            if e.step is not None and self.step_callback is not None:
                self.step_callback(e.step, x)
        return x

    def _generic_loop(self, ops, denoiser, x, cond, uc, plan, first_noise, bufs, noise_kw, scale):
        """The reference's call contract: an opaque `denoiser(x2, sigma2, cond2) -> denoised2` per evaluation with the
        guider's doubled inputs; guidance + update in one kernel (net_is_denoised)."""
        n = x.shape[0]
        self.last_timestep_indices = []
        if first_noise is not None:
            kw = noise_kw(first_noise)
            if kw:
                ops.sampler_step("input", x, **kw)
        for e in plan:
            point = bufs["x_eval"] if e.at_eval else x
            s_in = torch.full((n,), e.sigma, dtype=torch.float32, device=x.device)
            x2, s2, c2 = self.guider.prepare_inputs(point, s_in, cond, uc)
            den2 = denoiser(x2, s2, c2).float().contiguous()
            ops.sampler_step(e.mode, x, den2, None, scale=scale, net_is_denoised=True, **bufs, **e.kw, **noise_kw(e.noise))
            if e.step is not None and self.step_callback is not None:
                self.step_callback(e.step, x)
        return x


class EDMSampler(_Sampler):
    """sampling.py:85-133. With s_churn > 0, the steps whose sigma lies in [s_tmin, s_tmax] first move x to
    sigma_hat = sigma (1 + gamma) with fresh noise; that noise is added by the kernel that ends the step before (or by
    one extra kernel before the first evaluation)."""

    heun = False

    def __init__(self, discretization_config, num_steps=None, guider_config=None, verbose=False, device="cuda",
                 s_churn=0.0, s_tmin=0.0, s_tmax=float("inf"), s_noise=1.0):
        super().__init__(discretization_config, num_steps, guider_config, verbose, device)
        self.s_churn = s_churn
        self.s_tmin = s_tmin
        self.s_tmax = s_tmax
        self.s_noise = s_noise
        self.state_buffers = ("x_eval", "d") if self.heun else ()

    def _plan(self, sig):
        steps = len(sig) - 1
        churn = []
        for i in range(steps):
            gamma = U.edm_gamma(sig[i], self.s_churn, self.s_tmin, self.s_tmax, len(sig))
            hat, amp = U.edm_churn_scalars(sig[i], gamma)
            churn.append((gamma, hat, amp))

        def churn_noise(i):
            if i >= steps or not churn[i][0] > 0:
                return None
            return _Noise(self.s_noise, churn[i][2], draw=i)

        plan = []
        for i in range(steps):
            hat = churn[i][1]
            dt = U.sub32(sig[i + 1], hat)
            if self.heun and not sig[i + 1] < 1e-14:
                plan.append(_Eval(hat, "heun_a", kw={"sigma": hat, "dt": dt}))
                plan.append(_Eval(sig[i + 1], "heun_b", at_eval=True, step=i, kw={"sigma": sig[i + 1], "dt": dt},
                                  noise=churn_noise(i + 1)))
            else:
                plan.append(_Eval(hat, "euler", step=i, kw={"sigma": hat, "dt": dt}, noise=churn_noise(i + 1)))
        return churn_noise(0), plan


class EulerEDMSampler(EDMSampler):
    """sampling.py:214-218. With s_churn = 0 (the reference config) every step is one "euler" evaluation at
    sigma_hat = sigma, with no noise."""


class HeunEDMSampler(EDMSampler):
    """sampling.py:221-237: Euler predictor, then a second evaluation at the predictor and the trapezoidal correction;
    the last step (sigma_next = 0) stays an Euler step and saves the evaluation, like the reference."""

    heun = True


class AncestralSampler(_Sampler):
    """sampling.py:136-173. eta = 0 is supported as the deterministic limit (sigma_down = sigma_next, no noise and no
    noise_sampler call); the reference raises there (get_ancestral_step returns the float 0.0 for sigma_up, which
    append_dims cannot take)."""

    def __init__(self, discretization_config, num_steps=None, guider_config=None, verbose=False, device="cuda",
                 eta=1.0, s_noise=1.0):
        super().__init__(discretization_config, num_steps, guider_config, verbose, device)
        self.eta = eta
        self.s_noise = s_noise

    def _ancestral_noise(self, i, sigma_next, sigma_up):
        # torch.where evaluates both branches: the reference draws every step, and adds the draw where sigma_next > 0
        if not self.eta:
            return None
        return _Noise(self.s_noise, sigma_up, draw=i, apply=sigma_next > 0.0)


class EulerAncestralSampler(AncestralSampler):
    """sampling.py:240-247."""

    def _plan(self, sig):
        plan = []
        for i in range(len(sig) - 1):
            down, up = U.ancestral_scalars(sig[i], sig[i + 1], self.eta)
            plan.append(_Eval(sig[i], "euler", step=i, kw={"sigma": sig[i], "dt": U.sub32(down, sig[i])},
                              noise=self._ancestral_noise(i, sig[i + 1], up)))
        return None, plan


class DPMPP2SAncestralSampler(AncestralSampler):
    """sampling.py:250-287: a second evaluation at the exponential-integrator midpoint; where sigma_down = 0 the step is
    the ancestral Euler step with one evaluation, like the reference."""

    state_buffers = ("x_eval",)

    def _plan(self, sig):
        plan = []
        for i in range(len(sig) - 1):
            down, up = U.ancestral_scalars(sig[i], sig[i + 1], self.eta)
            noise = self._ancestral_noise(i, sig[i + 1], up)
            if down < 1e-14:
                plan.append(_Eval(sig[i], "euler", step=i, kw={"sigma": sig[i], "dt": U.sub32(down, sig[i])}, noise=noise))
                continue
            sigma_s, m = U.dpmpp2s_scalars(sig[i], down)
            plan.append(_Eval(sig[i], "dpmpp2s_a", kw={"m": m}))
            plan.append(_Eval(sigma_s, "dpmpp2s_b", at_eval=True, step=i, kw={"m": m}, noise=noise))
        return None, plan


class DPMPP2MSampler(_Sampler):
    """sampling.py:290-365: the second-order multistep update from the previous step's denoised latent (kept in a buffer
    of the sampler); the first step and the last one (sigma_next = 0) take the first-order update."""

    state_buffers = ("old_denoised",)

    def _plan(self, sig):
        plan = []
        for i in range(len(sig) - 1):
            m12, m34 = U.dpmpp2m_scalars(None if i == 0 else sig[i - 1], sig[i], sig[i + 1])
            plan.append(_Eval(sig[i], "dpmpp2m", step=i, kw={"m": m12 + (m34 or (0.0, 0.0)), "use_old": m34 is not None}))
        return None, plan


class LinearMultistepSampler(_Sampler):
    """sampling.py:176-211: linear multistep over the last `order` (<= 4) derivatives, kept in a ring of latent buffers."""

    state_buffers = ("d",)

    def __init__(self, discretization_config, num_steps=None, guider_config=None, verbose=False, device="cuda", order=4):
        super().__init__(discretization_config, num_steps, guider_config, verbose, device)
        if not 1 <= order <= 4:
            raise NotImplementedError("LinearMultistepSampler: order 1..4 are implemented")
        self.order = order
        self.lms_ring = order

    def _plan(self, sig):
        plan = []
        for i in range(len(sig) - 1):
            cur = min(i + 1, self.order)
            coeff = [U.linear_multistep_coeff(cur, sig, i, j) for j in range(cur)]
            plan.append(_Eval(sig[i], "lms", step=i, kw={"sigma": sig[i], "lms_coeff": coeff, "lms_ring": self.order,
                                                         "lms_slot": i % self.order}))
        return None, plan
