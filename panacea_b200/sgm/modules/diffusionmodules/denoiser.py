"""denoiser.py:31-63 DiscreteDenoiser with EpsScaling, for the eps-prediction network.

Host side: the ascending 1000-entry sigma table, sigma<->index snapping (`sigma_to_idx` = nearest table entry)
and the per-step scalars. Device side: `input * c_in` and `net * c_out + input * c_skip` are fused into
pn_sampler_step by the sampler; `__call__` below keeps the reference call signature for
callers that use the denoiser on its own (one elementwise kernel per call)."""
from __future__ import annotations

import numpy as np
import torch

from ...util import instantiate_from_config


class Denoiser:
    def __init__(self, weighting_config, scaling_config):
        self.weighting = instantiate_from_config(weighting_config)
        self.scaling = instantiate_from_config(scaling_config)

    def w(self, sigma):
        return self.weighting(sigma)


class DiscreteDenoiser(Denoiser):
    def __init__(self, weighting_config, scaling_config, num_idx, discretization_config, do_append_zero=False,
                 quantize_c_noise=True, flip=True):
        super().__init__(weighting_config, scaling_config)
        sigmas = instantiate_from_config(discretization_config)(num_idx, do_append_zero=do_append_zero, flip=flip)
        self.sigmas = sigmas.cpu()                               # ascending when flip=True
        self._sig_np = self.sigmas.numpy().astype(np.float32)
        self.quantize_c_noise = quantize_c_noise
        if not quantize_c_noise:
            raise NotImplementedError("continuous c_noise is not used by the reference config")

    # --- host-side table logic (reference denoiser.py:49-63)
    def sigma_to_idx(self, sigma):
        s = np.asarray(sigma.detach().cpu().numpy() if torch.is_tensor(sigma) else sigma, dtype=np.float32)
        idx = np.abs(s.reshape(1, -1) - self._sig_np[:, None]).argmin(axis=0)
        out = torch.from_numpy(idx.astype(np.int64)).reshape(s.shape)
        return out.to(sigma.device) if torch.is_tensor(sigma) else out

    def idx_to_sigma(self, idx):
        return self.sigmas.to(idx.device)[idx] if torch.is_tensor(idx) else self.sigmas[idx]

    def step_scalars(self, sigma: float):
        """(timestep index, quantised sigma, c_in) for one sampler sigma."""
        idx = int(np.abs(np.float32(sigma) - self._sig_np).argmin())
        sq = float(self._sig_np[idx])
        c_in = float(np.float32(1.0) / np.sqrt(np.float32(sq) * np.float32(sq) + np.float32(1.0)))
        return idx, sq, c_in

    @torch.no_grad()
    def __call__(self, network, input, sigma, cond):
        """Reference signature: returns the denoised sample network(input*c_in, idx, cond) * c_out + input."""
        from ....ops import NativeOps
        ops = getattr(self, "_ops", None) or NativeOps()
        self._ops = ops
        s0 = float(sigma.reshape(-1)[0])
        if not torch.all(sigma == sigma.reshape(-1)[0]):
            raise NotImplementedError("per-sample sigmas within one batch are not supported")
        idx, sq, c_in = self.step_scalars(s0)
        x = input.float().contiguous()
        x_in = ops.scale_dup(x, c_in, 1)
        t = torch.full((x.shape[0],), idx, dtype=torch.int64, device=x.device)
        eps = network(x_in, t, cond)
        out = ops.scale_dup(eps.float().contiguous(), -sq, 1)
        return ops.add_(out, x)
