"""guiders.py:8-40 VanillaCFG: batch doubling (unconditional half first) and x_u + scale (x_c - x_u).
The combine itself runs inside the fused sampler kernel (pn_sampler_step); this class carries the scale and
builds the doubled conditioning ONCE per sample instead of once per step."""
from __future__ import annotations

import torch

CFG_KEYS = ("vector", "crossattn", "concat", "cond_feat", "cond_bev_feat")


class VanillaCFG:
    def __init__(self, scale, dyn_thresh_config=None):
        if dyn_thresh_config is not None:
            raise NotImplementedError("only NoDynamicThresholding (the reference default) is implemented")
        self.scale = float(scale)

    def scale_schedule(self, sigma=None):
        return self.scale

    def prepare_cond(self, c: dict, uc: dict) -> dict:
        out = {}
        for k in c:
            if k in CFG_KEYS:
                out[k] = torch.cat((uc[k], c[k]), 0)
            else:
                assert c[k] == uc[k]
                out[k] = c[k]
        return out

    def prepare_inputs(self, x, s, c, uc):
        return torch.cat([x] * 2), torch.cat([s] * 2), self.prepare_cond(c, uc)


class IdentityGuider:
    scale = 1.0

    def prepare_cond(self, c, uc):
        return dict(c)

    def prepare_inputs(self, x, s, c, uc):
        return x, s, dict(c)
