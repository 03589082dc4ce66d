"""Cost of each sampler at the benchmarked shape: full-size UNet + ControlNet (bf16 fast path, one CUDA graph per
evaluation), T = 8 frames of 6 views of 32 x 56 latents, CFG scale 5, LegacyDDPM discretisation.

One JSON line per sampler: network evaluations per sample, the device time of pn_sampler_step per evaluation (CUDA
events around each update kernel alone) and the wall time of one whole sample at --steps (CUDA events around the
sampler call, after a warm-up sample that captures the graph).

    python tools/bench_samplers.py --steps 25 [--repeats 3] [--out profiles/bench_samplers.jsonl]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

SAMPLERS = {
    "euler": ("EulerEDMSampler", {}),
    "euler_churn": ("EulerEDMSampler", {"s_churn": 2.0, "s_tmin": 0.5, "s_tmax": 10.0}),
    "heun": ("HeunEDMSampler", {}),
    "euler_ancestral": ("EulerAncestralSampler", {"eta": 1.0}),
    "dpmpp2s_ancestral": ("DPMPP2SAncestralSampler", {"eta": 1.0}),
    "dpmpp2m": ("DPMPP2MSampler", {}),
    "lms": ("LinearMultistepSampler", {"order": 4}),
}


class TimedOps:
    """Forwards to the sampler's op set and brackets every pn_sampler_step with a pair of CUDA events."""

    def __init__(self, ops):
        self.ops = ops
        self.events = []

    def __getattr__(self, name):
        return getattr(self.ops, name)

    def sampler_step(self, *a, **k):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = self.ops.sampler_step(*a, **k)
        e.record()
        self.events.append((s, e))
        return out


def gpu_info() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return torch.cuda.get_device_name()


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=25)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args(argv)
    import bench as B
    from panacea_b200.sgm.modules.diffusionmodules.sampling import BoundDenoiser
    from panacea_b200.sgm.util import instantiate_from_config
    if not torch.cuda.is_available():
        raise RuntimeError("bench_samplers measures on a CUDA device; none is present")
    dev = torch.device("cuda", 0)
    seed = 3407
    pipe = B.build_pipeline(dev, seed)
    host = B.synth_inputs_host(seed)
    c = {"cond_feat": host["hint"].to(dev), "concat": host["concat"].to(dev), "crossattn": host["c_txt"].to(dev)}
    uc = dict(c, crossattn=host["uc_txt"].to(dev))
    noise = host["noise"].to(dev)
    fn = BoundDenoiser(pipe.denoiser, pipe.wrapper)
    info = gpu_info()
    lines = []
    for name, (cls, kw) in SAMPLERS.items():
        s = instantiate_from_config({"target": f"sgm.modules.diffusionmodules.sampling.{cls}", "params": dict(
            num_steps=a.steps, discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"},
            guider_config={"target": "sgm.modules.diffusionmodules.guiders.VanillaCFG", "params": {"scale": 5.0}}, **kw)})
        s.noise_seed = 1
        s(fn, noise.clone(), c, uc)                                  # warm-up: graph capture, conditioning, allocator
        timed = TimedOps(s.ops)
        s.ops = timed
        times = []
        for _ in range(a.repeats):
            x = noise.clone()
            st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            st.record()
            s(fn, x, c, uc)
            en.record()
            torch.cuda.synchronize()
            times.append(st.elapsed_time(en))
        evals = len(s.last_timestep_indices)
        upd = [st_.elapsed_time(en_) * 1e3 for st_, en_ in timed.events]
        rec = {"sampler": name, "class": cls, "kwargs": kw, "steps": a.steps, "evaluations_per_sample": evals,
               "update_kernels": len(upd) // a.repeats,
               "update_us_per_evaluation": sum(upd) / max(len(upd), 1),
               "ms_per_sample": min(times), "ms_per_sample_all": times, "ms_per_evaluation": min(times) / evals,
               "latent": list(noise.shape), "cfg_scale": 5.0, "precision": "bf16", "gpu": info}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
