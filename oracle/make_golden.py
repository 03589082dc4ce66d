"""TEST INFRASTRUCTURE — generates tests/golden/*.pt by running the UNMODIFIED reference modules
(/root/reference, imported through oracle/ref_loader.py) on the seeded cases of oracle/cases.py.

Run in the build container only:  python -m oracle.make_golden [--only name,...] [--skip-full]
Outputs are small (the reference OUTPUT tensors + known-answer values); inputs/weights are re-derived
from seeds by whoever consumes a fixture.
"""
from __future__ import annotations

import argparse
import gzip
import json
import sys
import time
from pathlib import Path

import torch

from . import cases as Cs
from . import ref_loader as R
from . import unet_port as P

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden"

# Every fixture stays below 1 MB. Larger eps outputs are stored as the fixed sample eps.flatten()[::EPS_SAMPLE_STRIDE];
# the stride is coprime with 2, 3 and 7, so the sample visits every frame, channel, row and column of the 32x336 and
# 32x384 latents.
EPS_FULL_MAX_ELEMENTS = 1 << 17
EPS_SAMPLE_STRIDE = 5


def shrink_eps(g: dict) -> dict:
    """A golden_eps() record whose output is too large to store whole -> the same record with a strided sample of it
    (`eps_shape` / `eps_stride` tell the consumer how to sample its own output the same way)."""
    eps = g["eps"]
    if eps.numel() <= EPS_FULL_MAX_ELEMENTS:
        return g
    return {**g, "eps": eps.flatten()[::EPS_SAMPLE_STRIDE].clone(), "eps_shape": tuple(eps.shape),
            "eps_stride": EPS_SAMPLE_STRIDE}


def trajectory_steps(num_steps: int) -> list[int]:
    """Steps whose start-of-step latent a sampler-loop fixture keeps: the first four (the CPU port follows the first
    three steps) and every eighth."""
    return sorted(set(range(min(4, num_steps))) | set(range(0, num_steps, 8)))


@torch.no_grad()
def golden_eps(case: Cs.EpsCase) -> dict:
    kw = case.unet_kwargs()
    model = R.build_reference_model(kw)
    sd = Cs.make_weights(case)
    missing = model.load_state_dict(sd, strict=True)
    x, t, c = Cs.make_inputs(case)
    t0 = time.time()
    with R.view_height_shim(case.H, case.w):
        eps = model(x, t, dict(c))
    dt = time.time() - t0
    return shrink_eps({"meta": case.meta(), "eps": eps.contiguous(), "seconds": dt, "torch": str(torch.__version__),
                       "threads": torch.get_num_threads()})


@torch.no_grad()
def golden_reference_model() -> dict:
    """What the reference's own modules say about the network itself: the state-dict key set with shapes (tiny_3to1
    case), the tensors its default init leaves at zero (the zero_module()'d tails), and the output of a freshly
    constructed model on the tiny_2to1 inputs."""
    case = Cs.GOLDEN_CASES[1]
    sd = R.build_reference_model(case.unet_kwargs()).state_dict()
    fresh_case = Cs.GOLDEN_CASES[0]
    fresh = R.build_reference_model(fresh_case.unet_kwargs())
    x, t, c = Cs.make_inputs(fresh_case)
    out = fresh(x, t, dict(c))
    return {"case": case.name, "state_spec": {k: list(v.shape) for k, v in sd.items()},
            "fresh_case": fresh_case.name,
            "fresh_zero_keys": sorted(k for k, v in fresh.state_dict().items() if not v.any()),
            "fresh_output_shape": list(out.shape), "fresh_output_max_abs": out.abs().max().item()}


@torch.no_grad()
def golden_kat() -> dict:
    """Known-answer values of the sampler stack and embeddings, from the reference classes."""
    ref = R.import_reference()
    disc = ref.discretizer.LegacyDDPMDiscretization()
    out = {"sigmas_25": disc(25), "sigmas_50": disc(50), "sigmas_10": disc(10)}
    den = ref.denoiser.DiscreteDenoiser(
        weighting_config={"target": "sgm.modules.diffusionmodules.denoiser_weighting.EpsWeighting"},
        scaling_config={"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
        num_idx=1000,
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"})
    out["denoiser_sigmas"] = den.sigmas.clone()
    out["idx_of_sigmas_25"] = den.sigma_to_idx(out["sigmas_25"][:-1])
    out["idx_of_sigmas_50"] = den.sigma_to_idx(out["sigmas_50"][:-1])
    out["pos_embed_T4_C8"] = ref.attention.create_1d_absolute_sin_cos_embedding(4, 8)
    out["pos_embed_T8_C64"] = ref.attention.create_1d_absolute_sin_cos_embedding(8, 64)
    out["timestep_embedding_320"] = ref.util.timestep_embedding(torch.tensor([0, 39, 500, 999]), 320)
    return out


@torch.no_grad()
def golden_sampler(case: Cs.EpsCase, num_steps: int = 10, scale: float = 5.0, use_last_frame: bool = False,
                   share_noise_level: float = 0.07, trajectory: bool = False) -> dict:
    """Full reference loop: EulerEDMSampler + VanillaCFG + DiscreteDenoiser around the reference wrapper.
    use_last_frame: BASELINE config 4 — the concat latent is zero except for the last frame
    (nuscenes_datasets_video.py:559-566) and the initial noise is mixed as DiffusionEngine3D.sample does
    (diffusion.py:242-249, restated below because the Lightning module itself needs the conditioner/VAE configs).
    trajectory: also record x at the start of every step (error-vs-step curves on the GPU)."""
    ref = R.import_reference()
    model = R.build_reference_model(case.unet_kwargs())
    model.load_state_dict(Cs.make_weights(case), strict=True)
    den = ref.denoiser.DiscreteDenoiser(
        weighting_config={"target": "sgm.modules.diffusionmodules.denoiser_weighting.EpsWeighting"},
        scaling_config={"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
        num_idx=1000,
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"})
    sampler = ref.sampling.EulerEDMSampler(
        num_steps=num_steps, device="cpu",
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"},
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.VanillaCFG", "params": {"scale": scale}})
    x, c, uc = sampler_inputs(case, use_last_frame)
    calls, traj = [], []
    if use_last_frame and share_noise_level > 0.0:
        # diffusion.py:244-249: randn = randn + repeat(concat[-1], "c h w -> t c h w") * share_noise_level
        x = x + c["concat"][-1].unsqueeze(0).expand_as(x) * share_noise_level

    def denoise(xx, sigma, cc):
        calls.append(int(den.sigma_to_idx(sigma)[0]))
        if trajectory:
            traj.append(xx[: xx.shape[0] // 2].clone())
        return den(model, xx, sigma, cc)

    with R.view_height_shim(case.H, case.w):
        out = sampler(denoise, x.clone(), c, uc)
    res = {"meta": case.meta(), "num_steps": num_steps, "scale": scale, "x_final": out, "timestep_indices": calls,
           "use_last_frame": use_last_frame, "share_noise_level": share_noise_level}
    if trajectory:
        # x as the guider sees it at the start of step x_steps_at[k] (already * sqrt(1+s0^2))
        res["x_steps_at"] = trajectory_steps(num_steps)
        res["x_steps"] = torch.stack([traj[i] for i in res["x_steps_at"]])
    return res


VAE_DDCONFIG = dict(double_z=True, z_channels=4, resolution=64, in_channels=3, out_ch=3, ch=64, ch_mult=[1, 2, 2], num_res_blocks=1,
                    attn_resolutions=[], dropout=0.0)


def vae_decoder_weights(spec: dict, seed: int = 7) -> dict:
    """Seeded non-degenerate decoder weights keyed like the reference's AutoencoderKL state dict."""
    import math
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd = {}
    for k in sorted(spec):
        shape = tuple(spec[k])
        if k.endswith(".bias"):
            sd[k] = 0.05 * torch.randn(shape, generator=g)
        elif len(shape) == 1:
            sd[k] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            sd[k] = torch.randn(shape, generator=g) / math.sqrt(math.prod(shape[1:]))
    return sd


def vae_decoder_input(seed: int = 8):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(2, 4, 8, 48, generator=g)           # 2 frames, latent 8 x (6 views x 8)


@torch.no_grad()
def golden_vae_decode() -> dict:
    """Reference `AutoencoderKL.decode` = Decoder(post_quant_conv(z)) (autoencoder.py:362-365; model.py:882-1030) on a
    shrunk ddconfig with seeded weights."""
    R.import_reference()
    import contextlib, io
    from sgm.modules.diffusionmodules import model as M
    from panacea_b200.vae import decoder_param_spec
    spec = decoder_param_spec(VAE_DDCONFIG, 4)
    sd = vae_decoder_weights(spec)
    with contextlib.redirect_stdout(io.StringIO()):
        dec = M.Decoder(**VAE_DDCONFIG).eval()
    pq = torch.nn.Conv2d(4, 4, 1)
    missing = dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    pq.load_state_dict({"weight": sd["post_quant_conv.weight"], "bias": sd["post_quant_conv.bias"]})
    z = vae_decoder_input()
    out = dec(pq(z))
    # encoder: moments = quant_conv(Encoder(x)) (autoencoder.py:352-357)
    from panacea_b200.vae import encoder_param_spec
    espec = encoder_param_spec(VAE_DDCONFIG, 4)
    esd = vae_decoder_weights(espec, seed=9)
    with contextlib.redirect_stdout(io.StringIO()):
        enc = M.Encoder(**VAE_DDCONFIG).eval()
    enc.load_state_dict({k[len("encoder."):]: v for k, v in esd.items() if k.startswith("encoder.")}, strict=True)
    qc = torch.nn.Conv2d(8, 8, 1)
    qc.load_state_dict({"weight": esd["quant_conv.weight"], "bias": esd["quant_conv.bias"]})
    x = vae_encoder_input()
    moments = qc(enc(x))
    return {"ddconfig": VAE_DDCONFIG, "image": out.contiguous(), "keys": sorted(spec), "moments": moments.contiguous(),
            "encoder_keys": sorted(espec)}


def vae_encoder_input(seed: int = 10):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.rand(2, 3, 32, 192, generator=g) * 2.0 - 1.0       # 2 frames, 32 x (6 views x 32) pixels


def sampler_inputs(case: Cs.EpsCase, use_last_frame: bool = False):
    """One sequence (case.b is ignored: the sampler doubles the batch itself): init noise, c and uc dicts."""
    g = torch.Generator(device="cpu").manual_seed(case.input_seed + 100)
    T, W = case.num_frames, 6 * case.w
    x = torch.randn(T, 4, case.H, W, generator=g)
    concat = torch.randn(T, 4, case.H, W, generator=g)
    if use_last_frame:
        concat[:-1].zero_()
    hint = torch.rand(T, 19, 8 * case.H, 8 * W, generator=g)
    c = {"concat": concat, "cond_feat": hint, "crossattn": torch.randn(1, 77, case.context_dim, generator=g)}
    uc = {"concat": concat, "cond_feat": hint, "crossattn": torch.randn(1, 77, case.context_dim, generator=g)}
    return x, c, uc


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    ap.add_argument("--skip-full", action="store_true")
    a = ap.parse_args(argv)
    only = set(filter(None, a.only.split(",")))
    GOLDEN.mkdir(parents=True, exist_ok=True)
    if not only or "kat" in only:
        torch.save(golden_kat(), GOLDEN / "kat.pt")
        print("kat.pt")
    if not only or "reference_model" in only:
        with gzip.GzipFile(GOLDEN / "reference_model.json.gz", "wb", mtime=0) as f:
            f.write(json.dumps(golden_reference_model(), indent=0).encode())
        print("reference_model.json.gz")
    for case in Cs.GOLDEN_CASES:
        if only and case.name not in only:
            continue
        if a.skip_full and case.model_channels >= 320:
            continue
        g = golden_eps(case)
        torch.save(g, GOLDEN / f"eps_{case.name}.pt")
        print(f"eps_{case.name}.pt  {tuple(g['eps'].shape)}  rms={g['eps'].pow(2).mean().sqrt():.4f}  {g['seconds']:.1f}s")
    if not only or "sampler" in only:
        case = Cs.GOLDEN_CASES[0]
        g = golden_sampler(case)
        torch.save(g, GOLDEN / f"sampler_{case.name}.pt")
        print(f"sampler_{case.name}.pt rms={g['x_final'].pow(2).mean().sqrt():.4f} idx={g['timestep_indices']}")
    if not only or "vae" in only:
        g = golden_vae_decode()
        torch.save(g, GOLDEN / "vae_decode_small.pt")
        print(f"vae_decode_small.pt {tuple(g['image'].shape)} rms={g['image'].pow(2).mean().sqrt():.4f}")
    # 25-step (the YAML's count, with use_last_frame share-noise init = BASELINE config 4) and 50-step (BASELINE
    # config 2) reference loops on the GPU-runnable head_dim-64 model, with the per-step trajectory
    for steps, ulf in ((25, True), (50, False)):
        name = f"sampler_{Cs.SAMPLER_CASE.name}_{steps}"
        if only and name not in only and "sampler_loops" not in only:
            continue
        t0 = time.time()
        g = golden_sampler(Cs.SAMPLER_CASE, num_steps=steps, use_last_frame=ulf, trajectory=True)
        torch.save(g, GOLDEN / f"{name}.pt")
        print(f"{name}.pt rms={g['x_final'].pow(2).mean().sqrt():.4f} {time.time() - t0:.1f}s")


if __name__ == "__main__":
    main(sys.argv[1:])
