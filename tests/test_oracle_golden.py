"""Pins the CPU oracle (oracle/unet_port.py, oracle/sampler_port.py) against golden outputs of the UNMODIFIED
reference (tests/golden/*.pt, produced by oracle/make_golden.py in the build container)."""
from pathlib import Path

import pytest
import torch

from oracle import cases as Cs
from oracle import sampler_port as SP
from oracle import unet_port as P

GOLDEN = Path(__file__).resolve().parent / "golden"


@pytest.mark.parametrize("name", ["tiny_2to1", "tiny_3to1", "small_hd64", "small_hd64_3to2"])
def test_eps_port_matches_reference_golden(name):
    case = [c for c in Cs.GOLDEN_CASES if c.name == name][0]
    g = torch.load(GOLDEN / f"eps_{name}.pt")
    assert {"last_frame_concat": False, **g["meta"]} == case.meta()     # fixtures made before the field existed lack it
    x, t, c = Cs.make_inputs(case)
    eps = P.wrapper_forward(Cs.make_weights(case), case.net_config(), x, t, c)
    assert eps.shape == g["eps"].shape
    assert (eps - g["eps"]).abs().max().item() < 2e-5      # fp32 vs fp32, different op order only


def test_state_spec_is_the_reference_key_set():
    cfg = P.NetConfig()
    spec = P.state_spec(cfg)
    assert len(spec) == 2478
    n = sum(int(torch.tensor(s).prod()) for s in spec.values())
    assert abs(n - 2237.5e6) < 0.1e6                        # SURVEY.md section 3.5: 2,237.5 M parameters


def test_sampler_known_answers():
    kat = torch.load(GOLDEN / "kat.pt")
    for n in (10, 25, 50):
        assert torch.equal(SP.legacy_ddpm_sigmas(n), kat[f"sigmas_{n}"])
    den = SP.DiscreteDenoiserPort()
    assert torch.equal(den.sigmas, kat["denoiser_sigmas"])
    assert torch.equal(den.sigma_to_idx(kat["sigmas_25"][:-1]), kat["idx_of_sigmas_25"])
    assert kat["idx_of_sigmas_25"].tolist() == list(range(999, 0, -40))
    assert torch.equal(P.temporal_pos_embedding(4, 8), kat["pos_embed_T4_C8"])
    assert torch.equal(P.temporal_pos_embedding(8, 64), kat["pos_embed_T8_C64"])
    te = P.timestep_embedding(torch.tensor([0, 39, 500, 999]), 320)
    assert (te - kat["timestep_embedding_320"]).abs().max().item() < 1e-6
    # SURVEY.md section 8c constants
    s25 = SP.legacy_ddpm_sigmas(25)
    assert abs(s25[0].item() - 14.61464) < 1e-4 and abs(s25[24].item() - 0.1963) < 1e-4 and s25[25].item() == 0.0


def test_sampler_loop_matches_reference_golden():
    from oracle.make_golden import sampler_inputs
    g = torch.load(GOLDEN / "sampler_tiny_2to1.pt")
    case = Cs.GOLDEN_CASES[0]
    sd, cfg = Cs.make_weights(case), case.net_config()
    x, c, uc = sampler_inputs(case)
    seen = []

    def net(xi, ti, ci):
        seen.append(int(ti[0]))
        return P.wrapper_forward(sd, cfg, xi, ti, ci)

    out = SP.euler_edm_sample(net, x.clone(), c, uc, g["num_steps"], g["scale"])
    assert seen == g["timestep_indices"]
    rel = ((out - g["x_final"]).norm() / g["x_final"].norm()).item()
    assert rel < 1e-4, rel


def test_sampler_port_follows_the_reference_25_step_trajectory():
    """First 3 steps of the reference's 25-step loop on the head_dim-64 model with the use_last_frame shared-noise init
    (diffusion.py:242-249): the oracle sampler port must land on the committed reference trajectory."""
    from oracle import sampler_port as SP
    from oracle.make_golden import sampler_inputs
    case = Cs.SAMPLER_CASE
    g = torch.load(GOLDEN / f"sampler_{case.name}_25.pt")
    assert g["use_last_frame"] and g["timestep_indices"] == list(range(999, 0, -40))
    x, c, uc = sampler_inputs(case, True)
    x = x + c["concat"][-1].unsqueeze(0).expand_as(x) * g["share_noise_level"]
    sd, cfg = Cs.make_weights(case), case.net_config()
    out = SP.euler_edm_sample(lambda xi, ti, ci: P.wrapper_forward(sd, cfg, xi, ti, ci), x, c, uc, 25, g["scale"], max_steps=3)
    ref = g["x_steps"][g["x_steps_at"].index(3)]
    assert ((out - ref).norm() / ref.norm()).item() < 1e-5
