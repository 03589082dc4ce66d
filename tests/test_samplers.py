"""CPU tests of the reference's samplers (sampling.py:85-365): host scalars against known-answer values of the
unmodified reference (tests/golden/sampler_family_kat.pt, python -m oracle.sampler_family), and the samplers' host
loops run through a torch restatement of the kernel modes (TorchRefOps.sampler_step) against the reference's own
trajectories."""
from pathlib import Path

import pytest
import torch

from oracle import cases as Cs
from oracle import sampler_family as MG
from oracle import sampler_port as SP
from oracle import unet_port as P
from torch_ref_ops import TorchRefOps

GOLDEN = Path(__file__).resolve().parent / "golden"
F32 = torch.float32


@pytest.fixture(scope="module")
def kat():
    return torch.load(GOLDEN / "sampler_family_kat.pt")


def test_edm_discretization_matches_reference(kat):
    from panacea_b200.sgm.modules.diffusionmodules.discretizer import EDMDiscretization
    for n, ref in kat["edm_sigmas"].items():
        assert torch.equal(EDMDiscretization()(n), ref), n
    assert torch.equal(EDMDiscretization(0.002, 14.6, 5.0)(12), kat["edm_sigmas_custom"])


def test_host_scalars_are_bit_equal_to_the_reference(kat):
    from panacea_b200.sgm.modules.diffusionmodules import sampling_utils as U
    for r in kat["ancestral_step"]:
        got = U.ancestral_scalars(float(r["sigma_from"]), float(r["sigma_to"]), r["eta"])
        assert got == (float(r["sigma_down"]), float(r["sigma_up"])), r
    for r in kat["dpmpp2s_mults"]:
        sigma_s, m = U.dpmpp2s_scalars(float(r["sigma"]), float(r["sigma_down"]))
        assert sigma_s == float(r["sigma_s"]) and m == tuple(float(v) for v in r["mult"]), r
    for r in kat["dpmpp2m_mults"]:
        prev = None if r["sigma_prev"] is None else float(r["sigma_prev"])
        m12, m34 = U.dpmpp2m_scalars(prev, float(r["sigma"]), float(r["sigma_next"]))
        assert m12 + (m34 or ()) == tuple(float(v) for v in r["mult"]), r
    # sigma_next = 0: the reference's inf mults select x_standard = 0 * x - (-1) * denoised
    sig = [float(s) for s in kat["sigmas"]]
    assert U.dpmpp2m_scalars(sig[-3], sig[-2], 0.0) == ((0.0, -1.0), None)
    assert U.ancestral_scalars(sig[-2], 0.0, 1.0) == (0.0, 0.0) and U.ancestral_scalars(sig[0], sig[1], 0) == (sig[1], 0.0)


def test_lms_coefficients_are_the_exact_integrals(kat):
    """On float64 nodes the reference's quad integrates a float64 polynomial: exact up to rounding. On the float32 sigmas
    the reference sampler passes, numpy >= 2 evaluates its integrand in float32 (Python floats are weakly typed, NEP 50):
    those values carry float32 rounding, and the exact integral is within a few float32 ulps of them."""
    from panacea_b200.sgm.modules.diffusionmodules import sampling_utils as U
    t64 = kat["sigmas"].double().numpy()
    for order, i, j, ref in kat["lms_coeff_f64_nodes"]:
        got = U.linear_multistep_coeff(order, t64, i, j)
        assert abs(got - ref) <= 1e-12 * abs(ref), (order, i, j, got, ref)
    for order, i, j, ref in kat["lms_coeff_f32_nodes"]:
        got = U.linear_multistep_coeff(order, kat["sigmas"].numpy(), i, j)
        assert abs(got - ref) <= 1e-6 * abs(ref), (order, i, j, got, ref)
    with pytest.raises(ValueError):
        U.linear_multistep_coeff(3, t64, 1, 0)


def test_reference_targets_instantiate():
    from panacea_b200.sgm.util import instantiate_from_config
    for name, (cls, kw) in MG.SAMPLER_FAMILY.items():
        s = _make(name)
        assert type(s).__name__ == cls and type(s).__module__.startswith("panacea_b200.")
    edm = instantiate_from_config({"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization"})
    assert type(edm).__module__.startswith("panacea_b200.")
    s = _make("dpmpp2m", MG.EDM_DISC)
    assert torch.equal(s.sigmas(5), edm(5))


def _make(name, disc=MG.LEGACY_DDPM, ops=None):
    from panacea_b200.sgm.util import instantiate_from_config
    cls, kw = MG.SAMPLER_FAMILY[name]
    s = instantiate_from_config({"target": f"sgm.modules.diffusionmodules.sampling.{cls}", "params": dict(
        num_steps=MG.FAMILY_STEPS, discretization_config=disc,
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.VanillaCFG", "params": {"scale": MG.FAMILY_SCALE}},
        **kw)})
    if ops is not None:
        s.ops = ops
    return s


def _run(name, disc, network, x, c, uc, fused):
    from panacea_b200.pipeline import DEFAULT_DENOISER
    from panacea_b200.sgm.modules.diffusionmodules.sampling import BoundDenoiser
    from panacea_b200.sgm.util import instantiate_from_config
    ops = TorchRefOps()
    sampler = _make(name, disc, ops)
    noise = MG.SeededNoise()
    sampler.noise_sampler = noise
    seen, traj = [], {}

    def net(xi, ti, ci):
        seen.append(int(ti[0]))
        return network(xi, ti, ci)

    sampler.step_callback = lambda i, xx: traj.__setitem__(i, xx.clone())
    if fused:
        den = BoundDenoiser(instantiate_from_config(DEFAULT_DENOISER), net)
    else:
        port = SP.DiscreteDenoiserPort()
        den = lambda xx, s, cc: port(net, xx, s, cc)        # noqa: E731
    out = sampler(den, x.clone(), c, uc)
    if fused:
        assert sampler.last_timestep_indices == seen
        assert ops.launches == 1 + len(seen)           # the first input, then one update kernel per evaluation
    return out, seen, noise.calls, traj


def _rel(a, b):
    return ((a - b).double().norm() / b.double().norm()).item()


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("name", list(MG.SAMPLER_FAMILY) + [n + "_edm" for n in MG.SAMPLER_FAMILY_EDM])
def test_closed_form_trajectories_match_reference(kat, name, fused):
    g = kat["trajectories"][name]
    disc = MG.EDM_DISC if name.endswith("_edm") else MG.LEGACY_DDPM
    x, c, uc = MG.closed_form_inputs()
    out, seen, calls, traj = _run(name.removesuffix("_edm"), disc, MG.closed_form_network, x, c, uc, fused)
    assert seen == g["timestep_indices"] and calls == g["noise_calls"]
    assert _rel(out, g["x_final"]) <= 1e-6
    for i, ref in zip(g["x_steps_at"], g["x_steps"]):       # x at the first evaluation of step i
        if i > 0:
            assert _rel(traj[i - 1], ref) <= 1e-6, i


def test_ancestral_eta_zero_is_the_euler_sampler():
    """eta = 0 (a crash in the reference) is the deterministic limit: EulerAncestralSampler equals EulerEDMSampler and never
    calls the noise source."""
    x, c, uc = MG.closed_form_inputs()
    port = SP.DiscreteDenoiserPort()
    den = lambda xx, s, cc: port(MG.closed_form_network, xx, s, cc)        # noqa: E731
    ea = _make("euler_ancestral", ops=TorchRefOps())
    ea.eta = 0.0
    ea.noise_sampler = lambda z: pytest.fail("noise drawn at eta = 0")
    eu = _make("euler_churn", ops=TorchRefOps())
    eu.s_churn = 0.0                # the reference config's Euler sampler
    a = ea(den, x.clone(), c, uc)
    b = SP.euler_edm_sample(MG.closed_form_network, x.clone(), c, uc, MG.FAMILY_STEPS, MG.FAMILY_SCALE)
    assert _rel(a, b) <= 1e-6
    assert _rel(eu(den, x.clone(), c, uc), b) <= 1e-6


@pytest.mark.slow
@pytest.mark.parametrize("name", list(MG.SAMPLER_FAMILY))
def test_sampler_loops_match_reference_on_tiny_network(name):
    """Every sampler around the CPU oracle of the network (tiny_2to1) against the reference's loop."""
    g = torch.load(GOLDEN / f"sampler_family_tiny_2to1_{name}.pt")
    case = Cs.GOLDEN_CASES[0]
    sd, cfg = Cs.make_weights(case), case.net_config()
    x, c, uc = MG.sampler_inputs(case)
    out, seen, calls, _ = _run(name, MG.LEGACY_DDPM, lambda xi, ti, ci: P.wrapper_forward(sd, cfg, xi, ti, ci), x, c, uc, False)
    assert seen == g["timestep_indices"] and calls == g["noise_calls"]
    assert _rel(out, g["x_final"]) <= 1e-4
