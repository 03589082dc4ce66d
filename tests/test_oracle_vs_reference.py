"""Comparison of the oracle port with the reference itself, through what the unmodified reference modules produced
(oracle/make_golden.py): its state-dict key set, the tensors its default init zeroes, its output on the tiny_3to1
case and the output of a freshly constructed reference model (tests/golden/reference_model.json.gz,
tests/golden/eps_tiny_3to1.pt)."""
import gzip
import json
from pathlib import Path

import torch

from oracle import cases as Cs
from oracle import unet_port as P

GOLDEN = Path(__file__).resolve().parent / "golden"


def _reference_model() -> dict:
    with gzip.open(GOLDEN / "reference_model.json.gz", "rt") as f:
        return json.load(f)


def test_reference_state_dict_keys_and_port_output():
    case = Cs.GOLDEN_CASES[1]                      # non-2:1 views -> exercises the view-height shim
    g = _reference_model()
    assert g["case"] == case.name
    assert {k: tuple(v) for k, v in g["state_spec"].items()} == P.state_spec(case.net_config())
    ref = torch.load(GOLDEN / f"eps_{case.name}.pt")["eps"]
    sd = Cs.make_weights(case)
    x, t, c = Cs.make_inputs(case)
    out = P.wrapper_forward(sd, case.net_config(), x, t, c)
    assert (out - ref).abs().max().item() < 2e-5


def test_fresh_reference_model_outputs_zero():
    """SURVEY.md section 0.3: zero_module'd tails make a fresh model predict exactly 0. The port with exactly the
    tensors the reference zeroes set to zero predicts 0 too, and a fresh drop-in model zeroes the same tensors."""
    from panacea_b200.pipeline import default_network_config
    from panacea_b200.sgm.modules.diffusionmodules import OpenAIWrapperControlLDM3D
    from panacea_b200.sgm.util import instantiate_from_config
    case = Cs.GOLDEN_CASES[0]
    g = _reference_model()
    assert g["fresh_case"] == case.name and g["fresh_output_max_abs"] == 0.0
    zero = set(g["fresh_zero_keys"])
    sd = {k: torch.zeros_like(v) if k in zero else v for k, v in Cs.make_weights(case).items()}
    x, t, c = Cs.make_inputs(case)
    out = P.wrapper_forward(sd, case.net_config(), x, t, c)
    assert list(out.shape) == g["fresh_output_shape"] and out.abs().max().item() == 0.0
    kw = case.unet_kwargs()
    model = instantiate_from_config(default_network_config(**{k: kw[k] for k in ("model_channels", "num_head_channels", "context_dim", "num_frames")}))
    fresh = OpenAIWrapperControlLDM3D(model).state_dict()
    assert {k for k, v in fresh.items() if not v.any()} == zero
