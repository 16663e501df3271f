"""Pins oracle/net.py (the torch-fp32 restatement) to the real reference network definition:
 - against tests/golden/net_<arch>.json and net_reference_live.json (outputs of the reference module, recorded by
   gen_net_golden.py)."""
import json
import os

import numpy as np
import pytest

from oracle import net as onet
from tests.golden.gen_net_golden import golden_input

GOLD = os.path.join(os.path.dirname(__file__), "golden")
ARCHS = {"risev2_34": onet.arch_risev2(34, 81), "risev33_52": onet.arch_risev33(52, 76, True),
         "risev2_63": onet.arch_risev2(63, 84)}


@pytest.mark.parametrize("name", sorted(ARCHS))
def test_oracle_net_matches_reference_golden(name):
    arch = ARCHS[name]
    with open(os.path.join(GOLD, f"net_{name}.json")) as f:
        g = json.load(f)
    out = onet.forward(onet.make_state_dict(arch, g["seed"]), arch, golden_input(arch, seed=g["input_seed"]))
    idx = np.array(g["logit_idx"])
    np.testing.assert_allclose(out["value"], g["value"], atol=2e-6)
    np.testing.assert_allclose(out["policy_logits"][:, idx], g["logits"], atol=2e-5)
    np.testing.assert_allclose(out["prob"][:, idx], g["prob"], rtol=1e-4, atol=1e-9)
    np.testing.assert_allclose(out["policy_logits"].sum(1), g["logits_sum"], rtol=1e-4, atol=1e-2)
    assert out["policy_logits"].argmax(1).tolist() == g["argmax"]
    if g["aux"] is not None:
        np.testing.assert_allclose(out["aux"], g["aux"], atol=2e-6)


@pytest.mark.parametrize("name", ["risev2_34", "risev33_52"])
def test_oracle_net_matches_imported_reference(name):
    """state_dict seed 7 on three positions against the imported reference module's outputs for them
    (tests/golden/net_reference_live.json, recorded by gen_net_golden.py)."""
    arch = ARCHS[name]
    with open(os.path.join(GOLD, "net_reference_live.json")) as f:
        g = json.load(f)[name]
    out = onet.forward(onet.make_state_dict(arch, g["seed"]), arch, golden_input(arch, n=g["n"], seed=g["input_seed"]))
    idx = np.array(g["logit_idx"])
    np.testing.assert_allclose(out["value"], g["value"], atol=2e-6)
    np.testing.assert_allclose(out["policy_logits"][:, idx].ravel(), g["logits"], atol=2e-5)
    np.testing.assert_allclose(out["policy_logits"].astype(np.float64).sum(1), g["logits_sum"], rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(np.abs(out["policy_logits"].astype(np.float64)).sum(1), g["logits_abs_sum"], rtol=1e-4, atol=1e-2)
    if g["aux"] is not None:
        np.testing.assert_allclose(out["aux"].ravel(), g["aux"], atol=2e-6)
