"""CPU: the oracle restatement (oracle/bt_oracle.py) against golden vectors minted from the
reference itself (tests/golden/make_golden.py), plus the Random123 KATs of the Philox restatement."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import bt_oracle as O
from oracle import philox_ref as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "meta.json")) as _f:
    _META = json.load(_f)
CASES = sorted(_META["cases"].keys())


def _opt(c, k):
    return c.get(k)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_bitexact(golden, name):
    c, m = golden.case(name), golden.meta["cases"][name]
    if m["kind"] == "linear":
        if m["flipout"]:
            y = O.linear_flipout(c["x"], c["mu_w"], c["rho_w"], c["eps_w"], c["sign_in"], c["sign_out"],
                                 _opt(c, "mu_b"), _opt(c, "rho_b"), _opt(c, "eps_b"))
        else:
            y = O.linear_reparam(c["x"], c["mu_w"], c["rho_w"], c["eps_w"], _opt(c, "mu_b"), _opt(c, "rho_b"),
                                 _opt(c, "eps_b"))
    else:
        kw = dict(stride=m["stride"], padding=m["padding"], dilation=m["dilation"], groups=m["groups"])
        if m["flipout"]:
            y = O.conv_flipout(m["nd"], c["x"], c["mu_w"], c["rho_w"], c["eps_w"], c["sign_in"], c["sign_out"],
                               _opt(c, "mu_b"), _opt(c, "rho_b"), _opt(c, "eps_b"), **kw)
        else:
            y = O.conv_reparam(m["nd"], c["x"], c["mu_w"], c["rho_w"], c["eps_w"], _opt(c, "mu_b"),
                               _opt(c, "rho_b"), _opt(c, "eps_b"), **kw)
    assert torch.equal(y, c["y"]), f"{name}: max abs {float((y - c['y']).abs().max())}"
    kl = O.kl_loss(c["mu_w"], c["rho_w"], m["prior_mean"], m["prior_variance"], _opt(c, "mu_b"), _opt(c, "rho_b"))
    # the reference fills fp32 prior tensors; the scalar restatement agrees to fp32 rounding
    assert abs(float(kl) - float(c["kl"])) <= 2e-6 * max(1.0, abs(float(c["kl"])))
    assert abs(float(c["kl_loss"]) - float(c["kl"])) <= 1e-6 * max(1.0, abs(float(c["kl"])))


def test_signs_are_plus_minus_one(golden):
    for name in golden.names():
        c = golden.case(name)
        if "sign_in" in c:
            assert set(torch.unique(c["sign_in"]).tolist()) <= {-1.0, 1.0}
            assert set(torch.unique(c["sign_out"]).tolist()) <= {-1.0, 1.0}


def test_kl_against_torch_distributions():
    torch.manual_seed(0)
    mu, rho = torch.randn(1000) * 0.1, torch.randn(1000) * 0.1 - 3
    sig = O.sigma_of_rho(rho)
    ref = torch.distributions.kl_divergence(torch.distributions.Normal(mu, sig),
                                            torch.distributions.Normal(torch.tensor(0.3), torch.tensor(0.8))).mean()
    assert abs(float(O.kl_div(mu, sig, 0.3, 0.8)) - float(ref)) < 1e-5


def test_get_rho_and_mc(golden):
    c = golden.case("get_rho")
    assert torch.equal(O.get_rho(c["w"], 0.5), c["rho"])
    c = golden.case("mc")
    mean, var = O.mc_aggregate(c["logits"])
    assert torch.allclose(mean, c["mean"], atol=1e-7)
    assert torch.equal(mean.argmax(-1), c["pred"])
    assert (var >= -1e-7).all()


@pytest.mark.parametrize("ctr,key,expect", P.KAT)
def test_philox_known_answers(ctr, key, expect):
    out = P.philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
    assert [int(v) for v in out] == list(expect)


def test_philox_normals_and_signs_distribution():
    z = P.weight_eps(512, 1024, seed=1234, layer_key=5, sample_idx=2).astype(np.float64)
    assert abs(z.mean()) < 5e-3 and abs(z.std() - 1.0) < 5e-3
    assert abs(((z ** 3).mean())) < 2e-2 and abs((z ** 4).mean() - 3.0) < 5e-2
    # distinct samples / layers / streams decorrelate
    z2 = P.weight_eps(512, 1024, seed=1234, layer_key=5, sample_idx=3).astype(np.float64)
    assert abs((z * z2).mean()) < 5e-3
    s = P.sign_bits(256, 300, 1, 2, 3, P.STREAM_SIGN_IN)
    assert set(np.unique(s)) == {-1.0, 1.0} and abs(s.mean()) < 2e-2
    # tiling independence: a sub-block equals the slice of the full tensor
    full = P.weight_eps(64, 256, 9, 1, 0)
    assert np.array_equal(P.weight_eps(64, 128, 9, 1, 0), full[:, :128])


def test_uncertainty_restatement_equals_reference_numpy_formulas():
    """oracle entropy / predictive_entropy / mutual_information (reference utils/util.py:41-60) against the same formulas
    in float64 numpy written out independently, and against the reference module's own results on the same
    probabilities (tests/golden/port.npz, minted by tests/golden/make_golden_port.py)."""
    g = torch.Generator().manual_seed(11)
    probs = torch.softmax(torch.randn(9, 6, 10, generator=g) * 3, -1)          # [N, B, C]
    p64 = probs.double().numpy()
    ent = lambda q: -np.sum(q * np.log(q + 1e-15), axis=-1)
    pe = ent(p64.mean(0))
    mi = pe - ent(p64).mean(0)
    assert np.allclose(O.predictive_entropy(probs).numpy(), pe, atol=1e-6)
    assert np.allclose(O.mutual_information(probs).numpy(), mi, atol=1e-6)
    assert (mi > -1e-9).all()
    z = np.load(os.path.join(ROOT, "tests", "golden", "port.npz"))
    probs = torch.from_numpy(z["util/probs"])
    assert np.allclose(z["util/predictive_entropy"], O.predictive_entropy(probs).numpy(), atol=1e-6)
    assert np.allclose(z["util/mutual_information"], O.mutual_information(probs).numpy(), atol=1e-6)
