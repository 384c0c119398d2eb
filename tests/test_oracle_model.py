"""CPU: the module-level port used for CPU timing (oracle/ref_model.py) replays the REFERENCE modules bit-exactly under
the same seed: same parameters and input, torch.manual_seed(5), then the port's forward must equal the reference
module's output stored in tests/golden/port.npz (minted by tests/golden/make_golden_port.py)."""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle.ref_model import OracleBayesLayer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_Z = np.load(os.path.join(ROOT, "tests", "golden", "port.npz"))

# (layer, deterministic module it replaces, input shape); the same list as tests/golden/make_golden_port.py
CASES = [("Conv2d", lambda: nn.Conv2d(8, 12, 3, stride=2, padding=1), (3, 8, 9, 9)),
         ("Linear", lambda: nn.Linear(20, 7), (5, 20)),
         ("Conv1d", lambda: nn.Conv1d(4, 6, 3, padding=1, bias=False), (2, 4, 11))]


@pytest.fixture
def one_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def test_port_replays_reference_modules_bitexact(one_thread):
    for flip, (kind, make, xshape) in ((f, c) for f in (False, True) for c in CASES):
        name = kind + ("Flipout" if flip else "Reparameterization")
        g = {k[len(f"port/{name}/"):]: torch.from_numpy(_Z[k]) for k in _Z.files if k.startswith(f"port/{name}/")}
        assert g, f"{name} missing from tests/golden/port.npz"
        x = g["x"]
        assert tuple(x.shape) == xshape, name
        det = make()
        port = OracleBayesLayer(det, flip)
        port.mu_w.data.copy_(g["mu_w"]); port.rho_w.data.copy_(g["rho_w"])
        if det.bias is not None:
            port.mu_b.data.copy_(g["mu_b"]); port.rho_b.data.copy_(g["rho_b"])
        torch.manual_seed(5)
        y = port(x)
        assert torch.equal(y, g["y"]), f"{name}: max abs {float((y - g['y']).abs().max())}"
        kl_ref = float(g["kl"])
        assert abs(float(port.kl_loss()) - kl_ref) < 1e-5 * abs(kl_ref), name
