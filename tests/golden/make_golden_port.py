#!/usr/bin/env python
"""Mint golden vectors for the module-level CPU port (oracle/ref_model.py) and the MC uncertainty formulas from the
REFERENCE ITSELF (IntelLabs/bayesian-torch @ aa7e57b), so that tests/test_oracle_model.py and
tests/test_oracle_golden.py compare against the reference without needing its source tree:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_port.py <bayesian-torch checkout>

Writes tests/golden/port.npz:
  port/<Name>/{x, mu_w, rho_w[, mu_b, rho_b], y, kl}  the reference module's parameters, its input, and its forward
                                                      output and KL after torch.manual_seed(5) (one thread)
  util/{probs, predictive_entropy, mutual_information} utils/util.py:45-60 of the reference on seeded probabilities
The case list must match tests/test_oracle_model.py::CASES.
"""
import importlib.util
import os
import sys

if len(sys.argv) != 2:
    raise SystemExit(__doc__)
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REF)
sys.dont_write_bytecode = True

import numpy as np
import torch
import torch.nn as nn

import bayesian_torch.layers as RL  # the REFERENCE package

assert RL.__file__.startswith(REF), RL.__file__
HERE = os.path.dirname(os.path.abspath(__file__))
torch.set_num_threads(1)

CASES = [("Conv2d", lambda: nn.Conv2d(8, 12, 3, stride=2, padding=1), (3, 8, 9, 9)),
         ("Linear", lambda: nn.Linear(20, 7), (5, 20)),
         ("Conv1d", lambda: nn.Conv1d(4, 6, 3, padding=1, bias=False), (2, 4, 11))]

out = {}
for flip in (False, True):
    for i, (kind, make, xshape) in enumerate(CASES):
        torch.manual_seed(100 + i)
        det, x = make(), torch.randn(*xshape)
        name = kind + ("Flipout" if flip else "Reparameterization")
        kw = dict(bias=det.bias is not None)
        if isinstance(det, nn.Linear):
            ref = getattr(RL, name)(det.in_features, det.out_features, **kw)
        else:
            ks = det.kernel_size if len(det.kernel_size) > 1 else det.kernel_size[0]
            ref = getattr(RL, name)(det.in_channels, det.out_channels, ks, stride=det.stride, padding=det.padding, **kw)
        w = "weight" if isinstance(det, nn.Linear) else "kernel"
        rec = {"x": x, "mu_w": getattr(ref, "mu_" + w), "rho_w": getattr(ref, "rho_" + w)}
        if det.bias is not None:
            rec.update(mu_b=ref.mu_bias, rho_b=ref.rho_bias)
        torch.manual_seed(5)
        y, kl = ref(x)
        rec.update(y=y, kl=kl)
        for k, v in rec.items():
            out[f"port/{name}/{k}"] = v.detach().numpy()

spec = importlib.util.spec_from_file_location("_ref_util", os.path.join(REF, "bayesian_torch", "utils", "util.py"))
util = importlib.util.module_from_spec(spec)
spec.loader.exec_module(util)
g = torch.Generator().manual_seed(11)
probs = torch.softmax(torch.randn(9, 6, 10, generator=g) * 3, -1).numpy()          # [N, B, C]
out["util/probs"] = probs
out["util/predictive_entropy"] = np.asarray(util.predictive_entropy(probs))
out["util/mutual_information"] = np.asarray(util.mutual_information(probs))

np.savez_compressed(os.path.join(HERE, "port.npz"), **out)
print(f"wrote {len(out)} arrays to tests/golden/port.npz")
