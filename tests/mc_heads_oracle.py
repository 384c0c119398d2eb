"""Float64 restatements of Monte-Carlo aggregation for dense (segmentation) and regression heads: what
bayesian_torch_b200.mc_predict(task=...) is checked against in tests/test_gpu_mc_heads.py and
tests/test_mc_heads_gloo.py.  Pure torch on the CPU; the per-pixel uncertainties are the reference's
utils/util.py:41-60 (oracle/bt_oracle.py entropy / predictive_entropy / mutual_information) applied to every pixel."""
import torch

from oracle import bt_oracle as O


def mc_aggregate_dense(logits):
    """logits [N_mc, B, C, *spatial] (any spatial rank, including none): softmax over the class axis, mean and
    variance over the MC axis, and per-pixel predictive entropy / mutual information -> float64
    (mean [B, C, *sp], var [B, C, *sp], pred_entropy [B, *sp], mutual_info [B, *sp])."""
    p = torch.softmax(logits.double(), dim=2)
    mean = p.mean(0)
    var = (p * p).mean(0) - mean * mean
    p_last = p.movedim(2, -1)                    # [N_mc, B, *sp, C]: entropy() reduces the last axis
    return mean, var, O.predictive_entropy(p_last), O.mutual_information(p_last)


def mc_regression_moments(y):
    """y [N_mc, B, *rest] -> float64 mean and (population) variance over the MC axis, two-pass: no cancellation."""
    y = y.double()
    mean = y.mean(0)
    return mean, (y - mean).pow(2).mean(0)
