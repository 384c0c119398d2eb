"""-m gpu: mc_predict for dense (segmentation), regression and large-vocabulary heads, and the kernels behind them
(csrc/bt_mc.cu: bt_mc_accumulate_large, bt_mc_regression_accumulate / _finalize), against the float64 restatements
of tests/mc_heads_oracle.py."""
import pytest
import torch
import torch.nn as nn

import bayesian_torch_b200 as btb
from bayesian_torch_b200 import _native
from mc_heads_oracle import mc_aggregate_dense, mc_regression_moments

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRM = {"prior_mu": 0.0, "prior_sigma": 1.0, "posterior_mu_init": 0.0, "posterior_rho_init": -3.0,
       "type": "Reparameterization", "moped_enable": False, "moped_delta": 0.5}
TYPES = ["Reparameterization", "Flipout"]


def _bnn(net, typ, seed=5):
    btb.dnn_to_bnn(net, dict(PRM, type=typ))
    btb.assign_layer_keys(net)
    btb.manual_seed(seed)
    return net.to(DEV).eval()


def _segmenter(typ, n_out=21):
    """encoder-decoder: two stride-2 convs down, two stride-2 transposed convs up -> [B, n_out, H, W]"""
    torch.manual_seed(3)
    net = nn.Sequential(nn.Conv2d(3, 16, 3, stride=2, padding=1), nn.ReLU(),
                        nn.Conv2d(16, 32, 3, stride=2, padding=1), nn.ReLU(),
                        nn.ConvTranspose2d(32, 16, 4, stride=2, padding=1), nn.ReLU(),
                        nn.ConvTranspose2d(16, n_out, 4, stride=2, padding=1))
    return _bnn(net, typ)


def _mlp(typ, n_out, width=64):
    torch.manual_seed(4)
    return _bnn(nn.Sequential(nn.Linear(32, width), nn.ReLU(), nn.Linear(width, n_out)), typ)


def _per_sample(model, x, offset, n):
    """the reference's loop: n single-sample forwards with the global sample indices offset + s -> [n, B, ...]"""
    outs = []
    with torch.no_grad():
        for s in range(n):
            with btb.mc_sample_context(1, x.shape[0], offset + s):
                outs.append(model(x).float().cpu())
    return torch.stack(outs)


def _maxdiff(a, b):
    return float((a.double().cpu() - b.double().cpu()).abs().max())


def _large_c_logits(S, B, C, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    base = torch.randn(B, C, device=DEV, generator=g) * 2
    return (base.repeat(S, 1) + 1.5 * torch.randn(S * B, C, device=DEV, generator=g)).to(dtype)


# ---------------------------------------------------------------- kernels against the float64 oracle
@pytest.mark.parametrize("C", [1025, 21841, 131072])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_large_c_kernel_matches_oracle(C, dtype):
    S, B = 8, 4
    logits = _large_c_logits(S, B, C, dtype, C)
    sums = torch.empty(2, B, C, device=DEV)
    ent = torch.empty(B, device=DEV)
    _native.mc_accumulate(logits, S, B, sums, accumulate=False, entropy_sum=ent)
    mean, var = torch.empty(B, C, device=DEV), torch.empty(B, C, device=DEV)
    _native.mc_finalize(sums, S, mean, var)
    pe, mi = torch.empty(B, device=DEV), torch.empty(B, device=DEV)
    _native.mc_uncertainty(sums, ent, S, pe, mi)
    rmean, rvar, rpe, rmi = mc_aggregate_dense(logits.float().cpu().view(S, B, C))
    assert _maxdiff(mean, rmean) <= 2e-6 and _maxdiff(var, rvar) <= 2e-6, (_maxdiff(mean, rmean), _maxdiff(var, rvar))
    # relative to the entropy scale: MI = H(mean p) - mean H(p_s) carries the absolute error of the entropies
    scale = float(rpe.abs().max())
    assert _maxdiff(pe, rpe) <= 1e-5 * scale and _maxdiff(mi, rmi) <= 1e-5 * scale, (_maxdiff(pe, rpe), _maxdiff(mi, rmi), scale)
    assert float(rmi.min()) > 1e-3 * scale           # the samples disagree: MI is not a vanishing difference
    # two chunks (the second starts from the stored sums) == one pass, and a repeated call is bit-identical
    s2 = torch.empty_like(sums)
    e2 = torch.empty_like(ent)
    _native.mc_accumulate(logits[:3 * B], 3, B, s2, accumulate=False, entropy_sum=e2)
    _native.mc_accumulate(logits[3 * B:], S - 3, B, s2, accumulate=True, entropy_sum=e2)
    assert _maxdiff(s2, sums) <= 1e-6 * S and _maxdiff(e2, ent) <= 1e-5 * S * scale
    s3, e3 = torch.empty_like(sums), torch.empty_like(ent)
    _native.mc_accumulate(logits, S, B, s3, accumulate=False, entropy_sum=e3)
    assert torch.equal(s3, sums) and torch.equal(e3, ent)


def _regression_check(y, S, got_mean, got_var):
    rmean, rvar = mc_regression_moments(y.float().cpu().view(S, -1))
    ymax = float(y.float().abs().max())
    dm = _maxdiff(got_mean.view(-1), rmean)
    dv = float(((got_var.view(-1).double().cpu() - rvar).abs() / rvar.clamp_min(1e-30)).max())
    assert dm <= 1e-6 * ymax and dv <= 1e-4, (dm, dv)
    return rvar


@pytest.mark.parametrize("dtype,n,misalign", [(torch.float32, 4096 * 16, 0), (torch.bfloat16, 4096 * 16, 0),
                                              (torch.float32, 1001, 1), (torch.bfloat16, 999, 3)])
def test_regression_kernel_matches_oracle(dtype, n, misalign):
    S = 12
    g = torch.Generator(device=DEV).manual_seed(n)
    store = (torch.randn(S * n + misalign, device=DEV, generator=g) * 3 + 1).to(dtype)
    y = store[misalign:]                             # misalign / odd n: the scalar-load instantiation
    sums = torch.empty(2 * n, dtype=torch.float64, device=DEV)
    _native.mc_regression_accumulate(y, S, sums, accumulate=False)
    mean, var = torch.empty(n, device=DEV), torch.empty(n, device=DEV)
    _native.mc_regression_finalize(sums, S, mean, var)
    _regression_check(y, S, mean, var)
    s2 = torch.empty_like(sums)
    _native.mc_regression_accumulate(y[:5 * n], 5, s2, accumulate=False)
    _native.mc_regression_accumulate(y[5 * n:], S - 5, s2, accumulate=True)
    assert _maxdiff(s2[:n], sums[:n]) <= 1e-12 * S * float(y.float().abs().max())
    s3 = torch.empty_like(sums)
    _native.mc_regression_accumulate(y, S, s3, accumulate=False)
    assert torch.equal(s3, sums)


def test_regression_fp64_survives_large_mean_small_spread():
    """mean 1e3, std 1e-2: the fp64 sums give the variance to 1e-4; the fp32 moments the classification path uses
    (sum y^2 / N - mean^2, csrc/bt_mc.cu::mc_finalize_kernel) do not."""
    S, n = 64, 4096
    g = torch.Generator(device=DEV).manual_seed(0)
    y = 1e3 + 1e-2 * torch.randn(S * n, device=DEV, generator=g)
    sums = torch.empty(2 * n, dtype=torch.float64, device=DEV)
    _native.mc_regression_accumulate(y, S, sums, accumulate=False)
    mean, var = torch.empty(n, device=DEV), torch.empty(n, device=DEV)
    _native.mc_regression_finalize(sums, S, mean, var)
    rvar = _regression_check(y, S, mean, var)
    ys = y.view(S, n)
    s32 = torch.zeros(2, 1, n, device=DEV)
    for s in range(S):                                # fp32 running sums in sample order
        s32[0, 0] += ys[s]
        s32[1, 0] += ys[s] * ys[s]
    m32, v32 = torch.empty(1, n, device=DEV), torch.empty(1, n, device=DEV)
    _native.mc_finalize(s32, S, m32, v32)
    rel32 = float(((v32.view(-1).double().cpu() - rvar).abs() / rvar).max())
    assert rel32 > 0.1, rel32                        # fp32 cancellation: the variance is lost


# ---------------------------------------------------------------- whole models through mc_predict
def test_default_2d_path_is_the_existing_kernel_bit_for_bit():
    model = _mlp("Reparameterization", 10)
    B, S = 16, 8
    x = torch.randn(B, 32, device=DEV)
    mean, var = btb.mc_predict(model, x, S)
    with torch.no_grad(), btb.mc_sample_context(S, B, 0):
        logits = model(x)
    sums = torch.empty(2, B, 10, device=DEV)
    _native.mc_accumulate(logits, S, B, sums, accumulate=False)
    m, v = torch.empty(B, 10, device=DEV), torch.empty(B, 10, device=DEV)
    _native.mc_finalize(sums, S, m, v)
    assert torch.equal(mean, m) and torch.equal(var, v)


@pytest.mark.parametrize("typ", TYPES)
def test_dense_segmenter_matches_per_sample_oracle(typ):
    model = _segmenter(typ)
    B, S, off = 2, 6, 11
    x = torch.randn(B, 3, 32, 32, device=DEV)
    mean, var, pe, mi = btb.mc_predict(model, x, S, sample_offset=off, return_uncertainty=True)
    assert mean.shape == (B, 21, 32, 32) and pe.shape == (B, 32, 32) and mi.shape == (B, 32, 32)
    rmean, rvar, rpe, rmi = mc_aggregate_dense(_per_sample(model, x, off, S))
    assert _maxdiff(mean, rmean) <= 2e-6 and _maxdiff(var, rvar) <= 2e-6, (_maxdiff(mean, rmean), _maxdiff(var, rvar))
    assert _maxdiff(pe, rpe) <= 1e-5 and _maxdiff(mi, rmi) <= 1e-5, (_maxdiff(pe, rpe), _maxdiff(mi, rmi))
    assert float(var.max()) > 0 and float(mi.max()) > 0
    # chunk=1 == chunk=S up to summation order; repeated call bit-identical
    c1 = btb.mc_predict(model, x, S, sample_offset=off, return_uncertainty=True, chunk=1)
    for a, b in zip(c1, (mean, var, pe, mi)):
        assert _maxdiff(a, b) <= 1e-5
    again = btb.mc_predict(model, x, S, sample_offset=off, return_uncertainty=True)
    for a, b in zip(again, (mean, var, pe, mi)):
        assert torch.equal(a, b)


def test_dense_head_in_nchw_layout_costs_one_copy_and_gives_the_same_result():
    seg = _segmenter("Reparameterization")

    class Nchw(nn.Module):                           # a head that hands back an NCHW-contiguous tensor
        def __init__(self):
            super().__init__()
            self.seg = seg

        def forward(self, x):
            return self.seg(x).contiguous()

    B, S = 2, 4
    x = torch.randn(B, 3, 32, 32, device=DEV)
    l0 = _native.launch_count
    ref = btb.mc_predict(seg, x, S, return_uncertainty=True)
    l1 = _native.launch_count
    got = btb.mc_predict(Nchw().eval(), x, S, return_uncertainty=True)
    l2 = _native.launch_count
    for a, b in zip(got, ref):
        assert torch.equal(a, b)
    assert (l2 - l1) - (l1 - l0) == 1


@pytest.mark.parametrize("typ", TYPES)
def test_regression_models_match_per_sample_oracle(typ):
    torch.manual_seed(6)
    dense = _bnn(nn.Sequential(nn.Conv2d(3, 16, 3, stride=2, padding=1), nn.ReLU(),
                               nn.ConvTranspose2d(16, 1, 4, stride=2, padding=1)), typ)
    B, S, off = 3, 6, 100
    for model, x in ((_mlp(typ, 7), torch.randn(B, 32, device=DEV)), (dense, torch.randn(B, 3, 16, 16, device=DEV))):
        mean, var = btb.mc_predict(model, x, S, sample_offset=off, task="regression")
        ys = _per_sample(model, x, off, S)
        assert mean.shape == ys.shape[1:] and var.shape == ys.shape[1:]
        rmean, rvar = mc_regression_moments(ys)
        ymax = float(ys.abs().max())
        assert _maxdiff(mean, rmean) <= 2e-6 * ymax and _maxdiff(var, rvar) <= 2e-6 * ymax * ymax, \
            (_maxdiff(mean, rmean), _maxdiff(var, rvar))
        assert float(var.min()) >= 0 and float(var.max()) > 0
        c1 = btb.mc_predict(model, x, S, sample_offset=off, task="regression", chunk=1)
        assert _maxdiff(c1[0], mean) <= 1e-6 * ymax and _maxdiff(c1[1], var) <= 1e-6 * ymax * ymax
        again = btb.mc_predict(model, x, S, sample_offset=off, task="regression")
        assert torch.equal(again[0], mean) and torch.equal(again[1], var)
        assert btb.mc_predict(model, x, S, sample_offset=off, task="regression", return_var=False)[1] is None


def test_large_c_classifier_end_to_end():
    model = _mlp("Reparameterization", 21841)
    B, S, off = 4, 8, 3
    x = torch.randn(B, 32, device=DEV)
    mean, var, pe, mi = btb.mc_predict(model, x, S, sample_offset=off, return_uncertainty=True, chunk=3)
    assert mean.shape == (B, 21841)
    rmean, rvar, rpe, rmi = mc_aggregate_dense(_per_sample(model, x, off, S))
    assert _maxdiff(mean, rmean) <= 2e-6 and _maxdiff(var, rvar) <= 2e-6, (_maxdiff(mean, rmean), _maxdiff(var, rvar))
    scale = float(rpe.abs().max())
    assert _maxdiff(pe, rpe) <= 1e-5 * scale and _maxdiff(mi, rmi) <= 1e-5 * scale, (_maxdiff(pe, rpe), _maxdiff(mi, rmi))


@pytest.mark.parametrize("head", ["dense", "regression", "large_c"])
def test_graph_replay_equals_eager_and_fresh_draws(head):
    B, S = 2, 4
    if head == "dense":
        model, x, kw = _segmenter("Flipout"), torch.randn(B, 3, 32, 32, device=DEV), {"return_uncertainty": True}
    elif head == "regression":
        model, x, kw = _mlp("Reparameterization", 5), torch.randn(B, 32, device=DEV), {"task": "regression"}
    else:
        model, x, kw = _mlp("Flipout", 3000), torch.randn(B, 32, device=DEV), {"return_uncertainty": True}
    eager = btb.mc_predict(model, x, S, sample_offset=7, **kw)
    g = btb.mc_predict(model, x, S, sample_offset=7, use_graph=True, **kw)
    g2 = btb.mc_predict(model, x, S, sample_offset=7, use_graph=True, **kw)
    for a, b, c in zip(eager, g, g2):
        assert torch.equal(a, b) and torch.equal(a, c)
    model._bt_mc_drawn = 0
    f1 = btb.mc_predict(model, x, S, use_graph=True, fresh=True, **kw)       # samples [0, S)
    f2 = btb.mc_predict(model, x, S, use_graph=True, fresh=True, **kw)       # samples [S, 2S): new draws
    e2 = btb.mc_predict(model, x, S, sample_offset=S, **kw)
    assert not torch.equal(f1[0], f2[0])
    for a, b in zip(f2, e2):
        assert torch.equal(a, b)
    btb.mc.drop_graphs(model)


def test_errors():
    model = _mlp("Reparameterization", 4)
    x = torch.randn(3, 32, device=DEV)
    with pytest.raises(ValueError, match="task"):
        btb.mc_predict(model, x, 2, task="segmentation")
    with pytest.raises(ValueError, match="classification"):
        btb.mc_predict(model, x, 2, task="regression", return_uncertainty=True)

    class DropsARow(nn.Module):
        def __init__(self):
            super().__init__()
            self.m = model

        def forward(self, x):
            return self.m(x)[1:]

    for task in ("classification", "regression"):
        with pytest.raises(RuntimeError, match="S\\*B"):
            btb.mc_predict(DropsARow().eval(), x, 2, task=task)

    class Flat(nn.Module):
        def __init__(self):
            super().__init__()
            self.m = model

        def forward(self, x):
            return self.m(x)[:, 0]

    with pytest.raises(RuntimeError, match="class axis"):
        btb.mc_predict(Flat().eval(), x, 2)
