"""CPU, world size 2 and 3 over gloo: the N>1 host logic of MC inference for dense-classification and regression heads
(bayesian_torch_b200/mc.py::_Moments).  Each rank fills its moment buffer -- allocated by mc_predict's own code from
the output geometry -- with what the kernels add for its contiguous block of global sample indices; ONE all-reduce of
that flat buffer must give the single-process result on every rank, bit-identical across ranks."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from bayesian_torch_b200.mc import _Moments, all_reduce_moments, shard_samples
from mc_heads_oracle import mc_aggregate_dense, mc_regression_moments
from oracle import bt_oracle as O

N, B, C, H, W, D = 7, 3, 5, 4, 6, 9


def _dense_logits(sample_idx):
    g = torch.Generator().manual_seed(2000 + sample_idx)   # keyed by the GLOBAL sample index
    return torch.randn(B, C, H, W, generator=g) * 2


def _regression_out(sample_idx):
    g = torch.Generator().manual_seed(3000 + sample_idx)
    return 1e3 + 1e-2 * torch.randn(B, D, H, generator=g, dtype=torch.float64)   # large mean, small spread


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        start, count = shard_samples(N, world, rank)
        cpu = torch.device("cpu")
        # dense classification: a channels-last head output, as a Bayesian ConvTranspose2d writes it
        out = _dense_logits(0).repeat(2, 1, 1, 1).contiguous(memory_format=torch.channels_last)
        dm = _Moments("classification", out, B, with_entropy=True, device=cpu, zero=True)
        assert dm.perm == [0, 2, 3, 1] and tuple(dm.sums.shape) == (2, B * H * W, C) and dm.ent.numel() == B * H * W
        # regression: fp64 [2, n] in the output's memory order
        rm = _Moments("regression", _regression_out(0).repeat(2, 1, 1), B, with_entropy=False, device=cpu, zero=True)
        assert rm.buf.dtype == torch.float64 and rm.buf.numel() == 2 * B * D * H
        for s in range(start, start + count):
            p = torch.softmax(_dense_logits(s), 1).permute(0, 2, 3, 1).reshape(-1, C)   # rows = pixels, classes last
            dm.sums[0] += p
            dm.sums[1] += p * p
            dm.ent += O.entropy(p)
            y = _regression_out(s).reshape(-1)
            rm.sums[:y.numel()] += y
            rm.sums[y.numel():] += y * y
        all_reduce_moments(dm.buf)          # ONE collective per call, whatever the head
        all_reduce_moments(rm.buf)
        mean = (dm.sums[0] / N).view(B, H, W, C).permute(0, 3, 1, 2)
        var = (dm.sums[1] / N).view(B, H, W, C).permute(0, 3, 1, 2) - mean * mean
        pe = O.entropy(dm.sums[0] / N).view(B, H, W)
        mi = pe - (dm.ent / N).view(B, H, W)
        n = rm.buf.numel() // 2
        rmean = rm.sums[:n] / N
        rvar = (rm.sums[n:] / N - rmean * rmean).clamp_min(0)
        ret[rank] = (mean, var, pe, mi, rmean.view(B, D, H), rvar.view(B, D, H))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_dense_and_regression_moments_equal_single_process(world):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    ref_mean, ref_var, ref_pe, ref_mi = mc_aggregate_dense(torch.stack([_dense_logits(s) for s in range(N)]))
    ref_rmean, ref_rvar = mc_regression_moments(torch.stack([_regression_out(s) for s in range(N)]))
    assert float(ref_rvar.min()) > 0
    for r in range(world):
        mean, var, pe, mi, rmean, rvar = ret[r]
        assert torch.allclose(mean.double(), ref_mean, atol=1e-6) and torch.allclose(var.double(), ref_var, atol=1e-6)
        assert torch.allclose(pe.double(), ref_pe, atol=1e-5) and torch.allclose(mi.double(), ref_mi, atol=1e-5)
        assert torch.allclose(rmean, ref_rmean, rtol=0, atol=1e-9)
        assert float(((rvar - ref_rvar).abs() / ref_rvar).max()) < 1e-4     # fp64 sums keep the 1e-4 variance
        for a, b in zip(ret[r], ret[0]):
            assert torch.equal(a, b)          # identical on all ranks
