#!/usr/bin/env python
"""Kernel time and bandwidth of the MC aggregation for the three non-classifier heads, and the end-to-end step of a
Bayesian segmentation net.  Prints ONE JSON line.

    python tools/bench_mc_heads.py [--passes 20] [--steps 20]

Workloads (the aggregation only, CUDA events around each launch, the median pass reported):
  dense      S=32, B=8, 21 classes, 128x128, bf16 logits (Pascal-VOC-sized segmentation head, channels-last)
  large_c    S=32, B=128, C=21841, bf16 logits (ImageNet-21k head)
  regression S=64, B=4096, D=256, fp32 outputs
Every working set is larger than the 126 MB L2, and a 160 MiB buffer is overwritten before each timed pass as well, so
the logits come from HBM.  Algorithmic bytes = logits read once + moment buffer written; achieved GB/s is compared with
a device-to-device copy measured in the same run.
End to end: mc_predict(use_graph=True) on the encoder-decoder of tests/test_gpu_mc_heads.py (fp32, B=8, 128x128, S=32)
against the reference-style loop through the same layers (S single-sample forwards -> torch.stack -> softmax -> mean).
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bayesian_torch_b200 as btb  # noqa: E402
from bayesian_torch_b200 import _native  # noqa: E402

DEV = "cuda:0"


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, passes, flush):
    """median milliseconds of fn() over `passes`, L2 overwritten before each pass (outside the events)"""
    for _ in range(3):
        fn()
    times = []
    for _ in range(passes):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2]


def kernel_workloads(passes, flush):
    out = {}
    g = torch.Generator(device=DEV).manual_seed(0)
    # dense: [S*B, 21, 128, 128] channels-last == [S, B*128*128, 21] class-contiguous rows (the existing warp kernel)
    S, B, C, P = 32, 8, 21, 128 * 128
    logits = torch.randn(S * B * P, C, device=DEV, generator=g).bfloat16()
    sums = torch.empty(2, B * P, C, device=DEV)
    ms = timed(lambda: _native.mc_accumulate(logits, S, B * P, sums, accumulate=False), passes, flush)
    out["dense"] = {"shape": "S=32 B=8 C=21 128x128 bf16", "ms": ms,
                    "bytes": logits.numel() * 2 + sums.numel() * 4}
    del logits, sums
    S, B, C = 32, 128, 21841
    logits = torch.randn(S * B, C, device=DEV, generator=g).bfloat16()
    sums = torch.empty(2, B, C, device=DEV)
    ms = timed(lambda: _native.mc_accumulate(logits, S, B, sums, accumulate=False), passes, flush)
    out["large_c"] = {"shape": "S=32 B=128 C=21841 bf16", "ms": ms, "launches": 2,
                      "bytes": logits.numel() * 2 + sums.numel() * 4}
    del logits, sums
    S, B, D = 64, 4096, 256
    y = torch.randn(S * B * D, device=DEV, generator=g)
    rs = torch.empty(2 * B * D, dtype=torch.float64, device=DEV)
    ms = timed(lambda: _native.mc_regression_accumulate(y, S, rs, accumulate=False), passes, flush)
    out["regression"] = {"shape": "S=64 B=4096 D=256 fp32", "ms": ms, "bytes": y.numel() * 4 + rs.numel() * 8}
    del y, rs
    src = torch.empty(1 << 28, device=DEV)                        # 1 GiB device-to-device copy
    dst = torch.empty_like(src)
    ms = timed(lambda: dst.copy_(src), passes, flush)
    copy_gbs = 2 * src.numel() * 4 / ms / 1e6
    for v in out.values():
        v["gb_s"] = v["bytes"] / v["ms"] / 1e6
        v["of_copy_bw"] = v["gb_s"] / copy_gbs
    out["d2d_copy_gb_s"] = copy_gbs
    return out


def end_to_end(steps):
    torch.manual_seed(3)
    net = nn.Sequential(nn.Conv2d(3, 16, 3, stride=2, padding=1), nn.ReLU(),
                        nn.Conv2d(16, 32, 3, stride=2, padding=1), nn.ReLU(),
                        nn.ConvTranspose2d(32, 16, 4, stride=2, padding=1), nn.ReLU(),
                        nn.ConvTranspose2d(16, 21, 4, stride=2, padding=1))
    btb.dnn_to_bnn(net, {"prior_mu": 0.0, "prior_sigma": 1.0, "posterior_mu_init": 0.0, "posterior_rho_init": -3.0,
                         "type": "Reparameterization", "moped_enable": False, "moped_delta": 0.5})
    btb.assign_layer_keys(net)
    btb.manual_seed(0)
    net = net.to(DEV).eval()
    B, S = 8, 32
    x = torch.randn(B, 3, 128, 128, device=DEV)

    def mc():
        return btb.mc_predict(net, x, S, use_graph=True, fresh=True)

    def loop():
        with torch.no_grad():
            outs = []
            for s in range(S):
                with btb.mc_sample_context(1, B, s):
                    outs.append(net(x))
            return torch.softmax(torch.stack(outs).float(), dim=2).mean(0)

    res = {}
    for name, fn in (("mc_predict_graph", mc), ("reference_loop", loop)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        b.synchronize()
        res[name + "_ms"] = a.elapsed_time(b) / steps
    l0 = _native.launch_count
    mc()
    res["mc_predict_launches"] = _native.launch_count - l0
    res["speedup"] = res["reference_loop_ms"] / res["mc_predict_graph_ms"]
    res["workload"] = "encoder-decoder (2 conv s2, 2 convT s2, C=21) fp32 B=8 128x128 S=32"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mc_heads.py measures on a CUDA device; none found")
    flush = torch.empty(160 * 1024 * 1024 // 4, device=DEV)       # 160 MiB > 126 MB L2
    rec = {"info": gpu_info(), "kernels": kernel_workloads(args.passes, flush), "end_to_end": end_to_end(args.steps)}
    rec["info"]["power_limit_after"] = gpu_info()["power_limit"]
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
