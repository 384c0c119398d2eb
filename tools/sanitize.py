#!/usr/bin/env python
"""One small launch of every kernel family, for compute-sanitizer (SURVEY.md section 5: memcheck / racecheck on the
hand-rolled mbarrier / TMEM / TMA protocols).

    compute-sanitizer --tool memcheck  python tools/sanitize.py
    compute-sanitizer --tool racecheck python tools/sanitize.py
    compute-sanitizer --tool synccheck python tools/sanitize.py

Prints the kernel family each launch took; tools/gpu_sanitize.sh keeps the sanitizer summaries."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ.setdefault("BT_DYNAMIC_ENV", "1")

import bayesian_torch_b200 as btb  # noqa: E402
from bayesian_torch_b200 import _native  # noqa: E402
from gpu_util import build_layer  # noqa: E402

DEV = "cuda:0"


def run(tag, layer, x, env=None, **kw):
    old = {}
    for k, v in (env or {}).items():
        old[k] = os.environ.get(k)
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    try:
        btb.manual_seed(1)
        y = layer._forward_impl(x, kw.pop("return_kl", False), **kw)
        torch.cuda.synchronize()
        y0 = y[0] if isinstance(y, tuple) else y
        print(f"{tag:34s} path={_native.last_forward_path():10s} out={tuple(y0.shape)} finite={bool(torch.isfinite(y0.float()).all())}",
              flush=True)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def main():
    torch.manual_seed(0)
    bf = torch.bfloat16
    only = set(sys.argv[1:])
    want = lambda t: not only or t in only

    if want("generic"):
        lay = build_layer("conv", 2, False, 16, 24, 3, 1, 1).to(DEV)
        run("generic tf32 conv + KL", lay, torch.randn(2, 16, 6, 6, device=DEV), return_kl=True)
        lay = build_layer("linear", 0, True, 72, 40, None).to(DEV).to(bf)
        run("generic bf16 flipout linear", lay, torch.randn(9, 72, device=DEV), return_kl=True)
    if want("fast"):
        lay = build_layer("conv", 2, True, 64, 64, 3, 2, 1).to(DEV).to(bf)
        run("fast flipout conv s2", lay, torch.randn(4, 64, 8, 8, device=DEV).to(bf), env={"BT_DISABLE_TMA": "1"})
        lay = build_layer("conv", 2, False, 128, 128, 3, 2, 1).to(DEV).to(bf)
        run("fast reparam conv s2", lay, torch.randn(4, 128, 4, 4, device=DEV).to(bf), env={"BT_DISABLE_TMA": "1"})
    if want("ws"):
        lay = build_layer("conv", 2, False, 64, 128, 1, 2, 0).to(DEV).to(bf)
        run("ws 1x1 s2", lay, torch.randn(16, 64, 8, 8, device=DEV).to(bf), env={"BT_DISABLE_TMA": "1"})
        lay = build_layer("conv", 2, False, 64, 64, 3, 1, 1).to(DEV).to(bf)
        run("ws tap-copy 3x3", lay, torch.randn(8, 64, 8, 8, device=DEV).to(bf), env={"BT_DISABLE_TMA": "1", "BT_DISABLE_DIRECT": "1"})
    if want("direct"):
        lay = build_layer("conv", 2, False, 64, 64, 3, 1, 1).to(DEV).to(bf)
        run("direct reparam 3x3", lay, torch.randn(8, 64, 8, 8, device=DEV).to(bf), env={"BT_FORCE_DIRECT": "1"})
        lay = build_layer("conv", 2, True, 64, 64, 3, 1, 1).to(DEV).to(bf)
        run("direct flipout 3x3", lay, torch.randn(8, 64, 8, 8, device=DEV).to(bf), env={"BT_FORCE_DIRECT": "1"})
    if want("tma"):
        lay = build_layer("conv", 2, False, 64, 64, 3, 2, 1).to(DEV).to(bf)
        run("tma resident bf16 conv", lay, torch.randn(8, 64, 8, 8, device=DEV).to(bf), env={"BT_TMA_PREFER": "1", "BT_TMA_MODE": "1"})
        run("tma stream bf16 conv", lay, torch.randn(8, 64, 8, 8, device=DEV).to(bf), env={"BT_TMA_PREFER": "1", "BT_TMA_MODE": "2"})
        lay = build_layer("linear", 0, False, 256, 96, None).to(DEV)
        run("tma resident tf32 linear", lay, torch.randn(200, 256, device=DEV), env={"BT_TMA_MODE": "1"})
        run("tma stream tf32 linear", lay, torch.randn(200, 256, device=DEV), env={"BT_TMA_MODE": "2"})
    if want("dtma"):
        lay = build_layer("conv", 2, False, 64, 64, 3, 1, 1).to(DEV).to(bf)
        lay._bt_ep_scale, lay._bt_ep_shift, lay._bt_ep_relu = torch.rand(64, device=DEV) + 0.5, torch.randn(64, device=DEV), True
        x = torch.randn(3 * 6, 64, 8, 8, device=DEV).to(bf)
        res = torch.randn(3 * 6, 64, 8, 8, device=DEV).to(bf).contiguous(memory_format=torch.channels_last)
        with btb.mc_sample_context(3, 6, 0):
            run("tma_direct bf16 3x3 + residual", lay, x, residual=res)
        lay = build_layer("conv", 2, False, 32, 64, 3, 1, 1).to(DEV)
        run("tma_direct tf32 3x3", lay, torch.randn(5, 32, 6, 6, device=DEV))
        lay = build_layer("conv", 2, True, 64, 64, 3, 1, 1).to(DEV).to(bf)
        run("tma_direct flipout 3x3", lay, torch.randn(4, 64, 8, 8, device=DEV).to(bf))
        lay = build_layer("linear", 0, True, 256, 128, None).to(DEV).to(bf)
        run("tma_stream flipout linear", lay, torch.randn(200, 256, device=DEV).to(bf))
    if want("cluster"):
        lay = build_layer("linear", 0, False, 256, 256, None).to(DEV).to(bf)
        run("tma_stream, 2-CTA cluster multicast", lay, torch.randn(300, 256, device=DEV).to(bf), env={"BT_TMA_MODE": "2"})
        lay = build_layer("conv", 2, False, 128, 256, 3, 2, 1).to(DEV)
        run("tma_stream tf32 conv, cluster", lay, torch.randn(6, 128, 4, 4, device=DEV), env={"BT_TMA_MODE": "2", "BT_TMA_PREFER": "1"})
    if want("pool"):
        lay = build_layer("conv", 2, False, 3, 64, 7, 2, 3).to(DEV).to(bf)
        lay._bt_ep_scale, lay._bt_ep_shift, lay._bt_ep_relu = torch.rand(64, device=DEV) + 0.5, torch.randn(64, device=DEV), True
        lay._bt_ep_pool = True
        with btb.mc_sample_context(5, 4, 0):
            run("tma resident + fused max-pool", lay, torch.randn(4, 3, 32, 32, device=DEV).to(bf),
                env={"BT_TMA_PREFER": "1", "BT_TMA_MODE": "1", "BT_DISABLE_DTMA": "1"})
    if want("aux"):
        lay = build_layer("linear", 0, False, 512, 256, None).to(DEV)
        print("kl", float(lay.kl_loss()))
        lay(torch.randn(4, 512, device=DEV))
        lay.materialize_eps(0)
        logits = torch.randn(3 * 8, 10, device=DEV)
        sums = torch.empty(2, 8, 10, device=DEV)
        _native.mc_accumulate(logits, 3, 8, sums, accumulate=False)
        mean, var = torch.empty(8, 10, device=DEV), torch.empty(8, 10, device=DEV)
        _native.mc_finalize(sums, 3, mean, var)
        xp = torch.randn(4, 8, 8, 16, device=DEV).to(bf)
        _native.maxpool2d_nhwc(xp, (3, 3), (2, 2), (1, 1))
        torch.cuda.synchronize()
        print("aux kernels ok", flush=True)
    if want("mc"):
        # large-C softmax moments (two kernels, chunk accumulate) and the fp64 regression moments + finalize
        logits = torch.randn(3 * 4, 1500, device=DEV).to(bf)
        sums, ent = torch.empty(2, 4, 1500, device=DEV), torch.empty(4, device=DEV)
        _native.mc_accumulate(logits[:8], 2, 4, sums, accumulate=False, entropy_sum=ent)
        _native.mc_accumulate(logits[8:], 1, 4, sums, accumulate=True, entropy_sum=ent)
        y = torch.randn(3 * 1000, device=DEV)
        rs = torch.empty(2 * 1000, dtype=torch.float64, device=DEV)
        _native.mc_regression_accumulate(y, 3, rs, accumulate=False)
        _native.mc_regression_accumulate(y[1:2998], 3, torch.empty(2 * 999, dtype=torch.float64, device=DEV), False)
        mean, var = torch.empty(1000, device=DEV), torch.empty(1000, device=DEV)
        _native.mc_regression_finalize(rs, 3, mean, var)
        torch.cuda.synchronize()
        print("mc head kernels ok", flush=True)


if __name__ == "__main__":
    main()
