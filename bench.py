#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 bayesian-torch hot path.

Workload (BASELINE.json configs[2], "C3"): MC inference through dnn_to_bnn(torchvision ResNet-18,
10 classes), Reparameterization layers, synthetic 3x32x32 inputs, batch B=128, N=64 Monte-Carlo
weight samples per input batch.  One "step" = one input batch -> predictive mean + variance
[2, B, C] over the N samples (fused layer kernels, fused softmax/moment kernel, ONE all-reduce).
Every step draws FRESH weight samples (the reference draws new eps on every forward).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference (baseline/_ref) on host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # N > 1: one rank per GPU, samples sharded
    python bench.py --config c4 ...                          # BASELINE.json configs[3]: ResNet-50 Flipout 3x224x224, N=32
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's mean / var as DIR/*.npy

Prints ONE JSON line (rank 0).  metric = MC image-samples/sec = B*N / t_step.
The HEADLINE line is the fp32 model (fp32 parameters and activations -> tcgen05 kind::tf32 operands, the reference's
default dtype); the same measurement of the bf16 model rides in the line's "bf16" object (labelled).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree: it writes nothing there

CONFIGS = {
    # name: (arch, layer type, image, batch, MC samples, classes, metric, workload text)
    "c3": ("resnet18", "Reparameterization", 32, 128, 64, 10, "mc_inference_image_samples_per_sec_N64_bayesian_resnet18",
           "C3: dnn_to_bnn(torchvision ResNet-18, 10 classes) Reparameterization, 3x32x32, B=128, N=64 MC samples/step, "
           "samples sharded over ranks, one all-reduce of [2,B,C]"),
    "c4": ("resnet50", "Flipout", 224, 128, 32, 1000, "mc_inference_image_samples_per_sec_N32_bayesian_resnet50_flipout",
           "C4: dnn_to_bnn(torchvision ResNet-50, 1000 classes) Flipout, 3x224x224, B=128, N=32 MC samples/step, "
           "samples sharded over ranks, one all-reduce of [2,B,C]"),
}
PRM = {"prior_mu": 0.0, "prior_sigma": 1.0, "posterior_mu_init": 0.0, "posterior_rho_init": -3.0,
       "type": "Reparameterization", "moped_enable": False, "moped_delta": 0.5}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------------- reference arm
def _import_reference():
    """the UNMODIFIED reference package, installed once with pip --target into baseline/_ref (git-ignored, travels to
    the GPU box); None when it is not there"""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "bayesian_torch")):
        return None
    for k in [k for k in sys.modules if k == "bayesian_torch" or k.startswith("bayesian_torch.")]:
        del sys.modules[k]                       # (the repo root holds a drop-in package of the same import name)
    sys.path.insert(0, ref)
    try:
        import bayesian_torch.models.dnn_to_bnn as ref_d2b
        assert os.path.abspath(ref_d2b.__file__).startswith(os.path.abspath(ref)), ref_d2b.__file__
        return ref_d2b
    finally:
        sys.path.remove(ref)


def time_cpu_reference(cfg, steps, warmup, mc_per_step):
    """The reference's own modules (baseline/_ref: dnn_to_bnn(torchvision ResNet) and the evaluate() loop of
    examples/main_bayesian_cifar_dnn2bnn.py:541-557 -- N sequential forwards, stack, softmax, mean) on the host cores;
    falls back to the validated port (oracle/ref_model.py) only if the reference tree did not travel."""
    arch, typ, res, B, N, classes, _, _ = CONFIGS[cfg]
    import torchvision
    avail = len(os.sched_getaffinity(0))
    ref = _import_reference()
    torch.manual_seed(0)
    net = getattr(torchvision.models, arch)(num_classes=classes)
    if ref is not None:
        ref.dnn_to_bnn(net, dict(PRM, type=typ))
        kind = "reference"
    else:
        from oracle.ref_model import oracle_dnn_to_bnn
        net = oracle_dnn_to_bnn(net, flipout=typ == "Flipout")
        kind = "port"
    net.eval()
    torch.manual_seed(0)
    x = torch.randn(B, 3, res, res)

    def evaluate(n):
        with torch.no_grad():
            outs = [net(x) for _ in range(n)]
            p = torch.softmax(torch.stack(outs), -1)
            return p.mean(0), p.var(0, unbiased=False)

    best = (None, float("inf"))
    for t in sorted({min(avail, c) for c in (8, 16, 32, 64, avail)}):   # ATen's pool degrades when oversubscribed
        torch.set_num_threads(t)
        evaluate(1)
        t0 = time.perf_counter()
        evaluate(1)
        dt1 = time.perf_counter() - t0
        if dt1 < best[1]:
            best = (t, dt1)
    cores = best[0]
    torch.set_num_threads(cores)
    for _ in range(warmup):
        evaluate(1)
    t0 = time.perf_counter()
    for _ in range(steps):
        evaluate(mc_per_step)
    dt = (time.perf_counter() - t0) / steps
    return {"value": B * mc_per_step / dt, "unit": "image-samples/s", "cores": cores, "kind": kind,
            "sample": f"B={B}, {mc_per_step} MC samples per step (of {N}), {steps} steps, fp32, {cores} threads (best of "
                      f"8/16/32/64/{avail} available); " + ("baseline/_ref = the unmodified reference package" if kind == "reference"
                                                            else "oracle/ref_model.py port (baseline/_ref absent)"),
            "ms_per_step": dt * 1e3, "mc_per_step": mc_per_step}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arch, typ, res, B, N, classes, metric, workload = CONFIGS[args.config]
    mc = N if args.config == "c3" else 1          # C3: the full N=64 evaluate() per step; C4: one forward (bounded sample)
    cb = time_cpu_reference(args.config, max(args.steps, 1), min(args.warmup, 2), mc)
    line = {"impl": "reference", "metric": metric, "value": cb["value"], "unit": cb["unit"], "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "global_batch": B, "mc_samples": N, "mc_samples_per_step": mc},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------- this repo
def build_model(cfg, device, dtype, fuse=True):
    import torchvision
    import bayesian_torch_b200 as btb
    arch, typ, res, B, N, classes, _, _ = CONFIGS[cfg]
    torch.manual_seed(0)
    net = getattr(torchvision.models, arch)(num_classes=classes)
    btb.dnn_to_bnn(net, dict(PRM, type=typ))
    btb.assign_layer_keys(net)
    net = net.eval().to(device).to(dtype).to(memory_format=torch.channels_last)
    if fuse:
        btb.fuse_inference(net)      # eval-mode BatchNorm / ReLU / residual add -> conv epilogues
    return net


def measure(args, cfg, dtype, dev, world, rank, local, want_roofline):
    """one model dtype: device-resident step time, end-to-end step time, launches, clocks and (rank 0, world 1) the
    per-family roofline pass"""
    import torch.distributed as dist
    import bayesian_torch_b200 as btb
    from bayesian_torch_b200 import _native
    arch, typ, res, B, N_MC, classes, metric, workload = CONFIGS[cfg]
    net = build_model(cfg, dev, dtype, fuse=not args.no_fuse)
    btb.manual_seed(0)
    torch.manual_seed(1234)
    x_host = torch.randn(B, 3, res, res).pin_memory()
    x_dev = x_host.to(dev).to(dtype).contiguous(memory_format=torch.channels_last)
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)      # 168 MB > the 126 MB L2 (a write-back L2: the memset replaces every line)
    chunk = args.chunk
    if chunk is None and cfg == "c4":
        chunk = 4                                                      # 4 x 128 images of 224^2 per pass
    use_graph = not args.no_graph

    def step_device(graph=use_graph):
        flush.zero_()
        return btb.mc_predict(net, x_dev, N_MC, chunk=chunk, use_graph=graph, fresh=True)

    def step_e2e():
        flush.zero_()
        xd = x_host.to(dev, non_blocking=True).to(dtype).contiguous(memory_format=torch.channels_last)
        mean, var = btb.mc_predict(net, xd, N_MC, chunk=chunk, use_graph=use_graph, fresh=True)
        return torch.stack((mean, var)).cpu()          # D2H read of the step's result (synchronises)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (ms per step, what the last step returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps, last

    if args.profile:          # under ncu: W warm-up passes + K steps of the device-resident step, nothing else
        for _ in range(args.warmup + args.steps):
            step_device(False)
        torch.cuda.synchronize()
        return None
    for _ in range(max(args.warmup, 3)):
        step_device()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = _native.launch_count
    ms_step, (mean, var) = timed(step_device, args.steps)
    launches = _native.launch_count - l0
    outputs = {"mean": mean.cpu(), "var": var.cpu()}          # [B, C] fp32 each, what mc_predict hands its caller
    sampler.stop_flag = True
    sampler.join(timeout=2)
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    out = {"ms_per_step": ms_step, "value": B * N_MC / (ms_step * 1e-3), "e2e_ms": ms_e2e,
           "e2e": {"value": B * N_MC / (ms_e2e * 1e-3), "unit": "image-samples/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": 2 * B * classes * 4},
           "gpu_launches": launches, "clocks": sampler.summary(), "chunk": chunk, "outputs": outputs}
    if not want_roofline:
        return out

    # ---- roofline pass: CUDA events around every Bayesian-layer launch of `steps` eager steps.  The device first
    # spins for a few ms (torch.cuda._sleep) so that the host enqueues the whole step ahead of it: no host latency
    # sits between the event records and the kernels they bracket.  Numerators come from the LOGICAL tensors
    # (SURVEY.md 8d): bytes = sizeof * (|x| + |out| + 2|W| + 2|b|) per MC sample, flops = 2 M N K (Flipout 4 M N K);
    # filter taps the kernels skip because they only see zero padding are reported separately.
    rec = []

    def hook(geom, x, mu_w, out, info):
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        S = geom.n_samples
        es_x, es_p = out.element_size(), mu_w.element_size()
        m_rows = out.numel() // geom.c_out
        k_nom = info["k_logical"]
        mult = 2.0 if info["flipout"] else 1.0
        nbytes = S * (es_x * (info["x_logical_numel"] + out.numel() // S) + 2 * es_p * (info["w_numel"] + info["b_numel"]))
        nmin = es_x * (info["x_logical_numel"] * (1 if geom.x_shared else S) + out.numel()) + 2 * es_p * (info["w_numel"] + info["b_numel"])
        rec.append({"ev": ev, "bytes": nbytes, "bytes_min": nmin, "flops": mult * 2.0 * m_rows * geom.c_out * k_nom,
                    "flops_exec": mult * 2.0 * m_rows * geom.c_out * info["k_used"], "info": info})
        return ev

    def post(path):
        rec[-1]["path"] = path

    _native.timing_hook, _native.timing_post = hook, post
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eager_ms = 0.0
    for _ in range(args.steps):
        torch.cuda._sleep(int(2e7))            # ~10 ms at 1.9 GHz: the host runs ahead of the device
        e0.record()
        step_device(False)                     # eager: per-launch events cannot live inside a captured graph
        e1.record()
        torch.cuda.synchronize()
        eager_ms += e0.elapsed_time(e1)
    _native.timing_hook = _native.timing_post = None
    eager_ms /= args.steps
    fam = {}
    tot = {"ms": 0.0, "bytes": 0.0, "bytes_min": 0.0, "flops": 0.0, "flops_exec": 0.0}
    for r in rec:
        ms = r["ev"][0].elapsed_time(r["ev"][1]) / args.steps
        f = fam.setdefault(r.get("path", "?"), {"launches": 0, "ms": 0.0, "bytes": 0.0, "bytes_min": 0.0, "flops": 0.0, "flops_exec": 0.0})
        f["launches"] += 1
        for k, v in (("ms", ms), ("bytes", r["bytes"] / args.steps), ("bytes_min", r["bytes_min"] / args.steps),
                     ("flops", r["flops"] / args.steps), ("flops_exec", r["flops_exec"] / args.steps)):
            f[k] += v
            tot[k] += v
    hbm_peak, tf_peak, peak_src = _peaks()
    tf_peak_eff = tf_peak * (0.5 if dtype == torch.float32 else 1.0)      # kind::tf32 runs at half the bf16 rate
    for f in fam.values():
        f["launches"] //= args.steps
        f["hbm_gbs"] = f["bytes"] / (f["ms"] * 1e-3) / 1e9
        f["hbm_frac"] = f["hbm_gbs"] / hbm_peak
        f["tflops_executed"] = f["flops_exec"] / (f["ms"] * 1e-3) / 1e12
        f["tensor_frac"] = f["tflops_executed"] / tf_peak_eff
    n_fused = len(rec) // args.steps
    traffic = None            # DRAM bytes per step of the same launches from the committed ncu --set full capture
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            with open(tpath) as tf:
                tj = json.load(tf)
            ent = tj.get("bf16" if dtype == torch.bfloat16 else "fp32", tj)
            if ent.get("launches") == n_fused:
                traffic = ent["dram_bytes_per_step"]
        except (OSError, ValueError, KeyError, AttributeError):
            traffic = None
    ach_gbs = tot["bytes"] / (tot["ms"] * 1e-3) / 1e9
    out["roofline"] = {
        "kernel": "all Bayesian-layer launches of a step (families below)", "bound": "hbm",
        "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak, "traffic": traffic,
        "traffic_source": "profiles/traffic.json (ncu dram__bytes_read+write, summed over the same launches of one step)" if traffic else None,
        "peak_source": peak_src, "launches_per_step": n_fused, "kernel_ms_per_step": tot["ms"],
        # numerator and denominator from the SAME pass (eager, event-bracketed): the share of that step spent inside the
        # Bayesian-layer kernels, <= 1 by construction.  Against the graph replay the event-bracketed kernel times can
        # exceed 1 by a percent or two: every event pair also brackets the launch gap that a graph replay overlaps.
        "eager_step_ms": eager_ms, "kernel_share_of_step": tot["ms"] / eager_ms,
        "graph_step_ms": ms_step, "kernel_ms_over_graph_step": tot["ms"] / ms_step,
        "algorithmic_bytes_per_step": tot["bytes"],
        "algorithmic_bytes_definition": "SURVEY 8d: sizeof * (|x| + |out| + 2|W| + 2|b|) per Bayesian layer and MC sample, LOGICAL tensors "
                                        "(the stem's materialised im2col matrix is not counted)",
        "min_bytes_per_step_weights_once_per_launch": tot["bytes_min"],
        "tensor": {"achieved_tflops_executed": tot["flops_exec"] / (tot["ms"] * 1e-3) / 1e12,
                   "nominal_tflops_incl_skipped_padding_taps": tot["flops"] / (tot["ms"] * 1e-3) / 1e12,
                   "peak_tflops": tf_peak_eff, "frac": tot["flops_exec"] / (tot["ms"] * 1e-3) / 1e12 / tf_peak_eff,
                   "flops_executed_per_step": tot["flops_exec"], "flops_nominal_per_step": tot["flops"]},
        "families": fam,
        "note": "the step is issue / latency bound (DRAM traffic < algorithmic bytes: the MC samples of a launch share mu/rho through L2)",
    }
    return out


def dump_outputs(dirname, by_dtype):
    """DIR/<dtype>_<output>.npy (float32) of the last timed step of every model dtype that was measured.  The inputs
    (image batch, parameters, Philox seed and sample offsets) depend only on the arguments, so two builds run with the
    same arguments can be compared array for array."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for dt, outs in by_dtype.items():
        for name, t in outs.items():
            np.save(os.path.join(dirname, f"{dt}_{name}.npy"), t.float().numpy())


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner to STDOUT on the first communicator (seen on the 2xB200 box): keep stdout to the ONE
        # JSON line of the contract -- fd 1 points at stderr while the communicator is created and warmed up
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    cfg = args.config
    arch, typ, res, B, N_MC, classes, metric, workload = CONFIGS[cfg]
    dtypes = {"fp32": [torch.float32], "bf16": [torch.bfloat16], "both": [torch.float32, torch.bfloat16]}[args.dtype]
    res_by = {}
    for dt in dtypes:
        res_by[dt] = measure(args, cfg, dt, dev, world, rank, local, want_roofline=(world == 1 or True))
        torch.cuda.empty_cache()
    if args.profile or rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {("fp32" if dt == torch.float32 else "bf16"): r["outputs"] for dt, r in res_by.items()})
    head = res_by[dtypes[0]]
    name = {torch.float32: "tf32 (fp32 parameters and activations, tcgen05 kind::tf32)", torch.bfloat16: "bf16"}
    line = {
        "metric": metric, "value": head["value"], "unit": "image-samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": name[dtypes[0]], "data": "synthetic",
        "config": {"workload": workload, "global_batch": B, "mc_samples": N_MC, "mc_chunk": head["chunk"] or "all",
                   "epilogue_fusion": not args.no_fuse, "cuda_graph": not args.no_graph, "fresh_eps_every_step": True,
                   "parallelism": f"mc-sample-shard{world}",
                   "l2": "flushed between steps (160 MiB memset > 126 MB L2, inside the timed region); per-step working set >> L2",
                   "images_per_sec_reference_style": B / (head["ms_per_step"] * 1e-3)},
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
    }
    if "roofline" in head:
        line["roofline"] = head["roofline"]
    if len(dtypes) > 1:
        b = res_by[dtypes[1]]
        line["bf16"] = {"label": "same workload, model.to(bfloat16): bf16 parameters and activations, kind::f16 operands "
                                 "(NOT the headline: narrower than the reference arm's fp32)",
                        "value": b["value"], "ms_per_step": b["ms_per_step"], "e2e": b["e2e"],
                        "gpu_launches": b["gpu_launches"], "clocks": b["clocks"]}
        if "roofline" in b:
            line["bf16"]["roofline"] = b["roofline"]
    if world == 1 and not args.no_cpu_baseline:
        cb = time_cpu_reference(cfg, 2, 1, 4 if cfg == "c3" else 1)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--dtype", default="both", choices=["both", "fp32", "bf16"],
                    help="both: fp32 headline + the bf16 model as a labelled sub-object")
    ap.add_argument("--chunk", type=int, default=None, help="MC samples per pass (default: all samples of the rank)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from python instead of replaying a CUDA graph")
    ap.add_argument("--no-fuse", action="store_true", help="keep BatchNorm/ReLU/residual as separate PyTorch kernels")
    ap.add_argument("--profile", action="store_true", help="profiling mode (ncu): only warmup+steps device steps, no JSON")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the predictive mean and variance of the last timed step as "
                         "DIR/<dtype>_{mean,var}.npy (float32, [B, C])")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.profile):
        ap.error("--dump-outputs writes the outputs of the timed B200 steps: not with --impl reference or --profile")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
