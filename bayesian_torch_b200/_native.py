"""ctypes binding of libbtb200.so (C ABI: include/btb200.h).

PyTorch is used for device memory and streams only: every wrapper hands raw device pointers and
the current CUDA stream handle to the library.  There is deliberately NO CPU fallback -- a CPU
tensor, a missing library or a non-sm_100 device raises.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BT_LIB_VARIANT") or os.path.join(_HERE, "libbtb200.so")   # (variant: A/B builds, tools/)

BT_F32, BT_BF16 = 0, 1
MODE_REPARAM, MODE_FLIPOUT = 0, 1
_DTYPES = {torch.float32: BT_F32, torch.bfloat16: BT_BF16}


class BtDebugIO(ctypes.Structure):
    _fields_ = [("eps_w_in", ctypes.c_void_p), ("eps_b_in", ctypes.c_void_p),
                ("sign_in", ctypes.c_void_p), ("sign_out", ctypes.c_void_p)]


class BtEpilogue(ctypes.Structure):
    _fields_ = [("scale", ctypes.c_void_p), ("shift", ctypes.c_void_p), ("residual", ctypes.c_void_p),
                ("relu", ctypes.c_int32)]


class BtLayerGeom(ctypes.Structure):
    _fields_ = [("n_samples", ctypes.c_int32), ("x_shared", ctypes.c_int32), ("batch", ctypes.c_int32),
                ("c_in", ctypes.c_int32), ("c_out", ctypes.c_int32), ("groups", ctypes.c_int32),
                ("in_dhw", ctypes.c_int32 * 3), ("out_dhw", ctypes.c_int32 * 3), ("k_dhw", ctypes.c_int32 * 3),
                ("stride", ctypes.c_int32 * 3), ("pad", ctypes.c_int32 * 3), ("dil", ctypes.c_int32 * 3),
                ("rho_is_sigma", ctypes.c_int32), ("transposed", ctypes.c_int32),
                ("pool_hw", ctypes.c_int32 * 2), ("sample_offset", ctypes.c_void_p)]


class BtForwardPlan(ctypes.Structure):
    _fields_ = [("path", ctypes.c_int32), ("block_n", ctypes.c_int32), ("m_subtiles", ctypes.c_int32),
                ("k_blocks", ctypes.c_int32), ("grid", ctypes.c_int32 * 3), ("threads", ctypes.c_int32),
                ("smem_bytes", ctypes.c_int32), ("tmem_cols", ctypes.c_int32), ("window_slots", ctypes.c_int32),
                ("window_rows", ctypes.c_int32), ("staged_epilogue", ctypes.c_int32), ("samples_per_cta", ctypes.c_int32),
                ("window_boxes", ctypes.c_int32), ("cluster_n", ctypes.c_int32), ("pool_fused", ctypes.c_int32)]


_lib = None
_lock = threading.Lock()
launch_count = 0          # kernels of libbtb200 launched by this process (bench.py reports it)
timing_hook = None        # optional callable(geom, x, mu_w, out, info) -> (start_event, end_event) (bench.py roofline pass)
timing_post = None        # optional callable(kernel_family_name), called right after the launch

# every symbol include/btb200.h declares: (name, restype, argtypes)
_vp, _i, _i64, _f, _u64, _u32 = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float,
                                 ctypes.c_uint64, ctypes.c_uint32)
SYMBOLS = [
    ("bt_version", _i, []),
    ("bt_last_error", ctypes.c_char_p, []),
    ("bt_device_check", _i, []),
    ("bt_sm_count", _i, []),
    ("bt_set_pointer_checks", _i, [_i]),
    ("bt_kl_workspace_bytes", _i64, []),
    ("bt_kl_gaussian", _i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _f, _f, _i, _vp, _i, _vp, _vp]),
    ("bt_forward_workspace_bytes", _i64, []),
    ("bt_layer_forward", _i, [_i, ctypes.POINTER(BtLayerGeom), _vp, _i, _vp, _vp, _vp, _vp, _i, _vp,
                              _vp, _f, _f, _u64, _u32, _u32, ctypes.POINTER(BtDebugIO), ctypes.POINTER(BtEpilogue),
                              _vp, _vp]),
    ("bt_layer_forward_plan", _i, [_i, ctypes.POINTER(BtLayerGeom), _i, _i, _i, _i, _i, _i, ctypes.POINTER(BtForwardPlan)]),
    ("bt_last_forward_path", _i, []),
    ("bt_tma_probe4d", _i, [_vp, _i, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32),
                            ctypes.POINTER(ctypes.c_int32), _u32, _vp, _vp]),
    ("bt_tma_probe", _i, [ctypes.POINTER(BtLayerGeom), _vp, _i, _i64, _i, _i, _i, _i, _vp, _vp]),
    ("bt_rng_export", _i, [_i, _vp, _i64, _i64, ctypes.c_int32, ctypes.c_int32, _u64, _u32, _u32, _vp]),
    ("bt_mc_accumulate", _i, [_vp, _i, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _vp, _i, _vp]),
    ("bt_mc_accumulate_ex", _i, [_vp, _i, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _vp, _vp, _i, _vp]),
    ("bt_mc_uncertainty", _i, [_vp, _vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _vp, _vp, _vp]),
    ("bt_mc_finalize", _i, [_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _vp, _vp, _vp]),
    ("bt_mc_accumulate_large", _i, [_vp, _i, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _vp, _vp, _i, _vp, _vp]),
    ("bt_mc_regression_accumulate", _i, [_vp, _i, ctypes.c_int32, _i64, _vp, _i, _vp]),
    ("bt_mc_regression_finalize", _i, [_vp, _i64, ctypes.c_int32, _vp, _vp, _vp]),
    ("bt_im2col2d", _i, [_vp, _i, _i64] + [ctypes.c_int32] * 3 + [ctypes.POINTER(ctypes.c_int64)] + [ctypes.c_int32] * 9 + [_vp, _vp]),
    ("bt_lstm_cell", _i, [_vp] * 7 + [_i] + [ctypes.c_int32] * 4 + [_vp]),
    ("bt_maxpool2d_nhwc", _i, [_vp, _i, _i64] + [ctypes.c_int32] * 9 + [_vp, _vp]),
]


def load():
    """dlopen the in-tree library; raise (never fall back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m bayesian_torch_b200.build` "
                "(nvcc, sm_100a).  bayesian_torch_b200 has no CPU / eager fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc):
    if rc != 0:
        msg = load().bt_last_error().decode("utf-8", "replace")
        if rc in (-1, -2):
            raise ValueError(f"libbtb200: {msg}")
        raise RuntimeError(f"libbtb200 (code {rc}): {msg}")


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(
            f"bayesian_torch_b200: `{name}` is on {t.device}; the B200 layers run on CUDA (sm_100a) only "
            "and have no CPU fallback (move the module and its inputs to cuda).")


def dtype_code(t, name):
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise ValueError(f"bayesian_torch_b200: `{name}` has dtype {t.dtype}; supported: float32, bfloat16")


_ws = {}


def _workspace(device, kind, nbytes):
    key = (device.index, kind, torch.cuda.current_stream(device).cuda_stream)
    w = _ws.get(key)
    if w is None or w.numel() * 4 < nbytes:
        w = torch.zeros((nbytes + 3) // 4, dtype=torch.float32, device=device)
        _ws[key] = w
    return w


def kl_gaussian(mu_w, rho_w, prior_mu_w=None, prior_sigma_w=None, mu_b=None, rho_b=None,
                prior_mu_b=None, prior_sigma_b=None, prior_mu=0.0, prior_sigma=1.0, out=None, accumulate=False):
    """mean-KL(weight) + mean-KL(bias) in ONE launch -> 0-d fp32 tensor."""
    lib = load()
    require_cuda(mu_w, "mu")
    dt = dtype_code(mu_w, "mu")
    for t in (rho_w, prior_mu_w, prior_sigma_w, mu_b, rho_b, prior_mu_b, prior_sigma_b):
        if t is not None and t.dtype != mu_w.dtype:
            raise ValueError("bayesian_torch_b200: KL tensors must share one dtype")
    dev = mu_w.device
    if out is None:
        out = torch.empty((), dtype=torch.float32, device=dev)
    ws = _workspace(dev, "kl", lib.bt_kl_workspace_bytes())
    global launch_count
    launch_count += 1
    with torch.cuda.device(dev):
        _check(lib.bt_kl_gaussian(_ptr(mu_w), _ptr(rho_w), mu_w.numel(), _ptr(prior_mu_w), _ptr(prior_sigma_w),
                                  _ptr(mu_b), _ptr(rho_b), 0 if mu_b is None else mu_b.numel(),
                                  _ptr(prior_mu_b), _ptr(prior_sigma_b), float(prior_mu), float(prior_sigma),
                                  dt, _ptr(out), int(bool(accumulate)), _ptr(ws), _stream(dev)))
    return out


def layer_forward(mode, geom, x, mu_w, rho_w, mu_b, rho_b, out, kl_out=None, prior_mu=0.0, prior_sigma=1.0,
                  seed=0, layer_key=0, sample0=0, eps_w_in=None, eps_b_in=None, sign_in=None, sign_out=None,
                  ep_scale=None, ep_shift=None, ep_residual=None, ep_relu=False, info=None):
    lib = load()
    dev = x.device
    dbg = None
    if any(t is not None for t in (eps_w_in, eps_b_in, sign_in, sign_out)):
        for t in (eps_w_in, eps_b_in, sign_in, sign_out):
            if t is not None and (t.dtype != torch.float32 or not t.is_cuda):
                raise ValueError("debug eps/sign tensors must be float32 CUDA tensors")
        dbg = BtDebugIO(*(None if t is None else t.data_ptr() for t in (eps_w_in, eps_b_in, sign_in, sign_out)))
    epi = None
    if ep_scale is not None or ep_residual is not None or ep_relu:
        if ep_scale is not None and (ep_scale.dtype != torch.float32 or ep_shift is None or ep_shift.dtype != torch.float32):
            raise ValueError("epilogue scale / shift must both be float32 tensors")
        if ep_residual is not None and (ep_residual.dtype != out.dtype or ep_residual.numel() != out.numel()):
            raise ValueError("epilogue residual must match the output in dtype and size")
        epi = BtEpilogue(None if ep_scale is None else ep_scale.data_ptr(),
                         None if ep_shift is None else ep_shift.data_ptr(),
                         None if ep_residual is None else ep_residual.data_ptr(), int(bool(ep_relu)))
    probe = os.environ.get("BT_DIRECT_TIMES") is not None      # tools/direct_probe.py: phase stamps of bt_direct_kernel
    ws = _workspace(dev, "fwd", lib.bt_forward_workspace_bytes()) if (kl_out is not None or probe) else None
    global launch_count
    launch_count += 1 if kl_out is None else 2
    hook = timing_hook(geom, x, mu_w, out, info or {}) if timing_hook is not None else None
    with torch.cuda.device(dev):
        if hook is not None:
            hook[0].record(torch.cuda.current_stream(dev))
        _check(lib.bt_layer_forward(int(mode), ctypes.byref(geom), _ptr(x), dtype_code(x, "input"),
                                    _ptr(mu_w), _ptr(rho_w), _ptr(mu_b), _ptr(rho_b), dtype_code(mu_w, "mu"),
                                    _ptr(out), _ptr(kl_out), float(prior_mu), float(prior_sigma),
                                    ctypes.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), ctypes.c_uint32(layer_key),
                                    ctypes.c_uint32(sample0 & 0xFFFFFFFF),
                                    None if dbg is None else ctypes.byref(dbg),
                                    None if epi is None else ctypes.byref(epi), _ptr(ws), _stream(dev)))
        if hook is not None:
            hook[1].record(torch.cuda.current_stream(dev))
            if timing_post is not None:
                timing_post(last_forward_path())
    return out


def plan_forward(mode, geom, x_dtype, p_dtype, with_kl=False, with_debug_hooks=False, with_residual=False, sm_count=148):
    """The tiling / kernel-selection decision of bt_layer_forward for `geom` (no GPU needed): dict of BtForwardPlan."""
    plan = BtForwardPlan()
    _check(load().bt_layer_forward_plan(int(mode), ctypes.byref(geom), _DTYPES[x_dtype], _DTYPES[p_dtype], int(with_kl),
                                        int(with_debug_hooks), int(with_residual), int(sm_count), ctypes.byref(plan)))
    d = {k: getattr(plan, k) for k, _ in BtForwardPlan._fields_ if k != "grid"}
    d["grid"] = tuple(plan.grid)
    d["path"] = PATH_NAMES[plan.path]
    return d


def tma_probe(geom, x, m0, sample=0, group=0, tap=0, slab=0):
    """the 16 KB shared-memory image of one TMA-staged activation tile (uint8 [128, 128]); see include/btb200.h"""
    out = torch.empty((128, 128), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _check(load().bt_tma_probe(ctypes.byref(geom), _ptr(x), dtype_code(x, "input"), int(m0), int(sample), int(group),
                                   int(tap), int(slab), _ptr(out), _stream(x.device)))
    return out


def tma_probe4d(x, dims, box, coords, dst_off):
    """uint8 [256, 128] image of the probe's 32 KB shared-memory buffer; see include/btb200.h::bt_tma_probe4d"""
    out = torch.empty((256, 128), dtype=torch.uint8, device=x.device)
    d = (ctypes.c_int64 * 4)(*dims)
    b = (ctypes.c_int32 * 4)(*box)
    c = (ctypes.c_int32 * 4)(*coords)
    with torch.cuda.device(x.device):
        _check(load().bt_tma_probe4d(_ptr(x), dtype_code(x, "input"), d, b, c, ctypes.c_uint32(dst_off), _ptr(out), _stream(x.device)))
    return out


def set_pointer_checks(enabled):
    """thread-local switch of the cudaPointerGetAttributes argument checks (off while a CUDA graph is captured)"""
    return int(load().bt_set_pointer_checks(int(bool(enabled))))


PATH_NAMES = {-1: "none", 0: "generic", 1: "fast", 2: "fast_ws", 3: "ws", 4: "direct", 5: "tma", 6: "tma_stream", 7: "tma_direct"}


def sm_count():
    """SM count of the current CUDA device (what bt_layer_forward's kernel selection uses)"""
    return int(load().bt_sm_count())


def last_forward_path():
    """name of the kernel family this thread's most recent layer_forward took (diagnostics / tests)"""
    return PATH_NAMES[int(load().bt_last_forward_path())]


def rng_export(what, out, rows, cols, taps, cols_per_group, seed, layer_key, sample_idx):
    lib = load()
    dev = out.device
    with torch.cuda.device(dev):
        _check(lib.bt_rng_export(int(what), _ptr(out), int(rows), int(cols), int(taps), int(cols_per_group),
                                 ctypes.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), ctypes.c_uint32(layer_key),
                                 ctypes.c_uint32(sample_idx & 0xFFFFFFFF), _stream(dev)))
    return out


MC_WARP_MAX_CLASSES = 1024     # bt_mc_accumulate_ex holds a row in one warp's registers; wider rows take the large-C path


def mc_accumulate(logits, n_samples, batch, sums, accumulate, entropy_sum=None):
    """logits: contiguous [S * batch, C] (batch = rows per sample); sums fp32 [2, batch, C], entropy_sum fp32 [batch]"""
    lib = load()
    require_cuda(logits, "logits")
    dev = logits.device
    n_classes = int(logits.shape[-1])
    global launch_count
    if n_classes > MC_WARP_MAX_CLASSES:
        ws = torch.empty(2 * int(n_samples) * int(batch), dtype=torch.float32, device=dev)
        launch_count += 2
        with torch.cuda.device(dev):
            _check(lib.bt_mc_accumulate_large(_ptr(logits), dtype_code(logits, "logits"), int(n_samples), int(batch),
                                              n_classes, _ptr(sums), _ptr(entropy_sum), int(bool(accumulate)), _ptr(ws),
                                              _stream(dev)))
        return sums
    launch_count += 1
    with torch.cuda.device(dev):
        _check(lib.bt_mc_accumulate_ex(_ptr(logits), dtype_code(logits, "logits"), int(n_samples), int(batch),
                                       n_classes, _ptr(sums), _ptr(entropy_sum), int(bool(accumulate)),
                                       _stream(dev)))
    return sums


def mc_regression_accumulate(y, n_samples, sums, accumulate):
    """y: the S samples' outputs, each sample's block of n elements contiguous in memory (sample-major);
    sums: fp64 [2 * n]"""
    lib = load()
    require_cuda(y, "y")
    if sums.dtype != torch.float64 or sums.numel() * int(n_samples) != 2 * y.numel():
        raise ValueError("mc_regression_accumulate: sums must be float64 [2 * elements per sample]")
    dev = y.device
    global launch_count
    launch_count += 1
    with torch.cuda.device(dev):
        _check(lib.bt_mc_regression_accumulate(_ptr(y), dtype_code(y, "y"), int(n_samples), sums.numel() // 2,
                                               _ptr(sums), int(bool(accumulate)), _stream(dev)))
    return sums


def mc_regression_finalize(sums, n_total, mean, var):
    """fp64 sums [2 * n] -> fp32 mean [n], var [n] (or None), in the sums' element order"""
    lib = load()
    dev = sums.device
    global launch_count
    launch_count += 1
    with torch.cuda.device(dev):
        _check(lib.bt_mc_regression_finalize(_ptr(sums), sums.numel() // 2, int(n_total), _ptr(mean), _ptr(var),
                                             _stream(dev)))
    return mean, var


def mc_uncertainty(sums, entropy_sum, n_total, pred_entropy, mutual_info):
    lib = load()
    dev = sums.device
    global launch_count
    launch_count += 1
    with torch.cuda.device(dev):
        _check(lib.bt_mc_uncertainty(_ptr(sums), _ptr(entropy_sum), int(sums.shape[1]), int(sums.shape[2]), int(n_total),
                                     _ptr(pred_entropy), _ptr(mutual_info), _stream(dev)))
    return pred_entropy, mutual_info


def mc_finalize(sums, n_total, mean, var):
    lib = load()
    dev = sums.device
    global launch_count
    launch_count += 1
    with torch.cuda.device(dev):
        _check(lib.bt_mc_finalize(_ptr(sums), int(sums.shape[1]), int(sums.shape[2]), int(n_total),
                                  _ptr(mean), _ptr(var), _stream(dev)))
    return mean, var


def im2col2d(x, ks, stride, padding, dilation, kpad):
    """x: logical [N, C, H, W] CUDA tensor (any strides) -> [N * OH * OW, kpad] im2col rows (include/btb200.h)"""
    lib = load()
    require_cuda(x, "input")
    n, c, h, w = x.shape
    oh = (h + 2 * padding[0] - dilation[0] * (ks[0] - 1) - 1) // stride[0] + 1
    ow = (w + 2 * padding[1] - dilation[1] * (ks[1] - 1) - 1) // stride[1] + 1
    out = torch.empty((n * oh * ow, kpad), dtype=x.dtype, device=x.device)
    st = (ctypes.c_int64 * 4)(*x.stride())
    global launch_count
    launch_count += 1
    with torch.cuda.device(x.device):
        _check(lib.bt_im2col2d(_ptr(x), dtype_code(x, "input"), n, c, h, w, st, ks[0], ks[1], stride[0], stride[1],
                               padding[0], padding[1], dilation[0], dilation[1], int(kpad), _ptr(out), _stream(x.device)))
    return out


def lstm_cell(gates_i, gates_h, c_prev, h_out, c_out, h_seq, c_seq, t):
    """one LSTM time step's pointwise stage (include/btb200.h::bt_lstm_cell); all tensors contiguous, same dtype"""
    lib = load()
    require_cuda(gates_i, "gates")
    b, h4 = gates_i.shape
    global launch_count
    launch_count += 1
    with torch.cuda.device(gates_i.device):
        _check(lib.bt_lstm_cell(_ptr(gates_i), _ptr(gates_h), _ptr(c_prev), _ptr(h_out), _ptr(c_out), _ptr(h_seq), _ptr(c_seq),
                                dtype_code(gates_i, "gates"), int(b), int(h4 // 4), int(h_seq.shape[1]), int(t),
                                _stream(gates_i.device)))
    return h_out, c_out


def maxpool2d_nhwc(x_phys, kernel, stride, padding):
    """x_phys: dense [N, H, W, C] CUDA tensor -> [N, OH, OW, C]."""
    lib = load()
    require_cuda(x_phys, "input")
    n, h, w, c = x_phys.shape
    oh = (h + 2 * padding[0] - kernel[0]) // stride[0] + 1
    ow = (w + 2 * padding[1] - kernel[1]) // stride[1] + 1
    out = torch.empty((n, oh, ow, c), dtype=x_phys.dtype, device=x_phys.device)
    global launch_count
    launch_count += 1
    with torch.cuda.device(x_phys.device):
        _check(lib.bt_maxpool2d_nhwc(_ptr(x_phys), dtype_code(x_phys, "input"), n, h, w, c, kernel[0], kernel[1],
                                     stride[0], stride[1], padding[0], padding[1], _ptr(out), _stream(x_phys.device)))
    return out
