"""Monte-Carlo inference driver: N weight samples per input batch, sharded over GPUs.

Replaces the sequential loop of the reference's evaluate()
(/root/reference/bayesian_torch/examples/main_bayesian_cifar_dnn2bnn.py:541-557:
`for mc_run in range(num_monte_carlo): model.forward(data)` -> stack -> softmax -> mean):

  * the MC-sample index is a GRID DIMENSION of every fused layer kernel: a chunk of S samples is
    evaluated in one pass through the model with the samples stacked along the batch dimension
    (eval-mode BatchNorm / ReLU / pooling are per-image, so stacking is exact);
  * softmax + running sums of p and p^2 are one kernel (csrc/bt_mc.cu), no per-sample D2H copy;
  * multi-GPU: one process per GPU, rank r evaluates a contiguous block of the N global sample
    indices (Philox counters use the GLOBAL index, so the result does not depend on the number of
    ranks up to fp32 summation order) and ONE all-reduce of the moment buffer crosses NVLink
    (fp32 [2, B, C] for a classifier, [2, B*pixels, C] for a dense head, fp64 [2, n] for a regressor).
    Nothing else is communicated.
"""
import torch
import torch.distributed as dist

from . import _native
from ._core import BayesLayerBase, mc_sample_context


def shard_samples(n_samples, world_size, rank):
    """Contiguous block [start, start+count) of the global MC sample indices owned by `rank`."""
    if n_samples < 1 or world_size < 1 or not (0 <= rank < world_size):
        raise ValueError(f"bad sharding request n={n_samples} world={world_size} rank={rank}")
    base, rem = divmod(n_samples, world_size)
    count = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, count


def all_reduce_moments(sums, group=None):
    """The ONE collective of the path: sum the flat moment buffer over ranks -- fp32 [2, R, C] (+ [R] per-sample
    entropy sums when uncertainties are requested) for classification, fp64 [2, n] for regression."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    return sums


TASKS = ("classification", "regression")


def _layout(out, task):
    """The physical order of `out`'s dims (outermost first) when the kernels can read it in place, else None.
    In place means: dim 0 outermost and the whole tensor dense, so each MC sample's block is contiguous; for
    classification the class axis (dim 1) innermost as well, so every pixel's C logits are one contiguous row.  A
    channels-last Bayesian conv / ConvTranspose head ([S*B, C, *sp], physically [S*B, *sp, C]) and any contiguous
    [S*B, C] or regression output qualify."""
    cls = 1 if task == "classification" else None
    rest = sorted((d for d in range(1, out.dim()) if d != cls), key=lambda d: -out.stride(d))
    perm = [0] + rest + ([cls] if cls is not None else [])
    return perm if out.permute(perm).is_contiguous() else None


class _Moments:
    """One flat buffer of running sums (what the single all-reduce carries) and the output geometry to read the
    result back in the model output's layout.
      classification: fp32 [2, R, C] sums of p and p^2, + [R] per-sample entropy sums when uncertainties are asked for,
                      R = B * prod(spatial) rows of C class-contiguous logits (R = B for a [S*B, C] head);
      regression:     fp64 [2, n] sums of y and y^2, n = B * prod(rest) elements in the output's memory order."""

    def __init__(self, task, out, batch, with_entropy, device, zero):
        self.task = task
        self.shape = (batch,) + tuple(out.shape[1:])
        self.perm = _layout(out, task) or self._canonical(out.dim())
        if task == "classification":
            self.n_classes = out.shape[1]
            self.rows = out[:batch].numel() // self.n_classes
            self.buf, self.sums, self.ent = _moment_buffer(self.rows, self.n_classes, device, with_entropy, zero)
        else:
            make = torch.zeros if zero else torch.empty
            self.buf = self.sums = make(2 * out[:batch].numel(), dtype=torch.float64, device=device)
            self.ent = None

    def _canonical(self, ndim):
        """the layout a copy produces when the output cannot be read in place: class-innermost / contiguous"""
        if self.task == "classification":
            return [0] + list(range(2, ndim)) + [1]
        return list(range(ndim))

    def accumulate(self, out, s, accumulate):
        if tuple(out.shape[1:]) != self.shape[1:]:
            raise RuntimeError(f"mc_predict: the model output changed shape between chunks: {tuple(out.shape)}")
        phys = out.permute(self.perm)
        if _layout(out, self.task) != self.perm:
            phys = phys.contiguous()      # ONE copy into a layout the kernels read (e.g. an NCHW deterministic head)
            _native.launch_count += 1
        if self.task == "classification":
            _native.mc_accumulate(phys.view(s * self.rows, self.n_classes), s, self.rows, self.sums,
                                  accumulate=accumulate, entropy_sum=self.ent)
        else:
            _native.mc_regression_accumulate(phys, s, self.sums, accumulate=accumulate)

    def _empty(self, keep, device):
        """fp32 tensor of the dims `keep` of the output geometry, stored in the output's physical order"""
        order = [d for d in self.perm if d in keep]
        phys = torch.empty([self.shape[d] for d in order], dtype=torch.float32, device=device)
        return phys, phys.permute([order.index(d) for d in keep])

    def finalize(self, n_samples, return_var, return_uncertainty, device):
        every = list(range(len(self.shape)))
        phys_mean, mean = self._empty(every, device)
        phys_var, var = self._empty(every, device) if return_var else (None, None)
        if self.task == "regression":
            _native.mc_regression_finalize(self.sums, n_samples, phys_mean, phys_var)
            return mean, var
        _native.mc_finalize(self.sums, n_samples, phys_mean, phys_var)
        if not return_uncertainty:
            return mean, var
        phys_pe, pred_entropy = self._empty([d for d in every if d != 1], device)
        phys_mi, mutual_info = self._empty([d for d in every if d != 1], device)
        _native.mc_uncertainty(self.sums, self.ent, n_samples, phys_pe, phys_mi)
        return mean, var, pred_entropy, mutual_info


def _forward_moments(model, x, start, count, chunk, sample_offset, with_entropy, task, sample_word=None):
    """This rank's share of the work: `count` samples from global index sample_offset + start, `chunk` per pass ->
    the _Moments of those samples.  With `sample_word` (int32 CUDA tensor [1]) the offset is NOT baked into the
    launches: the kernels add *sample_word at run time (CUDA-graph replays with fresh draws)."""
    batch = x.shape[0]
    mom = None
    done = 0
    base = start if sample_word is not None else sample_offset + start
    while done < count:
        s = min(chunk, count - done)
        with mc_sample_context(s, batch, base + done, sample_word, sample_offset if sample_word is not None else 0):
            out = model(x)
        _check_output(out, s, batch, task)
        if mom is None:
            mom = _Moments(task, out, batch, with_entropy, x.device, zero=False)
        mom.accumulate(out, s, accumulate=done > 0)
        done += s
    if mom is None:  # a rank with no samples (n_samples < world): contributes zeros of the output's geometry
        with mc_sample_context(1, batch, 0):
            out = model(x)
        _check_output(out, 1, batch, task)
        mom = _Moments(task, out, batch, with_entropy, x.device, zero=True)
    return mom


def _check_output(out, s, batch, task):
    if out.dim() < 1 or out.shape[0] != s * batch or out.numel() == 0:
        raise RuntimeError(f"mc_predict expects the model output [S*B, ...] with the S samples stacked along dim 0; got "
                           f"{tuple(out.shape)} for S={s}, B={batch} (is the first layer of the model a "
                           "bayesian_torch_b200 layer?)")
    if task == "classification" and out.dim() < 2:
        raise RuntimeError(f"mc_predict(task='classification') expects logits [S*B, C, *spatial] with the class axis at "
                           f"dim 1; got {tuple(out.shape)}")


class _MCGraph:
    """The whole per-rank MC pass (every layer launch, pooling, softmax/moments) captured ONCE as a CUDA graph and
    replayed per input batch: ~70 kernel launches through python + ctypes cost ~1.8 ms of host time per step, which
    is as long as the GPU needs at N = 1 and 2-3x longer than a rank needs at N = 4-8 GPUs (tools/small_s_check.py).
    The Philox seed and the rank's sample range are baked in, like the tensor shapes; the SAMPLE OFFSET is not: every
    layer kernel adds a device word (BtLayerGeom.sample_offset) that run() rewrites before the replay, so each replay
    can draw fresh eps -- the reference draws new eps on every forward (conv_variational.py:362).  The collective and the
    finalize stay outside the graph."""

    def __init__(self, model, x, start, count, chunk, sample_offset, with_entropy, task):
        self.static_x = x.clone()
        self.sample_word = torch.full((1,), int(sample_offset) & 0x7FFFFFFF, dtype=torch.int32, device=x.device)
        self.param_versions = _param_versions(model)
        args = (model, self.static_x, start, count, chunk, int(sample_offset) & 0x7FFFFFFF, with_entropy, task,
                self.sample_word)
        side = torch.cuda.Stream(device=x.device)           # warm-up off the capture stream (fills every host cache)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(side):
            _forward_moments(*args)
        torch.cuda.current_stream(x.device).wait_stream(side)
        l0 = _native.launch_count
        self.graph = torch.cuda.CUDAGraph()
        prev = _native.set_pointer_checks(False)             # (pointer-attribute queries are illegal during capture;
        try:                                                 #  the identical arguments were just checked eagerly)
            # thread-local capture mode: only THIS thread is held to the capture rules, so the NCCL watchdog thread
            # of a multi-GPU job may keep polling its events while the pass is being captured
            with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
                self.moments = _forward_moments(*args)
        finally:
            _native.set_pointer_checks(prev)
        self.n_launches = _native.launch_count - l0          # libbtb200 kernels per replay
        # python does not run at replay time: keep the layers' "last draw" bookkeeping (materialize_eps) in step with
        # the offset each replay uses
        self.capture_offset = int(sample_offset) & 0x7FFFFFFF
        self.layers = [m for m in model.modules() if isinstance(m, BayesLayerBase) and m._bt_last is not None]
        self.layer_base = [(m._bt_last["sample0"] - self.capture_offset) & 0xFFFFFFFF for m in self.layers]

    def run(self, x, sample_offset):
        if x.data_ptr() != self.static_x.data_ptr():
            self.static_x.copy_(x)
        self.sample_word.fill_(int(sample_offset) & 0x7FFFFFFF)
        self.graph.replay()
        for m, base in zip(self.layers, self.layer_base):
            m._bt_last["sample0"] = (base + (int(sample_offset) & 0x7FFFFFFF)) & 0xFFFFFFFF
        _native.launch_count += self.n_launches
        return self.moments


_graphs = {}


def _param_versions(model):
    return [p._version for p in model.parameters()]


def _graph_key(model, x, start, count, chunk, with_entropy, task):
    from ._core import current_seed
    return (id(model), tuple(x.shape), tuple(x.stride()), x.dtype, x.device, start, count, chunk, with_entropy,
            current_seed(), task)


def drop_graphs(model=None):
    """forget the captured CUDA graphs (of `model`, or all): they bake parameter pointers and cached transforms in"""
    for k in list(_graphs):
        if model is None or k[0] == id(model):
            _graphs.pop(k)


@torch.no_grad()
def mc_predict(model, x, n_samples, chunk=None, group=None, sample_offset=0, return_var=True,
               return_uncertainty=False, use_graph=False, fresh=False, task="classification"):
    """Predictive mean (and variance) of softmax(model(x)) -- or of model(x) itself -- over `n_samples` weight samples.

    x: [B, ...] CUDA tensor; the model returns its S samples stacked along dim 0: [S*B, ...].  Results are fp32 and
    identical on all ranks.
    task="classification" (default): logits [S*B, C] -> (mean [B, C], var [B, C] or None), or a dense head
    [S*B, C, *spatial] (segmentation; class axis at dim 1) -> mean / var [B, C, *spatial], per pixel.  Any number of
    classes.  The kernels read logits whose classes are contiguous per pixel in place (a channels-last Bayesian conv or
    ConvTranspose head is); any other layout (e.g. an NCHW-contiguous deterministic head) costs one copy per chunk.
    task="regression": output [S*B, *rest] -> (mean [B, *rest], var [B, *rest] or None): moments of the raw output,
    accumulated in fp64 (a large mean with a small spread keeps its variance), returned with the output's strides.
    chunk: samples evaluated per pass (default: all samples of this rank in one pass).
    return_uncertainty: also return (predictive_entropy [B], mutual_information [B]) of the MC ensemble -- the
    reference's utils/util.py:45-60 on the stacked per-sample probabilities -- computed on device from running sums
    that ride the same single all-reduce (SURVEY.md 8f rank 3); result = (mean, var, pred_entropy, mutual_info), the
    last two [B] (dense head: [B, *spatial], per pixel).  Classification only.
    use_graph: capture this rank's pass as a CUDA graph on first use (per model / shape / seed / sample range /
    parameter version) and replay it afterwards; the results are the same tensors' worth of numbers, the host cost per
    call drops from ~1.8 ms to a replay.  `sample_offset` is NOT part of the graph: it is written to a device word the
    kernels read, so replays with different offsets draw different eps and each equals the eager run with that offset.
    fresh: draw NEW weight samples on every call, like the reference's evaluate() (every forward draws new eps,
    conv_variational.py:362): the call uses sample_offset + (number of samples this model has drawn so far) and
    advances that counter by n_samples (identically on every rank).
    """
    if task not in TASKS:
        raise ValueError(f"mc_predict: unknown task {task!r}; expected one of {TASKS}")
    if return_uncertainty and task != "classification":
        raise ValueError("mc_predict: predictive entropy and mutual information are classification quantities; "
                         "task='regression' returns (mean, var)")
    if model.training:
        raise RuntimeError("mc_predict stacks MC samples along the batch dimension; call model.eval() first "
                           "(train-mode BatchNorm would mix statistics across samples)")
    _native.require_cuda(x, "input")
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    rank = dist.get_rank(group) if world > 1 else 0
    start, count = shard_samples(n_samples, world, rank)
    if chunk is None or chunk > count:
        chunk = max(count, 1)
    if fresh:
        drawn = getattr(model, "_bt_mc_drawn", 0)
        sample_offset = (sample_offset + drawn) & 0x7FFFFFFF
        model._bt_mc_drawn = drawn + n_samples
    if getattr(model, "_bt_fused_inference", False):
        from .fuse import refresh_epilogues
        refresh_epilogues(model)              # folded BatchNorm statistics changed (load_state_dict)? re-fold
    if use_graph:
        key = _graph_key(model, x, start, count, chunk, return_uncertainty, task)
        g = _graphs.get(key)
        if g is not None and g is not False and g.param_versions != _param_versions(model):
            g = None                                         # a parameter was updated in place: re-capture
        if g is None:
            if len(_graphs) >= 8:                            # bounded: graphs pin their activation pools
                _graphs.pop(next(iter(_graphs)))
            try:
                g = _MCGraph(model, x, start, count, chunk, sample_offset, return_uncertainty, task)
            except RuntimeError as e:                        # capture refused (e.g. an op that synchronises): stay eager
                import warnings
                warnings.warn(f"mc_predict: CUDA-graph capture failed, running eagerly ({e})", RuntimeWarning)
                g = False
            _graphs[key] = g
        if g is False:
            mom = _forward_moments(model, x, start, count, chunk, sample_offset, return_uncertainty, task)
        else:
            mom = g.run(x, sample_offset)
    else:
        mom = _forward_moments(model, x, start, count, chunk, sample_offset, return_uncertainty, task)
    all_reduce_moments(mom.buf, group)
    return mom.finalize(n_samples, return_var, return_uncertainty, x.device)


def _moment_buffer(batch, n_classes, device, with_entropy, zero):
    """One flat fp32 tensor: [2, B, C] sums of p and p^2, then (optionally) [B] sums of the per-sample entropies
    (B = rows: batch x pixels for a dense head)."""
    n = 2 * batch * n_classes
    make = torch.zeros if zero else torch.empty
    buf = make(n + (batch if with_entropy else 0), dtype=torch.float32, device=device)
    return buf, buf[:n].view(2, batch, n_classes), (buf[n:] if with_entropy else None)


def count_bayes_layers(model):
    return sum(1 for m in model.modules() if isinstance(m, BayesLayerBase))
