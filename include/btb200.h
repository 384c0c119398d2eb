/*
 * btb200.h -- C ABI of libbtb200.so: the B200 (sm_100a) implementation of the
 * bayesian-torch stochastic variational layer forward path and its Gaussian KL.
 *
 * The reference (IntelLabs/bayesian-torch, /root/reference) is pure Python on
 * PyTorch, so it has no FFI of its own; each entry point below names the
 * reference Python function whose arithmetic it replaces.  A maintainer binds
 * them with ctypes from the layer classes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no torch / CUDA-runtime types
 *     (a stream is passed as the raw cudaStream_t handle cast to void*).
 *   - Every pointer is a DEVICE pointer on the current device unless stated.
 *     The library never allocates or frees caller-visible memory, never
 *     synchronises, never calls cudaSetDevice; work is enqueued on `stream`.
 *   - Return value: 0 = BT_OK, negative = error; bt_last_error() gives the
 *     thread-local message.  There is NO CPU fallback: host pointers or a
 *     non-sm_100 device are errors.
 *   - Random numbers: counter-based Philox4x32-10 generated on chip; a launch
 *     is fully determined by (seed, layer_key, sample index) -- see
 *     oracle/philox_ref.py for the exact counter layout.
 */
#ifndef BTB200_H_
#define BTB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BT_VERSION 210 /* 0.2.1 */

/* status codes */
#define BT_OK 0
#define BT_ERR_BAD_SHAPE (-1)
#define BT_ERR_BAD_DTYPE (-2)
#define BT_ERR_UNSUPPORTED (-3)
#define BT_ERR_CUDA (-4)
#define BT_ERR_BAD_POINTER (-5)

/* element types */
#define BT_F32 0
#define BT_BF16 1

/* layer kind */
#define BT_MODE_REPARAM 0 /* *Reparameterization classes */
#define BT_MODE_FLIPOUT 1 /* *Flipout classes */

int bt_version(void);
const char* bt_last_error(void);
/* 0 if the current device is sm_100 (B200), else BT_ERR_UNSUPPORTED. */
int bt_device_check(void);
/*
 * Every entry point verifies with cudaPointerGetAttributes that its pointers are device pointers (there is no CPU
 * path).  That query is not allowed while the calling thread captures a CUDA graph in global capture mode; a caller
 * that captures launches it has already issued once eagerly (same arguments) turns the check off around the capture.
 * Thread-local; returns the previous setting.  NULL checks stay on.
 */
int bt_set_pointer_checks(int enabled);
/* number of SMs of the current device (148 on B200); negative on error. */
int bt_sm_count(void);

/*
 * bt_kl_gaussian -- mean-KL of a weight tensor plus mean-KL of an optional bias.
 * Replaces BaseVariationalLayer_.kl_div (layers/base_variational_layer.py:53-68)
 * as called by every layer's kl_loss() (e.g. layers/variational_layers/
 * linear_variational.py:144-155), including the softplus sigma = log1p(exp(rho)):
 *     out = mean_i KL(N(mu_i, sp(rho_i)) || N(pmu_i, psig_i)) [+ same over the bias]
 * prior_mu / prior_sigma: device tensors of the parameter's shape and dtype, or
 * NULL to use the scalars prior_mu_s / prior_sigma_s (the dnn_to_bnn case,
 * models/dnn_to_bnn.py:58-59).  n_b == 0 -> no bias term.
 * workspace: >= bt_kl_workspace_bytes() bytes, zero-initialised ONCE by the caller
 * (the kernel leaves it zeroed); deterministic two-stage reduction, fp32 accumulate.
 * One kernel launch.
 */
int64_t bt_kl_workspace_bytes(void);
int bt_kl_gaussian(const void* mu_w, const void* rho_w, int64_t n_w,
                   const void* prior_mu_w, const void* prior_sigma_w,
                   const void* mu_b, const void* rho_b, int64_t n_b,
                   const void* prior_mu_b, const void* prior_sigma_b,
                   float prior_mu_s, float prior_sigma_s, int dtype,
                   float* kl_out, int accumulate, void* workspace, void* stream);

/* Debug / parity hooks of the fused forward (all nullable, all DEVICE pointers). */
typedef struct BtDebugIO {
  const float* eps_w_in;   /* [Cout, K] in PHYSICAL (row, tap, channel) order: use instead of Philox  */
  const float* eps_b_in;   /* [Cout]                                                                  */
  const float* sign_in;    /* flipout: +-1 per element of x, same physical layout as x, fp32          */
  const float* sign_out;   /* flipout: +-1 per element of out, same physical layout as out, fp32      */
} BtDebugIO;

/*
 * Optional fused epilogue (NULL = none): what torchvision's BasicBlock / Bottleneck apply right after the
 * convolution in eval mode -- BatchNorm folded to a per-channel affine, the residual add and the ReLU
 * (SURVEY.md 8f rank 1).  Applied in this order:  y = relu( (conv + bias) * scale + shift + residual ).
 */
typedef struct BtEpilogue {
  const float* scale;    /* fp32 [C_out] or NULL */
  const float* shift;    /* fp32 [C_out] or NULL (both or neither) */
  const void* residual;  /* same physical layout and dtype as `out`, or NULL */
  int32_t relu;
} BtEpilogue;

/*
 * Geometry of one Bayesian layer forward seen as an (implicit) GEMM.
 * Linear layers are the degenerate conv with all spatial extents 1.
 * Activations are channels-last:  x   [S * B, ID, IH, IW, C_in ]
 *                                 out [S * B, OD, OH, OW, C_out]
 * weights are channels-last too:  mu/rho [C_out, KD, KH, KW, C_in / groups].
 */
typedef struct BtLayerGeom {
  int32_t n_samples;   /* S: MC weight samples evaluated by this launch (sample s uses rows [s*B, (s+1)*B)) */
  int32_t x_shared;    /* 1: x holds ONE sample's batch [B,...] that every sample reads (first layer)   */
  int32_t batch;       /* B */
  int32_t c_in, c_out, groups;
  int32_t in_dhw[3], out_dhw[3], k_dhw[3], stride[3], pad[3], dil[3];
  int32_t rho_is_sigma; /* 1: the `rho_w` argument already holds sigma = softplus(rho) (same dtype / layout): a caller
                           that evaluates many weight samples of FROZEN parameters (MC inference) computes it once
                           instead of once per sample and element.  Not allowed together with kl_out.  The bias
                           arguments always hold rho. */
  int32_t transposed;   /* 1: ConvTranspose{1,2,3}d (conv_variational.py:577-1094, conv_flipout.py:640-1228):
                           out[o] += x[i] * W[., k] for o = i*stride - pad + k*dil; out_dhw carries the output extent
                           (incl. output_padding).  The weight argument is the kernel-layout matrix
                           [C_out, KD, KH, KW, C_in / groups] (the caller repacks the reference's [C_in, C_out/g, k...]). */
  int32_t pool_hw[2];   /* {OH, OW} != {0, 0}: the output rows of one image are OH x OW pixels and torchvision's stem
                           max-pool (nn.MaxPool2d(3, stride=2, padding=1), resnet.py `self.maxpool`) is applied to the
                           epilogue's result inside the kernel: `out` is [S * n_img, OH/2, OW/2, C_out].  Only kernels
                           that keep whole output rows in one tile can do it (OW | 128, OH * OW a multiple of 128, no
                           residual): ask bt_layer_forward_plan (BtForwardPlan.pool_fused) first.               */
  const uint32_t* sample_offset; /* nullable DEVICE word: the launch uses global sample index sample_idx0 + *sample_offset
                           + s.  Read at run time, so a captured CUDA graph draws fresh eps on every replay when the
                           caller bumps the word between replays (the reference draws new eps on every forward,
                           conv_variational.py:362). */
} BtLayerGeom;

/*
 * bt_layer_forward -- ONE fused kernel per Bayesian layer forward.
 * Replaces LinearReparameterization.forward (linear_variational.py:157-201),
 * Conv{1,2,3}dReparameterization.forward (conv_variational.py:183-227/357-402/530-574),
 * LinearFlipout.forward (linear_flipout.py:145-197) and
 * Conv{1,2,3}dFlipout.forward (conv_flipout.py:175-244/370-439/568-637):
 *   reparam:  out = conv(x, mu + sp(rho) * eps) + (mu_b + sp(rho_b) * eps_b)
 *   flipout:  out = conv(x, mu) + mu_b + (conv(x * s_in, sp(rho) * eps) + sp(rho_b) * eps_b) * s_out
 * eps ~ N(0,1) and the +-1 signs are generated on chip (Philox), W is never
 * written to memory; the product runs on tcgen05 tensor cores with fp32 accumulation
 * in TMEM: kind::tf32 operands when parameters AND activations are fp32 (the reference's
 * default dtype), bf16 operands (kind::f16) otherwise.
 *   x_dtype / out dtype : BT_F32 or BT_BF16 (out has x's dtype)
 *   p_dtype             : dtype of mu/rho (weights and bias)
 *   kl_out (nullable)   : if non-NULL also writes mean-KL(weight)+mean-KL(bias) with
 *                         SCALAR priors (forward(return_kl=True)); needs `workspace`.
 *   seed, layer_key, sample_idx0 : Philox key/counter; sample s of the launch uses
 *                         global sample index sample_idx0 + s.
 *   max_ctas_hint       : 0 = automatic tiling.
 */
int64_t bt_forward_workspace_bytes(void);
int bt_layer_forward(int mode, const BtLayerGeom* geom,
                     const void* x, int x_dtype,
                     const void* mu_w, const void* rho_w,
                     const void* mu_b, const void* rho_b, int p_dtype,
                     void* out,
                     float* kl_out, float prior_mu_s, float prior_sigma_s,
                     uint64_t seed, uint32_t layer_key, uint32_t sample_idx0,
                     const BtDebugIO* dbg, const BtEpilogue* epi, void* workspace, void* stream);

/*
 * bt_layer_forward_plan -- the tiling / kernel-selection decision bt_layer_forward would take for this geometry on a
 * device with `sm_count` SMs, WITHOUT touching a device (pure host arithmetic; pointers are assumed 16-byte aligned).
 * Lets the host logic be tested where there is no GPU (tests/test_host_api.py) and lets a caller size its launches.
 */
typedef struct BtForwardPlan {
  int32_t path;          /* BT_PATH_* below                                                              */
  int32_t block_n;       /* output columns per CTA (UMMA N)                                              */
  int32_t m_subtiles;    /* 128-row M-subtiles that share one sampled weight tile (1 for WS / direct)     */
  int32_t k_blocks;      /* 64-wide k-blocks iterated, after dropping filter taps that only see padding   */
  int32_t grid[3];       /* x = M-groups / row-tile stride, y = N tiles (x groups), z = MC samples        */
  int32_t threads;       /* threads per CTA                                                              */
  int32_t smem_bytes;    /* dynamic shared memory per CTA                                                */
  int32_t tmem_cols;     /* TMEM columns allocated per CTA                                               */
  int32_t window_slots;  /* direct kernel: input-window ring depth                                       */
  int32_t window_rows;   /* direct kernel: rows (padded pixels) per window                               */
  int32_t staged_epilogue; /* direct kernel: 1 = epilogue goes through its shared-memory staging buffer   */
  int32_t samples_per_cta; /* TMA resident kernel: MC samples whose W_s one CTA keeps (shared x); else 0 / 1 */
  int32_t window_boxes;  /* TMA direct kernel: TMA boxes per window and 128-byte channel slab (1 when the tiles are whole
                            padded images: no halo boxes)                                                          */
  int32_t cluster_n;     /* TMA streaming kernel: thread-block cluster size along the n-tiles (2 = the two CTAs read the same
                            activation tiles, each loads half and multicasts); else 1                              */
  int32_t pool_fused;    /* 1 = BtLayerGeom.pool_hw is honoured (max-pool inside the epilogue); 0 = the caller must
                            clear pool_hw and pool separately (bt_layer_forward refuses otherwise)                 */
} BtForwardPlan;
int bt_layer_forward_plan(int mode, const BtLayerGeom* geom, int x_dtype, int p_dtype, int with_kl,
                          int with_debug_hooks, int with_residual, int sm_count, BtForwardPlan* plan);

/*
 * Which kernel the calling thread's most recent bt_layer_forward took (diagnostics / tests; -1 = none yet).
 * All of them compute the same function; they differ in how the operands reach the tensor core.
 */
#define BT_PATH_GENERIC 0  /* bt_fused_kernel, generic instantiation (debug hooks, KL side output, scalar gathers) */
#define BT_PATH_FAST 1     /* bt_fused_kernel, branch-free sampler                                                 */
#define BT_PATH_FAST_WS 2  /* bt_fused_kernel, weight-stationary schedule                                          */
#define BT_PATH_WS 3       /* bt_ws_kernel: persistent weight-stationary, cp.async im2col / tap-copy               */
#define BT_PATH_DIRECT 4   /* bt_direct_kernel: A operand read in place from a shared-memory input window          */
#define BT_PATH_TMA 5      /* bt_tma_kernel: A operand staged by TMA (tiled / im2col tensor maps), W_s resident    */
#define BT_PATH_TMA_STREAM 6 /* bt_tms_kernel: A by TMA, one sampled weight tile per k-block shared by 1-4 row tiles */
#define BT_PATH_TMA_DIRECT 7 /* bt_dtma_kernel: A read in place from an input window staged by tiled TMA boxes      */
int bt_last_forward_path(void);

/*
 * bt_tma_probe -- test hook of the TMA operand path (bt_tma_kernel): loads ONE activation tile -- 128 consecutive
 * output rows starting at row m0 of MC sample `sample`, channel group `group`, filter tap number `tap` (in kd, kh, kw
 * order) and k-block `slab` inside the tap -- through exactly the tensor map (cuTensorMapEncodeTiled / Im2col) and
 * cp.async.bulk.tensor instruction the kernel uses, and copies the 16 KB shared-memory image (128 rows x 128 bytes,
 * 16-byte chunk c of row r at r*128 + ((c ^ (r & 7)) << 4)) to `out`.  tests/test_gpu_tma.py compares it with the
 * im2col rows of the oracle.  x_dtype BT_BF16: 64 channels per row; BT_F32: 32.
 */
int bt_tma_probe(const BtLayerGeom* geom, const void* x, int x_dtype, int64_t m0, int sample, int group, int tap,
                 int slab, void* out, void* stream);

/*
 * bt_tma_probe4d -- test hook: one TILED 4-D TMA load (tensor dims {C, W, H, N} of a dense channels-last tensor, box
 * {C_box, W_box, H_box, 1} with C_box * sizeof = 128 bytes, 128B swizzle) at `coords` into a 1024-aligned 32 KB
 * shared-memory buffer (pre-filled with 0xA5) at byte offset dst_off (multiple of 128); the whole buffer is copied to
 * `out`.  Pins the out-of-range zero fill and the address-based swizzle of a destination that is not 1024-aligned.
 */
int bt_tma_probe4d(const void* x, int x_dtype, const int64_t* dims, const int32_t* box, const int32_t* coords,
                   uint32_t dst_off, void* out, void* stream);

/*
 * bt_rng_export -- regenerate, into global memory, exactly the random draws a
 * bt_layer_forward launch with the same (seed, layer_key, sample index) uses.
 * This is how the reference's `eps_weight / eps_kernel / eps_bias` buffers
 * (linear_variational.py:161,173) are materialised on demand.
 *   what = 0: weight eps -> fp32 [rows, taps*cpt] written in the REFERENCE's logical
 *             (Cout, Cin/g, k...) order (cpt = channels per tap, taps = prod(k))
 *   what = 1: bias eps   -> fp32 [rows]
 *   what = 2/3: input / output signs -> fp32 +-1, [rows, cols] (row = pixel resp. output row
 *             inside the sample, col = channel; for output signs of grouped convs
 *             cols_per_group = C_out / groups, else pass cols_per_group = cols)
 */
int bt_rng_export(int what, float* out, int64_t rows, int64_t cols, int32_t taps,
                  int32_t cols_per_group, uint64_t seed, uint32_t layer_key,
                  uint32_t sample_idx, void* stream);

/*
 * bt_mc_accumulate -- Monte-Carlo aggregation.  Replaces torch.stack + softmax + mean of
 * examples/main_bayesian_cifar_dnn2bnn.py:545-557 (and the per-sample D2H copy of
 * examples/main_bayesian_imagenet.py:617-624): logits [S*B, C] (sample-major) ->
 *   sums[0, b, c] (+)= sum_s softmax(logits[s,b,:])[c]
 *   sums[1, b, c] (+)= sum_s softmax(...)[c]^2
 * sums is fp32 [2, B, C]; it is what the single all-reduce over GPUs carries.
 */
int bt_mc_accumulate(const void* logits, int dtype, int32_t n_samples, int32_t batch,
                     int32_t n_classes, float* sums, int accumulate, void* stream);

/*
 * bt_mc_accumulate_ex -- as bt_mc_accumulate, and (entropy_sum != NULL, fp32 [B]) also
 *   entropy_sum[b] (+)= sum_s -sum_c p_s[b,c] log(p_s[b,c] + 1e-15)
 * i.e. utils/util.py:41-42 `entropy` of every MC member, the second term of mutual_information
 * (utils/util.py:54-60).  Laid out right behind `sums` it rides the same single all-reduce.
 */
int bt_mc_accumulate_ex(const void* logits, int dtype, int32_t n_samples, int32_t batch,
                        int32_t n_classes, float* sums, float* entropy_sum, int accumulate, void* stream);

/*
 * bt_mc_uncertainty -- predictive_entropy (utils/util.py:45-50) and mutual_information (utils/util.py:53-60)
 * of the MC ensemble from the (all-reduced) buffers, replacing the host/numpy post-processing of
 * examples/main_bayesian_imagenet.py:617-624:
 *   pred_entropy[b] = H(mean_s p_s[b,:]),   mutual_info[b] = pred_entropy[b] - mean_s H(p_s[b,:])
 * mutual_info may be NULL (then entropy_sum may be NULL too).
 */
int bt_mc_uncertainty(const float* sums, const float* entropy_sum, int32_t batch, int32_t n_classes,
                      int32_t n_total, float* pred_entropy, float* mutual_info, void* stream);

/* sums [2,B,C] + total sample count -> mean [B,C], var [B,C] (predictive mean / variance). */
int bt_mc_finalize(const float* sums, int32_t batch, int32_t n_classes, int32_t n_total,
                   float* mean, float* var, void* stream);

/*
 * bt_mc_accumulate_large -- bt_mc_accumulate_ex for any number of classes (bt_mc_accumulate_ex takes C <= 1024):
 * logits [S * rows, C] (sample-major, each row of C classes contiguous) -> the same sums [2, rows, C] and optional
 * entropy_sum [rows].  A dense head [S*B, C, *spatial] stored class-innermost is this with rows = B * prod(spatial).
 * Two launches, each reading every logit once: the per-(sample, row) log-sum-exp and entropy, then the class sums.
 * With `accumulate` the stored sums are the starting value and this call's samples are added to them in order.
 * workspace: fp32, >= 2 * S * rows elements (S * rows without entropy_sum).  Deterministic (no atomics).
 */
int bt_mc_accumulate_large(const void* logits, int dtype, int32_t n_samples, int32_t rows, int32_t n_classes,
                           float* sums, float* entropy_sum, int accumulate, float* workspace, void* stream);

/*
 * bt_mc_regression_accumulate -- Monte-Carlo moments of a regression output, elementwise:
 *   sums[0, i] (+)= sum_s y[s * n + i],   sums[1, i] (+)= sum_s y[s * n + i]^2      (i < n_elem)
 * y: the S samples' outputs, sample s occupying elements [s*n, (s+1)*n) in memory order (fp32 or bf16); sums fp64 [2, n].
 * fp64 keeps the variance of outputs with a large mean and a small spread (fp32 sum y^2 / N - mean^2 cancels).
 * Samples are added in order; the result has y's memory order, so a caller gets the output's strides for free.
 */
int bt_mc_regression_accumulate(const void* y, int dtype, int32_t n_samples, int64_t n_elem, double* sums,
                                int accumulate, void* stream);

/* fp64 sums [2, n] + total sample count -> fp32 mean [n], var [n] (var >= 0; var may be NULL). */
int bt_mc_regression_finalize(const double* sums, int64_t n_elem, int32_t n_total, float* mean, float* var,
                              void* stream);

/*
 * bt_maxpool2d_nhwc -- channels-last 2-D max pooling (floor mode, dilation 1) of x [n_img, H, W, C] into
 * out [n_img, OH, OW, C]; C % 8 == 0 (bf16) / C % 4 == 0 (fp32).  Replaces the nn.MaxPool2d that follows
 * the first Bayesian conv of a torchvision ResNet when the model was prepared with fuse_inference()
 * (SURVEY.md 8f rank 1); ATen's NHWC max-pool is far from HBM-bound on the MC-stacked batch.
 */
int bt_maxpool2d_nhwc(const void* x, int dtype, int64_t n_img, int32_t H, int32_t W, int32_t C,
                      int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t ph, int32_t pw,
                      void* out, void* stream);

/*
 * bt_im2col2d -- materialised im2col of a few-channel 2-D convolution input (the RGB stem): x [N, C, H, W] with element
 * strides `strides_nchw` -> out [N * OH * OW, kpad] (row-major), column k = (kh, kw, c), zero for k >= KH*KW*C.
 * The Bayesian conv then runs as a linear layer over these rows (weights repacked to [C_out, kpad] by the layer class,
 * eps counters in that matrix).  kpad: multiple of 8 (bf16) / 4 (fp32).  One launch; replaces F.pad + unfold + copy_.
 */
int bt_im2col2d(const void* x, int dtype, int64_t n_img, int32_t C, int32_t H, int32_t W, const int64_t* strides_nchw,
                int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t ph, int32_t pw, int32_t dh, int32_t dw,
                int32_t kpad, void* out, void* stream);

/*
 * bt_lstm_cell -- the pointwise stage of one LSTM time step (rnn_variational.py:127-141, rnn_flipout.py:127-141):
 *   gates = gates_i + gates_h ([B, 4H], order i | f | g | o);  c' = sig(f) c + sig(i) tanh(g);  h' = sig(o) tanh(c')
 * h' / c' go to h_out / c_out ([B, H]) and into row t of the [B, T, H] sequences h_seq / c_seq.  The two gate GEMMs
 * are bt_layer_forward launches on the layer's `ih` / `hh` Bayesian linears (fresh weight sample per time step, as in
 * the reference).  All tensors share `dtype`.
 */
int bt_lstm_cell(const void* gates_i, const void* gates_h, const void* c_prev, void* h_out, void* c_out,
                 void* h_seq, void* c_seq, int dtype, int32_t batch, int32_t hidden, int32_t seq_len, int32_t t,
                 void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BTB200_H_ */
