// Monte-Carlo aggregation on device: softmax of every sample's logits, running sum of p and p^2.
//
// Replaces   output_ = torch.stack(output_mc); softmax; mean(0)
// (/root/reference/bayesian_torch/examples/main_bayesian_cifar_dnn2bnn.py:545-557) and the
// per-sample `.cpu().numpy()` round trip of examples/main_bayesian_imagenet.py:617-624.
// The [2,B,C] fp32 result is the ONLY thing that crosses GPUs (one NCCL all-reduce).
#include "bt_common.cuh"

namespace {

template <typename T>
__device__ __forceinline__ float ld_logit(const T* p);
template <>
__device__ __forceinline__ float ld_logit<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ld_logit<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

// one warp per batch row b; loops over the S samples in order (deterministic).
// CPL = classes per lane held in registers (C <= 32 * CPL)
// ent_sum (nullable, [B]): running sum over the samples of the per-sample entropy  -sum_c p log(p + 1e-15)
// (utils/util.py:41-42 applied to every MC member, the second term of mutual_information, util.py:54-60).
template <typename T, int CPL>
__global__ void mc_accumulate_kernel(const T* __restrict__ logits, int S, int B, int C,
                                     float* __restrict__ sums, float* __restrict__ ent_sum, int accumulate) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B) return;
  float a1[CPL], a2[CPL];
  float ent = 0.f;
#pragma unroll
  for (int j = 0; j < CPL; ++j) a1[j] = a2[j] = 0.f;
  // The samples are ACCUMULATED strictly in order (deterministic, bit-identical for any batching), but their logits are
  // LOADED SB samples at a time: one dependent global load per sample made this kernel a 64-long latency chain (46 us per
  // step for 8192 x 10 logits, profiles/r02_launches_bf16.md).
  constexpr int SB = CPL == 1 ? 8 : (CPL == 4 ? 4 : 1);
  for (int s0 = 0; s0 < S; s0 += SB) {
    float vv[SB][CPL];
#pragma unroll
    for (int u = 0; u < SB; ++u) {
      const int su = s0 + u < S ? s0 + u : S - 1;
      const T* row = logits + ((long long)su * B + warp) * C;
#pragma unroll
      for (int j = 0; j < CPL; ++j) {
        const int c = lane + 32 * j;
        vv[u][j] = c < C ? ld_logit<T>(row + c) : -INFINITY;
      }
    }
#pragma unroll
    for (int u = 0; u < SB; ++u) {
    if (s0 + u >= S) break;
    float v[CPL];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
      v[j] = vv[u][j];
      mx = fmaxf(mx, v[j]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float den = 0.f;
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
      v[j] = (lane + 32 * j < C) ? __expf(v[j] - mx) : 0.f;
      den += v[j];
    }
    den = bt_warp_sum(den);
    const float inv = 1.0f / den;
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
      const float p = v[j] * inv;
      a1[j] += p;
      a2[j] = fmaf(p, p, a2[j]);
      if (ent_sum != nullptr && lane + 32 * j < C) ent = fmaf(-p, __logf(p + 1e-15f), ent);
    }
    }
  }
  if (ent_sum != nullptr) {
    ent = bt_warp_sum(ent);
    if (lane == 0) ent_sum[warp] = accumulate ? ent_sum[warp] + ent : ent;
  }
  float* o1 = sums + (long long)warp * C;
  float* o2 = sums + ((long long)B + warp) * C;
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    const int c = lane + 32 * j;
    if (c < C) {
      o1[c] = accumulate ? o1[c] + a1[j] : a1[j];
      o2[c] = accumulate ? o2[c] + a2[j] : a2[j];
    }
  }
}

__global__ void mc_finalize_kernel(const float* __restrict__ sums, long long n, float inv_total,
                                   float* __restrict__ mean, float* __restrict__ var) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float m = sums[i] * inv_total;
    mean[i] = m;
    if (var) var[i] = fmaxf(sums[n + i] * inv_total - m * m, 0.f);
  }
}

// predictive entropy  H(mean_s p_s)  and mutual information  H(mean p) - mean_s H(p_s)  (utils/util.py:45-60)
// from the (all-reduced) moment buffer: one warp per batch row.
__global__ void mc_uncertainty_kernel(const float* __restrict__ sums, const float* __restrict__ ent_sum, int B, int C,
                                      float inv_total, float* __restrict__ pred_entropy, float* __restrict__ mutual_info) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B) return;
  float h = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float m = sums[(long long)warp * C + c] * inv_total;
    h = fmaf(-m, __logf(m + 1e-15f), h);
  }
  h = bt_warp_sum(h);
  if (lane == 0) {
    pred_entropy[warp] = h;
    if (mutual_info != nullptr) mutual_info[warp] = h - ent_sum[warp] * inv_total;
  }
}

template <typename T>
int launch_acc(const void* logits, int S, int B, int C, float* sums, float* ent, int acc, cudaStream_t st) {
  const int threads = 128;  // 4 rows per block
  const unsigned blocks = (unsigned)((B + 3) / 4);
  const T* l = static_cast<const T*>(logits);
  if (C <= 32) mc_accumulate_kernel<T, 1><<<blocks, threads, 0, st>>>(l, S, B, C, sums, ent, acc);
  else if (C <= 128) mc_accumulate_kernel<T, 4><<<blocks, threads, 0, st>>>(l, S, B, C, sums, ent, acc);
  else if (C <= 1024) mc_accumulate_kernel<T, 32><<<blocks, threads, 0, st>>>(l, S, B, C, sums, ent, acc);
  else {
    bt_set_error("bt_mc_accumulate: n_classes %d > 1024 not supported (bt_mc_accumulate_large takes any C)", C);
    return BT_ERR_UNSUPPORTED;
  }
  BT_CHECK_CUDA(cudaGetLastError());
  return BT_OK;
}

// ---------------------------------------------------------------- large-C softmax moments (C > 1024)
// A warp cannot hold such a row in registers, and re-reading the [2, rows, C] sums once per sample would cost 8x the
// logit bytes at C = 21841.  Two kernels instead, each reading every logit once:
//   A  one CTA per (sample, row): max m, sum e^{l-m} and sum e^{l-m} (l-m) in one pass (online rescaling), i.e. the
//      log-sum-exp and the exact per-sample entropy H_s = log(sum e^{l-m}) - E_p[l-m];
//   B  one CTA per (row, 1024-class slice): streams the samples in order, p = exp(l - lse_s), sum p and p^2 in
//      registers, writes (or adds to) its slice of the sums once.
// Fixed reduction trees and in-order sample loops: a repeated call gives the same bits.
constexpr int LC_A_THREADS = 256;
constexpr int LC_B_THREADS = 128;
constexpr int LC_B_CPT = 8;                                 // classes per thread
constexpr int LC_SLICE = LC_B_THREADS * LC_B_CPT;           // classes per CTA of kernel B

// (m, s, t) <- merge with (m2, s2, t2), where s = sum e^{l-m} and t = sum e^{l-m} (l-m) of disjoint element sets
__device__ __forceinline__ void lse_merge(float& m, float& s, float& t, float m2, float s2, float t2) {
  if (m2 == -INFINITY) return;
  if (m == -INFINITY) {
    m = m2; s = s2; t = t2;
    return;
  }
  const float mn = fmaxf(m, m2);
  const float d1 = m - mn, d2 = m2 - mn;
  const float a = expf(d1), b = expf(d2);
  t = a * fmaf(d1, s, t) + b * fmaf(d2, s2, t2);
  s = a * s + b * s2;
  m = mn;
}

template <typename T>
__global__ void __launch_bounds__(LC_A_THREADS) mc_large_lse_kernel(const T* __restrict__ logits, int rows, int C,
                                                                     float* __restrict__ lse, float* __restrict__ hs) {
  const long long sr = blockIdx.x;                          // s * rows + r: the logits row of (sample s, row r)
  const T* row = logits + sr * C;
  constexpr int U = 8;                                      // loads in flight per thread
  float m = -INFINITY, s = 0.f, t = 0.f;
  for (int c0 = threadIdx.x; c0 < C; c0 += U * LC_A_THREADS) {
    float v[U];
    float cm = -INFINITY;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = c0 + u * LC_A_THREADS;
      v[u] = c < C ? ld_logit<T>(row + c) : -INFINITY;
      cm = fmaxf(cm, v[u]);
    }
    if (cm > m) {                                           // rescale the running sums to the new maximum
      if (m != -INFINITY) {
        const float d = m - cm, a = expf(d);
        t = a * fmaf(d, s, t);
        s *= a;
      }
      m = cm;
    }
    if (m == -INFINITY) continue;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const float d = v[u] - m;
      const float e = expf(d);
      s += e;
      t += e > 0.f ? e * d : 0.f;                           // (a -inf logit contributes nothing, not -inf * 0)
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o),
                t2 = __shfl_xor_sync(0xffffffffu, t, o);
    lse_merge(m, s, t, m2, s2, t2);
  }
  __shared__ float sm[3][LC_A_THREADS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sm[0][warp] = m; sm[1][warp] = s; sm[2][warp] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < LC_A_THREADS / 32; ++w) lse_merge(m, s, t, sm[0][w], sm[1][w], sm[2][w]);
    const float ls = logf(s);
    lse[sr] = m + ls;
    if (hs != nullptr) hs[sr] = ls - t / s;
  }
}

template <typename T>
__global__ void __launch_bounds__(LC_B_THREADS) mc_large_moments_kernel(const T* __restrict__ logits,
    const float* __restrict__ lse, const float* __restrict__ hs, int S, int rows, int C, float* __restrict__ sums,
    float* __restrict__ ent_sum, int accumulate) {
  const int r = blockIdx.x;
  const int cb = blockIdx.y * LC_SLICE + threadIdx.x;
  float* o1 = sums + (long long)r * C;
  float* o2 = sums + ((long long)rows + r) * C;
  float a1[LC_B_CPT], a2[LC_B_CPT];
#pragma unroll
  for (int k = 0; k < LC_B_CPT; ++k) {
    const int c = cb + k * LC_B_THREADS;
    a1[k] = accumulate && c < C ? o1[c] : 0.f;
    a2[k] = accumulate && c < C ? o2[c] : 0.f;
  }
  constexpr int SB = 2;                                     // samples loaded per step, accumulated in order
  for (int s0 = 0; s0 < S; s0 += SB) {
    float v[SB][LC_B_CPT], L[SB];
#pragma unroll
    for (int u = 0; u < SB; ++u) {
      const int su = s0 + u < S ? s0 + u : S - 1;
      const long long sr = (long long)su * rows + r;
      const T* row = logits + sr * C;
      L[u] = lse[sr];
#pragma unroll
      for (int k = 0; k < LC_B_CPT; ++k) {
        const int c = cb + k * LC_B_THREADS;
        v[u][k] = c < C ? ld_logit<T>(row + c) : -INFINITY;
      }
    }
#pragma unroll
    for (int u = 0; u < SB; ++u) {
      if (s0 + u >= S) break;
#pragma unroll
      for (int k = 0; k < LC_B_CPT; ++k) {
        const float p = bt_ex2((v[u][k] - L[u]) * 1.4426950408889634f);
        a1[k] += p;
        a2[k] = fmaf(p, p, a2[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < LC_B_CPT; ++k) {
    const int c = cb + k * LC_B_THREADS;
    if (c < C) {
      o1[c] = a1[k];
      o2[c] = a2[k];
    }
  }
  if (ent_sum != nullptr && blockIdx.y == 0 && threadIdx.x == 0) {
    float e = accumulate ? ent_sum[r] : 0.f;
    for (int s = 0; s < S; ++s) e += hs[(long long)s * rows + r];
    ent_sum[r] = e;
  }
}

// ---------------------------------------------------------------- regression moments
// y: S blocks of n elements (sample s = elements [s*n, (s+1)*n) in memory order); sums fp64 [2, n].
// fp64 because sum y^2 / N - mean^2 in fp32 cancels catastrophically for outputs with a large mean and a small spread
// (mean 1e3, std 1e-2: y^2 ~ 1e6 carries an fp32 rounding of ~0.06, the variance is 1e-4).
template <typename T, int VEC>
struct RegVec;
template <>
struct RegVec<float, 4> {
  static __device__ __forceinline__ void load(const float* p, float* v) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
};
template <>
struct RegVec<__nv_bfloat16, 8> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float* v) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] = bt_bf16_lo(w[j]);
      v[2 * j + 1] = bt_bf16_hi(w[j]);
    }
  }
};
template <typename T>
struct RegVec<T, 1> {
  static __device__ __forceinline__ void load(const T* p, float* v) { v[0] = ld_logit<T>(p); }
};

template <typename T, int VEC>
__global__ void mc_reg_accumulate_kernel(const T* __restrict__ y, int S, long long n, double* __restrict__ sums,
                                         int accumulate) {
  const long long nv = n / VEC;                             // (n % VEC == 0 when VEC > 1)
  constexpr int SB = 4;                                     // samples loaded per step, accumulated in order
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    const long long e0 = i * VEC;
    double a1[VEC], a2[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      a1[j] = accumulate ? sums[e0 + j] : 0.0;
      a2[j] = accumulate ? sums[n + e0 + j] : 0.0;
    }
    for (int s0 = 0; s0 < S; s0 += SB) {
      float v[SB][VEC];
#pragma unroll
      for (int u = 0; u < SB; ++u) {
        const int su = s0 + u < S ? s0 + u : S - 1;
        RegVec<T, VEC>::load(y + (long long)su * n + e0, v[u]);
      }
#pragma unroll
      for (int u = 0; u < SB; ++u) {
        if (s0 + u >= S) break;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const double d = v[u][j];
          a1[j] += d;
          a2[j] = fma(d, d, a2[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      sums[e0 + j] = a1[j];
      sums[n + e0 + j] = a2[j];
    }
  }
}

__global__ void mc_reg_finalize_kernel(const double* __restrict__ sums, long long n, double inv_total,
                                       float* __restrict__ mean, float* __restrict__ var) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const double m = sums[i] * inv_total;
    mean[i] = (float)m;
    if (var) var[i] = (float)fmax(sums[n + i] * inv_total - m * m, 0.0);
  }
}

unsigned grid_stride_blocks(long long work, int threads) {
  const long long b = (work + threads - 1) / threads;
  return (unsigned)(b > 148 * 16 ? 148 * 16 : (b < 1 ? 1 : b));
}

template <typename T>
int launch_reg(const void* y, int S, long long n, double* sums, int acc, cudaStream_t st) {
  constexpr int V = 16 / sizeof(T);                         // 16-byte loads when every sample block is 16-byte aligned
  const T* p = static_cast<const T*>(y);
  if (reinterpret_cast<uintptr_t>(y) % 16 == 0 && n % V == 0)
    mc_reg_accumulate_kernel<T, V><<<grid_stride_blocks(n / V, 256), 256, 0, st>>>(p, S, n, sums, acc);
  else
    mc_reg_accumulate_kernel<T, 1><<<grid_stride_blocks(n, 256), 256, 0, st>>>(p, S, n, sums, acc);
  BT_CHECK_CUDA(cudaGetLastError());
  return BT_OK;
}

}  // namespace

extern "C" {

int bt_mc_accumulate_ex(const void* logits, int dtype, int32_t n_samples, int32_t batch,
                        int32_t n_classes, float* sums, float* entropy_sum, int accumulate, void* stream) {
  BT_REQUIRE(n_samples > 0 && batch > 0 && n_classes > 0, BT_ERR_BAD_SHAPE,
             "bt_mc_accumulate: bad shape S=%d B=%d C=%d", n_samples, batch, n_classes);
  BT_REQUIRE(dtype == BT_F32 || dtype == BT_BF16, BT_ERR_BAD_DTYPE, "bt_mc_accumulate: dtype %d", dtype);
  int rc;
  if ((rc = bt_check_device_ptr(logits, "logits")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(sums, "sums")) != BT_OK) return rc;
  if (entropy_sum != nullptr && (rc = bt_check_device_ptr(entropy_sum, "entropy_sum")) != BT_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dtype == BT_F32 ? launch_acc<float>(logits, n_samples, batch, n_classes, sums, entropy_sum, accumulate, st)
                         : launch_acc<__nv_bfloat16>(logits, n_samples, batch, n_classes, sums, entropy_sum,
                                                     accumulate, st);
}

int bt_mc_accumulate(const void* logits, int dtype, int32_t n_samples, int32_t batch,
                     int32_t n_classes, float* sums, int accumulate, void* stream) {
  return bt_mc_accumulate_ex(logits, dtype, n_samples, batch, n_classes, sums, nullptr, accumulate, stream);
}

int bt_mc_uncertainty(const float* sums, const float* entropy_sum, int32_t batch, int32_t n_classes, int32_t n_total,
                      float* pred_entropy, float* mutual_info, void* stream) {
  BT_REQUIRE(batch > 0 && n_classes > 0 && n_total > 0, BT_ERR_BAD_SHAPE, "bt_mc_uncertainty: bad shape");
  BT_REQUIRE(mutual_info == nullptr || entropy_sum != nullptr, BT_ERR_BAD_POINTER,
             "bt_mc_uncertainty: mutual information needs the per-sample entropy sums");
  int rc;
  if ((rc = bt_check_device_ptr(sums, "sums")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(pred_entropy, "pred_entropy")) != BT_OK) return rc;
  const unsigned blocks = (unsigned)((batch + 3) / 4);
  mc_uncertainty_kernel<<<blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      sums, entropy_sum, batch, n_classes, 1.0f / (float)n_total, pred_entropy, mutual_info);
  BT_CHECK_CUDA(cudaGetLastError());
  return BT_OK;
}

int bt_mc_finalize(const float* sums, int32_t batch, int32_t n_classes, int32_t n_total,
                   float* mean, float* var, void* stream) {
  BT_REQUIRE(batch > 0 && n_classes > 0 && n_total > 0, BT_ERR_BAD_SHAPE, "bt_mc_finalize: bad shape");
  int rc;
  if ((rc = bt_check_device_ptr(sums, "sums")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(mean, "mean")) != BT_OK) return rc;
  const long long n = (long long)batch * n_classes;
  const unsigned blocks = (unsigned)((n + 255) / 256 > 1184 ? 1184 : (n + 255) / 256);
  mc_finalize_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      sums, n, 1.0f / (float)n_total, mean, var);
  BT_CHECK_CUDA(cudaGetLastError());
  return BT_OK;
}

int bt_mc_accumulate_large(const void* logits, int dtype, int32_t n_samples, int32_t rows, int32_t n_classes,
                           float* sums, float* entropy_sum, int accumulate, float* workspace, void* stream) {
  BT_REQUIRE(n_samples > 0 && rows > 0 && n_classes > 0, BT_ERR_BAD_SHAPE,
             "bt_mc_accumulate_large: bad shape S=%d rows=%d C=%d", n_samples, rows, n_classes);
  BT_REQUIRE((long long)n_samples * rows <= 0x7FFFFFFFLL, BT_ERR_BAD_SHAPE,
             "bt_mc_accumulate_large: S * rows = %lld exceeds the grid", (long long)n_samples * rows);
  BT_REQUIRE((n_classes + LC_SLICE - 1) / LC_SLICE <= 65535, BT_ERR_BAD_SHAPE,
             "bt_mc_accumulate_large: n_classes %d exceeds the grid", n_classes);
  BT_REQUIRE(dtype == BT_F32 || dtype == BT_BF16, BT_ERR_BAD_DTYPE, "bt_mc_accumulate_large: dtype %d", dtype);
  int rc;
  if ((rc = bt_check_device_ptr(logits, "logits")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(sums, "sums")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(workspace, "workspace")) != BT_OK) return rc;
  if (entropy_sum != nullptr && (rc = bt_check_device_ptr(entropy_sum, "entropy_sum")) != BT_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* lse = workspace;
  float* hs = entropy_sum != nullptr ? workspace + (long long)n_samples * rows : nullptr;
  const dim3 grid_b((unsigned)rows, (unsigned)((n_classes + LC_SLICE - 1) / LC_SLICE));
  if (dtype == BT_F32) {
    const float* l = static_cast<const float*>(logits);
    mc_large_lse_kernel<float><<<(unsigned)(n_samples * rows), LC_A_THREADS, 0, st>>>(l, rows, n_classes, lse, hs);
    mc_large_moments_kernel<float><<<grid_b, LC_B_THREADS, 0, st>>>(l, lse, hs, n_samples, rows, n_classes, sums,
                                                                     entropy_sum, accumulate);
  } else {
    const __nv_bfloat16* l = static_cast<const __nv_bfloat16*>(logits);
    mc_large_lse_kernel<__nv_bfloat16><<<(unsigned)(n_samples * rows), LC_A_THREADS, 0, st>>>(l, rows, n_classes,
                                                                                               lse, hs);
    mc_large_moments_kernel<__nv_bfloat16><<<grid_b, LC_B_THREADS, 0, st>>>(l, lse, hs, n_samples, rows, n_classes,
                                                                             sums, entropy_sum, accumulate);
  }
  BT_CHECK_CUDA(cudaGetLastError());
  return BT_OK;
}

int bt_mc_regression_accumulate(const void* y, int dtype, int32_t n_samples, int64_t n_elem, double* sums,
                                int accumulate, void* stream) {
  BT_REQUIRE(n_samples > 0 && n_elem > 0, BT_ERR_BAD_SHAPE, "bt_mc_regression_accumulate: bad shape S=%d n=%lld",
             n_samples, (long long)n_elem);
  BT_REQUIRE(n_elem <= (1LL << 62) / n_samples, BT_ERR_BAD_SHAPE, "bt_mc_regression_accumulate: S * n overflows");
  BT_REQUIRE(dtype == BT_F32 || dtype == BT_BF16, BT_ERR_BAD_DTYPE, "bt_mc_regression_accumulate: dtype %d", dtype);
  int rc;
  if ((rc = bt_check_device_ptr(y, "y")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(sums, "sums")) != BT_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dtype == BT_F32 ? launch_reg<float>(y, n_samples, n_elem, sums, accumulate, st)
                         : launch_reg<__nv_bfloat16>(y, n_samples, n_elem, sums, accumulate, st);
}

int bt_mc_regression_finalize(const double* sums, int64_t n_elem, int32_t n_total, float* mean, float* var,
                              void* stream) {
  BT_REQUIRE(n_elem > 0 && n_total > 0, BT_ERR_BAD_SHAPE, "bt_mc_regression_finalize: bad shape");
  int rc;
  if ((rc = bt_check_device_ptr(sums, "sums")) != BT_OK) return rc;
  if ((rc = bt_check_device_ptr(mean, "mean")) != BT_OK) return rc;
  if (var != nullptr && (rc = bt_check_device_ptr(var, "var")) != BT_OK) return rc;
  mc_reg_finalize_kernel<<<grid_stride_blocks(n_elem, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      sums, n_elem, 1.0 / (double)n_total, mean, var);
  BT_CHECK_CUDA(cudaGetLastError());
  return BT_OK;
}

}  // extern "C"
