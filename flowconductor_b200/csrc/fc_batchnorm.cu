// fc_batchnorm.cu — batch normalisation as a flow layer (BatchNorm, flowcon/transforms/normalization.py, 2-D inputs).
//
// With w = softplus(unconstrained_weight) + eps and σ = sqrt(v + eps) per feature:
//   forward  y = w · ((x − μ) / σ) + bias,       logabsdet = Σ_d (log w_d − ½ log(v_d + eps))
//   inverse  y = σ · ((x − bias) / w) + μ,       logabsdet = −Σ_d (log w_d − ½ log(v_d + eps))
// where (μ, v) are the batch mean and UNBIASED variance in training mode and the running buffers in eval mode.
//
// Every kernel walks the same layout: CTA g owns the rows [g R, (g + 1) R); thread (tx, ty) owns the V-wide column groups
// tx, tx + cw, ... (V = 4: 128-bit accesses when D, the strides and the pointers allow) and the rows ty, ty + ry, ...,
// U rows in flight.  cw = min(D / V, 256) exactly (not rounded up to a power of two), so a warp reads whole rows.
// The subtraction comes first and the scale second (y = s · (x − μ) + b, never s · x + (b − s μ)): the composed shift
// cancels catastrophically when |μ| >> σ.  w and σ are computed from the parameters and buffers inside the kernels, so a
// CUDA graph replays against their current values.
//
// Reductions are deterministic (no atomics): each CTA reduces its rows per column in a fixed order into a workspace, and
// a finish kernel (one CTA per column) merges the blocks in a fixed order.  The batch statistics are Welford means and
// sums of squared deviations per thread, merged with Chan's formula — never Σx² − Bμ² — all in fp64: an fp32 running
// mean loses ~√n ulps of |μ| over n rows, which is the whole signal when |μ| >> σ.  The kernel stays HBM-bound (five
// fp64 operations per 4-byte element).
#include <type_traits>

#include "fc_common.cuh"

namespace fc {

constexpr int kBnThreads = 256;
constexpr int kBnMaxD = 4096;  // 16 columns per thread (scalar) or 4 groups of 4 (vector)
constexpr int kBnFinishThreads = 128;

enum BnKernel { kBnStats = 0, kBnApply = 1, kBnGrad = 2, kBnGradX = 3 };

struct BnArgs {
  const float* x;
  const float* gy;
  const float* gl;  // may be null
  float* out;       // y (apply) or grad_x (grad with write_out, grad_x pass)
  float* lad;
  const float* mean;
  const float* var;
  const float* uw;
  const float* bias;
  float* ws;
  int64_t xs, gys, outs, B, rows_per_block;
  int D, cw, blocks, inverse, write_out;
  float eps;
};

__device__ __forceinline__ float bn_weight(float uw, float eps) {
  return (uw > 20.f ? uw : log1pf(expf(uw))) + eps;  // F.softplus (threshold 20) + eps
}

// (n, m, q) <- merge of (n, m, q) and (nb, mb, qb): counts, means, sums of squared deviations (Chan et al.)
__device__ __forceinline__ void chan_merge(double& n, double& m, double& q, double nb, double mb, double qb) {
  if (nb == 0.0) return;
  const double nt = n + nb;
  const double delta = mb - m;
  const double f = nb / nt;
  m = fma(delta, f, m);
  q = q + qb + delta * delta * n * f;
  n = nt;
}

// Rows [r_lo, r_hi) of CTA g; the number of them that row lane y visits.
__device__ __forceinline__ double bn_lane_rows(int64_t rows, int y, int ry) {
  return rows > y ? (double)((rows - y + ry - 1) / ry) : 0.0;
}

// G: column groups per thread (1 when D <= 256 V, else kBnMaxD / 256 / V).
template <int K, int V, int G>
__global__ void __launch_bounds__(kBnThreads) bn_rows_kernel(const BnArgs a) {
  extern __shared__ float sm[];  // [D] scale, [D] subtrahend, [D] addend, [D] k2, then [ry][2][D] partials
  const int D = a.D, cw = a.cw;
  float* sc = sm;
  float* sub = sm + D;
  float* add = sm + 2 * D;
  float* k2 = sm + 3 * D;
  using Acc = std::conditional_t<K == kBnStats, double, float>;
  Acc* red = reinterpret_cast<Acc*>(sm + 4 * D);
  const int ry = kBnThreads / cw, tx = threadIdx.x % cw, ty = threadIdx.x / cw;
  const int64_t r_lo = (int64_t)blockIdx.x * a.rows_per_block;
  int64_t r_hi = r_lo + a.rows_per_block;
  r_hi = r_hi < a.B ? r_hi : a.B;

  if constexpr (K != kBnStats) {
    __shared__ float parts[kBnThreads];
    float part = 0.f;
    for (int d = threadIdx.x; d < D; d += kBnThreads) {
      if constexpr (K == kBnGradX) {
        const float* coef = a.ws + (size_t)a.blocks * 2 * D + a.blocks;  // [3][D]: k1, k0, k2 from the finish kernel
        sc[d] = coef[d], add[d] = coef[D + d], k2[d] = coef[2 * D + d], sub[d] = __ldg(a.mean + d);
      } else {
        const float w = bn_weight(__ldg(a.uw + d), a.eps), ve = __ldg(a.var + d) + a.eps, s = sqrtf(ve);
        const float mu = __ldg(a.mean + d), b = __ldg(a.bias + d);
        sc[d] = a.inverse ? s / w : w / s;
        sub[d] = a.inverse ? b : mu;
        add[d] = a.inverse ? mu : b;
        part += logf(w) - 0.5f * logf(ve);
      }
    }
    if constexpr (K == kBnApply) {  // Σ_d logabsdet_d in a fixed order: per-thread partials, then thread 0
      parts[threadIdx.x] = part;
      __syncthreads();
      if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < kBnThreads; ++i) t += parts[i];
        parts[0] = a.inverse ? -t : t;
      }
    }
    __syncthreads();
    if constexpr (K == kBnApply) {
      const float total = parts[0];
      for (int64_t r = r_lo + threadIdx.x; r < r_hi; r += kBnThreads) a.lad[r] = total;
    }
  }

  constexpr bool kLoadG = K == kBnGrad || K == kBnGradX;
  constexpr int U = V == 4 ? 2 : (kLoadG || G > 1 ? 4 : 8);  // rows in flight per thread
  Acc acc0[G][V], acc1[G][V];
#pragma unroll
  for (int c = 0; c < G; ++c)
#pragma unroll
    for (int v = 0; v < V; ++v) acc0[c][v] = acc1[c][v] = 0;
  int n = 0;
  if (ty < ry) {
    for (int64_t r0 = r_lo + ty; r0 < r_hi; r0 += (int64_t)U * ry) {
      const int64_t left = (r_hi - r0 + ry - 1) / ry;
      const int nu = left < U ? (int)left : U;
      double inv[U];
      if constexpr (K == kBnStats) {
#pragma unroll
        for (int u = 0; u < U; ++u) inv[u] = 1.0 / (double)(n + u + 1);
      }
#pragma unroll
      for (int c = 0; c < G; ++c) {
        const int d = (tx + c * cw) * V;
        if (d < D) {
          float xv[U][V], gv[U][V];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (u < nu) {
              const int64_t r = r0 + (int64_t)u * ry;
              if constexpr (V == 4) {
                *reinterpret_cast<float4*>(xv[u]) = __ldcs(reinterpret_cast<const float4*>(a.x + r * a.xs + d));
                if constexpr (kLoadG)
                  *reinterpret_cast<float4*>(gv[u]) = __ldcs(reinterpret_cast<const float4*>(a.gy + r * a.gys + d));
              } else {
                xv[u][0] = __ldcs(a.x + r * a.xs + d);
                if constexpr (kLoadG) gv[u][0] = __ldcs(a.gy + r * a.gys + d);
              }
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (u < nu) {
              const int64_t r = r0 + (int64_t)u * ry;
              float o[V];
#pragma unroll
              for (int v = 0; v < V; ++v) {
                const float x = xv[u][v];
                if constexpr (K == kBnStats) {
                  const double delta = (double)x - acc0[c][v];
                  acc0[c][v] = fma(delta, inv[u], acc0[c][v]);
                  acc1[c][v] = fma(delta, (double)x - acc0[c][v], acc1[c][v]);
                } else if constexpr (K == kBnApply) {
                  o[v] = fmaf(sc[d + v], x - sub[d + v], add[d + v]);
                } else if constexpr (K == kBnGrad) {
                  const float g = gv[u][v];
                  acc0[c][v] = fmaf(g, x - sub[d + v], acc0[c][v]);
                  acc1[c][v] += g;
                  o[v] = g * sc[d + v];
                } else {
                  o[v] = fmaf(sc[d + v], gv[u][v], fmaf(k2[d + v], x - sub[d + v], add[d + v]));
                }
              }
              if (K == kBnApply || K == kBnGradX || (K == kBnGrad && a.write_out)) {
                if constexpr (V == 4) {
                  __stcs(reinterpret_cast<float4*>(a.out + r * a.outs + d), *reinterpret_cast<float4*>(o));
                } else {
                  a.out[r * a.outs + d] = o[0];
                }
              }
            }
          }
        }
      }
      n += nu;
    }
  }
  if constexpr (K == kBnStats || K == kBnGrad) {
    if (ty < ry) {
#pragma unroll
      for (int c = 0; c < G; ++c) {
        const int d = (tx + c * cw) * V;
        if (d < D) {
#pragma unroll
          for (int v = 0; v < V; ++v) {
            red[(ty * 2 + 0) * D + d + v] = acc0[c][v];
            red[(ty * 2 + 1) * D + d + v] = acc1[c][v];
          }
        }
      }
    }
    __syncthreads();
    Acc* out = reinterpret_cast<Acc*>(a.ws) + (size_t)blockIdx.x * 2 * D;  // stats: fp64 (mean, M2) per block
    for (int d = threadIdx.x; d < D; d += kBnThreads) {
      Acc t0 = 0, t1 = 0;
      if constexpr (K == kBnStats) {  // Chan merge of the row lanes in order
        double cnt = 0.0;
        for (int y = 0; y < ry; ++y)
          chan_merge(cnt, t0, t1, bn_lane_rows(r_hi - r_lo, y, ry), red[(y * 2 + 0) * D + d], red[(y * 2 + 1) * D + d]);
      } else {
        for (int y = 0; y < ry; ++y) {
          t0 += red[(y * 2 + 0) * D + d];
          t1 += red[(y * 2 + 1) * D + d];
        }
      }
      out[d] = t0;
      out[D + d] = t1;
    }
    if constexpr (K == kBnGrad) {  // Σ grad_logabsdet over the CTA's rows
      if (a.gl) {
        __shared__ float gparts[kBnThreads];
        float t = 0.f;
        for (int64_t r = r_lo + threadIdx.x; r < r_hi; r += kBnThreads) t += a.gl[r];
        gparts[threadIdx.x] = t;
        __syncthreads();
        if (threadIdx.x == 0) {
          float s = 0.f;
          for (int i = 0; i < kBnThreads; ++i) s += gparts[i];
          a.ws[(size_t)a.blocks * 2 * D + blockIdx.x] = s;
        }
      }
    }
  }
}

// One CTA per column: the blocks' (mean, M2) merged in a fixed order (strided per thread, then a fixed shuffle tree and
// the warps in order); writes the batch mean and the unbiased variance M2 / (B - 1) (NaN for B = 1, as torch.var), each
// rounded once to fp32.
__global__ void __launch_bounds__(kBnFinishThreads) bn_stats_finish_kernel(const double* ws, int blocks, int D, int64_t B,
                                                                           int64_t rows_per_block, float* mean,
                                                                           float* var) {
  const int d = blockIdx.x;
  double n = 0.0, m = 0.0, q = 0.0;
  for (int b = threadIdx.x; b < blocks; b += kBnFinishThreads) {
    const int64_t lo = (int64_t)b * rows_per_block, left = B - lo;
    const double nb = (double)(left < rows_per_block ? (left > 0 ? left : 0) : rows_per_block);
    chan_merge(n, m, q, nb, ws[(size_t)b * 2 * D + d], ws[(size_t)b * 2 * D + D + d]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double nb = __shfl_down_sync(0xffffffffu, n, o), mb = __shfl_down_sync(0xffffffffu, m, o);
    const double qb = __shfl_down_sync(0xffffffffu, q, o);
    chan_merge(n, m, q, nb, mb, qb);
  }
  __shared__ double parts[3][kBnFinishThreads / 32];
  if ((threadIdx.x & 31) == 0) {
    parts[0][threadIdx.x >> 5] = n;
    parts[1][threadIdx.x >> 5] = m;
    parts[2][threadIdx.x >> 5] = q;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tn = 0.0, tm = 0.0, tq = 0.0;
    for (int w = 0; w < kBnFinishThreads / 32; ++w) chan_merge(tn, tm, tq, parts[0][w], parts[1][w], parts[2][w]);
    mean[d] = (float)tm;
    var[d] = (float)(tq / (double)(B - 1));
  }
}

// One CTA per column: the blocks' Σ g (x − sub) and Σ g, and Σ grad_logabsdet, summed in a fixed order; then the
// parameter gradients and, in training mode, the coefficients of the grad_x pass (grad_x = k1 g + k0 + k2 (x − μ)).
__global__ void __launch_bounds__(kBnFinishThreads) bn_grad_finish_kernel(const BnArgs a, int mode, float* g_uw,
                                                                          float* g_bias) {
  const int d = blockIdx.x, D = a.D, blocks = a.blocks;
  const float* ws = a.ws;
  const bool has_gl = a.gl != nullptr;
  float t0 = 0.f, t1 = 0.f, g = 0.f;
  for (int b = threadIdx.x; b < blocks; b += kBnFinishThreads) {
    t0 += ws[(size_t)b * 2 * D + d];
    t1 += ws[(size_t)b * 2 * D + D + d];
    if (has_gl) g += ws[(size_t)blocks * 2 * D + b];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    t0 += __shfl_xor_sync(0xffffffffu, t0, o);
    t1 += __shfl_xor_sync(0xffffffffu, t1, o);
    g += __shfl_xor_sync(0xffffffffu, g, o);
  }
  __shared__ float parts[3][kBnFinishThreads / 32];
  if ((threadIdx.x & 31) == 0) {
    parts[0][threadIdx.x >> 5] = t0;
    parts[1][threadIdx.x >> 5] = t1;
    parts[2][threadIdx.x >> 5] = g;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  float sa = 0.f, sb = 0.f, G = 0.f;
  for (int w = 0; w < kBnFinishThreads / 32; ++w) {
    sa += parts[0][w];
    sb += parts[1][w];
    G += parts[2][w];
  }
  const float uw = a.uw[d], w = bn_weight(uw, a.eps), ve = a.var[d] + a.eps, s = sqrtf(ve);
  float gw, gb;
  if (mode == FC_BATCHNORM_EVAL_INVERSE) {  // sa = Σ g (x − bias)
    gw = -s * sa / (w * w) - G / w;
    gb = -(s / w) * sb;
  } else {  // sa = Σ g (x − μ): Σ g x̂ = sa / σ
    const float gxh = sa / s;
    gw = gxh + G / w;
    gb = sb;
    if (mode == FC_BATCHNORM_TRAIN) {
      float* coef = a.ws + (size_t)blocks * 2 * D + blocks;
      const float k1 = w / s;
      coef[d] = k1;
      coef[D + d] = -k1 * (sb / (float)a.B);
      coef[2 * D + d] = -(w * gxh + G) / ((float)(a.B - 1) * ve);
    }
  }
  g_uw[d] = gw / (1.f + expf(-uw));  // d weight / d unconstrained_weight = sigmoid(unconstrained_weight)
  g_bias[d] = gb;
}

static int bn_blocks(int64_t B) {
  const int64_t want = (B + 127) / 128;  // at least 128 rows per CTA
  const int cap = 8 * device_info().sm_count;
  return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Launch bn_rows_kernel<K, V> with the layout for (D, vector width); vec: D, strides and pointers allow float4.
template <int K>
static int bn_launch(BnArgs& a, bool vec, cudaStream_t st) {
  const int V = vec ? 4 : 1;
  a.cw = a.D / V < kBnThreads ? a.D / V : kBnThreads;
  const int ry = kBnThreads / a.cw;
  const size_t smem = sizeof(float) * (size_t)4 * a.D + sizeof(double) * (size_t)ry * 2 * a.D;
  constexpr int kWide4 = kBnMaxD / kBnThreads / 4, kWide1 = kBnMaxD / kBnThreads;
  auto kern = vec ? (a.D > 4 * kBnThreads ? bn_rows_kernel<K, 4, kWide4> : bn_rows_kernel<K, 4, 1>)
                  : (a.D > kBnThreads ? bn_rows_kernel<K, 1, kWide1> : bn_rows_kernel<K, 1, 1>);
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return FC_ERR_CUDA;
  kern<<<a.blocks, kBnThreads, smem, st>>>(a);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

static BnArgs bn_args(int64_t B, int32_t D, float eps) {
  BnArgs a = {};
  a.B = B, a.D = D, a.eps = eps;
  a.blocks = bn_blocks(B);
  a.rows_per_block = (B + a.blocks - 1) / a.blocks;
  return a;
}

}  // namespace fc

using namespace fc;

extern "C" int64_t fc_batchnorm_workspace_floats(int64_t B, int32_t D) {
  if (B < 0 || D < 1) return FC_ERR_INVALID_ARGUMENT;
  if (D > kBnMaxD) return FC_ERR_UNSUPPORTED;
  const int blocks = bn_blocks(B);
  return (int64_t)blocks * 4 * D + blocks + 3 * (int64_t)D;  // stats: fp64 [blocks][2][D]; backward: fp32, smaller
}

extern "C" int fc_batchnorm_stats(const float* x, int64_t x_row_stride, float* mean, float* var, float* workspace,
                                  int64_t B, int32_t D, void* stream) {
  if (B < 1 || D < 1 || !x || !mean || !var || !workspace || x_row_stride < D) return FC_ERR_INVALID_ARGUMENT;
  if (D > kBnMaxD) return FC_ERR_UNSUPPORTED;
  BnArgs a = bn_args(B, D, 0.f);
  a.x = x, a.xs = x_row_stride, a.ws = workspace;
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && aligned16(x);
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = bn_launch<kBnStats>(a, vec, st);
  if (rc != FC_OK) return rc;
  bn_stats_finish_kernel<<<D, kBnFinishThreads, 0, st>>>(reinterpret_cast<const double*>(workspace), a.blocks, D, B, a.rows_per_block, mean, var);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int fc_batchnorm_apply(const float* x, int64_t x_row_stride, const float* mean, const float* var,
                                  const float* unconstrained_weight, const float* bias, float eps, float* y,
                                  int64_t y_row_stride, float* logabsdet, int64_t B, int32_t D, int32_t inverse,
                                  void* stream) {
  if (B < 0 || D < 1 || !mean || !var || !unconstrained_weight || !bias) return FC_ERR_INVALID_ARGUMENT;
  if (B > 0 && (!x || !y || !logabsdet || x_row_stride < D || y_row_stride < D)) return FC_ERR_INVALID_ARGUMENT;
  if (D > kBnMaxD) return FC_ERR_UNSUPPORTED;
  if (B == 0) return FC_OK;
  BnArgs a = bn_args(B, D, eps);
  a.x = x, a.xs = x_row_stride, a.out = y, a.outs = y_row_stride, a.lad = logabsdet;
  a.mean = mean, a.var = var, a.uw = unconstrained_weight, a.bias = bias, a.inverse = inverse != 0;
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && (y_row_stride & 3) == 0 && aligned16(x) && aligned16(y);
  return bn_launch<kBnApply>(a, vec, (cudaStream_t)stream);
}

extern "C" int fc_batchnorm_backward(const float* x, int64_t x_row_stride, const float* mean, const float* var,
                                     const float* unconstrained_weight, const float* bias, float eps,
                                     const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet,
                                     float* grad_x, int64_t gx_row_stride, float* grad_unconstrained_weight,
                                     float* grad_bias, float* workspace, int64_t B, int32_t D, int32_t mode,
                                     void* stream) {
  if (B < 0 || D < 1 || !mean || !var || !unconstrained_weight || !bias || !grad_unconstrained_weight || !grad_bias)
    return FC_ERR_INVALID_ARGUMENT;
  if (mode != FC_BATCHNORM_TRAIN && mode != FC_BATCHNORM_EVAL_FORWARD && mode != FC_BATCHNORM_EVAL_INVERSE)
    return FC_ERR_INVALID_ARGUMENT;
  if (B > 0 && (!x || !grad_y || !grad_x || !workspace || x_row_stride < D || gy_row_stride < D || gx_row_stride < D))
    return FC_ERR_INVALID_ARGUMENT;
  if (D > kBnMaxD) return FC_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) {
    if (cudaMemsetAsync(grad_unconstrained_weight, 0, sizeof(float) * D, st) != cudaSuccess) return FC_ERR_CUDA;
    if (cudaMemsetAsync(grad_bias, 0, sizeof(float) * D, st) != cudaSuccess) return FC_ERR_CUDA;
    return FC_OK;
  }
  BnArgs a = bn_args(B, D, eps);
  a.x = x, a.xs = x_row_stride, a.gy = grad_y, a.gys = gy_row_stride, a.gl = grad_logabsdet;
  a.out = grad_x, a.outs = gx_row_stride, a.ws = workspace;
  a.mean = mean, a.var = var, a.uw = unconstrained_weight, a.bias = bias;
  a.inverse = mode == FC_BATCHNORM_EVAL_INVERSE;
  a.write_out = mode != FC_BATCHNORM_TRAIN;  // training mode needs the column sums before grad_x
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && (gy_row_stride & 3) == 0 && (gx_row_stride & 3) == 0 &&
                   aligned16(x) && aligned16(grad_y) && aligned16(grad_x);
  int rc = bn_launch<kBnGrad>(a, vec, st);
  if (rc != FC_OK) return rc;
  bn_grad_finish_kernel<<<D, kBnFinishThreads, 0, st>>>(a, mode, grad_unconstrained_weight, grad_bias);
  FC_CHECK_LAUNCH();
  if (mode == FC_BATCHNORM_TRAIN) return bn_launch<kBnGradX>(a, vec, st);
  return FC_OK;
}
