// fc_pointwise.cu — element-wise squashing layers (Sigmoid / Logit, Tanh, LeakyReLU, Exp, CauchyCDF,
// flowcon/transforms/nonlinearities.py).  The per-element arithmetic is in fc_pointwise.cuh.
//
// Forward / inverse (pw_apply_kernel): the row layout of dn_log_prob_kernel (fc_diagnormal.cu).  seg =
// min(32, next_pow2(D / V)) lanes cover one row (V = 4: 128-bit accesses when D, the strides and the pointers allow, else
// V = 1), a warp covers 32 / seg rows per pass, and the row's log-det is an xor-shuffle sum over its lanes.  Domain
// violations are collected per thread and OR-ed into the status word once at the end.
// Backward (pw_backward_kernel): the same layout, element-wise at the layer's input.  With the temperature gradient,
// every thread sums its elements' ∂/∂T terms, the CTA sums its threads in a fixed order (xor tree per warp, then the
// warps in order) into workspace[blockIdx.x], and pw_finish_kernel sums the CTA partials in a fixed order: no atomics.
#include "fc_common.cuh"
#include "fc_pointwise.cuh"

namespace fc {

constexpr int kPwThreads = 256;
constexpr int64_t kPwMaxBlocks = 2048;  // bound on the grid, and so on the temperature-gradient workspace

struct PwArgs {
  const float* x;
  float* y;
  float* lad;
  const float* gy;
  const float* gl;
  float* gx;
  float* gt;    // grad_temperature (backward, optional)
  float* part;  // [gridDim.x] temperature partials
  int32_t* status;
  const float* temperature;
  int64_t xs, ys, gys, gxs, B;
  int D, accumulate;
  float s, log_s, eps;
};

template <int V>
__device__ __forceinline__ void pw_load_cs(float (&v)[V], const float* p) {
  if constexpr (V == 4) {
    *reinterpret_cast<float4*>(v) = __ldcs(reinterpret_cast<const float4*>(p));
  } else {
    v[0] = __ldcs(p);
  }
}

template <int V>
__device__ __forceinline__ void pw_store_cs(float* p, const float (&v)[V]) {
  if constexpr (V == 4) {
    __stcs(reinterpret_cast<float4*>(p), *reinterpret_cast<const float4*>(v));
  } else {
    __stcs(p, v[0]);
  }
}

__device__ __forceinline__ PwScalars pw_scalars(const PwArgs& a) {
  PwScalars c;
  c.T = a.temperature ? __ldg(a.temperature) : 1.f;
  c.log_T = logf(c.T);
  c.s = a.s, c.log_s = a.log_s, c.eps = a.eps;
  return c;
}

template <int OP, bool INV, int V>
__global__ void __launch_bounds__(kPwThreads) pw_apply_kernel(const PwArgs a, int seg) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rpw = 32 / seg, sub = lane / seg, j0 = lane % seg;
  const int64_t groups = (a.B + rpw - 1) / rpw;
  const int D = a.D;
  const PwScalars c = pw_scalars(a);
  bool bad = false;
  for (int64_t w = (int64_t)blockIdx.x * kWarps + warp; w < groups; w += (int64_t)gridDim.x * kWarps) {
    const int64_t row = w * rpw + sub;
    const bool row_ok = row < a.B;
    float sum = 0.f;
    if (row_ok) {
      const float* xr = a.x + row * a.xs;
      float* yr = a.y + row * a.ys;
      for (int d = j0 * V; d < D; d += seg * V) {
        float xv[V], yv[V];
        pw_load_cs<V>(xv, xr + d);
#pragma unroll
        for (int v = 0; v < V; ++v) {
          float l;
          pw_eval<OP, INV>(xv[v], c, yv[v], l, bad);
          sum += l;
        }
        pw_store_cs<V>(yr + d, yv);
      }
    }
    sum = seg_reduce_sum(sum, seg);
    if (row_ok && j0 == 0) a.lad[row] = a.accumulate ? a.lad[row] + sum : sum;
  }
  if (bad && a.status) atomicOr(a.status, FC_STATUS_INPUT_OUTSIDE_DOMAIN);
}

template <int OP, bool INV, int V, bool WANT_T>
__global__ void __launch_bounds__(kPwThreads) pw_backward_kernel(const PwArgs a, int seg) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rpw = 32 / seg, sub = lane / seg, j0 = lane % seg;
  const int64_t groups = (a.B + rpw - 1) / rpw;
  const int D = a.D;
  const PwScalars c = pw_scalars(a);
  float acc_t = 0.f;
  for (int64_t w = (int64_t)blockIdx.x * kWarps + warp; w < groups; w += (int64_t)gridDim.x * kWarps) {
    const int64_t row = w * rpw + sub;
    if (row >= a.B) continue;  // warp-uniform loop: every lane still reaches the reduction below
    const float* xr = a.x + row * a.xs;
    const float* gyr = a.gy ? a.gy + row * a.gys : nullptr;
    float* gxr = a.gx + row * a.gxs;
    const float gl = a.gl ? __ldg(a.gl + row) : 0.f;
    for (int d = j0 * V; d < D; d += seg * V) {
      float xv[V], gv[V], out[V];
      pw_load_cs<V>(xv, xr + d);
      if (gyr) {
        pw_load_cs<V>(gv, gyr + d);
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) gv[v] = 0.f;
      }
#pragma unroll
      for (int v = 0; v < V; ++v) {
        float dy, dl, dyT, dlT;
        pw_grad<OP, INV>(xv[v], c, dy, dl, dyT, dlT);
        out[v] = fmaf(gl, dl, gv[v] * dy);
        if constexpr (WANT_T) acc_t += fmaf(gl, dlT, gv[v] * dyT);
      }
      pw_store_cs<V>(gxr + d, out);
    }
  }
  if constexpr (WANT_T) {
    __shared__ float red[kWarps];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc_t += __shfl_xor_sync(0xffffffffu, acc_t, o);
    if (lane == 0) red[warp] = acc_t;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int k = 0; k < kWarps; ++k) t += red[k];
      if (gridDim.x == 1)
        *a.gt = t;
      else
        a.part[blockIdx.x] = t;
    }
  }
}

// one warp: the CTA partials, lane-strided, then a fixed xor tree
__global__ void pw_finish_kernel(const float* part, int n, float* out) {
  float t = 0.f;
  for (int k = threadIdx.x; k < n; k += 32) t += part[k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if (threadIdx.x == 0) *out = t;
}

static bool pw_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int64_t pw_blocks(int64_t B, int seg) {
  const int64_t rows_per_cta = (int64_t)(32 / seg) * kWarps;
  int64_t cap = 8 * (int64_t)device_info().sm_count;
  if (cap > kPwMaxBlocks) cap = kPwMaxBlocks;
  const int64_t want = (B + rows_per_cta - 1) / rows_per_cta;
  return want < cap ? want : cap;
}

// Arguments shared by both entries; FC_OK or FC_ERR_INVALID_ARGUMENT.
static int pw_check_config(const fc_pointwise_config* cfg, int64_t B, int64_t D) {
  if (!cfg || B < 0 || D < 1 || D > 0x7fffffff) return FC_ERR_INVALID_ARGUMENT;
  if (cfg->op < FC_POINTWISE_SIGMOID || cfg->op > FC_POINTWISE_CAUCHY_CDF) return FC_ERR_INVALID_ARGUMENT;
  if (cfg->op == FC_POINTWISE_SIGMOID && !cfg->temperature) return FC_ERR_INVALID_ARGUMENT;
  if (cfg->op == FC_POINTWISE_LEAKY_RELU && !(cfg->slope > 0.f)) return FC_ERR_INVALID_ARGUMENT;
  return FC_OK;
}

static void pw_scalar_args(PwArgs& a, const fc_pointwise_config* cfg) {
  a.temperature = cfg->op == FC_POINTWISE_SIGMOID ? cfg->temperature : nullptr;
  a.eps = cfg->eps;
  a.log_s = logf(cfg->slope);  // the reference's fp32 log_negative_slope, for both directions
  a.s = cfg->inverse ? (float)(1.0 / (double)cfg->slope) : cfg->slope;
}

template <int OP, bool INV>
static void pw_launch_apply(const PwArgs& a, bool vec, bool, int64_t blocks, int seg, cudaStream_t st) {
  if (vec)
    pw_apply_kernel<OP, INV, 4><<<(unsigned)blocks, kPwThreads, 0, st>>>(a, seg);
  else
    pw_apply_kernel<OP, INV, 1><<<(unsigned)blocks, kPwThreads, 0, st>>>(a, seg);
}

template <int OP, bool INV>
static void pw_launch_backward(const PwArgs& a, bool vec, bool want_t, int64_t blocks, int seg, cudaStream_t st) {
  if (want_t) {
    if (vec)
      pw_backward_kernel<OP, INV, 4, true><<<(unsigned)blocks, kPwThreads, 0, st>>>(a, seg);
    else
      pw_backward_kernel<OP, INV, 1, true><<<(unsigned)blocks, kPwThreads, 0, st>>>(a, seg);
  } else {
    if (vec)
      pw_backward_kernel<OP, INV, 4, false><<<(unsigned)blocks, kPwThreads, 0, st>>>(a, seg);
    else
      pw_backward_kernel<OP, INV, 1, false><<<(unsigned)blocks, kPwThreads, 0, st>>>(a, seg);
  }
}

using PwLaunch = void (*)(const PwArgs&, bool, bool, int64_t, int, cudaStream_t);

#define FC_PW_TABLE(L)                                                                           \
  {{L<FC_POINTWISE_SIGMOID, false>, L<FC_POINTWISE_SIGMOID, true>},                              \
   {L<FC_POINTWISE_TANH, false>, L<FC_POINTWISE_TANH, true>},                                    \
   {L<FC_POINTWISE_LEAKY_RELU, false>, L<FC_POINTWISE_LEAKY_RELU, true>},                        \
   {L<FC_POINTWISE_EXP, false>, L<FC_POINTWISE_EXP, true>},                                      \
   {L<FC_POINTWISE_CAUCHY_CDF, false>, L<FC_POINTWISE_CAUCHY_CDF, true>}}
static const PwLaunch kPwApply[5][2] = FC_PW_TABLE(pw_launch_apply);
static const PwLaunch kPwBackward[5][2] = FC_PW_TABLE(pw_launch_backward);
#undef FC_PW_TABLE

}  // namespace fc

using namespace fc;

extern "C" int fc_pointwise_apply(const float* x, int64_t x_row_stride, float* y, int64_t y_row_stride,
                                  float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int64_t D,
                                  const fc_pointwise_config* cfg, int32_t* status, void* stream) {
  if (pw_check_config(cfg, B, D) != FC_OK) return FC_ERR_INVALID_ARGUMENT;
  if (!x || !y || !logabsdet || x_row_stride < D || y_row_stride < D) return FC_ERR_INVALID_ARGUMENT;
  if (B == 0) return FC_OK;
  PwArgs a = {};
  a.x = x, a.xs = x_row_stride, a.y = y, a.ys = y_row_stride, a.lad = logabsdet, a.accumulate = accumulate_logabsdet;
  a.status = status, a.B = B, a.D = (int)D;
  pw_scalar_args(a, cfg);
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && (y_row_stride & 3) == 0 && pw_aligned16(x) &&
                   pw_aligned16(y);
  const int seg = lane_map((int)(vec ? D / 4 : D)).seg;
  const int64_t blocks = pw_blocks(B, seg);
  cudaStream_t st = (cudaStream_t)stream;
  kPwApply[cfg->op][cfg->inverse != 0](a, vec, false, blocks, seg, st);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int64_t fc_pointwise_workspace_floats(int64_t B, int64_t D) {
  if (B < 0 || D < 1) return FC_ERR_INVALID_ARGUMENT;
  const int64_t n = (B + kWarps - 1) / kWarps;  // a CTA covers at least kWarps rows per pass
  return n < 1 ? 1 : (n < kPwMaxBlocks ? n : kPwMaxBlocks);
}

extern "C" int fc_pointwise_backward(const float* x, int64_t x_row_stride, const float* grad_y, int64_t gy_row_stride,
                                     const float* grad_logabsdet, float* grad_x, int64_t gx_row_stride,
                                     float* grad_temperature, float* workspace, int64_t B, int64_t D,
                                     const fc_pointwise_config* cfg, void* stream) {
  if (pw_check_config(cfg, B, D) != FC_OK) return FC_ERR_INVALID_ARGUMENT;
  if (!x || !grad_x || x_row_stride < D || gx_row_stride < D || (grad_y && gy_row_stride < D))
    return FC_ERR_INVALID_ARGUMENT;
  const bool want_t = grad_temperature != nullptr;
  if (want_t && (cfg->op != FC_POINTWISE_SIGMOID || !workspace)) return FC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) {
    if (want_t && cudaMemsetAsync(grad_temperature, 0, sizeof(float), st) != cudaSuccess) return FC_ERR_CUDA;
    return FC_OK;
  }
  PwArgs a = {};
  a.x = x, a.xs = x_row_stride, a.gy = grad_y, a.gys = gy_row_stride, a.gl = grad_logabsdet, a.gx = grad_x;
  a.gxs = gx_row_stride, a.gt = grad_temperature, a.part = workspace, a.B = B, a.D = (int)D;
  pw_scalar_args(a, cfg);
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && (gx_row_stride & 3) == 0 && pw_aligned16(x) &&
                   pw_aligned16(grad_x) && (!grad_y || ((gy_row_stride & 3) == 0 && pw_aligned16(grad_y)));
  const int seg = lane_map((int)(vec ? D / 4 : D)).seg;
  const int64_t blocks = pw_blocks(B, seg);
  kPwBackward[cfg->op][cfg->inverse != 0](a, vec, want_t, blocks, seg, st);
  FC_CHECK_LAUNCH();
  if (want_t && blocks > 1) {
    pw_finish_kernel<<<1, 32, 0, st>>>(workspace, (int)blocks, grad_temperature);
    FC_CHECK_LAUNCH();
  }
  return FC_OK;
}
