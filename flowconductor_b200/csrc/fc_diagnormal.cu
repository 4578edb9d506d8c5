// fc_diagnormal.cu — diagonal Gaussian base densities (DiagonalNormal, ConditionalDiagonalNormal,
// flowcon/distributions/normal.py).
//
// One parameter format: P [C, 2D] row-major with any row stride (>= 2D), means in columns [0, D), log standard
// deviations in columns [D, 2D) (the blocked layout of the reference's `_compute_params`; a context encoder's output is
// read in place).  Data row r uses parameter row r / G, G the group size: G = 1 for the conditional log-density, G = n
// for n draws per context row, G = R for one shared row (DiagonalNormal).  The last group may be partial.
//   log_prob   out[r] = −½ Σ_d z² − Σ_d s − log_z (+ logabsdet[r]),   z = (x − m) · e^{−s}
//   sample     y[r]   = m + e^{s} · ε[r]
// The backward kernels reduce the parameter gradients over the rows of each group without atomics:
//   per lane  (G <= kDnLaneG): one row lane walks every row of a group in order and writes the group's gradient;
//   segments  (G > kDnLaneG):  a CTA owns a run of rows inside one group; its row lanes are summed in a fixed order and
//             written directly when the run is the whole group, else to a workspace row that dn_finish_kernel sums in a
//             fixed order (the ActNorm / BatchNorm scheme).  Two calls are bitwise equal.
// Layout as fc_batchnorm.cu: thread (tx, ty) owns the V-wide column groups tx, tx + cw, ... (V = 4: 128-bit accesses
// when D, the strides and the pointers allow) of the rows ty, ty + ry, ...; wider rows are walked in column tiles of
// cw · V, so any D works.
#include "fc_common.cuh"

namespace fc {

constexpr int kDnThreads = 256;
constexpr int64_t kDnLaneG = 32;       // largest group reduced by one row lane
constexpr int64_t kDnSegRows = 256;    // least rows per segment of a large group

enum DnKernel { kDnLogProbBwd = 0, kDnSampleBwd = 1 };

struct DnArgs {
  const float* x;    // log_prob: x; sample: noise ε
  const float* p;    // parameters [C, 2D]
  const float* g;    // log_prob backward: upstream gradient [R]; sample backward: grad_samples [R, D]
  const float* lad;  // log_prob: optional logabsdet [R]
  float* out;        // log_prob: [R]; sample: samples; log_prob backward: grad_x
  float* gp;         // backward: grad_params [C, 2D] (dense)
  float* ws;         // backward, segments: [C · nseg][2D]
  int64_t xs, ps, gs, outs;
  int64_t R, G, C, nseg, seg_rows, units_per_block;
  int D, cw;
  float log_z;
};

// parameter row of data row r; 32-bit division whenever the row index allows it
__device__ __forceinline__ int64_t dn_prow(int64_t r, int64_t G) {
  if (G == 1) return r;
  if (((uint64_t)r | (uint64_t)G) <= 0xffffffffull) return (int64_t)((uint32_t)r / (uint32_t)G);
  return r / G;
}

template <int V>
__device__ __forceinline__ void dn_load(float (&v)[V], const float* p) {
  if constexpr (V == 4) {
    *reinterpret_cast<float4*>(v) = __ldg(reinterpret_cast<const float4*>(p));
  } else {
    v[0] = __ldg(p);
  }
}

template <int V>
__device__ __forceinline__ void dn_load_cs(float (&v)[V], const float* p) {
  if constexpr (V == 4) {
    *reinterpret_cast<float4*>(v) = __ldcs(reinterpret_cast<const float4*>(p));
  } else {
    v[0] = __ldcs(p);
  }
}

template <int V>
__device__ __forceinline__ void dn_store(float* p, const float (&v)[V]) {
  if constexpr (V == 4) {
    __stcs(reinterpret_cast<float4*>(p), *reinterpret_cast<const float4*>(v));
  } else {
    __stcs(p, v[0]);
  }
}

// log_prob: seg = min(32, next_pow2(D / V)) lanes per row (lane_map), a warp covers 32 / seg rows per pass; the row's
// two sums are xor-shuffle reductions over its lanes.
template <int V>
__global__ void __launch_bounds__(kDnThreads) dn_log_prob_kernel(const DnArgs a, int seg) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rpw = 32 / seg, sub = lane / seg, j0 = lane % seg;
  const int64_t groups = (a.R + rpw - 1) / rpw;
  const int D = a.D;
  for (int64_t w = (int64_t)blockIdx.x * kWarps + warp; w < groups; w += (int64_t)gridDim.x * kWarps) {
    const int64_t row = w * rpw + sub;
    const bool row_ok = row < a.R;
    float zz = 0.f, ss = 0.f;
    if (row_ok) {
      const float* xr = a.x + row * a.xs;
      const float* pr = a.p + dn_prow(row, a.G) * a.ps;
      for (int d = j0 * V; d < D; d += seg * V) {
        float xv[V], m[V], s[V];
        dn_load_cs<V>(xv, xr + d);
        dn_load<V>(m, pr + d);
        dn_load<V>(s, pr + D + d);
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float z = (xv[v] - m[v]) * expf(-s[v]);
          zz = fmaf(z, z, zz);
          ss += s[v];
        }
      }
    }
    zz = seg_reduce_sum(zz, seg);
    ss = seg_reduce_sum(ss, seg);
    if (row_ok && j0 == 0) {
      const float lp = (-0.5f * zz - ss) - a.log_z;  // the reference's order: −½Σz², −= Σs, −= log_z
      a.out[row] = a.lad ? lp + a.lad[row] : lp;
    }
  }
}

// sample: element-wise over the CTA's rows [r_lo, r_hi) (units_per_block rows per CTA).
template <int V>
__global__ void __launch_bounds__(kDnThreads) dn_sample_kernel(const DnArgs a) {
  const int cw = a.cw, ry = kDnThreads / cw, tx = threadIdx.x % cw, ty = threadIdx.x / cw, D = a.D;
  if (ty >= ry) return;
  const int64_t r_lo = (int64_t)blockIdx.x * a.units_per_block;
  const int64_t r_hi = r_lo + a.units_per_block < a.R ? r_lo + a.units_per_block : a.R;
  for (int64_t r = r_lo + ty; r < r_hi; r += ry) {
    const float* pr = a.p + dn_prow(r, a.G) * a.ps;
    for (int d = tx * V; d < D; d += cw * V) {
      float e[V], m[V], s[V], y[V];
      dn_load_cs<V>(e, a.x + r * a.xs + d);
      dn_load<V>(m, pr + d);
      dn_load<V>(s, pr + D + d);
#pragma unroll
      for (int v = 0; v < V; ++v) y[v] = fmaf(expf(s[v]), e[v], m[v]);
      dn_store<V>(a.out + r * a.outs + d, y);
    }
  }
}

// One row's contribution at columns [d, d + V): accumulates (grad_mean, grad_log_std) and, for the log_prob backward,
// writes grad_x.
template <int K, int V>
__device__ __forceinline__ void dn_row(const DnArgs& a, int64_t r, const float* pr, int d, float (&am)[V],
                                       float (&as)[V]) {
  float xv[V], m[V], s[V];
  dn_load_cs<V>(xv, a.x + r * a.xs + d);
  dn_load<V>(s, pr + a.D + d);
  if constexpr (K == kDnLogProbBwd) {
    dn_load<V>(m, pr + d);
    const float g = __ldg(a.g + r);
    float gx[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const float e = expf(-s[v]);
      const float z = (xv[v] - m[v]) * e;
      const float gz = g * z * e;
      gx[v] = -gz;
      am[v] += gz;
      as[v] = fmaf(g, fmaf(z, z, -1.f), as[v]);
    }
    dn_store<V>(a.out + r * a.outs + d, gx);
  } else {
    float gy[V];
    dn_load_cs<V>(gy, a.g + r * a.gs + d);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      am[v] += gy[v];
      as[v] = fmaf(gy[v] * expf(s[v]), xv[v], as[v]);
    }
  }
}

template <int V>
__device__ __forceinline__ void dn_put(float* dst, int D, int d, const float (&am)[V], const float (&as)[V]) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    dst[d + v] = am[v];
    dst[D + d + v] = as[v];
  }
}

// Backward.  lane mode (nseg == 0): CTA b owns groups [b U, (b + 1) U), row lane ty walks groups ty, ty + ry, ...
// segment mode: CTA b owns segment b % nseg of group b / nseg (seg_rows rows).
template <int K, int V>
__global__ void __launch_bounds__(kDnThreads) dn_backward_kernel(const DnArgs a) {
  __shared__ float red[2][kDnThreads * 4];
  const int cw = a.cw, ry = kDnThreads / cw, tx = threadIdx.x % cw, ty = threadIdx.x / cw, D = a.D;
  if (a.nseg == 0) {
    if (ty >= ry) return;
    const int64_t c_lo = (int64_t)blockIdx.x * a.units_per_block;
    const int64_t c_hi = c_lo + a.units_per_block < a.C ? c_lo + a.units_per_block : a.C;
    for (int64_t c = c_lo + ty; c < c_hi; c += ry) {
      const float* pr = a.p + c * a.ps;
      const int64_t r_lo = c * a.G, r_hi = r_lo + a.G < a.R ? r_lo + a.G : a.R;
      for (int d = tx * V; d < D; d += cw * V) {
        float am[V], as[V];
#pragma unroll
        for (int v = 0; v < V; ++v) am[v] = as[v] = 0.f;
#pragma unroll 4
        for (int64_t r = r_lo; r < r_hi; ++r) dn_row<K, V>(a, r, pr, d, am, as);
        dn_put<V>(a.gp + c * 2 * D, D, d, am, as);
      }
    }
    return;
  }
  const int64_t c = blockIdx.x / a.nseg, k = blockIdx.x % a.nseg;
  const float* pr = a.p + c * a.ps;
  const int64_t g_hi = (c + 1) * a.G < a.R ? (c + 1) * a.G : a.R;
  const int64_t r_lo = c * a.G + k * a.seg_rows;
  const int64_t r_hi = r_lo + a.seg_rows < g_hi ? r_lo + a.seg_rows : g_hi;
  float* dst = a.nseg == 1 ? a.gp + c * 2 * D : a.ws + (size_t)blockIdx.x * 2 * D;
  const int tile = cw * V;
  for (int d0 = 0; d0 < D; d0 += tile) {
    const int d = d0 + tx * V;
    float am[V], as[V];
#pragma unroll
    for (int v = 0; v < V; ++v) am[v] = as[v] = 0.f;
    if (ty < ry && d < D) {
#pragma unroll 2
      for (int64_t r = r_lo + ty; r < r_hi; r += ry) dn_row<K, V>(a, r, pr, d, am, as);
    }
    if (ty < ry) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        red[0][ty * tile + tx * V + v] = am[v];
        red[1][ty * tile + tx * V + v] = as[v];
      }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * tile; t += kDnThreads) {  // the row lanes summed in order
      const int h = t / tile, col = t % tile;
      if (d0 + col < D) {
        float sum = 0.f;
        for (int y = 0; y < ry; ++y) sum += red[h][y * tile + col];
        dst[h * D + d0 + col] = sum;
      }
    }
    __syncthreads();
  }
}

// One warp per output (c, column of 2D): the nseg segment partials, lane-strided, then a fixed xor tree.
__global__ void __launch_bounds__(kDnThreads) dn_finish_kernel(const float* ws, float* gp, int64_t C, int64_t nseg,
                                                               int D) {
  const int64_t w = ((int64_t)blockIdx.x * kDnThreads + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= C * 2 * D) return;  // whole warps leave together
  const int64_t c = w / (2 * D);
  const int col = (int)(w % (2 * D));
  float sum = 0.f;
  for (int64_t k = lane; k < nseg; k += 32) sum += ws[(size_t)(c * nseg + k) * 2 * D + col];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) gp[c * 2 * D + col] = sum;
}

static bool dn_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int dn_cap() { return 8 * device_info().sm_count; }

// Segments per group for the backward (0: lane mode).
static int64_t dn_nseg(int64_t R, int64_t G) {
  if (G <= kDnLaneG) return 0;
  const int64_t C = (R + G - 1) / G;
  int64_t want = (G + kDnSegRows - 1) / kDnSegRows;
  const int64_t fill = (dn_cap() + C - 1) / C;  // enough CTAs to fill the device, no more
  if (want > fill) want = fill;
  return want < 1 ? 1 : want;
}

static void dn_layout(DnArgs& a, bool vec) {
  const int nv = vec ? a.D / 4 : a.D;
  a.cw = nv < kDnThreads ? nv : kDnThreads;
}

// CTAs for `units` rows (or groups) handled `ry` at a time: at least 128 rows' worth each, at most 8 CTAs per SM.
static int64_t dn_blocks(int64_t units, int64_t rows_per_unit) {
  const int64_t rows = units * rows_per_unit;
  int64_t want = (rows + 127) / 128;
  if (want > dn_cap()) want = dn_cap();
  if (want > units) want = units;
  return want < 1 ? 1 : want;
}

}  // namespace fc

using namespace fc;

extern "C" int fc_diagnormal_log_prob(const float* x, int64_t x_row_stride, const float* params,
                                      int64_t params_row_stride, const float* logabsdet, float* out, int64_t R,
                                      int32_t D, int64_t group, void* stream) {
  if (R < 0 || D < 1 || group < 1) return FC_ERR_INVALID_ARGUMENT;
  if (R == 0) return FC_OK;
  if (!x || !params || !out || x_row_stride < D || (params_row_stride < 2 * (int64_t)D && R > group))
    return FC_ERR_INVALID_ARGUMENT;
  DnArgs a = {};
  a.x = x, a.xs = x_row_stride, a.p = params, a.ps = params_row_stride, a.lad = logabsdet, a.out = out;
  a.R = R, a.D = D, a.G = group;
  a.log_z = (float)(0.5 * (double)D * log(2.0 * 3.14159265358979323846));  // the fp64 buffer, applied in fp32
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && (params_row_stride & 3) == 0 && dn_aligned16(x) &&
                   dn_aligned16(params);
  const int seg = lane_map(vec ? D / 4 : D).seg;
  int64_t blocks = (R + (32 / seg) * kWarps - 1) / ((32 / seg) * kWarps);
  if (blocks > dn_cap()) blocks = dn_cap();
  cudaStream_t st = (cudaStream_t)stream;
  if (vec)
    dn_log_prob_kernel<4><<<(int)blocks, kDnThreads, 0, st>>>(a, seg);
  else
    dn_log_prob_kernel<1><<<(int)blocks, kDnThreads, 0, st>>>(a, seg);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int fc_diagnormal_sample(const float* noise, int64_t noise_row_stride, const float* params,
                                    int64_t params_row_stride, float* samples, int64_t samples_row_stride, int64_t R,
                                    int32_t D, int64_t group, void* stream) {
  if (R < 0 || D < 1 || group < 1) return FC_ERR_INVALID_ARGUMENT;
  if (R == 0) return FC_OK;
  if (!noise || !params || !samples || noise_row_stride < D || samples_row_stride < D ||
      (params_row_stride < 2 * (int64_t)D && R > group))
    return FC_ERR_INVALID_ARGUMENT;
  DnArgs a = {};
  a.x = noise, a.xs = noise_row_stride, a.p = params, a.ps = params_row_stride, a.out = samples;
  a.outs = samples_row_stride, a.R = R, a.D = D, a.G = group;
  const bool vec = (D & 3) == 0 && (noise_row_stride & 3) == 0 && (params_row_stride & 3) == 0 &&
                   (samples_row_stride & 3) == 0 && dn_aligned16(noise) && dn_aligned16(params) &&
                   dn_aligned16(samples);
  dn_layout(a, vec);
  const int64_t blocks = dn_blocks(R, 1);
  a.units_per_block = (R + blocks - 1) / blocks;
  cudaStream_t st = (cudaStream_t)stream;
  if (vec)
    dn_sample_kernel<4><<<(int)blocks, kDnThreads, 0, st>>>(a);
  else
    dn_sample_kernel<1><<<(int)blocks, kDnThreads, 0, st>>>(a);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int64_t fc_diagnormal_workspace_floats(int64_t R, int32_t D, int64_t group) {
  if (R < 0 || D < 1 || group < 1) return FC_ERR_INVALID_ARGUMENT;
  const int64_t nseg = dn_nseg(R, group);
  if (nseg <= 1) return 0;
  return ((R + group - 1) / group) * nseg * 2 * (int64_t)D;
}

template <int K>
static int dn_backward(DnArgs& a, bool vec, float* grad_params, float* workspace, cudaStream_t st) {
  const int64_t C = (a.R + a.G - 1) / a.G;
  a.C = C, a.gp = grad_params, a.ws = workspace;
  a.nseg = dn_nseg(a.R, a.G);
  if (a.nseg > 1 && !workspace) return FC_ERR_INVALID_ARGUMENT;
  dn_layout(a, vec);
  int64_t blocks;
  if (a.nseg == 0) {
    blocks = dn_blocks(C, a.G);
    a.units_per_block = (C + blocks - 1) / blocks;
  } else {
    a.seg_rows = (a.G + a.nseg - 1) / a.nseg;
    blocks = C * a.nseg;
  }
  if (blocks > 0x7fffffff) return FC_ERR_UNSUPPORTED;
  auto kern = vec ? dn_backward_kernel<K, 4> : dn_backward_kernel<K, 1>;
  kern<<<(unsigned)blocks, kDnThreads, 0, st>>>(a);
  FC_CHECK_LAUNCH();
  if (a.nseg > 1) {
    const int64_t warps = C * 2 * a.D, fblocks = (warps * 32 + kDnThreads - 1) / kDnThreads;
    if (fblocks > 0x7fffffff) return FC_ERR_UNSUPPORTED;
    dn_finish_kernel<<<(unsigned)fblocks, kDnThreads, 0, st>>>(workspace, grad_params, C, a.nseg, a.D);
    FC_CHECK_LAUNCH();
  }
  return FC_OK;
}

extern "C" int fc_diagnormal_log_prob_backward(const float* x, int64_t x_row_stride, const float* params,
                                               int64_t params_row_stride, const float* grad_out, float* grad_x,
                                               int64_t gx_row_stride, float* grad_params, float* workspace, int64_t R,
                                               int32_t D, int64_t group, void* stream) {
  if (R < 0 || D < 1 || group < 1) return FC_ERR_INVALID_ARGUMENT;
  if (R == 0) return FC_OK;
  if (!x || !params || !grad_out || !grad_x || !grad_params || x_row_stride < D || gx_row_stride < D ||
      (params_row_stride < 2 * (int64_t)D && R > group))
    return FC_ERR_INVALID_ARGUMENT;
  DnArgs a = {};
  a.x = x, a.xs = x_row_stride, a.p = params, a.ps = params_row_stride, a.g = grad_out, a.out = grad_x;
  a.outs = gx_row_stride, a.R = R, a.D = D, a.G = group;
  const bool vec = (D & 3) == 0 && (x_row_stride & 3) == 0 && (params_row_stride & 3) == 0 &&
                   (gx_row_stride & 3) == 0 && dn_aligned16(x) && dn_aligned16(params) && dn_aligned16(grad_x);
  return dn_backward<kDnLogProbBwd>(a, vec, grad_params, workspace, (cudaStream_t)stream);
}

extern "C" int fc_diagnormal_sample_backward(const float* noise, int64_t noise_row_stride, const float* params,
                                             int64_t params_row_stride, const float* grad_samples, int64_t gs_row_stride,
                                             float* grad_params, float* workspace, int64_t R, int32_t D, int64_t group,
                                             void* stream) {
  if (R < 0 || D < 1 || group < 1) return FC_ERR_INVALID_ARGUMENT;
  if (R == 0) return FC_OK;
  if (!noise || !params || !grad_samples || !grad_params || noise_row_stride < D || gs_row_stride < D ||
      (params_row_stride < 2 * (int64_t)D && R > group))
    return FC_ERR_INVALID_ARGUMENT;
  DnArgs a = {};
  a.x = noise, a.xs = noise_row_stride, a.p = params, a.ps = params_row_stride, a.g = grad_samples;
  a.gs = gs_row_stride, a.R = R, a.D = D, a.G = group;
  const bool vec = (D & 3) == 0 && (noise_row_stride & 3) == 0 && (params_row_stride & 3) == 0 &&
                   (gs_row_stride & 3) == 0 && dn_aligned16(noise) && dn_aligned16(params) &&
                   dn_aligned16(grad_samples);
  return dn_backward<kDnSampleBwd>(a, vec, grad_params, workspace, (cudaStream_t)stream);
}
