// fc_lulinear.cu — the dense D x D map of LULinear (transforms/lu.py) for 1 <= D < 64:
//   forward   y = x · Mᵀ + c,   lad[b] = *logdet (or lad[b] += *logdet)
//   backward  grad_x = grad_y · M,   grad_M = grad_yᵀ · x,   grad_c = Σ_b grad_y[b]
// M, c and logdet are device data composed by the caller (the LU factors, their inverse, ±Σ log upper_diag), so nothing
// here synchronises with the host and a layer call can be captured into a CUDA graph.
//
// One streaming pass over row tiles.  A tile of TR rows is copied into shared memory TRANSPOSED (s[k * TRp + r]) with
// 4-byte cp.async (any row stride, any alignment, any D; two tiles in flight per CTA, so the next tile's loads overlap the
// current tile's arithmetic and stores).  The transposed layout is what the packed FMA wants: a lane reads four
// consecutive rows of one input column as one 16-byte load and pairs them in fp32x2 FMAs ((x[r], x[r+1]) * (w, w)), so per
// input column a warp issues NR + NC 16-byte shared loads for 8 * NR * NC FFMA2 — the loop is bound by the FMA pipe, not
// by shared-memory wavefronts (the trap described at made_kloop, fc_made_inverse.cuh).  The outputs are written over the
// warp's own rows of the tile and leave with coalesced stores in row order.
#include "fc_common.cuh"

namespace fc {

constexpr int kLuThreads = 256;
constexpr int kLuWarps = kLuThreads / 32;
constexpr int kLuMaxD = 63;
constexpr int kLuWCols = 64;          // output columns of the shared weight tile (zero beyond D)
constexpr int kLuTileFloats = 6144;   // input floats per tile (24 KB), rounded to whole passes

struct LuArgs {
  const float* x;       // [B, D], row stride xs
  const float* g;       // backward: grad_y [B, D], row stride gs
  const float* M;       // [D, D] row-major
  const float* c;       // forward: [D]
  const float* logdet;  // forward: device scalar
  float* y;             // forward: y; backward: grad_x  (row stride ys)
  float* lad;           // forward: [B]
  float* ws;            // backward: [gridDim.x][D * D + D] per-CTA partial sums
  int64_t xs, gs, ys, B, num_tiles;
  int D, TR, TRp, accumulate;
};

__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// rows [0, rows) of a row-major matrix with row stride ld -> s[k * TRp + r]; consecutive threads take consecutive
// elements in row order, so the global reads are coalesced whatever D is.
__device__ __forceinline__ void lu_load(float* s, const float* src, int64_t ld, int rows, int D, int TRp) {
  int r = threadIdx.x / D, k = threadIdx.x - r * D;
  const int dr = kLuThreads / D, dk = kLuThreads - dr * D;
  for (int i = threadIdx.x; i < rows * D; i += kLuThreads) {
    cp_async4(s + k * TRp + r, src + (int64_t)r * ld + k);
    r += dr, k += dk;
    if (k >= D) k -= D, ++r;
  }
}

__device__ __forceinline__ void lu_store(float* dst, int64_t ld, const float* s, int rows, int D, int TRp) {
  int r = threadIdx.x / D, k = threadIdx.x - r * D;
  const int dr = kLuThreads / D, dk = kLuThreads - dr * D;
  for (int i = threadIdx.x; i < rows * D; i += kLuThreads) {
    __stcs(dst + (int64_t)r * ld + k, s[k * TRp + r]);
    r += dr, k += dk;
    if (k >= D) k -= D, ++r;
  }
}

// Rows [rb, rb + 16 NR) of the tile, in place: s[j][r] <- cs[j] + Σ_k W[k][j] s[k][r].  Lane (g = lane & 7, q = lane >> 3)
// owns the output columns 32 c + 4 g + e (c < NC, e < 4) of the rows rb + 16 n + 4 q + i (n < NR, i < 4); acc[.][.][e][h]
// holds the row pair (2h, 2h + 1).  The 8 column groups of a warp read 128 contiguous bytes of W, the 4 row groups 64
// contiguous bytes of s: one wavefront per load.  Only the warp itself touches these rows, so __syncwarp orders the
// in-place write.
template <int NC, int NR>
__device__ __forceinline__ void lu_rows(float* s, const float* __restrict__ W, const float* __restrict__ cs, int D, int TRp,
                                        int rb, int lane) {
  const int g = lane & 7, q = lane >> 3;
  float2 acc[NR][NC][4][2];
#pragma unroll
  for (int c = 0; c < NC; ++c)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float b = cs[32 * c + 4 * g + e];
#pragma unroll
      for (int n = 0; n < NR; ++n) acc[n][c][e][0] = acc[n][c][e][1] = make_float2(b, b);
    }
  const float* xp = s + rb + 4 * q;
  const float* wp = W + 4 * g;
#pragma unroll 4
  for (int k = 0; k < D; ++k) {
    float4 xv[NR], wv[NC];
#pragma unroll
    for (int n = 0; n < NR; ++n) xv[n] = *reinterpret_cast<const float4*>(xp + k * TRp + 16 * n);
#pragma unroll
    for (int c = 0; c < NC; ++c) wv[c] = *reinterpret_cast<const float4*>(wp + k * kLuWCols + 32 * c);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const float w[4] = {wv[c].x, wv[c].y, wv[c].z, wv[c].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 w2 = make_float2(w[e], w[e]);
#pragma unroll
        for (int n = 0; n < NR; ++n) {
          acc[n][c][e][0] = __ffma2_rn(make_float2(xv[n].x, xv[n].y), w2, acc[n][c][e][0]);
          acc[n][c][e][1] = __ffma2_rn(make_float2(xv[n].z, xv[n].w), w2, acc[n][c][e][1]);
        }
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < NC; ++c)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = 32 * c + 4 * g + e;
      if (j < D) {
#pragma unroll
        for (int n = 0; n < NR; ++n)
          *reinterpret_cast<float4*>(s + j * TRp + rb + 16 * n + 4 * q) =
              make_float4(acc[n][c][e][0].x, acc[n][c][e][0].y, acc[n][c][e][1].x, acc[n][c][e][1].y);
      }
    }
  __syncwarp();
}

// Shared memory: W [D][64] (W[k][j]: weight of input k in output j), cs [64], then 2 stages of the tile (backward: x and
// grad_y).  Forward W[k][j] = M[j][k]; backward (grad_x = grad_y · M) W[j][k] = M[j][k].
template <int NC, int NR, bool kBwd>
__global__ void __launch_bounds__(kLuThreads, kBwd ? 1 : 2) lulinear_kernel(const LuArgs a) {
  extern __shared__ __align__(16) float lu_sm[];
  const int D = a.D, TR = a.TR, TRp = a.TRp;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* const W = lu_sm;
  float* const cs = W + D * kLuWCols;
  float* const tiles = cs + kLuWCols;
  const int stage_floats = (kBwd ? 2 : 1) * D * TRp;
  const int64_t nt = a.num_tiles;

  auto issue = [&](int64_t t, int stage) {
    if (t < nt) {
      const int64_t row0 = t * TR;
      const int rows = (int)min((int64_t)TR, a.B - row0);
      float* st = tiles + stage * stage_floats;
      lu_load(st, a.x + row0 * a.xs, a.xs, rows, D, TRp);
      if (kBwd) lu_load(st + D * TRp, a.g + row0 * a.gs, a.gs, rows, D, TRp);
    }
    cp_async_commit();  // an empty group when there is no tile: the wait counts below stay uniform
  };
  issue(blockIdx.x, 0);
  issue(blockIdx.x + gridDim.x, 1);

  for (int i = threadIdx.x; i < D * kLuWCols; i += kLuThreads) {
    const int k = i / kLuWCols, j = i - k * kLuWCols;
    W[i] = j < D ? __ldg(a.M + (kBwd ? k * D + j : j * D + k)) : 0.f;
  }
  for (int j = threadIdx.x; j < kLuWCols; j += kLuThreads) cs[j] = (!kBwd && j < D) ? __ldg(a.c + j) : 0.f;
  const float logdet = kBwd ? 0.f : __ldg(a.logdet);

  // backward: lane block (jb, kb) of the NB x NB blocks of 4 x 4 entries of grad_M, row split sp of S (rows 4 sp, 4 sp + 4 S, ...)
  const int NB = (D + 3) >> 2, NB2 = NB * NB;
  const int S = kBwd ? max(1, kLuThreads / NB2) : 1;
  const int blk = threadIdx.x % NB2, sp = threadIdx.x / NB2;
  const int jb = blk / NB, kb = blk - jb * NB;
  const bool gm_thread = kBwd && sp < S;
  float2 gacc[4][4];
  float gcacc[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    gcacc[u] = 0.f;
#pragma unroll
    for (int v = 0; v < 4; ++v) gacc[u][v] = make_float2(0.f, 0.f);
  }

  constexpr int kPass = 16 * NR * kLuWarps;
  int it = 0;
  for (int64_t t = blockIdx.x; t < nt; t += gridDim.x, ++it) {
    const int stage = it & 1;
    const int64_t row0 = t * TR;
    const int rows = (int)min((int64_t)TR, a.B - row0);
    float* const sx = tiles + stage * stage_floats;
    float* const so = kBwd ? sx + D * TRp : sx;  // the tile the outputs are computed from and written over
    cp_async_wait1();
    __syncthreads();

    if (kBwd) {
      if (gm_thread) {
        for (int r = 4 * sp; r < rows; r += 4 * S) {
          float4 gv[4], xv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int j = 4 * jb + u, k = 4 * kb + u;
            gv[u] = j < D ? *reinterpret_cast<const float4*>(so + j * TRp + r) : make_float4(0.f, 0.f, 0.f, 0.f);
            xv[u] = k < D ? *reinterpret_cast<const float4*>(sx + k * TRp + r) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          if (r + 4 > rows) {  // ragged last quad: the rows past the end hold stale data
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              if (r + 1 >= rows) gv[u].y = xv[u].y = 0.f;
              if (r + 2 >= rows) gv[u].z = xv[u].z = 0.f;
              gv[u].w = xv[u].w = 0.f;
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int v = 0; v < 4; ++v) {
              gacc[u][v] = __ffma2_rn(make_float2(gv[u].x, gv[u].y), make_float2(xv[v].x, xv[v].y), gacc[u][v]);
              gacc[u][v] = __ffma2_rn(make_float2(gv[u].z, gv[u].w), make_float2(xv[v].z, xv[v].w), gacc[u][v]);
            }
            gcacc[u] += (gv[u].x + gv[u].y) + (gv[u].z + gv[u].w);
          }
        }
      }
      __syncthreads();  // grad_M has read the tile before grad_x overwrites grad_y
    }

    for (int rb = warp * 16 * NR; rb < rows; rb += kPass) lu_rows<NC, NR>(so, W, cs, D, TRp, rb, lane);
    __syncthreads();
    lu_store(a.y + row0 * a.ys, a.ys, so, rows, D, TRp);
    if (!kBwd)
      for (int r = threadIdx.x; r < rows; r += kLuThreads) {
        float* l = a.lad + row0 + r;
        *l = a.accumulate ? *l + logdet : logdet;
      }
    __syncthreads();  // the stage is read out before it is refilled
    issue(t + 2 * (int64_t)gridDim.x, stage);
  }

  if (kBwd) {
    // the S row splits of every entry, summed in split order (deterministic), then one partial per entry for this CTA
    cp_async_wait0();
    __syncthreads();
    float* red = tiles;                   // [S][NB2][16]
    float* gcred = tiles + S * NB2 * 16;  // [S][NB][4]
    if (gm_thread) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int v = 0; v < 4; ++v) red[(sp * NB2 + blk) * 16 + u * 4 + v] = gacc[u][v].x + gacc[u][v].y;
        if (kb == 0) gcred[(sp * NB + jb) * 4 + u] = gcacc[u];
      }
    }
    __syncthreads();
    float* out = a.ws + (size_t)blockIdx.x * (D * D + D);
    for (int e = threadIdx.x; e < NB2 * 16; e += kLuThreads) {
      const int b = e >> 4, u = (e >> 2) & 3, v = e & 3;
      const int j = 4 * (b / NB) + u, k = 4 * (b % NB) + v;
      if (j < D && k < D) {
        float sum = 0.f;
        for (int s = 0; s < S; ++s) sum += red[(s * NB2 + b) * 16 + u * 4 + v];
        out[j * D + k] = sum;
      }
    }
    for (int j = threadIdx.x; j < D; j += kLuThreads) {
      float sum = 0.f;
      for (int s = 0; s < S; ++s) sum += gcred[s * NB * 4 + j];
      out[D * D + j] = sum;
    }
  }
}

// Second stage of the backward: one CTA per entry of [grad_M | grad_c] sums the per-CTA partials in a fixed order
// (strided partial sums per thread, then shuffles and one thread over the warps), as actnorm_finish_kernel does, so replays
// of a captured training step stay bitwise equal.
constexpr int kLuFinishThreads = 128;
__global__ void __launch_bounds__(kLuFinishThreads) lulinear_finish_kernel(const float* ws, int blocks, int D,
                                                                           float* grad_M, float* grad_c) {
  const int e = blockIdx.x, n = D * D + D;
  float t = 0.f;
  for (int b = threadIdx.x; b < blocks; b += kLuFinishThreads) t += ws[(size_t)b * n + e];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  __shared__ float parts[kLuFinishThreads / 32];
  if ((threadIdx.x & 31) == 0) parts[threadIdx.x >> 5] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < kLuFinishThreads / 32; ++w) s += parts[w];
    if (e < D * D) grad_M[e] = s;
    else grad_c[e - D * D] = s;
  }
}

struct LuPlan {
  int TR, TRp, grid;
  size_t smem;
  int64_t num_tiles;
};

// Tile rows: whole passes of the CTA (128 rows for D > 32, 256 below), about kLuTileFloats inputs.  CTAs: forward as many
// per SM (at most 2) as the shared memory allows; backward one (its grad_M accumulators take 160-170 registers), all of
// them resident.  The grid depends only on (B, D, the device), so the backward's workspace size is known before the launch.
static LuPlan lu_plan(int64_t B, int D, bool bwd) {
  LuPlan p;
  const int pass = 16 * kLuWarps * (D <= 32 ? 2 : 1);
  p.TR = (kLuTileFloats / D) / pass * pass;
  if (p.TR < pass) p.TR = pass;
  p.TRp = p.TR + 4;  // ≡ 4 (mod 32): the 16-byte rows of different columns start in different banks
  p.smem = sizeof(float) * ((size_t)D * kLuWCols + kLuWCols + (size_t)2 * (bwd ? 2 : 1) * D * p.TRp);
  int per_sm = (int)((size_t)(227 * 1024) / (p.smem + 1024));
  per_sm = (bwd || per_sm < 1) ? 1 : (per_sm > 2 ? 2 : per_sm);
  p.num_tiles = (B + p.TR - 1) / p.TR;
  const int64_t cap = (int64_t)device_info().sm_count * per_sm;
  p.grid = (int)(p.num_tiles < cap ? (p.num_tiles < 1 ? 1 : p.num_tiles) : cap);
  return p;
}

template <bool kBwd>
static int lu_launch(const LuArgs& a, const LuPlan& p, cudaStream_t st) {
  auto kern = a.D <= 32 ? lulinear_kernel<1, 2, kBwd> : lulinear_kernel<2, 1, kBwd>;
  if (p.smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem) != cudaSuccess)
    return FC_ERR_CUDA;
  kern<<<p.grid, kLuThreads, p.smem, st>>>(a);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

}  // namespace fc

using namespace fc;

extern "C" int fc_lulinear_apply(const float* x, int64_t x_row_stride, const float* M, const float* c,
                                 const float* logdet, float* y, int64_t y_row_stride, float* logabsdet,
                                 int32_t accumulate_logabsdet, int64_t B, int32_t D, void* stream) {
  if (B < 0 || D < 1 || D > kLuMaxD || !M || !c || !logdet) return FC_ERR_INVALID_ARGUMENT;
  if (B == 0) return FC_OK;
  if (!x || !y || !logabsdet || x_row_stride < D || y_row_stride < D) return FC_ERR_INVALID_ARGUMENT;
  const LuPlan p = lu_plan(B, D, false);
  LuArgs a = {};
  a.x = x; a.M = M; a.c = c; a.logdet = logdet; a.y = y; a.lad = logabsdet;
  a.xs = x_row_stride; a.ys = y_row_stride; a.B = B; a.num_tiles = p.num_tiles;
  a.D = D; a.TR = p.TR; a.TRp = p.TRp; a.accumulate = accumulate_logabsdet != 0;
  return lu_launch<false>(a, p, (cudaStream_t)stream);
}

extern "C" int64_t fc_lulinear_workspace_floats(int64_t B, int32_t D) {
  if (B < 0 || D < 1 || D > kLuMaxD) return FC_ERR_INVALID_ARGUMENT;
  return (int64_t)lu_plan(B, D, true).grid * (D * D + D);
}

extern "C" int fc_lulinear_backward(const float* x, int64_t x_row_stride, const float* M, const float* grad_y,
                                    int64_t gy_row_stride, float* grad_x, int64_t gx_row_stride, float* grad_M,
                                    float* grad_c, float* workspace, int64_t B, int32_t D, void* stream) {
  if (B < 0 || D < 1 || D > kLuMaxD || !M || !grad_M || !grad_c) return FC_ERR_INVALID_ARGUMENT;
  if (B > 0 && (!x || !grad_y || !grad_x || !workspace || x_row_stride < D || gy_row_stride < D || gx_row_stride < D))
    return FC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) {
    if (cudaMemsetAsync(grad_M, 0, sizeof(float) * D * D, st) != cudaSuccess) return FC_ERR_CUDA;
    if (cudaMemsetAsync(grad_c, 0, sizeof(float) * D, st) != cudaSuccess) return FC_ERR_CUDA;
    return FC_OK;
  }
  const LuPlan p = lu_plan(B, D, true);
  LuArgs a = {};
  a.x = x; a.g = grad_y; a.M = M; a.y = grad_x; a.ws = workspace;
  a.xs = x_row_stride; a.gs = gy_row_stride; a.ys = gx_row_stride; a.B = B; a.num_tiles = p.num_tiles;
  a.D = D; a.TR = p.TR; a.TRp = p.TRp;
  const int rc = lu_launch<true>(a, p, st);
  if (rc != FC_OK) return rc;
  lulinear_finish_kernel<<<D * D + D, kLuFinishThreads, 0, st>>>(workspace, p.grid, D, grad_M, grad_c);
  FC_CHECK_LAUNCH();
  return FC_OK;
}
