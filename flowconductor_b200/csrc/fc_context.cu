// fc_context.cu — the context terms of a conditional conditioner, g = ctx Wc^T + bc for every context layer of the net
// at once (DESIGN.md 4.12, "context terms"), for contexts narrower than the tensor-core GEMM's minimum reduction.
//
// Wc stacks the `context_layer`s of a ResidualNet (resnet.py:24-25, one per block) or a residual MADE (made.py:121-122 and
// one per block, made.py:139-140); the fused conditioner kernel reads the terms in the T128 layout (one row thread owns a
// row, so a warp reads 512 contiguous bytes per float4), and this kernel writes that layout directly.
//
// One CTA = one 128-row tile, one thread = one row: the row's C context values sit in registers, the weights of 32 output
// columns at a time in shared memory (every thread reads the same word: broadcast).  fp32 FMA chains in k order: the
// precision of an fp32 GEMM (the tensor-core path of fc_linear.cu takes over from C = 64 on, tc_autograd.MIN_K).
#include "fc_common.cuh"

namespace fc {

constexpr int kCtxRows = 128;
constexpr int kCtxCols = 32;  // output columns per weight chunk

template <int CP>  // context width padded to a multiple of 16
__global__ void __launch_bounds__(kCtxRows) context_terms_kernel(const float* __restrict__ ctx, long long ldc, long long B,
                                                                 int C, const float* __restrict__ W,
                                                                 const float* __restrict__ bias, int T,
                                                                 float* __restrict__ out) {
  __shared__ float xs[kCtxRows * (CP + 1)];  // odd row pitch: thread r reads word r (CP + 1) + k without bank conflicts
  __shared__ __align__(16) float ws[kCtxCols * CP];
  __shared__ float bs[kCtxCols];
  const int r = threadIdx.x;
  const long long row0 = (long long)blockIdx.x * kCtxRows;
  const int rows = (int)min((long long)kCtxRows, B - row0);
  for (int i = r; i < kCtxRows * C; i += kCtxRows) {
    const int rr = i / C, k = i - rr * C;
    xs[rr * (CP + 1) + k] = rr < rows ? ctx[(row0 + rr) * ldc + k] : 0.f;
  }
  for (int i = r; i < kCtxRows * (CP - C); i += kCtxRows) {
    const int rr = i / (CP - C), k = C + i - rr * (CP - C);
    xs[rr * (CP + 1) + k] = 0.f;
  }
  __syncthreads();
  float x[CP];
#pragma unroll
  for (int k = 0; k < CP; ++k) x[k] = xs[r * (CP + 1) + k];
  float* const tile = out + (long long)blockIdx.x * kCtxRows * T;
  for (int n0 = 0; n0 < T; n0 += kCtxCols) {
    const int nc = min(kCtxCols, T - n0);
    __syncthreads();  // the previous chunk's weights have been read
    for (int i = r; i < kCtxCols * CP; i += kCtxRows) {
      const int j = i / CP, k = i - j * CP;
      ws[i] = (j < nc && k < C) ? W[(long long)(n0 + j) * C + k] : 0.f;
    }
    if (r < kCtxCols) bs[r] = (r < nc && bias) ? bias[n0 + r] : 0.f;
    __syncthreads();
    if (r >= rows) continue;
    for (int j0 = 0; j0 < nc; j0 += 4) {
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4* w4 = reinterpret_cast<const float4*>(ws + (j0 + i) * CP);
        float acc = bs[j0 + i];
#pragma unroll
        for (int k4 = 0; k4 < CP / 4; ++k4) {
          const float4 w = w4[k4];
          acc = fmaf(x[4 * k4 + 0], w.x, acc);
          acc = fmaf(x[4 * k4 + 1], w.y, acc);
          acc = fmaf(x[4 * k4 + 2], w.z, acc);
          acc = fmaf(x[4 * k4 + 3], w.w, acc);
        }
        v[i] = acc;
      }
      // T128: element (r, c) at ((c / 4) * 128 + r) * 4 + c % 4 inside the tile
      reinterpret_cast<float4*>(tile)[((n0 + j0) >> 2) * kCtxRows + r] = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

}  // namespace fc

using namespace fc;

extern "C" int fc_context_terms(const float* ctx, int64_t ldc, int64_t B, int32_t C, const float* W, const float* bias,
                                int32_t T, float* out, void* stream) {
  if (B < 0 || C <= 0 || C > 64 || T <= 0 || (T & 15) || ldc < C) return FC_ERR_INVALID_ARGUMENT;
  if (B == 0) return FC_OK;
  if (!ctx || !W || !out) return FC_ERR_INVALID_ARGUMENT;
  if (reinterpret_cast<uintptr_t>(out) & 15) return FC_ERR_UNSUPPORTED;
  const long long tiles = (B + kCtxRows - 1) / kCtxRows;
  if (tiles >= (1ll << 31)) return FC_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)tiles);
  if (C <= 16) {
    context_terms_kernel<16><<<grid, kCtxRows, 0, st>>>(ctx, ldc, B, C, W, bias, T, out);
  } else if (C <= 32) {
    context_terms_kernel<32><<<grid, kCtxRows, 0, st>>>(ctx, ldc, B, C, W, bias, T, out);
  } else if (C <= 48) {
    context_terms_kernel<48><<<grid, kCtxRows, 0, st>>>(ctx, ldc, B, C, W, bias, T, out);
  } else {
    context_terms_kernel<64><<<grid, kCtxRows, 0, st>>>(ctx, ldc, B, C, W, bias, T, out);
  }
  FC_CHECK_LAUNCH();
  return FC_OK;
}
