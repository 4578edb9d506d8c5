// fc_made_inverse.cuh — the INVERSE of a masked autoregressive layer (sampling direction) in ONE kernel, with the MADE
// conditioner evaluated incrementally (SURVEY.md 8(f) n2; DESIGN.md 4.13).
//
// Replaces AutoregressiveTransform.inverse (flowcon/transforms/autoregressive/autoregressive.py:44-53): the reference
// runs the WHOLE conditioner D times, each pass on the partially inverted outputs, and keeps one more correct feature
// per pass.  Feature f's parameters depend only on features < f (the masks of flowcon/transforms/made.py:28-51), and in
// a MADE whose hidden units are ordered by degree every masked weight row is a PREFIX of its input: a hidden unit of
// degree m reads the units of degree <= m of the layer below.  So pass f only has to compute the hidden units that
// become valid with feature f - 1 (about H / (D - 1) per layer) from the prefix computed so far, and the P outputs of
// feature f.  Summed over the D passes that is HALF of one conditioner evaluation instead of D of them (cfg 3: 32 x
// fewer multiply-adds), and nothing but the inputs and outputs touches HBM.
//
// The host (flowconductor_b200/made_inverse.py) turns a residual MADE into a straight-line PROGRAM of phases and lays
// the masked, degree-sorted weights out in the order the kernel consumes them.  A phase is a [rows x width] weight
// matrix whose column groups are TASKS, one per warp: "units [j0, j0 + nj) of array `out` (+)= W . act(array `in`
// [k0, k0 + kn))".  Per pass there is one WIDE phase — everything that depends only on earlier passes: for every
// layer the products of the pass's new units with the units that were already final (the bulk of the work), the
// first layer of the new units, and the same for the feature's parameters — followed by one NARROW phase per layer
// for the dependent chain (the new units of one layer times the new units of the layer below: H / (D - 1) k-values)
// and the inversion of the feature.  The kernel is an interpreter for that program:
//
//   * one CTA = 32 rows (lane = row).  The row tile's state lives in shared memory as [unit][32 rows] fp32 arrays:
//     the features inverted so far, one array per hidden layer output (1 + 2 x blocks arrays of H units, holding
//     partial sums until a unit is final), the parameter tile of the feature being inverted.  That state (5 KB per
//     row at cfg 3) is what limits a CTA to 32 rows, and is why this is an fp32 CUDA-core kernel: the products are
//     32 x <=24 x k slivers on a serial chain, far below a tcgen05 tile.
//   * the weights are one linear stream, identical for every row tile: a producer warp walks the program and feeds a
//     ring of 8 KB slots (a few rows of the phase's matrix) with 1-D TMA bulk copies on mbarriers; it runs ahead
//     across phases and row tiles.
//   * the 8 compute warps each own one task of the phase (a slice of the OUTPUTS, so no cross-warp reduction): per
//     k-value one conflict-free activation load, the task's weights broadcast as 128-bit loads, packed fp32x2 FMAs
//     into <= 24 accumulators; bias / the partial sum of the wide phase / the skip connection are added when the
//     task stores its units.  One CTA barrier per phase.
//   * warp 0 then inverts the feature (same element arithmetic as the layer kernels: fc_math.cuh) and the next pass
//     starts.  log|det J| is the sum of the per-feature terms (what the reference's last pass returns).
//   * a conditional MADE (kCtx): the context enters as precomputed terms Wc ctx + bc, which do not depend on x; the
//     hidden arrays that consume them are prefilled with bias + act(term) when a row tile starts, and the program's tasks
//     accumulate onto that value.  Nothing else changes.
//
// This header holds the kernel and its launch plumbing; every bijection family instantiates it in its own .cu with an Op
//   struct Op { __device__ void eval(float z, const float* pc, float& x, float& lad, unsigned& status) const; }
// where pc points at the row's column of the parameter tile ([P][32 rows]: parameter i at pc[32 i], see made_load_params).
#pragma once
#include "fc_common.cuh"
#include "fc_tc.cuh"

namespace fc {


constexpr int kMR = 32;                 // rows per CTA
constexpr int kMW = FC_MADE_TASKS;      // compute warps = tasks per phase (8; 16 measured: no faster — the wide phases are
                                        // bound by shared-memory wavefronts, not by latency)
constexpr int kMThreads = (kMW + 1) * 32;
constexpr int kMJT = FC_MADE_MAX_NJ;    // outputs per task (24)
constexpr int kMJL = kMJT / 4;          // ... per lane (6)
constexpr int kMMaxStages = 8;
constexpr int kMSlotBytes = 8192;       // ring slot: floor(2048 / width) rows of the phase's matrix
constexpr int kMSlotFloats = kMSlotBytes / 4;
constexpr int kMPhaseInt4 = (4 + 12 * kMW) / 4;  // one fc_made_phase = header + 8 tasks = 25 x int4
constexpr int kMRecFloats = FC_MADE_RECORD_FLOATS;  // the phase record at the head of the phase's weights (padded to 512 B)

struct MadeKernelArgs {
  const int4* phases;  // fc_made_phase[n_phases]
  int n_phases;
  const float* weights;
  const float* bias;
  int n_bias;
  int D, P, n_arrays, hidden, stages;
  const float* z;
  long long ldz;
  float* x;
  long long ldx;
  float* lad;
  int accumulate;
  long long M;
  int num_tiles;
  int32_t* status;
};
// Conditional MADE (kCtx): this call's context terms [M, term_width] in T128 and the hidden arrays that start from them.
// A kernel parameter of its own, so that the context-free kernels keep their parameter layout and code.
struct MadeTerms {
  const float* terms;
  int term_width, n_term_arrays;
  int4 arrays[FC_MADE_MAX_TERM_ARRAYS];  // (array, first column in `terms`, bias offset, relu)
};
struct MadeArgs : MadeKernelArgs {
  MadeTerms ctx;
};

// Experiments only (-DFC_MADE_PROFILE=1: FC_LINEAR_PROFILE_BUILD=1 python -m flowconductor_b200.build --force): cycles warps 0
// and 5 of CTA 0 spend in each part of the interpreter loop; fc_made_inverse_profile() reads them back.
#ifndef FC_MADE_PROFILE
#define FC_MADE_PROFILE 0
#endif
static __device__ unsigned long long g_made_prof[32];  // per translation unit; fc_made_inverse_profile reads fc_made_inverse.cu's
#if FC_MADE_PROFILE
// clock read that cannot be scheduled before `dep` is available
__device__ __forceinline__ long long made_clock_after(int dep) {
  long long t;
  asm volatile("{.reg .u64 c; mov.u64 c, %%clock64; add.u64 %0, c, %1;}" : "=l"(t) : "l"((long long)(dep >> 30)) : "memory");
  return t;
}
#define MPROF_T(t, dep) const long long t = made_clock_after(dep)
#define MPROF_ADD(i, t1, t0) prof[pb + (i)] += (t1) - (t0)
#else
#define MPROF_T(t, dep)
#define MPROF_ADD(i, t1, t0)
#endif

// Bounded mbarrier wait: a protocol error ends the kernel with a trap (the launch fails) instead of hanging the GPU.
__device__ __forceinline__ void made_wait(uint32_t bar, uint32_t parity) {
  if (tc::mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!tc::mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}

// One task's share of a ring slot.  A lane owns 4 rows x JL outputs (register tile: a broadcast-only mapping — lane = row,
// every weight read by all 32 lanes — is bound by shared-memory wavefronts, 4 per 128-bit broadcast load; measured):
//   acc[i] (rows 0,1) and acc[kMJL + i] (rows 2,3) += act(in[r][4 rows]) * w[r][i]   for r in [0, n), i in [0, JL)
// `in` advances 32 floats per k-value, `w` one row (`width` floats) of the phase's matrix.
template <int JL>
__device__ __forceinline__ void made_kloop(float2 (&acc)[2 * kMJL], const float* __restrict__ in, const float* __restrict__ w,
                                           int width, int n, bool relu) {
#pragma unroll(JL <= 2 ? 8 : 4)
  for (int r = 0; r < n; ++r) {
    float4 a4 = *reinterpret_cast<const float4*>(in + r * kMR);
    if (relu) {
      a4.x = fmaxf(a4.x, 0.f);
      a4.y = fmaxf(a4.y, 0.f);
      a4.z = fmaxf(a4.z, 0.f);
      a4.w = fmaxf(a4.w, 0.f);
    }
    const float2 a01 = make_float2(a4.x, a4.y), a23 = make_float2(a4.z, a4.w);
    const float* wr = w + r * width;
    float wv[JL];
    if constexpr (JL % 4 == 0) {
#pragma unroll
      for (int i = 0; i < JL; i += 4) {
        const float4 t = *reinterpret_cast<const float4*>(wr + i);
        wv[i] = t.x, wv[i + 1] = t.y, wv[i + 2] = t.z, wv[i + 3] = t.w;
      }
    } else if constexpr (JL % 2 == 0) {
#pragma unroll
      for (int i = 0; i < JL; i += 2) {
        const float2 t = *reinterpret_cast<const float2*>(wr + i);
        wv[i] = t.x, wv[i + 1] = t.y;
      }
    } else {
#pragma unroll
      for (int i = 0; i < JL; ++i) wv[i] = wr[i];
    }
#pragma unroll
    for (int i = 0; i < JL; ++i) {
      const float2 w2 = make_float2(wv[i], wv[i]);
      acc[i] = __ffma2_rn(a01, w2, acc[i]);
      acc[kMJL + i] = __ffma2_rn(a23, w2, acc[kMJL + i]);
    }
  }
}

struct MadeSmem {
  // [ring: stages x 8 KB][X: D x 32][H: n_arrays x hidden x 32][PT: P x 32][bias: n_bias (padded to 4)][barriers]
  static __host__ __device__ size_t floats_after_ring(int D, int P, int n_arrays, int hidden, int n_bias) {
    return (size_t)D * kMR + (size_t)n_arrays * hidden * kMR + (size_t)P * kMR + (size_t)((n_bias + 3) & ~3);
  }
  static __host__ __device__ size_t total(int stages, int D, int P, int n_arrays, int hidden, int n_bias) {
    return (size_t)stages * kMSlotBytes + 4 * floats_after_ring(D, P, n_arrays, hidden, n_bias) + 8 * 2 * kMMaxStages + 128;
  }
};

template <class Op, bool kCtx>
__global__ void __launch_bounds__(kMThreads, 1) made_inverse_kernel(const MadeKernelArgs a, const Op op, const MadeTerms ct) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const uint32_t raw_s = tc::s32(smem_raw);
  const uint32_t base = (raw_s + 127u) & ~127u;
  unsigned char* const gbase = smem_raw + (base - raw_s);
  const int stages = a.stages;
  float* const ring_g = reinterpret_cast<float*>(gbase);
  float* const X = reinterpret_cast<float*>(gbase + (size_t)stages * kMSlotBytes);  // [D][32]: z until a feature is inverted, then x
  float* const H = X + a.D * kMR;                                                    // [n_arrays][hidden][32]
  float* const PT = H + (size_t)a.n_arrays * a.hidden * kMR;                         // [P][32] parameters of the feature
  float* const BS = PT + a.P * kMR;                                                  // every layer's bias
  const uint32_t bars = base + (uint32_t)(stages * kMSlotBytes) +
                        4u * (uint32_t)MadeSmem::floats_after_ring(a.D, a.P, a.n_arrays, a.hidden, a.n_bias);
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (kMMaxStages + s); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      tc::mbar_init(full_bar(s), 1);
      tc::mbar_init(empty_bar(s), kMW);
    }
    tc::fence_mbar_init();
  }
  for (int i = threadIdx.x; i < a.n_bias; i += kMThreads) BS[i] = __ldg(a.bias + i);
  __syncthreads();

  if (warp == kMW) {
    // ------------------------------------------------------------------ weight producer
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
        int4 hd = __ldg(a.phases);
        for (int p = 0; p < a.n_phases; ++p) {
          const int rows = hd.x, width = hd.y;
          const float* src = a.weights + (size_t)(unsigned)hd.z * 4;
          if (p + 1 < a.n_phases) hd = __ldg(a.phases + (size_t)(p + 1) * kMPhaseInt4);  // in flight while this phase is fed
          // first slot: the phase record (kMRecFloats) + as many rows as fit behind it; then whole slots of rows
          int r0 = 0, cap = (kMSlotFloats - kMRecFloats) / width, lead = kMRecFloats;
          do {
            const int nr = rows - r0 < cap ? rows - r0 : cap;
            const uint32_t bytes = (uint32_t)((lead + nr * width) * 4);
            made_wait(empty_bar(s), ph ^ 1u);
            tc::mbar_expect_tx(full_bar(s), bytes);
            tc::bulk_load_1d(base + (uint32_t)(s * kMSlotBytes), src, bytes, full_bar(s));
            src += lead + nr * width;
            r0 += nr;
            cap = kMSlotFloats / width;
            lead = 0;
            if (++s == stages) {
              s = 0;
              ph ^= 1u;
            }
          } while (r0 < rows);
        }
      }
    }
    return;
  }

  // -------------------------------------------------------------------- compute warps
  const int tid = threadIdx.x;  // 0..255
  const int jg = lane >> 3, rg = lane & 7;  // this lane's outputs jg * JL .. and rows 4 rg .. 4 rg + 3
  int s = 0;
  uint32_t ph = 0;
  unsigned status = 0;
#if FC_MADE_PROFILE
  long long prof[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // [0..7] wide phases, [8..15] narrow phases
  const long long prof_begin = clock64();
#endif
  const int D = a.D;
  const size_t arr_floats = (size_t)a.hidden * kMR;
  for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
    const long long row0 = (long long)tile * kMR;
    for (int i = tid; i < kMR * D; i += kMW * 32) {
      const int r = i / D, f = i - r * D;
      X[f * kMR + r] = (row0 + r < a.M) ? __ldg(a.z + (row0 + r) * a.ldz + f) : 0.f;
    }
    if constexpr (kCtx) {
      // The context terms do not depend on x: every unit of a context array starts the tile at bias + act(term) (MADE
      // initial layer: act = ReLU, made.py:138-140; first layer of a block: identity, made.py:100-102), and the tasks that
      // write those units accumulate onto it (the host clears FC_MADE_INIT_BIAS on them).  Lane = row: one float4 of the
      // T128 matrix per (row, 4 units), 512 contiguous bytes per warp, conflict-free [unit][32 rows] stores.  Rows past M
      // get the bias alone (the T128 rows there were never written).
      const int groups = (a.hidden + 3) >> 2;
      const float* tile_terms = ct.terms + (row0 >> 7) * 128ll * ct.term_width + (row0 & 127) * 4;
      for (int i = tid; i < ct.n_term_arrays * groups * kMR; i += kMW * 32) {
        const int r = i & (kMR - 1), q = i >> 5, g = q % groups;
        const int4 ta = ct.arrays[q / groups];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + r < a.M) v = __ldg(reinterpret_cast<const float4*>(tile_terms + (size_t)((ta.y >> 2) + g) * 512 + r * 4));
        if (ta.w) v = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
        const float t[4] = {v.x, v.y, v.z, v.w};
        const int j0 = 4 * g, n = a.hidden - j0 < 4 ? a.hidden - j0 : 4;
        float* h = H + (size_t)(ta.x - 1) * arr_floats + (size_t)j0 * kMR + r;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (e < n) h[e * kMR] = BS[ta.z + j0 + e] + t[e];
      }
    }
    float lad_acc = 0.f;
    tc::named_barrier_sync(1, kMW * 32);
    for (int p = 0; p < a.n_phases; ++p) {
      MPROF_T(p_t0, p);
      // the phase record travels at the head of the phase's first weight slot (a global read of it here would cost an L2
      // round trip per phase on the serial chain: measured)
      made_wait(full_bar(s), ph);
      const int4* rec = reinterpret_cast<const int4*>(ring_g + s * kMSlotFloats);
      const int4 hd = rec[0], t0 = rec[1 + 3 * warp], t1 = rec[2 + 3 * warp], t2 = rec[3 + 3 * warp];
      const int rows = hd.x, width = hd.y, feature = hd.w;
      const int in_array = t0.x, out_array = t0.y, k0 = t0.z, kn = t0.w;
      const int j0 = t1.x, nj = t1.y, c0 = t1.z, flags = t1.w;
      const int res_array = t2.x, b_off = t2.y;
      const int jl = (nj + 3) >> 2;  // outputs per lane
      const bool relu = (flags & FC_MADE_RELU_IN) != 0;
#if FC_MADE_PROFILE
      const int pb = rows > 40 ? 0 : 8;
#endif
      MPROF_T(p_t1, rows + width + kn + b_off);
      MPROF_ADD(0, p_t1, p_t0);
      float2 acc[2 * kMJL];
#pragma unroll
      for (int j = 0; j < 2 * kMJL; ++j) acc[j] = make_float2(0.f, 0.f);
      const float* in = (in_array == 0 ? X : H + (size_t)(in_array - 1) * arr_floats) + (size_t)k0 * kMR + 4 * rg;
      int r0 = 0, cap = (kMSlotFloats - kMRecFloats) / width, lead = kMRecFloats;
      do {
        const int nr = rows - r0 < cap ? rows - r0 : cap;
        MPROF_T(s_t0, r0);
        if (r0 > 0) made_wait(full_bar(s), ph);
        MPROF_T(s_t1, r0);
        MPROF_ADD(1, s_t1, s_t0);
        int n = kn - r0;  // this task's k-values inside the slot
        n = n < nr ? n : nr;
        if (nj > 0 && n > 0) {
          const float* w = ring_g + s * kMSlotFloats + lead + c0 + jg * jl;
          const float* in_r = in + (size_t)r0 * kMR;
          switch (jl) {
            case 1: made_kloop<1>(acc, in_r, w, width, n, relu); break;
            case 2: made_kloop<2>(acc, in_r, w, width, n, relu); break;
            case 3: made_kloop<3>(acc, in_r, w, width, n, relu); break;
            case 4: made_kloop<4>(acc, in_r, w, width, n, relu); break;
            case 5: made_kloop<5>(acc, in_r, w, width, n, relu); break;
            default: made_kloop<6>(acc, in_r, w, width, n, relu); break;
          }
        }
        __syncwarp();
        MPROF_T(s_t2, __float_as_int(acc[0].x + acc[3].y + acc[7].x + acc[11].y));
        MPROF_ADD(2, s_t2, s_t1);
        if (lane == 0) tc::mbar_arrive(empty_bar(s));
        if (++s == stages) {
          s = 0;
          ph ^= 1u;
        }
        r0 += nr;
        cap = kMSlotFloats / width;
        lead = 0;
      } while (r0 < rows);
      MPROF_T(p_t2, p);
      // this task's units: bias or the partial sum stored by an earlier phase, skip connection
      if (nj > 0) {
        float* out = (out_array > 0 ? H + (size_t)(out_array - 1) * arr_floats : PT) + (size_t)j0 * kMR + 4 * rg;
        const float* res = res_array > 0 ? H + (size_t)(res_array - 1) * arr_floats + (size_t)j0 * kMR + 4 * rg : nullptr;
        const bool init = (flags & FC_MADE_INIT_BIAS) != 0;
#pragma unroll
        for (int i = 0; i < kMJL; ++i) {
          const int j = jg * jl + i;
          if (i < jl && j < nj) {
            float4 v = make_float4(acc[i].x, acc[i].y, acc[kMJL + i].x, acc[kMJL + i].y);
            float4* o = reinterpret_cast<float4*>(out + j * kMR);
            if (init) {
              const float b = BS[b_off + j];
              v.x += b, v.y += b, v.z += b, v.w += b;
            } else {
              const float4 t = *o;
              v.x += t.x, v.y += t.y, v.z += t.z, v.w += t.w;
            }
            if (res) {
              const float4 t = *reinterpret_cast<const float4*>(res + j * kMR);
              v.x += t.x, v.y += t.y, v.z += t.z, v.w += t.w;
            }
            *o = v;
          }
        }
      }
      MPROF_T(p_t3, p);
      MPROF_ADD(3, p_t3, p_t2);
      tc::named_barrier_sync(1, kMW * 32);
      MPROF_T(p_t4, p);
      MPROF_ADD(4, p_t4, p_t3);
      if (feature >= 0) {
        // the feature's parameters are complete: invert it (autoregressive.py:50-52 for the one column that becomes final)
        if (warp == 0) {
          const float zf = X[feature * kMR + lane];
          float xf, lf;
          op.eval(zf, PT + lane, xf, lf, status);
          X[feature * kMR + lane] = xf;
          lad_acc += lf;
        }
        tc::named_barrier_sync(1, kMW * 32);
        MPROF_T(p_t5, __float_as_int(lad_acc));
        MPROF_ADD(5, p_t5, p_t4);
      }
#if FC_MADE_PROFILE
      {
        MPROF_T(p_t6, p);
        prof[pb + 6] += p_t6 - p_t0;
        prof[pb + 7] += 1;
      }
#endif
    }
    for (int i = tid; i < kMR * D; i += kMW * 32) {
      const int r = i / D, f = i - r * D;
      if (row0 + r < a.M) a.x[(row0 + r) * a.ldx + f] = X[f * kMR + r];
    }
    if (warp == 0 && row0 + lane < a.M) {
      const long long row = row0 + lane;
      a.lad[row] = a.accumulate ? a.lad[row] + lad_acc : lad_acc;
    }
    tc::named_barrier_sync(1, kMW * 32);
  }
  if (warp == 0 && status != 0 && a.status) atomicOr(a.status, (int)status);
#if FC_MADE_PROFILE
  if (blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 5)) {  // (a light and a heavy warp of the wide phases)
    unsigned long long* o = g_made_prof + (warp == 0 ? 0 : 16);
    for (int i = 0; i < 16; ++i) o[i] = (unsigned long long)prof[i];
    (void)prof_begin;
  }
#endif
}

inline int made_stages(int D, int P, int n_arrays, int hidden, int n_bias) {
  const size_t fixed = MadeSmem::total(0, D, P, n_arrays, hidden, n_bias);
  const size_t limit = (size_t)device_info().max_smem_optin;
  if (fixed + 2 * kMSlotBytes > limit) return 0;
  const size_t st = (limit - fixed) / kMSlotBytes;
  return (int)(st > kMMaxStages ? kMMaxStages : st);
}

inline int made_check(const fc_made_program* prog, const float* z, int64_t ldz, float* x, int64_t ldx, float* lad, int64_t B,
                      int P, MadeArgs& a) {
  if (!prog || !prog->phases || !prog->weights || !prog->bias || prog->n_phases <= 0) return FC_ERR_INVALID_ARGUMENT;
  if (prog->features <= 0 || prog->hidden <= 0 || prog->n_arrays <= 0 || prog->params_per_feature != P || prog->n_bias <= 0)
    return FC_ERR_INVALID_ARGUMENT;
  if (B < 0) return FC_ERR_INVALID_ARGUMENT;
  if (B > 0 && (!z || !x || !lad)) return FC_ERR_INVALID_ARGUMENT;
  if (ldz < prog->features || ldx < prog->features) return FC_ERR_INVALID_ARGUMENT;
  if ((reinterpret_cast<uintptr_t>(prog->weights) & 15) || (reinterpret_cast<uintptr_t>(prog->phases) & 15)) return FC_ERR_UNSUPPORTED;
  if (B >= ((int64_t)1 << 31) * kMR) return FC_ERR_UNSUPPORTED;
  a.phases = reinterpret_cast<const int4*>(prog->phases);
  a.n_phases = prog->n_phases;
  a.weights = prog->weights;
  a.bias = prog->bias;
  a.n_bias = prog->n_bias;
  a.D = prog->features;
  a.P = P;
  a.n_arrays = prog->n_arrays;
  a.hidden = prog->hidden;
  a.z = z;
  a.ldz = ldz;
  a.x = x;
  a.ldx = ldx;
  a.lad = lad;
  a.M = B;
  a.num_tiles = (int)((B + kMR - 1) / kMR);
  const int nt = prog->n_term_arrays;
  if (nt < 0 || nt > FC_MADE_MAX_TERM_ARRAYS) return FC_ERR_INVALID_ARGUMENT;
  if (nt > 0) {
    if (!prog->terms || (reinterpret_cast<uintptr_t>(prog->terms) & 15) || prog->term_width <= 0 || prog->term_width % 16)
      return FC_ERR_INVALID_ARGUMENT;
    for (int t = 0; t < nt; ++t) {
      const fc_made_term_array& ta = prog->term_arrays[t];
      if (ta.array < 1 || ta.array > prog->n_arrays) return FC_ERR_INVALID_ARGUMENT;
      for (int u = 0; u < t; ++u)
        if (prog->term_arrays[u].array == ta.array) return FC_ERR_INVALID_ARGUMENT;
      if (ta.column < 0 || ta.column % 4 || (int64_t)ta.column + prog->hidden > prog->term_width) return FC_ERR_INVALID_ARGUMENT;
      if (ta.b_off < 0 || (int64_t)ta.b_off + prog->hidden > prog->n_bias) return FC_ERR_INVALID_ARGUMENT;
      a.ctx.arrays[t] = make_int4(ta.array, ta.column, ta.b_off, ta.relu != 0);
    }
    a.ctx.terms = prog->terms;
    a.ctx.term_width = prog->term_width;
  }
  a.ctx.n_term_arrays = nt;
  a.stages = made_stages(a.D, a.P, a.n_arrays, a.hidden, a.n_bias);
  if (a.stages < 2) return FC_ERR_UNSUPPORTED;
  return FC_OK;
}

template <class Op>
inline int launch_made(const MadeArgs& a, const Op& op, cudaStream_t stream) {
  auto kern = a.ctx.n_term_arrays > 0 ? made_inverse_kernel<Op, true> : made_inverse_kernel<Op, false>;
  const size_t smem = MadeSmem::total(a.stages, a.D, a.P, a.n_arrays, a.hidden, a.n_bias);
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return FC_ERR_CUDA;
  const int sms = device_info().sm_count;
  const int grid = a.num_tiles < sms ? a.num_tiles : sms;
  kern<<<grid, kMThreads, smem, stream>>>(a, op, a.ctx);
  FC_CHECK_LAUNCH();
  return FC_OK;
}


// Copy the feature's P parameters of this row out of the parameter tile into a local array.
template <int PMAX>
__device__ __forceinline__ void made_load_params(const float* pc, int P, float (&p)[PMAX]) {
  for (int i = 0; i < P && i < PMAX; ++i) p[i] = pc[i * kMR];
}

}  // namespace fc
