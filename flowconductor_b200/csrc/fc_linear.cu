// fc_linear.cu — the conditioner's dense layers on the 5th-gen tensor cores (tcgen05 / TMEM / TMA), fp32-faithful.
//
// Replaces nn.Linear / MaskedLinear.forward of the conditioner networks
// (flowcon/nn/nets/resnet.py:39-56,90-99, flowcon/transforms/made.py:71-72,266-272) and — for the final layer —
// the element-wise bijection that consumes its output (rational_quadratic.py:13-181, coupling.py:279-293,549-582):
// the spline runs in the GEMM epilogue straight out of tensor memory, so the [B, D_t*P] parameter tensor
// (2.9 GB per layer at cfg 2) never exists in HBM.
//
// Precision: the reference computes these GEMMs in fp32 (no TF32).  One tf32 UMMA per product would lose 13
// mantissa bits, so every operand is split  a = a_hi + a_lo  (both tf32-representable, |a - a_hi - a_lo| <=
// 2^-24 |a|) and the product is accumulated as  a_lo*b_hi + a_hi*b_lo + a_hi*b_hi  in the fp32 TMEM accumulator
// ("3xTF32": error ~2^-21 per product, the same size as the summation-order noise of an fp32 GEMM with K = 256).
//   * weights: split once by fc_linear_pack into a [hi | lo] pair of K-major planes (also folds the MADE mask,
//     the per-feature padding P -> P_pad and the coupling column scatter into the layout);
//   * activations: TMA lands the raw fp32 tile in shared memory; four converter warps split it (optionally after
//     ReLU — the residual blocks are pre-activation, resnet.py:41-47) and write (a_hi, a_lo) into a tensor-memory
//     operand ring (TS kernels) or back into shared memory (a_hi in place, a_lo next to it).
//
// Accumulation: the tensor core truncates (rounds toward zero) every time an MMA result is added to the fp32
// accumulator in TMEM; over the K/8 = 32 dependent additions of a K = 256 dot product that is a systematic error
// of ~1.5e-6 relative, 5x the rounding noise of an fp32 FMA chain.  The accumulator is therefore drained every
// `chunk` pipeline stages (default 32 k-values = 4 UMMA k-steps): the MMA warp starts a fresh partial sum in the
// other TMEM buffer while the epilogue warps add the finished partial into fp32 REGISTER accumulators with
// round-to-nearest.  The partials are 8x smaller and 8x shorter, which brings the GEMM error down to that of the
// fp32 cuBLAS GEMM the reference runs (measured on K = 256 Gaussian operands, scripts/check_linear.py: rms error
// 1.8e-6 undrained, 4.6e-7 at 64, 2.5e-7 at 32; cuBLAS fp32 2.9e-7).
//
// Kernel: persistent, one CTA per SM, 16 warps (24 with the spline warps; register budget re-balanced with setmaxnreg):
//   warp 0      TMA producer   : per stage one box of A (128 x BK) and the hi/lo boxes of W (BN x BK each)
//   warp 1      UMMA issuer    : 3 x BK/8 tcgen05.mma (128 x BN x 8, kind::tf32) per stage, commit -> barriers
//   warp 2      TMEM allocator
//   warps 4-7   converters     : raw A tile -> (a_hi, a_lo)
//   warps 8-15  epilogue       : tcgen05.ld each partial accumulator (double-buffered in TMEM, so draining chunk i
//                                overlaps the MMAs of chunk i+1) into registers, then + bias and either
//                                ReLU/residual/store, the hand-over of the parameter tile to the spline warps, or the
//                                affine transform of 32 features per 64 columns.
//   warps 16-23 spline warps (EPI 1): the rational-quadratic spline of 8 (K=8) / 4 (K=16) features per 192-column tile.
//   warp 3      staging manager (EPI 3): brings the skip connection into the staging tile and stores the finished tile —
//                                one bulk copy for a T128 tile, four 2-D tensor-map boxes (128 rows x 32 columns,
//                                128-byte swizzled rows) for a row-major result; split-K ranges land in consecutive
//                                row blocks of one partials matrix.
// Operand forms of A (LinArgs::a_tiled): 0 row-major [M, K] (swizzled TMA boxes), 1 the T128 activation layout,
// 2 TRANSPOSED [K, M] row-major — the weight-gradient product grad_y^T x reads grad_y as it lies: converter thread m
// (= TMEM lane m) reads column m of every k-row of an un-swizzled BK x 128 box, and can accumulate the column sums
// (the bias gradient) on the way (LinArgs::colsum).  StoreEpi::res_mask turns the staged skip-connection tile into a
// gate (ReLU backward of an input-gradient product).
// DESIGN.md 4.6 (inference) and 4.8 (training) have the measurements behind each of these choices.
#include <atomic>

#include "fc_common.cuh"
#include "fc_tc.cuh"

namespace fc {

using namespace tc;

constexpr int kBaseThreads = 256;  // warps 0-7: producer, MMA issuer, allocator, spare, 4 converters
constexpr int kBM = 128;
constexpr int kConvWarp0 = 4;
constexpr int kEpiWarp0 = 8;
constexpr int kNumConv = 128;  // converter threads (warps 4-7)
constexpr int kEpiWarps = 8;   // epilogue warps 8-15: two column groups, 4 warps (TMEM lane quarters) each

// Kernel forms per epilogue (see the kernel comment): every kernel but the plain store (EPI 0) takes its activation
// operand from tensor memory (TS), and the spline (EPI 1) runs on 8 warps of its own (SW).
constexpr bool operand_in_tmem(int epi) { return epi != 0; }
constexpr int spline_warps(int epi) { return epi == 1 ? 8 : 0; }

// setmaxnreg budgets per warpgroup (the register file holds 65536):
//   8 epilogue warps: 512 threads launch with 128;  128*40 + 128*56 + 256*208 = 65536
//   8 epilogue + 8 spline warps: 768 threads launch with 80;  128*32 + 128*64 + 256*120 + 256*72 = 61440 (= 768 * 80,
//   the CTA's pool)
template <int SW>
struct RegBudget {
  static constexpr int kProducer = SW ? 32 : 40, kConverter = SW ? 64 : 56, kEpilogue = SW ? 120 : 208, kSpline = 72;
};

struct LinArgs {
  int M;
  int num_k_stages;  // pipeline stages (BK k-values each) per output tile
  int chunk;         // stages per partial accumulator
  int num_m_tiles, num_n_tiles;
  int n_pad;         // rows of one weight plane (lo plane starts at row n_pad of the weight tensor map)
  int relu_in;       // ReLU applied to A while splitting
  int a_tiled;       // 1: A is stored in the T128 activation layout (include/flowcon_b200.h); 2: A is given TRANSPOSED,
                     //    [K, M] row-major (weight gradients: grad_y [B, N] is the A operand of grad_y^T x as it lies)
  int k_slices;      // split-K: the reduction is cut into k_slices ranges of num_k_stages slots, one work unit each
  int debug;         // FC_LINEAR_DEBUG: 4 = record the cycle counters (only in builds with -DFC_LINEAR_PROFILE=1)
  const float* bias;  // [n_pad]
  float* colsum;      // a_tiled == 2 only, may be null: column sums of A^T per reduction range, [k_slices][slice rows]
                      // (the bias gradient grad_y.sum(0) comes for free while grad_y passes through the converters)
};

struct StoreEpi {
  float* out;
  int64_t ldo;
  const float* residual;
  int64_t ldr;
  int n_out;
  int relu_out;
  int tiled;  // out (and residual) are stored in the T128 layout; ldo / ldr are then their logical widths
  int res_mask;  // staged kernel: `residual` is not added, it gates: out = residual > 0 ? out : 0 (the ReLU backward
                 // of an input-gradient product, masked by the saved pre-activation)
  int64_t slice_stride;  // split-K: floats between the partial results of consecutive reduction ranges
};

struct RqsEpi {
  const float* x;
  int64_t ldx;
  float* y;
  int64_t ldy;
  float* lad;
  int accumulate;
  const int32_t* tcols;
  const int32_t* ccols;
  int n_copy;
  int D_t;
  RqsParams c;
  int32_t* status;
  int activation;  // EPI 2 (affine): FC_SCALE_*; c.inverse carries the direction
};

template <int EPI, int BN, int BK, int STAGES, int CTAS>
struct LinSmem {
  static constexpr int A_BYTES = kBM * BK * 4;
  static constexpr int B_BYTES = (BN / CTAS) * BK * 4;  // a CTA pair splits the rows of every weight box
  static constexpr int A_PLANES = operand_in_tmem(EPI) ? 1 : 2;  // TS: the converted operand lives in tensor memory
  static constexpr int STAGE_BYTES = A_PLANES * A_BYTES + 2 * B_BYTES;
  // parameter tile (spline warps) / staging tile (EPI 3)
  static constexpr int PARAMS_BYTES = (spline_warps(EPI) || EPI == 3) ? kBM * BN * 4 : 0;
  static constexpr int BAR_BYTES = 8 * (4 * STAGES + 6) + 16;
  // per-row partial log-dets of the second thread group, double-buffered (spline warps: one row block per buffer; drain
  // warps: buffers 3 row blocks apart, of which only the first is written)
  static constexpr int LAD_BYTES = (spline_warps(EPI) ? 2 : 2 * 3) * kBM * 4;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + PARAMS_BYTES + BAR_BYTES + LAD_BYTES + 1024;  // + alignment slack
  static_assert(A_BYTES % 1024 == 0 && B_BYTES % 1024 == 0, "operand tiles must keep 1024-byte alignment");
};

// Experiments only: cycles the MMA-issuing thread / one epilogue warp of CTA 0 spend waiting (FC_LINEAR_DEBUG & 4).
// The counters cost registers in the hot loops, so they are compiled in only with -DFC_LINEAR_PROFILE=1
// (FC_LINEAR_PROFILE_BUILD=1 python -m flowconductor_b200.build --force); otherwise the record stays zero.
#ifndef FC_LINEAR_PROFILE
#define FC_LINEAR_PROFILE 0
#endif
__device__ unsigned long long g_lin_prof[16];

template <int N>
__device__ __forceinline__ void set_max_regs_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void set_max_regs_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// acc[0..N) (=|+=) N consecutive TMEM columns of this thread's lane.  16 columns per tcgen05.ld, software-pipelined:
// the additions of group j run while the load of group j+1 is in flight.
template <int N, bool kFirst>
__device__ __forceinline__ void drain_partial(uint32_t taddr, float* acc) {
  static_assert(N % 16 == 0, "column count per thread must be a multiple of 16");
  if (kFirst) {
#pragma unroll
    for (int j = 0; j < N; j += 16) tmem_ld16(taddr + (uint32_t)j, reinterpret_cast<uint32_t*>(acc + j));
    tmem_wait_ld();
    return;
  }
  uint32_t v[2][16];
  tmem_ld16(taddr, v[0]);
  tmem_wait_ld();
#pragma unroll
  for (int j = 0; j < N; j += 16) {
    const int cur = (j >> 4) & 1;
    if (j + 16 < N) tmem_ld16(taddr + (uint32_t)(j + 16), v[cur ^ 1]);
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[j + i] += __uint_as_float(v[cur][i]);
    if (j + 16 < N) tmem_wait_ld();
  }
}

// EPI: 0 = store (bias, optional residual / ReLU), 1 = rational-quadratic spline with KC bins,
//      2 = affine (PPAD = 2 accumulator columns per feature: raw scale, shift),
//      3 = store of T128 outputs through a shared-memory staging tile: the skip connection comes IN by one TMA bulk
//          load and the result goes OUT by one TMA bulk store per 128 x 128 tile (contiguous 64 KB in the T128
//          layout), issued by the otherwise idle warp 3; the epilogue warps never touch global memory.
// RQS tile geometry: FEATS features of PPAD accumulator columns each (BN = FEATS * PPAD).
// Without PAIR every CTA works on its own row tile.
// PAIR: clusters of two CTAs (the two SMs of a TPC) that issue ONE tcgen05.mma.cta_group::2 (256 x BN x 8) per
//   product: each CTA stages its own 128 rows of A but only HALF of every weight box, so the weight traffic (L2 ->
//   shared memory AND shared memory -> tensor core) per SM is halved and the ring is 1.5x deeper.  Rank 0 (the leader)
//   issues the MMAs; rank 1's converter and drain warps arrive on the leader's barriers.  Only TS kernels pair.
// TS (EPI 1, 2, 3): the converters write the (hi, lo) split of the activation tile into TENSOR MEMORY (tcgen05.st; ring
//   of STAGES slots of 2*BK columns behind the two partial accumulators) and the MMAs take their A operand from there.
//   Per 8 k-values the shared memory then serves 3 weight-tile reads + the TMA writes + one raw-tile read instead of
//   3 x (A + B) reads + TMA writes + raw read + two converted writes: 132 instead of 201 B/cycle at BN = 192 (the
//   SMEM port delivers 128), and no generic->async proxy hand-off is needed.
// SW (EPI 1): the bijection runs on 8 extra warps.  The drain warps only accumulate the partial sums and drop the
//   finished parameter tile (128 rows x BN columns, column-major so that a warp's 32 rows are 32 consecutive words)
//   into shared memory; the spline warps evaluate it while the MMAs and drains of the NEXT tile run.  Without this the
//   MMA warp can only run two partial accumulators ahead of the ~6k cycles the spline of a tile takes, and waits a
//   third of the time.
template <int EPI, int BN, int BK, int STAGES, int KC, int PPAD, bool PAIR>
__global__ void __launch_bounds__(kBaseThreads + 32 * (kEpiWarps + spline_warps(EPI)), 1)
    linear_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmR,
                         const LinArgs la, const StoreEpi se, const RqsEpi re) {
  constexpr int CTAS = PAIR ? 2 : 1;  // CTAs per MMA = cluster size = row tiles per work unit
  constexpr bool TS = operand_in_tmem(EPI);
  constexpr int SW = spline_warps(EPI);
  using SM = LinSmem<EPI, BN, BK, STAGES, CTAS>;
  static_assert(EPI != 3 || BN == 128, "staged store: 128-wide tiles");
  static_assert(!PAIR || TS, "CTA pairs take the activation operand from tensor memory");
  static_assert(!TS || 2 * BN + STAGES * 2 * BK <= 512, "TS: operand ring must fit behind the accumulators");
  constexpr uint32_t kTmemA0 = 2 * BN;  // first column of the operand ring (TS)
  extern __shared__ unsigned char smem_raw[];
  const uint32_t raw_s = s32(smem_raw);
  const uint32_t base = (raw_s + 1023u) & ~1023u;
  unsigned char* const gbase = smem_raw + (base - raw_s);
  const uint32_t params_s = base + STAGES * SM::STAGE_BYTES;  // parameter tile (SW > 0)
  const uint32_t bars = params_s + SM::PARAMS_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto conv_bar = [&](int s) { return bars + 8u * (STAGES + s); };
  auto empty_bar = [&](int s) { return bars + 8u * (2 * STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (4 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (4 * STAGES + 2 + a); };  // leader's is the one in use
  const uint32_t pfull_bar = bars + 8u * (4 * STAGES + 4), pempty_bar = bars + 8u * (4 * STAGES + 5);
  const uint32_t tmem_slot = bars + 8u * (4 * STAGES + 6);
  unsigned char* const gbars = gbase + STAGES * SM::STAGE_BYTES + SM::PARAMS_BYTES;
  volatile uint32_t* const tmem_slot_g = reinterpret_cast<volatile uint32_t*>(gbars + 8 * (4 * STAGES + 6));
  float* const lad_x = reinterpret_cast<float*>(gbars + SM::BAR_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t kTmemCols = 512;
  static_assert(2 * BN <= 512, "two partial accumulators must fit in tensor memory");
  const int rank = CTAS == 2 ? (int)cluster_ctarank() : 0;
  const int unit0 = (int)blockIdx.x / CTAS, unit_step = (int)gridDim.x / CTAS;  // cluster index / count
  const int ks_n = la.k_slices;                                                   // reduction ranges (split-K), else 1
  const int n_units = ((la.num_m_tiles + CTAS - 1) / CTAS) * ks_n;             // work units: (row tile(s), range)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(conv_bar(s), 4 * CTAS);  // one arrival per converter warp (of both CTAs of a pair, in the leader)
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), kEpiWarps * CTAS);
    }
    // SW: parameter tile full (drain warps) / empty (spline warps).  EPI 3: staging tile ready to be written (manager,
    // possibly through the skip connection's TMA bytes) / written by all epilogue warps
    mbar_init(pfull_bar, EPI == 3 ? 1 : kEpiWarps);
    mbar_init(pempty_bar, EPI == 3 ? kEpiWarps : (SW > 0 ? SW : 1));
    fence_mbar_init();
  }
  if (warp == 2) {
    if (CTAS == 2) {
      tmem_alloc_pair(tmem_slot, kTmemCols);
    } else {
      tmem_alloc(tmem_slot, kTmemCols);
    }
  }
  tc_fence_before();
  if (CTAS == 2) {
    cluster_sync_all();  // barriers of both CTAs initialised before any remote arrive
  } else {
    __syncthreads();
  }
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_g;

  const int nk = la.num_k_stages;
  const int n_tiles = la.num_n_tiles;
  const int chunk = la.chunk;
  const int n_chunks = (nk + chunk - 1) / chunk;

  if (warp < kConvWarp0) {
    set_max_regs_dec<RegBudget<SW>::kProducer>();
    if (warp == 0) {
      // ---------------------------------------------------------------- TMA producer
      if (lane == 0) {
        int s = 0;
        uint32_t ph = 0;
        for (int mp = unit0; mp < n_units; mp += unit_step) {
          const int mt = (mp / ks_n) * CTAS + rank;
          const int k_base = (mp % ks_n) * nk;  // first ring slot of this unit's reduction range (split-K)
          // The skip connection of the NEXT row tile of this CTA (one contiguous block in either layout) is pulled
          // into L2 slice by slice while this tile is computed: fetched by the epilogue in one burst from HBM it
          // would stall the tile for ~6k cycles (128 KB at one SM's share of the HBM bandwidth).
          const char* pf_base = nullptr;
          uint32_t pf_bytes = 0, pf_slice = 0;
          if (EPI == 0 && se.residual != nullptr) {
            const int mt_next = ((mp + unit_step) / ks_n) * CTAS + rank;
            if (mt_next < la.num_m_tiles) {
              const int64_t rows_left = (int64_t)la.M - (int64_t)mt_next * kBM;
              const int rows = se.tiled ? kBM : (rows_left < kBM ? (int)rows_left : kBM);
              pf_base = reinterpret_cast<const char*>(se.residual + (int64_t)mt_next * kBM * se.ldr);
              pf_bytes = (uint32_t)rows * (uint32_t)se.ldr * 4u;
              pf_slice = ((pf_bytes / (uint32_t)(nk * n_tiles)) + 15u) & ~15u;
            }
          }
          uint32_t pf_done = 0;
          for (int nt = 0; nt < n_tiles; ++nt) {
            const int brow = nt * BN + rank * (BN / CTAS);  // this CTA's share of the weight rows of the tile
            for (int kc = 0; kc < nk; ++kc) {
              if (pf_done < pf_bytes) {
                const uint32_t nb = pf_bytes - pf_done < pf_slice ? pf_bytes - pf_done : pf_slice;
                bulk_prefetch_l2(pf_base + pf_done, nb);
                pf_done += nb;
              }
              if (CTAS == 2) {
                mbar_wait_cluster(empty_bar(s), ph ^ 1u);
              } else {
                mbar_wait(empty_bar(s), ph ^ 1u);
              }
              const uint32_t st = base + s * SM::STAGE_BYTES;
              mbar_expect_tx(full_bar(s), SM::A_BYTES + 2 * SM::B_BYTES);
              if (la.a_tiled == 2) {
                tma_load_2d(st, &tmA, mt * kBM, (k_base + kc) * BK, full_bar(s));  // BK rows of 128 values, as they lie
              } else if (la.a_tiled) {
                tma_load_4d(st, &tmA, 0, 0, (k_base + kc) * (BK / 4), mt, full_bar(s));
              } else {
                tma_load_2d(st, &tmA, (k_base + kc) * BK, mt * kBM, full_bar(s));
              }
              tma_load_2d(st + SM::A_PLANES * SM::A_BYTES, &tmB, (k_base + kc) * BK, brow, full_bar(s));
              tma_load_2d(st + SM::A_PLANES * SM::A_BYTES + SM::B_BYTES, &tmB, (k_base + kc) * BK, la.n_pad + brow,
                          full_bar(s));
              if (++s == STAGES) {
                s = 0;
                ph ^= 1u;
              }
            }
          }
        }
      }
    } else if (warp == 3 && EPI == 3) {
      // ---------------------------------------------------------------- staging manager (EPI 3)
      if (lane == 0) {
        constexpr uint32_t kTileBytes = kBM * BN * 4;
        uint32_t ph = 0;
        for (int mp = unit0; mp < n_units; mp += unit_step) {
          const int mt = (mp / ks_n) * CTAS + rank;
          for (int nt = 0; nt < n_tiles; ++nt) {
            // a T128 tile of 128 rows x BN columns is contiguous: tile mt, column groups nt*BN/4 ..;
            // a row-major tile moves as BN/32 boxes of 128 rows x 32 columns (128-byte swizzled rows in the staging
            // tile, tensor maps tmO / tmR; rows and columns outside the matrix are zero-filled / clipped by the TMA)
            const int64_t off = (int64_t)mt * kBM * se.ldo + (int64_t)nt * kBM * BN;
            if (se.residual != nullptr) {
              mbar_expect_tx(pfull_bar, kTileBytes);
              if (se.tiled) {
                bulk_load_1d(params_s, se.residual + (int64_t)mt * kBM * se.ldr + (int64_t)nt * kBM * BN, kTileBytes,
                             pfull_bar);
              } else {
#pragma unroll
                for (int cb = 0; cb < BN / 32; ++cb)
                  tma_load_2d(params_s + (uint32_t)(cb * kBM * 128), &tmR, nt * BN + cb * 32, mt * kBM, pfull_bar);
              }
            } else {
              mbar_arrive(pfull_bar);  // nothing to bring in: the tile may be written right away
            }
            mbar_wait(pempty_bar, ph);  // all epilogue warps have written their part (generic -> async fenced)
            if (se.tiled) {
              bulk_store_1d(se.out + off, params_s, kTileBytes);
            } else {
#pragma unroll
              for (int cb = 0; cb < BN / 32; ++cb)
                if (nt * BN + cb * 32 < se.n_out)  // split-K: range i writes rows [i * slice_rows, ...) of the partials
                  tma_store_2d(&tmO, nt * BN + cb * 32, (mp % ks_n) * (int)se.slice_stride + mt * kBM,
                               params_s + (uint32_t)(cb * kBM * 128));
              bulk_commit_group();
            }
            bulk_store_wait_read();     // the staging tile may be overwritten (next skip connection / next result)
            ph ^= 1u;
          }
        }
        bulk_store_wait_all();
      }
    } else if (warp == 1) {
      // ---------------------------------------------------------------- UMMA issuer (leader) / relay (peer)
      if (CTAS == 1 || rank == 0) {
        // The WHOLE warp walks the loop and waits on the barriers, one elected lane issues: with warp-uniform control
        // flow the descriptors stay in uniform registers.  (Issued from inside `if (lane == 0)` every tcgen05.mma
        // was preceded by a ~12-instruction vector->uniform register "waterfall" loop, ~130 dependent instructions
        // per stage, which is as long as the six MMAs of a stage take to execute: the issuing thread, not the
        // tensor pipe, set the pace.)
        constexpr uint32_t idesc = make_idesc_tf32(kBM * CTAS, BN);
        int s = 0, acc = 0;
        uint32_t ph = 0, aph = 0;
        const bool prof = FC_LINEAR_PROFILE && (la.debug & 4) && blockIdx.x == 0;
        long long t_tempty = 0, t_conv = 0, t_stages = 0;
        const long long t_begin = clock64();
        // descriptors of ring slot 0; slot s adds s * STAGE_BYTES to the 16-byte-granular address field
        const bool tiled = la.a_tiled != 0;
        const uint64_t a_hi0 = tiled ? make_smem_desc_noswizzle(base, kBM * 16, 128) : make_smem_desc(base, BK * 4);
        const uint64_t a_lo0 = tiled ? make_smem_desc_noswizzle(base + SM::A_BYTES, kBM * 16, 128)
                                     : make_smem_desc(base + SM::A_BYTES, BK * 4);
        const uint64_t b_hi0 = make_smem_desc(base + SM::A_PLANES * SM::A_BYTES, BK * 4);
        const uint64_t b_lo0 = make_smem_desc(base + SM::A_PLANES * SM::A_BYTES + SM::B_BYTES, BK * 4);
        // 8 k-values further along K: T128 operands (no swizzle) jump two column groups, swizzled ones 32 bytes
        const uint64_t a_step = tiled ? (uint64_t)((2 * kBM * 16) >> 4) : 2ull;
        for (int mp = unit0; mp < n_units; mp += unit_step) {
          for (int nt = 0; nt < n_tiles; ++nt) {
            for (int k0 = 0; k0 < nk; k0 += chunk) {
              const int k1 = k0 + chunk < nk ? k0 + chunk : nk;
              long long t0 = prof ? clock64() : 0;
              if (CTAS == 2) {
                mbar_wait_cluster(tempty_bar(acc), aph ^ 1u);
              } else {
                mbar_wait(tempty_bar(acc), aph ^ 1u);
              }
              if (prof) t_tempty += clock64() - t0;
              tc_fence_after();
              const uint32_t d = tmem_base + (uint32_t)(acc * BN);
              for (int kc = k0; kc < k1; ++kc) {
                if (prof) t0 = clock64();
                // the converters (of both CTAs of a pair) arrive only after THEIR wait on full_bar, so conv_bar also
                // covers the TMA boxes
                if (CTAS == 2) {
                  mbar_wait_cluster(conv_bar(s), ph);
                } else {
                  mbar_wait(conv_bar(s), ph);
                }
                if (prof) {
                  const long long t1 = clock64();
                  t_conv += t1 - t0;
                  t0 = t1;
                }
                if (prof) ++t_stages;
                tc_fence_after();
                const uint64_t so = (uint64_t)((uint32_t)s * (uint32_t)(SM::STAGE_BYTES >> 4));
                const uint64_t a_hi = a_hi0 + so, a_lo = a_lo0 + so, b_hi = b_hi0 + so, b_lo = b_lo0 + so;
                if (elect_one()) {
#pragma unroll
                  for (int kk = 0; kk < BK / 8; ++kk) {
                    const uint64_t o = (uint64_t)(kk * 2);  // 8 tf32 = 32 bytes = 2 x 16 B inside the swizzle span
                    const uint64_t oa = a_step * (uint64_t)kk;
                    const uint32_t first = (kc > k0 || kk > 0) ? 1u : 0u;
                    // small terms first, so they are not absorbed by the large one before they have been summed
                    if (TS) {
                      const uint32_t ta_hi = tmem_base + kTmemA0 + (uint32_t)(s * 2 * BK + kk * 8);
                      const uint32_t ta_lo = ta_hi + (uint32_t)BK;
                      if (CTAS == 2) {
                        umma_tf32_ts_pair(d, ta_lo, b_hi + o, idesc, first);
                        umma_tf32_ts_pair(d, ta_hi, b_lo + o, idesc, 1u);
                        umma_tf32_ts_pair(d, ta_hi, b_hi + o, idesc, 1u);
                      } else {
                        umma_tf32_ts(d, ta_lo, b_hi + o, idesc, first);
                        umma_tf32_ts(d, ta_hi, b_lo + o, idesc, 1u);
                        umma_tf32_ts(d, ta_hi, b_hi + o, idesc, 1u);
                      }
                    } else {
                      umma_tf32_ss(d, a_lo + oa, b_hi + o, idesc, first);
                      umma_tf32_ss(d, a_hi + oa, b_lo + o, idesc, 1u);
                      umma_tf32_ss(d, a_hi + oa, b_hi + o, idesc, 1u);
                    }
                  }
                  if (CTAS == 2) {
                    umma_commit_pair(empty_bar(s), 3);
                  } else {
                    umma_commit(empty_bar(s));
                  }
                  if (kc == k1 - 1) {
                    if (CTAS == 2) {
                      umma_commit_pair(tfull_bar(acc), 3);
                    } else {
                      umma_commit(tfull_bar(acc));
                    }
                  }
                }
                __syncwarp();
                if (++s == STAGES) {
                  s = 0;
                  ph ^= 1u;
                }
              }
              if (++acc == 2) {
                acc = 0;
                aph ^= 1u;
              }
            }
          }
        }
        if (prof && lane == 0) {
          g_lin_prof[0] = (unsigned long long)(clock64() - t_begin);
          g_lin_prof[1] = (unsigned long long)t_tempty;
          g_lin_prof[2] = 0;
          g_lin_prof[3] = (unsigned long long)t_conv;
          g_lin_prof[4] = 0;
          g_lin_prof[5] = (unsigned long long)t_stages;
        }
      }
    }
  } else if (warp < kEpiWarp0) {
    // ------------------------------------------------------------------ converters: raw fp32 -> (hi, lo) tf32
    set_max_regs_dec<RegBudget<SW>::kConverter>();
    const int ct = threadIdx.x - kConvWarp0 * 32;
    int s = 0;
    uint32_t ph = 0;
    const bool relu = la.relu_in != 0;
    const bool cprof = FC_LINEAR_PROFILE && (la.debug & 4) && blockIdx.x == 0 && warp == kConvWarp0;
    long long c_wait = 0, c_work = 0, c_t = cprof ? clock64() : 0;
    for (int mp = unit0; mp < n_units; mp += unit_step) {
      float csum = 0.f;  // column sum of this thread's operand row over the unit's reduction range (a_tiled == 2)
      for (int it = 0; it < n_tiles * nk; ++it) {
        mbar_wait(full_bar(s), ph);
        if (cprof) {
          const long long t = clock64();
          c_wait += t - c_t;
          c_t = t;
        }
        const uint32_t st = base + s * SM::STAGE_BYTES;
        if (TS) {
          tc_fence_after();  // the slot's previous MMAs completed (empty -> TMA -> full): order the stores after them
          // one thread = one row (= its TMEM lane): read the row's BK raw values, split, store into the operand ring
          static_assert(!TS || BK == 16 || BK == 32, "TS converter: 64- or 128-byte operand rows");
          const int r = (warp & 3) * 32 + lane;
          const uint32_t ta = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kTmemA0 + (uint32_t)(s * 2 * BK);
#pragma unroll
          for (int h = 0; h < BK / 16; ++h) {  // 16 k-values at a time
            float f[16];
            if (la.a_tiled == 2) {
              // transposed operand: the tile is [BK k-rows][128 values]; this thread's row is column r of every k-row
              // (a warp reads 32 consecutive words: conflict-free)
#pragma unroll
              for (int i = 0; i < 16; ++i) f[i] = lds32(st + (uint32_t)((h * 16 + i) * (kBM * 4) + r * 4));
              if (la.colsum != nullptr && it < nk) {  // first column tile only: later tiles re-read the same operand
                // pairwise inside the 16 values: the sequential chain is 16x shorter than the range
                const float s0 = (f[0] + f[1]) + (f[2] + f[3]), s1 = (f[4] + f[5]) + (f[6] + f[7]);
                const float s2 = (f[8] + f[9]) + (f[10] + f[11]), s3 = (f[12] + f[13]) + (f[14] + f[15]);
                csum += (s0 + s1) + (s2 + s3);
              }
            } else
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int cc = h * 4 + c;  // 16-byte chunk of the row
              // row-major tile: BK*4-byte rows, chunk cc of row r sits at chunk cc ^ swz(r) (TMA 64B / 128B swizzle)
              // T128 tile     : [BK/4 column groups][128 rows][16 B]
              const int swz = BK == 16 ? ((r >> 1) & 3) : (r & 7);
              const uint32_t off = la.a_tiled ? (uint32_t)(cc * kBM * 16 + r * 16)
                                              : (uint32_t)(r * (BK * 4) + ((cc ^ swz) << 4));
              const float4 t = lds128(st + off);
              f[4 * c + 0] = t.x;
              f[4 * c + 1] = t.y;
              f[4 * c + 2] = t.z;
              f[4 * c + 3] = t.w;
            }
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              split_tf32(relu ? fmaxf(f[i], 0.f) : f[i], hi[i], lo[i]);
            }
            tmem_st16(ta + (uint32_t)(h * 16), hi);
            tmem_st16(ta + (uint32_t)(BK + h * 16), lo);
          }
          tmem_wait_st();
          tc_fence_before();
        } else
#pragma unroll
        for (int v = ct; v < SM::A_BYTES / 16; v += kNumConv) {
          const uint32_t addr = st + (uint32_t)v * 16u;
          float4 f = lds128(addr);
          if (relu) {
            f.x = fmaxf(f.x, 0.f);
            f.y = fmaxf(f.y, 0.f);
            f.z = fmaxf(f.z, 0.f);
            f.w = fmaxf(f.w, 0.f);
          }
          uint32_t h0, h1, h2, h3, l0, l1, l2, l3;
          split_tf32(f.x, h0, l0);
          split_tf32(f.y, h1, l1);
          split_tf32(f.z, h2, l2);
          split_tf32(f.w, h3, l3);
          sts128(addr, h0, h1, h2, h3);
          sts128(addr + SM::A_BYTES, l0, l1, l2, l3);
        }
        if (!TS) fence_proxy_async_smem();  // (TS: nothing was written to shared memory)
        __syncwarp();
        if (lane == 0) {
          if (CTAS == 2) {
            mbar_arrive_remote_relaxed(conv_bar(s), 0);  // operand went to tensor memory: ordered by the tcgen05 fence
          } else {
            mbar_arrive(conv_bar(s));
          }
        }
        if (++s == STAGES) {
          s = 0;
          ph ^= 1u;
        }
        if (cprof) {
          const long long t = clock64();
          c_work += t - c_t;
          c_t = t;
        }
      }
      if (TS && la.a_tiled == 2 && la.colsum != nullptr) {
        const int mt = (mp / ks_n) * CTAS + rank;
        la.colsum[(int64_t)(mp % ks_n) * se.slice_stride + mt * kBM + (warp & 3) * 32 + lane] = csum;
      }
    }
    if (cprof && lane == 0) {
      g_lin_prof[12] = (unsigned long long)c_wait;
      g_lin_prof[13] = (unsigned long long)c_work;
    }
  } else if (warp < kEpiWarp0 + kEpiWarps) {
    // ------------------------------------------------------------------ epilogue / drain warps
    set_max_regs_inc<RegBudget<SW>::kEpilogue>();
    uint32_t pph = 0;  // phase of the parameter-tile hand-off (SW > 0) / staging tile (EPI 3)
    constexpr int NG = kEpiWarps / 4;          // column groups: 4 warps (one per TMEM lane quarter) each
    constexpr int NCOL = BN / NG;              // accumulator columns (and registers) per thread
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int half = (warp - kEpiWarp0) >> 2;  // which column group of the tile (columns / features)
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    int acc = 0;
    uint32_t aph = 0;
    int parity = 0;
    const bool eprof = FC_LINEAR_PROFILE && (la.debug & 4) && blockIdx.x == 0 && warp == kEpiWarp0;
    long long e_init = 0, e_wait = 0, e_drain = 0, e_final = 0, e_t = 0;
    const long long e_begin = clock64();
    for (int mp = unit0; mp < n_units; mp += unit_step) {
      const int mt = (mp / ks_n) * CTAS + rank;
      const int64_t row = (int64_t)mt * kBM + q * 32 + lane;
      const bool valid = row < la.M;
      float lad_acc = 0.f;
      for (int nt = 0; nt < n_tiles; ++nt) {
        float av[NCOL];
        if (eprof) e_t = clock64();
        // Start of the tile, while its first MMAs are still running: the register accumulators start from the bias
        // (+ the skip connection), and the affine transform's inputs are fetched, so that no global-load latency is
        // left between the last partial accumulator and the stores.
        const int rt = q * 32 + lane;
        int64_t o_base = 0, r_base = 0, n_mul = 1;
        float xv[EPI == 2 ? (BN / PPAD) / NG : 1];
        int xcol[EPI == 2 ? (BN / PPAD) / NG : 1];
        if (EPI == 3) {
          const float4* b4 = reinterpret_cast<const float4*>(la.bias + nt * BN + half * NCOL);
#pragma unroll
          for (int j = 0; j < NCOL / 4; ++j) {
            const float4 b = __ldg(b4 + j);
            av[4 * j + 0] = b.x;
            av[4 * j + 1] = b.y;
            av[4 * j + 2] = b.z;
            av[4 * j + 3] = b.w;
          }
        } else if (EPI == 0) {
          // T128: element (r, n) of tile mt at mt*128*W + ((n/4)*128 + r)*4: a warp's 32 rows of one column group
          // are 512 contiguous bytes (coalesced); row-major: 32 rows x 16 B scattered over 32 lines
          o_base = (se.tiled ? (int64_t)mt * kBM * se.ldo + rt * 4 : row * se.ldo) + (int64_t)(mp % ks_n) * se.slice_stride;
          r_base = se.tiled ? (int64_t)mt * kBM * se.ldr + rt * 4 : row * se.ldr;
          n_mul = se.tiled ? kBM : 1;  // float offset per unit of n (n is a multiple of 4)
          const int n0 = nt * BN + half * NCOL;
          const float4* b4 = reinterpret_cast<const float4*>(la.bias + n0);
          const bool res = se.residual != nullptr && (valid || se.tiled);
          // skip connection first, straight into the accumulator registers: 32 independent 16-byte loads in flight
          // (with the bias first the compiler funnels the residual through one temporary and serialises them).
          // The producer warp prefetched this tile's residual block into L2 while the previous tile was computed.
#pragma unroll
          for (int j = 0; j < NCOL / 4; ++j) {
            const int n = n0 + 4 * j;
            float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
            if (res && n < se.n_out) r = __ldg(reinterpret_cast<const float4*>(se.residual + r_base + n * n_mul));
            av[4 * j + 0] = r.x;
            av[4 * j + 1] = r.y;
            av[4 * j + 2] = r.z;
            av[4 * j + 3] = r.w;
          }
#pragma unroll
          for (int j = 0; j < NCOL / 4; ++j) {
            const float4 b = __ldg(b4 + j);
            av[4 * j + 0] += b.x;
            av[4 * j + 1] += b.y;
            av[4 * j + 2] += b.z;
            av[4 * j + 3] += b.w;
          }
        } else {
          constexpr int FEATS = BN / PPAD;
          constexpr int FH = FEATS / NG;
          if (EPI == 2 && nt == 0 && half == 0 && re.n_copy > 0 && re.y != re.x) {
            // identity columns (coupling.py:96-98): the warp copies its 32 rows one row per step (coalesced)
            const int64_t row0 = (int64_t)mt * kBM + q * 32;
            for (int i0 = 0; i0 < re.n_copy; i0 += 32) {
              const int cc = (i0 + lane < re.n_copy) ? __ldg(re.ccols + i0 + lane) : -1;
#pragma unroll 8
              for (int r = 0; r < 32; ++r) {
                if (cc >= 0 && row0 + r < la.M) re.y[(row0 + r) * re.ldy + cc] = __ldg(re.x + (row0 + r) * re.ldx + cc);
              }
            }
          }
#pragma unroll
          for (int f = 0; f < FH; ++f) {
            const int fl = half * FH + f;    // feature within the tile
            const int fg = nt * FEATS + fl;  // feature of the layer
            const bool live = fg < re.D_t;
            if (EPI == 2) {
              xcol[f] = live ? (re.tcols ? __ldg(re.tcols + fg) : fg) : 0;
              xv[f] = (valid && live) ? __ldg(re.x + row * re.ldx + xcol[f]) : 0.f;
            }
            if constexpr (PPAD % 4 == 0) {
              const float4* bp = reinterpret_cast<const float4*>(la.bias + (nt * BN + fl * PPAD));
#pragma unroll
              for (int i = 0; i < PPAD / 4; ++i) {
                const float4 b = __ldg(bp + i);
                av[f * PPAD + 4 * i + 0] = b.x;
                av[f * PPAD + 4 * i + 1] = b.y;
                av[f * PPAD + 4 * i + 2] = b.z;
                av[f * PPAD + 4 * i + 3] = b.w;
              }
            } else {
              const float2 b = __ldg(reinterpret_cast<const float2*>(la.bias + (nt * BN + fl * PPAD)));
              av[f * PPAD + 0] = b.x;
              av[f * PPAD + 1] = b.y;
            }
          }
        }
        if (eprof) {
          const long long t = clock64();
          e_init += t - e_t;
          e_t = t;
        }
        for (int ch = 0; ch < n_chunks; ++ch) {
          if (CTAS == 2) {
            mbar_wait_cluster(tfull_bar(acc), aph);
          } else {
            mbar_wait(tfull_bar(acc), aph);
          }
          if (eprof) {
            const long long t = clock64();
            e_wait += t - e_t;
            e_t = t;
          }
          tc_fence_after();
          const uint32_t tacc = tmem_base + lane_sel + (uint32_t)(acc * BN + half * NCOL);
          drain_partial<NCOL, false>(tacc, av);
          tc_fence_before();  // partial accumulator fully read by this warp: hand it back to the MMA warp
          __syncwarp();
          if (lane == 0) {
            if (CTAS == 2) {
              mbar_arrive_remote_relaxed(tempty_bar(acc), 0);  // ordered by the tcgen05 fence above
            } else {
              mbar_arrive(tempty_bar(acc));
            }
          }
          if (++acc == 2) {
            acc = 0;
            aph ^= 1u;
          }
          if (eprof) {
            const long long t = clock64();
            e_drain += t - e_t;
            e_t = t;
          }
        }
        if (EPI == 3) {
          // finished tile -> staging tile (same [column group][row][4 floats] order as the T128 layout); the skip
          // connection is already there (TMA), the manager warp stores the tile with one bulk copy
          mbar_wait(pfull_bar, pph);
          const uint32_t sb = params_s + (uint32_t)(((half * (NCOL / 4)) * kBM + rt) * 16);
          const bool res = se.residual != nullptr;
          const bool otiled = se.tiled != 0;
#pragma unroll
          for (int j = 0; j < NCOL / 4; ++j) {
            float4 o = make_float4(av[4 * j + 0], av[4 * j + 1], av[4 * j + 2], av[4 * j + 3]);
            // row-major staging: box cb = 32 columns, row rt = 128 bytes, 16-byte chunk ci at ci ^ (rt & 7)
            const int cg = half * (NCOL / 4) + j;  // 4-column group inside the tile
            const uint32_t a = otiled ? sb + (uint32_t)(j * kBM * 16)
                                      : params_s + (uint32_t)((cg >> 3) * kBM * 128 + rt * 128 + (((cg & 7) ^ (rt & 7)) << 4));
            if (res) {
              const float4 r = lds128(a);
              if (se.res_mask) {
                o.x = r.x > 0.f ? o.x : 0.f;
                o.y = r.y > 0.f ? o.y : 0.f;
                o.z = r.z > 0.f ? o.z : 0.f;
                o.w = r.w > 0.f ? o.w : 0.f;
              } else {
                o.x += r.x;
                o.y += r.y;
                o.z += r.z;
                o.w += r.w;
              }
            }
            if (se.relu_out) {
              o.x = fmaxf(o.x, 0.f);
              o.y = fmaxf(o.y, 0.f);
              o.z = fmaxf(o.z, 0.f);
              o.w = fmaxf(o.w, 0.f);
            }
            sts128(a, __float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(o.w));
          }
          fence_proxy_async_smem();  // the bulk store reads the tile through the async proxy
          __syncwarp();
          if (lane == 0) mbar_arrive(pempty_bar);
          pph ^= 1u;
        } else if (EPI == 0) {
          const int n0 = nt * BN + half * NCOL;
#pragma unroll
          for (int j = 0; j < NCOL / 4; ++j) {
            float4 o = make_float4(av[4 * j + 0], av[4 * j + 1], av[4 * j + 2], av[4 * j + 3]);
            const int n = n0 + 4 * j;
            if ((valid || se.tiled) && n < se.n_out) {  // T128 buffers hold whole tiles: tail rows are written too
              if (se.relu_out) {
                o.x = fmaxf(o.x, 0.f);
                o.y = fmaxf(o.y, 0.f);
                o.z = fmaxf(o.z, 0.f);
                o.w = fmaxf(o.w, 0.f);
              }
              *reinterpret_cast<float4*>(se.out + o_base + n * n_mul) = o;
            }
          }
        } else if (EPI == 1) {
          // hand the finished parameter tile to the spline warps: column-major [BN][128 rows] words
          mbar_wait(pempty_bar, pph ^ 1u);
          const uint32_t pbase = params_s + (uint32_t)((half * NCOL) * kBM + q * 32 + lane) * 4u;
#pragma unroll
          for (int j = 0; j < NCOL; ++j) sts32(pbase + (uint32_t)(j * kBM * 4), av[j]);
          __syncwarp();
          if (lane == 0) mbar_arrive(pfull_bar);
          pph ^= 1u;
        } else {
          constexpr int FEATS = BN / PPAD;
          constexpr int FH = FEATS / NG;
          static_assert(FH * PPAD == NCOL && FH >= 1, "feature groups must tile the column group exactly");
#pragma unroll
          for (int f = 0; f < FH; ++f) {
            const int fg = nt * FEATS + half * FH + f;  // feature of the layer
            if (fg < re.D_t) {
              float yv, lv;
              affine_eval(xv[f], av[f * PPAD], av[f * PPAD + 1], re.activation, re.c.inverse, yv, lv);
              if (valid) re.y[row * re.ldy + xcol[f]] = yv;
              lad_acc += lv;
            }
          }
        }
      }
      if (EPI == 2) {
        // per-sample log|det J| (sum_except_batch, utils/torchutils.py:25-30): this thread summed its features in
        // order; the two column halves of a row are combined in a fixed order through shared memory
        float* ex = lad_x + parity * 3 * kBM;
        if (half > 0) ex[q * 32 + lane] = lad_acc;
        named_barrier_sync(1, 32 * kEpiWarps);
        if (half == 0 && valid) {
          const float tot = lad_acc + ex[q * 32 + lane];
          re.lad[row] = re.accumulate ? re.lad[row] + tot : tot;
        }
        parity ^= 1;
      }
    }
    if (eprof && lane == 0) {
      g_lin_prof[8] = (unsigned long long)(clock64() - e_begin);
      g_lin_prof[9] = (unsigned long long)e_init;
      g_lin_prof[10] = (unsigned long long)e_wait;
      g_lin_prof[11] = (unsigned long long)e_drain;
    }
  } else {
    // ------------------------------------------------------------------ spline warps (SW > 0)
    if constexpr (SW > 0) {
      set_max_regs_dec<RegBudget<SW>::kSpline>();
      constexpr int FEATS = BN / PPAD;
      constexpr int FG = FEATS / 2;             // features per thread and tile: two thread groups of 128 rows
      const int t = threadIdx.x - 32 * (kEpiWarp0 + kEpiWarps);
      const int r = t & (kBM - 1), g = t >> 7;  // row of the tile, feature group
      uint32_t pph = 0;
      unsigned status = 0;
      int parity = 0;
      for (int mp = unit0; mp < n_units; mp += unit_step) {
        const int mt = (mp / ks_n) * CTAS + rank;
        const int64_t row = (int64_t)mt * kBM + r;
        const bool valid = row < la.M;
        float lad_acc = 0.f;
        if (re.n_copy > 0 && re.y != re.x) {
          // identity columns (coupling.py:96-98): each warp copies its 32 rows, one row per step (coalesced)
          const int64_t row0 = (int64_t)mt * kBM + (r & ~31);
          if (g == 0) {
            for (int i0 = 0; i0 < re.n_copy; i0 += 32) {
              const int cc = (i0 + lane < re.n_copy) ? __ldg(re.ccols + i0 + lane) : -1;
#pragma unroll 8
              for (int rr = 0; rr < 32; ++rr) {
                if (cc >= 0 && row0 + rr < la.M) re.y[(row0 + rr) * re.ldy + cc] = __ldg(re.x + (row0 + rr) * re.ldx + cc);
              }
            }
          }
        }
        for (int nt = 0; nt < n_tiles; ++nt) {
          float xv[FG];
          int xcol[FG];
#pragma unroll
          for (int f = 0; f < FG; ++f) {  // inputs first: their latency hides behind the wait for the parameters
            const int fg = nt * FEATS + g * FG + f;
            const bool live = fg < re.D_t;
            xcol[f] = live ? (re.tcols ? __ldg(re.tcols + fg) : fg) : 0;
            xv[f] = (valid && live) ? __ldg(re.x + row * re.ldx + xcol[f]) : 0.f;
          }
          mbar_wait(pfull_bar, pph);
#pragma unroll 1
          for (int f = 0; f < FG; ++f) {
            const int fg = nt * FEATS + g * FG + f;
            float p[PPAD];
            const uint32_t pb = params_s + (uint32_t)(((g * FG + f) * PPAD) * kBM + r) * 4u;
#pragma unroll
            for (int i = 0; i < PPAD; ++i) p[i] = lds32(pb + (uint32_t)(i * kBM * 4));
            if (fg < re.D_t) {
              float xval = xv[0];
              int xc = xcol[0];
#pragma unroll
              for (int k = 1; k < FG; ++k) {
                xval = (k == f) ? xv[k] : xval;
                xc = (k == f) ? xcol[k] : xc;
              }
              float yv, lv;
              rqs_eval<KC, true>(re.c, xval, p, yv, lv, status);
              if (valid) re.y[row * re.ldy + xc] = yv;
              lad_acc += lv;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(pempty_bar);
          pph ^= 1u;
        }
        // per-sample log|det J|: the two feature groups of a row are combined in a fixed order
        float* ex = lad_x + parity * kBM;
        if (g == 1) ex[r] = lad_acc;
        named_barrier_sync(2, 32 * SW);
        if (g == 0 && valid) {
          const float tot = lad_acc + ex[r];
          re.lad[row] = re.accumulate ? re.lad[row] + tot : tot;
        }
        parity ^= 1;
      }
      if (status != 0 && re.status) atomicOr(re.status, (int)status);
    }
  }

  __syncwarp();  // the role branches leave most warps diverged; the cluster barrier is warp-aligned
  tc_fence_before();
  if (CTAS == 2) {
    cluster_sync_all();  // no CTA leaves (or frees tensor memory) while its partner can still signal it
  } else {
    __syncthreads();
  }
  if (warp == 2) {
    tc_fence_after();
    if (CTAS == 2) {
      tmem_dealloc_pair(tmem_base, kTmemCols);
    } else {
      tmem_dealloc(tmem_base, kTmemCols);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess) p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// [rows, cols] fp32 row-major matrix with row stride `ld` elements; box = box_rows x bk, swizzle span = bk * 4 bytes
static int make_map(CUtensorMap* m, const float* ptr, uint64_t rows, uint64_t cols, uint64_t ld, int box_rows, int bk) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return FC_ERR_CUDA;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {ld * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = bk == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? FC_OK : FC_ERR_CUDA;
}

// un-swizzled 2-D map: boxes of box_rows x box_cols (box_cols * 4 bytes a multiple of 16)
static int make_map_plain(CUtensorMap* m, const float* ptr, uint64_t rows, uint64_t cols, uint64_t ld, int box_rows,
                          int box_cols) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return FC_ERR_CUDA;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {ld * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? FC_OK : FC_ERR_CUDA;
}

// T128 activation buffer [tiles][W/4 column groups][128 rows][4 floats]: one (tile, column group) is 2 KB contiguous,
// described as 8 rows of 256 B so that the TMA moves wide rows; box = BK/4 column groups of one tile.
static int make_map_t128(CUtensorMap* m, const float* ptr, uint64_t tiles, uint64_t width, int bk) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return FC_ERR_CUDA;
  const cuuint64_t dims[4] = {64, 8, width / 4, tiles};
  const cuuint64_t strides[3] = {256, 2048, (cuuint64_t)kBM * width * sizeof(float)};
  const cuuint32_t box[4] = {64, 8, (cuuint32_t)(bk / 4), 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? FC_OK : FC_ERR_CUDA;
}

// k-values per partial accumulator (see "Accumulation" at the top).  Short dot products leave less room between
// the tensor core's truncation error and the (smaller) rounding noise of an fp32 FMA chain of the same length, so
// they are drained after every stage.
static int chunk_k(int K) { return K <= 64 ? 16 : 32; }

template <int EPI, int BN, int BK, int STAGES, int KC, int PPAD, bool PAIR>
static int launch_linear(const float* A, int64_t lda, int64_t M, int K, const fc_linear_weights* w, LinArgs la,
                         const StoreEpi& se, const RqsEpi& re, cudaStream_t stream) {
  constexpr int CTAS = PAIR ? 2 : 1;
  using SM = LinSmem<EPI, BN, BK, STAGES, CTAS>;
  static_assert(SM::TOTAL <= 232448, "shared memory per CTA");
  if (w->n_pad % BN != 0 || w->k_pad % 32 != 0) return FC_ERR_INVALID_ARGUMENT;
  CUtensorMap tmA, tmB;
  int rc = la.a_tiled == 2 ? make_map_plain(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, BK, kBM)
           : la.a_tiled    ? make_map_t128(&tmA, A, (uint64_t)((M + kBM - 1) / kBM), (uint64_t)lda, BK)
                           : make_map(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, kBM, BK);
  if (rc != FC_OK) return rc;
  rc = make_map(&tmB, w->w, (uint64_t)2 * w->n_pad, (uint64_t)w->k_pad, (uint64_t)w->k_pad, BN / CTAS, BK);
  if (rc != FC_OK) return rc;
  CUtensorMap tmO = tmA, tmR = tmA;  // only the staged store kernel with a row-major result reads these
  if (EPI == 3 && !se.tiled) {
    // (split-K: the partial products of all ranges form one matrix of k_slices * slice_stride rows)
    const uint64_t out_rows = la.k_slices > 1 ? (uint64_t)la.k_slices * (uint64_t)se.slice_stride : (uint64_t)M;
    rc = make_map(&tmO, se.out, out_rows, (uint64_t)se.n_out, (uint64_t)se.ldo, kBM, 32);
    if (rc != FC_OK) return rc;
    if (se.residual) {
      rc = make_map(&tmR, se.residual, (uint64_t)M, (uint64_t)se.n_out, (uint64_t)se.ldr, kBM, 32);
      if (rc != FC_OK) return rc;
    }
  }
  la.M = (int)M;
  la.num_k_stages = (K + BK - 1) / BK;
  if (la.k_slices < 1) la.k_slices = 1;
  if (la.k_slices > 1) la.num_k_stages = (la.num_k_stages + la.k_slices - 1) / la.k_slices;  // slots per range
  la.chunk = chunk_k(K) / BK > 0 ? chunk_k(K) / BK : 1;
  la.num_m_tiles = (int)((M + kBM - 1) / kBM);
  la.n_pad = w->n_pad;
  la.bias = w->bias;
  static const int debug = [] {
    const char* e = getenv("FC_LINEAR_DEBUG");
    return e ? atoi(e) : 0;
  }();
  la.debug = debug;
  auto kern = linear_tf32x3_kernel<EPI, BN, BK, STAGES, KC, PPAD, PAIR>;
  // the opt-in shared-memory size is a per-device function attribute: set it once per (instantiation, device)
  static std::atomic<uint64_t> configured{0};
  int dev_id = 0;
  cudaGetDevice(&dev_id);
  const uint64_t dev_bit = 1ull << (dev_id & 63);
  if (!(configured.load(std::memory_order_acquire) & dev_bit)) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL) != cudaSuccess)
      return FC_ERR_CUDA;
    configured.fetch_or(dev_bit, std::memory_order_release);
  }
  const int units = ((la.num_m_tiles + CTAS - 1) / CTAS) * la.k_slices;
  const int max_units = device_info().sm_count / CTAS;
  const int grid = (units < max_units ? units : max_units) * CTAS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kBaseThreads + 32 * (kEpiWarps + spline_warps(EPI)));
  cfg.dynamicSmemBytes = SM::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTAS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmO, tmR, la, se, re) != cudaSuccess) return FC_ERR_CUDA;
  FC_CHECK_LAUNCH();
  return FC_OK;
}

static int check_operand(const float* A, int64_t lda, int64_t M, int K, const fc_linear_weights* w, int a_tiled) {
  if (M == 0 && w && K > 0) return FC_OK;  // empty batch: nothing to read (the pointer may be null)
  if (!A || !w || !w->w || !w->bias || M < 0 || K <= 0) return FC_ERR_INVALID_ARGUMENT;
  if (M >= (int64_t)1 << 31) return FC_ERR_UNSUPPORTED;
  if (K > w->k_pad) return FC_ERR_INVALID_ARGUMENT;
  if (a_tiled && (lda != K || (K & 15))) return FC_ERR_INVALID_ARGUMENT;  // T128: width == K, a multiple of 16
  // TMA: 16-byte aligned base and row pitch
  if ((reinterpret_cast<uintptr_t>(A) & 15) || (lda & 3) || lda < K) return FC_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(w->w) & 15) || (reinterpret_cast<uintptr_t>(w->bias) & 15)) return FC_ERR_UNSUPPORTED;
  return FC_OK;
}

__global__ void pack_kernel(const float* __restrict__ W, int64_t ldw, const float* __restrict__ mask, int64_t ldm,
                            const float* __restrict__ bias, const int32_t* __restrict__ row_map,
                            const int32_t* __restrict__ col_map, int N, int K, int n_pad, int k_pad,
                            float* __restrict__ out_w, float* __restrict__ out_b) {
  const int64_t total = (int64_t)N * K;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i / K), k = (int)(i % K);
    float wv = W[n * ldw + k];
    if (mask) wv = wv * mask[n * ldm + k];  // MaskedLinear: weight * mask (made.py:72)
    const int rn = row_map ? row_map[n] : n;
    const int ck = col_map ? col_map[k] : k;
    const uint32_t hi = tc::to_tf32(wv);
    const uint32_t lo = tc::to_tf32(wv - __uint_as_float(hi));
    out_w[(int64_t)rn * k_pad + ck] = __uint_as_float(hi);
    out_w[((int64_t)n_pad + rn) * k_pad + ck] = __uint_as_float(lo);
    if (k == 0) out_b[rn] = bias ? bias[n] : 0.f;
  }
}

// Transposing weight producer for the split-K weight-gradient product: the reduction axis (the batch) has to be the
// contiguous one.  128 x 32 tiles through shared memory, coalesced on both sides.
//   dst[0][c][r] = tf32_hi(src[r][c]), dst[1][c][r] = tf32(src[r][c] - hi)   (x [B, K] -> packed planes)
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ src, int64_t lds, int64_t rows, int cols,
                                                        float* __restrict__ dst, int64_t ldd, int64_t plane_stride,
                                                        int relu) {
  // 128 rows x 32 columns per block: 16 independent 128-byte row reads in flight per warp, then 16-byte vector
  // writes along the (contiguous) row axis of the transposed result.  tile_t[c][r], row stride 132 floats: the
  // vector reads are conflict-free, the scalar writes 4-way (shared memory is not the limit here, HBM is).
  __shared__ __align__(16) float tile_t[32][132];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.x * 128;
  const int c0 = blockIdx.y * 32;
  float v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int64_t r = r0 + warp + 8 * i;
    const int c = c0 + lane;
    v[i] = (r < rows && c < cols) ? __ldcs(src + r * lds + c) : 0.f;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) tile_t[lane][warp + 8 * i] = relu ? fmaxf(v[i], 0.f) : v[i];
  __syncthreads();
  const bool vec = (ldd & 3) == 0 && (plane_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + warp * 4 + i;
    const int64_t r = r0 + 4 * lane;
    if (c >= cols || r >= rows) continue;
    const float4 t = *reinterpret_cast<const float4*>(&tile_t[warp * 4 + i][4 * lane]);
    const float e[4] = {t.x, t.y, t.z, t.w};
    float hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t h = tc::to_tf32(e[j]);
      hi[j] = __uint_as_float(h);
      lo[j] = __uint_as_float(tc::to_tf32(e[j] - hi[j]));
    }
    float* d = dst + (int64_t)c * ldd + r;
    if (vec && r + 3 < rows) {
      *reinterpret_cast<float4*>(d) = make_float4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<float4*>(d + plane_stride) = make_float4(lo[0], lo[1], lo[2], lo[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (r + j < rows) {
          d[j] = hi[j];
          d[plane_stride + j] = lo[j];
        }
      }
    }
  }
}

}  // namespace fc

using namespace fc;

extern "C" int fc_linear_pack_transposed(const float* X, int64_t x_row_stride, int64_t B, int32_t K, int32_t n_pad,
                                         int32_t k_pad, int32_t relu, float* w_packed, float* bias_packed,
                                         void* stream) {
  if (B <= 0 || K <= 0 || !X || !w_packed || !bias_packed || n_pad < K || k_pad < B || (k_pad % 32) || (n_pad % 16))
    return FC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  // the padding (rows K..n_pad of both planes, columns B..k_pad) must read as zero
  if ((n_pad != K || k_pad != B) &&
      cudaMemsetAsync(w_packed, 0, sizeof(float) * 2 * (size_t)n_pad * k_pad, st) != cudaSuccess)
    return FC_ERR_CUDA;
  if (cudaMemsetAsync(bias_packed, 0, sizeof(float) * (size_t)n_pad, st) != cudaSuccess) return FC_ERR_CUDA;
  const dim3 grid((unsigned)((B + 127) / 128), (unsigned)((K + 31) / 32));
  transpose_kernel<<<grid, 256, 0, st>>>(X, x_row_stride, B, K, w_packed, k_pad, (int64_t)n_pad * k_pad, relu);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int fc_linear_debug_profile(unsigned long long* out16) {
  if (!out16) return FC_ERR_INVALID_ARGUMENT;
  if (cudaMemcpyFromSymbol(out16, g_lin_prof, sizeof(unsigned long long) * 16) != cudaSuccess) return FC_ERR_CUDA;
  return FC_OK;
}

extern "C" int fc_linear_pack(const float* W, int64_t w_row_stride, const float* mask, int64_t mask_row_stride,
                              const float* bias, int32_t N, int32_t K, const int32_t* row_map, const int32_t* col_map,
                              int32_t n_pad, int32_t k_pad, float* w_packed, float* bias_packed, void* stream) {
  if (!W || !w_packed || !bias_packed || N <= 0 || K <= 0 || n_pad < N || k_pad < K) return FC_ERR_INVALID_ARGUMENT;
  if (k_pad % 32 != 0 || n_pad % 16 != 0) return FC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(w_packed, 0, sizeof(float) * 2 * (size_t)n_pad * k_pad, st) != cudaSuccess) return FC_ERR_CUDA;
  if (cudaMemsetAsync(bias_packed, 0, sizeof(float) * (size_t)n_pad, st) != cudaSuccess) return FC_ERR_CUDA;
  const int64_t total = (int64_t)N * K;
  const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_kernel<<<blocks, 256, 0, st>>>(W, w_row_stride, mask, mask_row_stride, bias, row_map, col_map, N, K, n_pad, k_pad,
                                      w_packed, bias_packed);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int fc_linear_apply(const float* A, int64_t lda, int64_t M, int32_t K, const fc_linear_weights* w,
                               int32_t relu_in, float* out, int64_t ldo, int32_t n_out, int32_t relu_out,
                               const float* residual, int64_t ldr, int32_t layouts, void* stream) {
  const int a_tiled = (layouts & FC_LINEAR_A_T128) != 0, o_tiled = (layouts & FC_LINEAR_OUT_T128) != 0;
  const int res_mask = (layouts & FC_LINEAR_RESIDUAL_GATES) != 0;
  if (res_mask && !residual) return FC_ERR_INVALID_ARGUMENT;
  int rc = check_operand(A, lda, M, K, w, a_tiled);
  if (rc != FC_OK) return rc;
  if (M == 0) return FC_OK;  // empty batch (null data pointers are fine)
  if (!out || n_out <= 0 || n_out > w->n_pad) return FC_ERR_INVALID_ARGUMENT;
  if ((n_out & 3) || (ldo & 3) || (reinterpret_cast<uintptr_t>(out) & 15)) return FC_ERR_UNSUPPORTED;
  if (residual && ((ldr & 3) || (reinterpret_cast<uintptr_t>(residual) & 15))) return FC_ERR_UNSUPPORTED;
  if (o_tiled && (ldo != n_out || (residual && ldr != n_out))) return FC_ERR_INVALID_ARGUMENT;
  if (M == 0) return FC_OK;
  LinArgs la{};
  la.relu_in = relu_in;
  la.a_tiled = a_tiled;
  StoreEpi se{out, ldo, residual, ldr, n_out, relu_out, o_tiled, res_mask, 0};
  RqsEpi re{};
  constexpr int BN = 256;
  if (w->n_pad % BN != 0) return FC_ERR_INVALID_ARGUMENT;
  la.num_n_tiles = (n_out + BN - 1) / BN;
  cudaStream_t st = (cudaStream_t)stream;
  if (!o_tiled || n_out % 128 == 0) {
    // staged kernel (operand in TMEM, CTA pairs): a T128 output in whole 128-wide tiles leaves by TMA bulk copies, a
    // row-major one (the staging tile and the skip connection) through 2-D tensor maps
    la.num_n_tiles = (n_out + 127) / 128;
    // (short reductions keep 16-value slots: their partial accumulators are drained every 16 k-values)
    if (K > 64) return launch_linear<3, 128, 32, 4, 0, 32, true>(A, lda, M, K, w, la, se, re, st);
    return launch_linear<3, 128, 16, 8, 0, 32, true>(A, lda, M, K, w, la, se, re, st);
  }
  if (res_mask) return FC_ERR_UNSUPPORTED;  // only the staged kernel gates
  return launch_linear<0, BN, 16, 4, 0, 32, false>(A, lda, M, K, w, la, se, re, st);
}

extern "C" int fc_linear_rqs_apply(const float* hidden, int64_t ldh, int64_t B, int32_t H, const fc_linear_weights* w,
                                   int32_t relu_in, const float* x, int64_t x_row_stride, float* y,
                                   int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int32_t D_t,
                                   fc_cols tcols, fc_cols ccols, const fc_rqs_config* cfg, int32_t* status,
                                   int32_t layouts, void* stream) {
  RqsParams c;
  int rc = make_rqs_params(cfg, c);
  if (rc != FC_OK) return rc;
  const int a_tiled = (layouts & FC_LINEAR_A_T128) != 0;
  rc = check_operand(hidden, ldh, B, H, w, a_tiled);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  if (!x || !y || !logabsdet || D_t <= 0) return FC_ERR_INVALID_ARGUMENT;
  if (tcols.idx && tcols.n != D_t) return FC_ERR_INVALID_ARGUMENT;
  if (c.tails != FC_TAILS_LINEAR) return FC_ERR_UNSUPPORTED;  // fused epilogue: linear tails (P = 3K-1) only
  if (B == 0) return FC_OK;
  LinArgs la{};
  la.relu_in = relu_in;
  la.a_tiled = a_tiled;
  StoreEpi se{};
  RqsEpi re{x, x_row_stride, y, y_row_stride, logabsdet, accumulate_logabsdet, tcols.idx, ccols.idx, ccols.n, D_t, c, status};
  if (c.K != 8 && c.K != 16) return FC_ERR_UNSUPPORTED;
  constexpr int BN = 192;
  const int feats = BN / (3 * c.K);  // features per tile: 3K - 1 parameters padded to PP = 3K columns each
  la.num_n_tiles = (D_t + feats - 1) / feats;
  if (w->n_pad < la.num_n_tiles * BN) return FC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  if (c.K == 8) return launch_linear<1, BN, 16, 4, 8, 24, true>(hidden, ldh, B, H, w, la, se, re, st);
  return launch_linear<1, BN, 16, 4, 16, 48, true>(hidden, ldh, B, H, w, la, se, re, st);
}

extern "C" int fc_linear_affine_apply(const float* hidden, int64_t ldh, int64_t B, int32_t H, const fc_linear_weights* w,
                                      int32_t relu_in, const float* x, int64_t x_row_stride, float* y,
                                      int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int32_t D_t,
                                      fc_cols tcols, fc_cols ccols, int32_t activation, int32_t inverse,
                                      int32_t layouts, void* stream) {
  const int a_tiled = (layouts & FC_LINEAR_A_T128) != 0;
  int rc = check_operand(hidden, ldh, B, H, w, a_tiled);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  if (!x || !y || !logabsdet || D_t <= 0) return FC_ERR_INVALID_ARGUMENT;
  if (tcols.idx && tcols.n != D_t) return FC_ERR_INVALID_ARGUMENT;
  if (activation < FC_SCALE_SIGMOID2 || activation > FC_SCALE_SOFTPLUS_EPS) return FC_ERR_INVALID_ARGUMENT;
  if (B == 0) return FC_OK;
  LinArgs la{};
  la.relu_in = relu_in;
  la.a_tiled = a_tiled;
  StoreEpi se{};
  RqsEpi re{x, x_row_stride, y, y_row_stride, logabsdet, accumulate_logabsdet, tcols.idx, ccols.idx, ccols.n, D_t, {}, nullptr,
            activation};
  re.c.inverse = inverse;
  constexpr int BN = 64;  // 32 features per tile: the affine final layer is narrow (2 columns per feature)
  la.num_n_tiles = (2 * D_t + BN - 1) / BN;
  if (w->n_pad < la.num_n_tiles * BN) return FC_ERR_INVALID_ARGUMENT;
  return launch_linear<2, BN, 16, 8, 0, 2, false>(hidden, ldh, B, H, w, la, se, re, (cudaStream_t)stream);
}

// Weight-gradient form of the split-K product: At is the A operand TRANSPOSED, [K, M] row-major (grad_y [B, N] as the
// backward pass holds it), so no transposed copy of it is ever written.  The tile goes to tensor memory through the
// converter warps (thread m of a row tile reads column m of every k-row), the result leaves through the staged store:
// partials[i] (rows [i * slice_rows, i * slice_rows + M) of a [k_slices * slice_rows, ldo] matrix, slice_rows a multiple of
// 256 >= M) holds the product over reduction range i.  colsum (optional, [k_slices][slice_rows]) receives the column
// sums of At over each range: summed over the ranges they are the bias gradient grad_y.sum(0).
extern "C" int fc_linear_splitk_t_apply(const float* At, int64_t ldat, int64_t M, int64_t K, const fc_linear_weights* w,
                                        int32_t k_slices, float* partials, int64_t slice_rows, int64_t ldo,
                                        int32_t n_out, float* colsum, void* stream) {
  if (!At || !w || !w->w || !w->bias || M <= 0 || K <= 0 || M >= ((int64_t)1 << 31) || K >= ((int64_t)1 << 31))
    return FC_ERR_INVALID_ARGUMENT;
  if (!partials || n_out <= 0 || n_out > w->n_pad || k_slices < 1) return FC_ERR_INVALID_ARGUMENT;
  if (K > w->k_pad || ldat < M) return FC_ERR_INVALID_ARGUMENT;
  if ((ldat & 3) || (reinterpret_cast<uintptr_t>(At) & 15) || (n_out & 3) || (ldo & 3) ||
      (reinterpret_cast<uintptr_t>(partials) & 15))
    return FC_ERR_UNSUPPORTED;
  if (slice_rows < M || (slice_rows % 256) || (int64_t)k_slices * slice_rows >= ((int64_t)1 << 31)) return FC_ERR_INVALID_ARGUMENT;
  if (w->n_pad % 128 != 0) return FC_ERR_INVALID_ARGUMENT;
  LinArgs la{};
  la.k_slices = k_slices;
  la.a_tiled = 2;
  la.colsum = colsum;
  StoreEpi se{partials, ldo, nullptr, 0, n_out, 0, 0, 0, slice_rows};
  RqsEpi re{};
  la.num_n_tiles = (n_out + 127) / 128;
  return launch_linear<3, 128, 32, 4, 0, 32, true>(At, ldat, M, (int)K, w, la, se, re, (cudaStream_t)stream);
}
