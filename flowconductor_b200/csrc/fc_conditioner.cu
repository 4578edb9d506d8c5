// fc_conditioner.cu — a WHOLE conditioner network and the bijection it parameterises in ONE persistent kernel
// (SURVEY.md 8(f) n1; DESIGN.md 4.12).
//
// Replaces, per flow layer, ResidualNet.forward (flowcon/nn/nets/resnet.py:92-100: initial layer, pre-activation
// residual blocks :39-56, final layer) or the residual MADE (flowcon/transforms/made.py:274-283, blocks :170-181,
// MaskedLinear :71-72) TOGETHER WITH the rational-quadratic spline that consumes its output
// (flowcon/transforms/splines/rational_quadratic.py:13-181 through coupling.py:549-582 / autoregressive.py:578-615).
// The per-layer kernels of fc_linear.cu write every [B, H] activation to HBM and read it back (12.8 GB per flow layer
// at cfg 2); here a 128-row activation tile never leaves the SM:
//
//   registers      fp32 accumulators of the layer being computed (one thread = one row x 64 columns per N tile)
//   tensor memory  the layer's A operand [128 rows x K <= 256] as fp16 (hi, lo) planes (256 columns), and two partial
//                  accumulators of 128 columns (256 columns)
//   shared memory  the residual stream h [256 columns][128 rows] fp32 (128 KB, touched only by the thread that owns
//                  the entry), a ring of weight slots streamed from L2 by 1-D TMA bulk copies, barriers
//
// Arithmetic: "3xFP16".  The reference computes these products in fp32.  Every operand is split a = hi + lo with hi, lo
// fp16 (11 significant bits each, like the tf32 split of fc_linear.cu) after scaling by an exact power of two — per
// (row, 64-value chunk) for the activations, per layer for the weights — so that the largest magnitude sits in
// [2^7, 2^14) (activations; the sum of the chunk's magnitudes is scaled into [2^13, 2^14)) or [2^13, 2^14) (weights):
// hi + lo then reproduces the scaled value to 2^-22 relative (2^-32 of the chunk's maximum for small entries), and
// nothing overflows fp16.  Products  lo*hi + hi*lo + hi*hi  run as tcgen05.mma.kind::f16 (twice the
// tf32 rate, measured: scripts/microbench/tmem_rate.cu) into an fp32 accumulator in tensor memory.  As in
// fc_linear.cu the tensor core truncates on accumulation, so every 64 k-values (12 MMAs) the partial sum is handed
// to the row's thread, which adds  partial * 2^-e(row, chunk)  into a register accumulator with round-to-nearest while
// the next partial is computed in the other TMEM buffer; the weight scale 2^-e(n) is applied together with the bias.
//
// The thread that owns (row, 64 columns) applies bias / skip connection / ReLU to its finished values, converts them
// to the (hi, lo) operand of the NEXT layer and writes that straight into tensor memory (tcgen05.st): there are no
// converter warps and no activation traffic at all.  The final layer runs in N tiles of 96 columns (4 features x 24
// padded parameters for 8 bins, 2 x 48 for 16 bins): the row threads only accumulate its partial sums and drop each
// finished 128 x 96 parameter tile into shared memory (two buffers in the residual stream's space, which is dead by
// then); four more warps — one thread per row — evaluate the splines from there while the tensor core and the row
// threads are already on the next N tile (and, for the last N tiles, on the next row tile's first layers).  Measured
// before this split: with the spline inside the row threads the final layer took 2.3x its MMA time.
//
// CTA pairs (cta_group::2): one MMA covers 256 rows (128 per SM); each SM stages half of every weight slot.
// Warps: 0 TMA producer, 1 MMA issuer (leader CTA), 2 TMEM allocator, 3 relay ("my half of the slot has landed" to
// the leader), 4-11 row threads (two per row), 12-15 bijection threads (one per row).  Every mbarrier wait is bounded
// (kTimeoutCycles): a protocol error ends the kernel with a code in the error word instead of hanging the GPU.
#include <atomic>
#include <cstdlib>
#include <cuda_fp16.h>

#include "fc_common.cuh"
#include "fc_tc.cuh"

namespace fc {

using namespace tc;

constexpr int kCM = 128;              // rows per CTA (= TMEM lanes)
constexpr int kSlotBytes = 16384;     // ring slot per CTA: (hi | lo) planes of <= 64 weight rows x 64 fp16
constexpr int kCondStages = 4;
constexpr int kCondThreads = 512;     // 4 control warps, 8 row warps, 4 bijection warps
constexpr int kRowWarps = 8, kBijWarps = 4;
constexpr int kVecBytes = 20480;      // bias of every output column of every layer (fp32), then 1 / weight scale per layer
constexpr int kMaxCondLayers = FC_COND_MAX_LAYERS;
constexpr uint32_t kTmemAcc = 0;      // two partial accumulators, 128 columns apart
constexpr uint32_t kTmemA = 256;      // operand: hi plane (128 columns = 256 fp16), lo plane 128 columns further
constexpr long long kTimeoutCycles = 4000000000ll;

struct CondLayerDev {
  int n_tiles;       // N tiles of the layer
  int bn;            // columns per N tile: 128 (hidden layers), 96 (final layer)
  int k_chunks;      // 64-value reduction chunks = ring slots per N tile
  int k_steps_last;  // 16-value MMA steps in the last chunk (1..4)
  int kind;          // FC_COND_*: 0 initial (h = out), 1 first of a block (operand only), 2 second of a block (h += out),
                     // 3 final (parameters)
  int relu_next;     // the next layer's operand is relu(result)
  unsigned w_off16;  // first slot of the layer inside the packed weights, in 16-byte units
  unsigned cta_bytes;  // bytes per slot and CTA: 2 planes x bn/2 rows x 128 B
  int col0;            // first column of the layer in the shared-memory bias / exponent vectors
  const float* bias;   // [n_tiles * bn]
  const float* winv;   // [1] exact power of two: 1 / the layer's weight scale
  int term_mode;       // FC_COND_TERM_*: context terms consumed by this layer
  const float* terms;  // T128 context terms from the layer's first column on
  long long term_tile; // floats per 128-row tile of the term matrix (128 x its width)
};

struct CondArgs {
  const unsigned char* weights;
  const float* a;  // conditioner input [M, k_in] row-major
  long long lda;
  int k_in;
  long long M;
  int num_tiles;  // 256-row tiles (one per CTA pair and step)
  int n_layers;
  int has_terms;  // some layer consumes context terms
  int slots_per_tile;
  int total_cols;  // output columns of all layers (a multiple of 4): size of the bias / scale-exponent vectors in shared memory
  CondLayerDev L[kMaxCondLayers];
  // bijection
  const float* x;
  long long ldx;
  float* y;
  long long ldy;
  float* lad;
  int accumulate;
  const int32_t* tcols;
  const int32_t* ccols;
  int n_copy;
  int D_t;
  RqsParams c;
  int hand_period;   // every hand_period-th final N tile a row thread hands ALL its features to the bijection warps (0: never)
  float sos_offset;  // sum-of-sigmoids bijection: added to the outputs (autoregressive.py:309: -0.5; conditional.py: 0)
  int affine_activation, affine_inverse;  // affine bijection (FC_SCALE_*, direction)
  float* params_out;      // CondStore: the final layer's outputs [M][store_n] instead of a bijection
  long long ldp;
  int store_n;
  int32_t* status;
  int32_t* error;  // device word: 0, or the code of the first wait that timed out
};

// The bijection a kernel instantiation evaluates from a register-resident parameter vector p[0 .. PPAD).
// G: features per accumulator slot of PPAD columns (1 for the splines / sum of sigmoids; the affine transform has two
// parameters per feature, so a 24-column slot carries 12 features).
template <int KC>
struct CondRqs {  // rational-quadratic spline, KC bins, linear tails (rational_quadratic.py:13-181)
  static constexpr int G = 1;
  static constexpr bool kStore = false;
  template <int PPAD>
  static __device__ __forceinline__ void eval(const CondArgs& a, float x, const float (&p)[PPAD], float& y, float& lad,
                                              unsigned& status) {
    // raw derivative entries behind the 2 KC width / height parameters: KC - 1 with linear tails, KC + 1 without (an
    // instantiation whose PPAD leaves room for KC - 1 only is launched for linear tails only)
    constexpr int NPD = PPAD - 2 * KC >= KC + 1 ? KC + 1 : KC - 1;
    static_assert(PPAD - 2 * KC >= KC - 1, "parameters per feature");
    rqs_eval<KC, true, NPD>(a.c, x, p, y, lad, status);
  }
};
template <int NC>
struct CondSos {  // sum of NC sigmoids + extended softplus (adaptive_sigmoids.py:111-142, nonlinearities.py:543-552), forward
  static constexpr int G = 1;
  static constexpr bool kStore = false;
  template <int PPAD>
  static __device__ __forceinline__ void eval(const CondArgs& a, float x, const float (&p)[PPAD], float& y, float& lad,
                                              unsigned&) {
    static_assert(3 * NC + 1 <= PPAD, "parameters per feature");
    float lj;
    sos_eval_t<NC>(x, p, NC, y, lj);
    y += a.sos_offset;
    lad = lj;
  }
};

__device__ int32_t g_cond_error;

// Experiments only (-DFC_COND_PROFILE=1: FC_LINEAR_PROFILE_BUILD=1 python -m flowconductor_b200.build --force): cycles CTA 0's
// MMA-issuing warp and its first row warp spend in each phase; fc_conditioner_profile() reads them back.
#ifndef FC_COND_PROFILE
#define FC_COND_PROFILE 0
#endif
__device__ unsigned long long g_cond_prof[32];
#if FC_COND_PROFILE
#define CPROF_DECL(name) long long name = 0
#define CPROF_T0(t) const long long t = clock64()
#define CPROF_ADD(name, t) name += clock64() - (t)
#else
#define CPROF_DECL(name)
#define CPROF_T0(t)
#define CPROF_ADD(name, t)
#endif

template <int N>
__device__ __forceinline__ void cond_set_max_regs_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void cond_set_max_regs_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {  // A, B = f16 (format 0), D = f32, K-major
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// 256 x N x 16 across the pair, A (this CTA's 128 rows, 8 packed f16x2 columns) from tensor memory
__device__ __forceinline__ void umma_f16_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Bounded waits.  `abort_s` is a shared-memory flag of this CTA: once any role has given up, the others stop waiting too.
__device__ __forceinline__ bool cond_wait(uint32_t bar, uint32_t parity, volatile int* abort_s) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (*abort_s != 0 || clock64() - t0 > kTimeoutCycles) return false;
  }
  return true;
}
__device__ __forceinline__ bool try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool cond_wait_cluster(uint32_t bar, uint32_t parity, volatile int* abort_s) {
  if (try_wait_cluster(bar, parity)) return true;
  const long long t0 = clock64();
  while (!try_wait_cluster(bar, parity)) {
    if (*abort_s != 0 || clock64() - t0 > kTimeoutCycles) return false;
  }
  return true;
}

// acc[0..N) += inv_s * (N consecutive TMEM columns of this thread's lane): all loads in flight, one wait
template <int N>
__device__ __forceinline__ void drain_scaled(uint32_t taddr, float inv_s, float* acc) {
  static_assert(N % 16 == 0, "16 columns per load");
  // packed fp32x2 arithmetic (sm_100: one issue slot for two IEEE fmas); at most 32 columns in flight (registers)
  const float2 s2 = make_float2(inv_s, inv_s);
#pragma unroll
  for (int j0 = 0; j0 < N; j0 += 32) {
    constexpr int kStep = 32;
    const int n = N - j0 < kStep ? N - j0 : kStep;
    uint32_t v[kStep];
#pragma unroll
    for (int j = 0; j < kStep; j += 16)
      if (j < n) tmem_ld16(taddr + (uint32_t)(j0 + j), v + j);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < kStep; j += 2) {
      if (j < n) {
        const float2 r = __ffma2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), s2,
                                    make_float2(acc[j0 + j], acc[j0 + j + 1]));
        acc[j0 + j] = r.x;
        acc[j0 + j + 1] = r.y;
      }
    }
  }
}

// 64 fp32 values of one row -> packed (hi, lo) fp16 words of one operand chunk (w[0..32) hi plane, w[32..64) lo plane),
// scaled by the power of two that puts the largest magnitude into [2^13, 2^14).  Returns 1 / scale (exact).
__device__ __forceinline__ float convert_chunk(const float* v, uint32_t* w) {
  // The scale only has to put the chunk's largest magnitude somewhere into [2^7, 2^14) (see the header comment: hi + lo
  // then still carries 2^-22 relative, 2^-32 of the maximum for small entries).  The sum of the magnitudes bounds the
  // maximum from above within a factor of 64, and costs 64 full-rate additions in four independent chains; a running
  // maximum compiles to a chain of 3-input min/max instructions that issue once per ~8 cycles (measured:
  // scripts/microbench/alu_rate.cu, 320 -> 75 cycles per chunk).
  float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f;
#pragma unroll
  for (int j = 0; j < 64; j += 4) {
    m0 += fabsf(v[j]);
    m1 += fabsf(v[j + 1]);
    m2 += fabsf(v[j + 2]);
    m3 += fabsf(v[j + 3]);
  }
  float m = fminf(fmaxf((m0 + m1) + (m2 + m3), 1e-30f), 1e30f);
  const uint32_t E = __float_as_uint(m) >> 23;  // biased exponent (m > 0)
  const float s = __uint_as_float((267u - E) << 23);      // 2^(13 - (E - 127))
  const float inv_s = __uint_as_float((E - 13u) << 23);   // 2^((E - 127) - 13)
  const float2 s2 = make_float2(s, s), neg1 = make_float2(-1.f, -1.f);
#pragma unroll
  for (int p = 0; p < 32; ++p) {
    const float2 a2 = __fmul2_rn(make_float2(v[2 * p], v[2 * p + 1]), s2);
    const __half2 h2 = __floats2half2_rn(a2.x, a2.y);  // k even in the low half
    const float2 r2 = __ffma2_rn(__half22float2(h2), neg1, a2);  // a - hi, exact
    const __half2 l2 = __floats2half2_rn(r2.x, r2.y);
    w[p] = *reinterpret_cast<const uint32_t*>(&h2);
    w[32 + p] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  return inv_s;
}
// ... into tensor memory: hi plane at ta_chunk (32 columns), lo plane 128 columns further
__device__ __forceinline__ void store_chunk(const uint32_t* w, uint32_t ta_chunk) {
  tmem_st16(ta_chunk, w);
  tmem_st16(ta_chunk + 16u, w + 16);
  tmem_st16(ta_chunk + 128u, w + 32);
  tmem_st16(ta_chunk + 144u, w + 48);
}
__device__ __forceinline__ float produce_chunk(const float* v, uint32_t ta_chunk) {
  uint32_t w[64];
  const float inv_s = convert_chunk(v, w);
  store_chunk(w, ta_chunk);
  return inv_s;
}

struct CondSmem {
  static constexpr int RING_BYTES = kCondStages * kSlotBytes;
  static constexpr int H_BYTES = 256 * kCM * 4;      // residual stream [256 columns][128 rows]
  static constexpr int SC_BYTES = 2 * 4 * kCM * 4;   // 1 / operand scale: [layer parity][chunk][row]
  static constexpr int LAD_BYTES = 2 * 2 * kCM * 4;  // per-row log-det partial sums of the two row threads, double-buffered
  static constexpr int BAR_BYTES = 8 * (3 * kCondStages + 12) + 16;
  static constexpr int TOTAL = RING_BYTES + H_BYTES + SC_BYTES + LAD_BYTES + kVecBytes + BAR_BYTES + 1024;
};

struct CondAffine {  // y = x * scale(raw) + shift and its inverse (coupling.py:224-252, autoregressive.py:97-129): a slot of 24
  static constexpr int G = 12;  // columns holds (raw scale, shift) of 12 consecutive features
  static constexpr bool kStore = false;
  // feature g of the slot
  template <int PPAD>
  static __device__ __forceinline__ void eval_g(const CondArgs& a, int g, float x, const float (&p)[PPAD], float& y, float& lad) {
    affine_eval(x, p[2 * g], p[2 * g + 1], a.affine_activation, a.affine_inverse, y, lad);
  }
};

// No bijection: the conditioner's outputs are written out, output column 96 t + c from column c of final tile t
// (ResidualNet.forward / MADE.forward as ONE launch, for the bijections that run as element-wise kernels afterwards).  A row thread owns (row, 48
// columns): stored from there, 32 lanes would write 4 bytes each a row pitch apart (measured: 2.5x slower than the per-layer
// kernels).  Instead EVERY final tile goes through the shared-memory parameter tile (HAND, period 1; its column stride is
// padded to 129 words here so that both the row threads' column-wise writes and the row-wise reads below are free of bank
// conflicts) and the four bijection warps copy it out row by row, 32 lanes on 32 consecutive outputs of one row.
struct CondStore {
  static constexpr int G = 1;
  static constexpr bool kStore = true;
  template <int PPAD>
  static __device__ __forceinline__ void eval(const CondArgs&, float, const float (&)[PPAD], float& y, float& lad, unsigned&) {
    y = 0.f;
    lad = 0.f;
  }
};

// Bij the bijection, PPAD accumulator columns per feature, NT = hidden width / 128
// HAND: every hand_period-th final tile is handed to the bijection warps entirely (instantiated where it pays)
// CTX: the hidden layers consume context terms (FC_COND_TERM_*; a separate instantiation, so that the code of nets without
// context stays exactly as it is)
template <class Bij, int PPAD, int NT, bool HAND, bool CTX>
__global__ void __launch_bounds__(kCondThreads, 1) conditioner_f16x3_kernel(const CondArgs a) {
  constexpr int KCH = 2 * NT;         // 64-value chunks of a hidden-width reduction
  constexpr int FEATS = 96 / PPAD;    // features per final N tile
  constexpr int NF = FEATS / 2;       // ... per row thread (two threads share a row)
  // Of the NF features of an N tile whose parameters a row thread accumulates it evaluates its first one itself and hands
  // the others to its row's bijection thread; on every hand_period-th tile it hands over ALL of them (measured: the row
  // threads are the critical resource — drains, conversions and one spline per tile keep them ~80 % busy while the
  // bijection warps wait 60 % of the time —, so part of the row threads' splines moves there).
  constexpr int NF_OWN = 1;
  constexpr int G = Bij::G;           // features per slot (see the bijection policies)
  constexpr int kPS = Bij::kStore ? kCM + 1 : kCM;  // column stride (words) of the handed-over parameter tile
  static_assert(!Bij::kStore || (HAND && NF == 1), "the store variant hands every tile over");
  static_assert(NF >= 1 && NF * 2 * PPAD == 96, "final N tile: 96 columns");
  static_assert(G == 1 || 2 * G <= PPAD, "grouped features: two parameters each");
  // (compile-time "never" for tiles of several features per thread: measured to be best there, and the kernel keeps
  // the leaner code — one own spline per row thread, NF - 1 per bijection thread and half)
  auto tile_own = [&](int nt) -> int {
    if constexpr (HAND && NF == 1) {
      return (a.hand_period > 0 && (nt + 1) % a.hand_period == 0) ? 0 : NF_OWN;
    } else {
      return NF_OWN;
    }
  };
  extern __shared__ unsigned char smem_raw[];
  const uint32_t raw_s = s32(smem_raw);
  const uint32_t base = (raw_s + 1023u) & ~1023u;
  unsigned char* const gbase = smem_raw + (base - raw_s);
  float* const hs = reinterpret_cast<float*>(gbase + CondSmem::RING_BYTES);
  float* const scs = reinterpret_cast<float*>(gbase + CondSmem::RING_BYTES + CondSmem::H_BYTES);
  float* const ladx = scs + 2 * 4 * kCM;  // [tile parity][column half][row]
  // bias[total_cols], then 1 / weight scale of each layer
  float* const vbias = ladx + 2 * 2 * kCM;
  float* const vwinv = vbias + a.total_cols;
  const uint32_t bars = base + CondSmem::RING_BYTES + CondSmem::H_BYTES + CondSmem::SC_BYTES + CondSmem::LAD_BYTES + kVecBytes;
  unsigned char* const gbars = gbase + (bars - base);
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto ready_bar = [&](int s) { return bars + 8u * (kCondStages + s); };   // leader's: both halves have landed
  auto empty_bar = [&](int s) { return bars + 8u * (2 * kCondStages + s); };
  auto tfull_bar = [&](int i) { return bars + 8u * (3 * kCondStages + i); };
  auto tempty_bar = [&](int i) { return bars + 8u * (3 * kCondStages + 2 + i); };  // leader's
  auto opnd_bar = [&](int g) { return bars + 8u * (3 * kCondStages + 4 + g); };    // leader's
  // parameter tiles (final layer): written by the row warps / consumed by the bijection warps
  auto pfull_bar = [&](int b) { return bars + 8u * (3 * kCondStages + 6 + b); };
  auto pempty_bar = [&](int b) { return bars + 8u * (3 * kCondStages + 8 + b); };
  const uint32_t lad_bar = bars + 8u * (3 * kCondStages + 10);  // the row threads' log-det partial sums of a row tile are written
  const uint32_t tmem_slot = bars + 8u * (3 * kCondStages + 11);
  volatile uint32_t* const tmem_slot_g = reinterpret_cast<volatile uint32_t*>(gbars + 8 * (3 * kCondStages + 11));
  volatile int* const abort_s = reinterpret_cast<volatile int*>(gbars + 8 * (3 * kCondStages + 11) + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int cl0 = (int)blockIdx.x >> 1, cl_step = (int)gridDim.x >> 1;

  if (threadIdx.x == 0) {
    *abort_s = 0;
    for (int s = 0; s < kCondStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(ready_bar(s), 2);
      mbar_init(empty_bar(s), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 2 * kRowWarps);  // the row warps of both CTAs
      mbar_init(opnd_bar(i), 2 * kRowWarps);
      mbar_init(pfull_bar(i), kRowWarps);
      mbar_init(pempty_bar(i), kBijWarps);
    }
    mbar_init(lad_bar, kRowWarps);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
  // per-column vectors of every layer -> shared memory (read in every row tile by every row thread)
  for (int l = 0; l < a.n_layers; ++l) {
    const CondLayerDev& L = a.L[l];
    const int n = L.n_tiles * L.bn;
    for (int i = threadIdx.x; i < n; i += kCondThreads) vbias[L.col0 + i] = __ldg(L.bias + i);
    if (threadIdx.x == 0) vwinv[l] = __ldg(L.winv);
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_g;

#define COND_FAIL(code)                                  \
  {                                                      \
    *abort_s = 1;                                        \
    atomicCAS(a.error, 0, (int)(code) + 100 * warp);     \
    goto teardown;                                       \
  }

  if (warp < 4) {
    cond_set_max_regs_dec<40>();
    if (warp == 0) {
      // ---------------------------------------------------------------- weight producer
      if (lane == 0) {
        int s = 0;
        uint32_t ph = 0;
        // the context terms of a row tile -> L2 ahead of the row threads (in T128 a layer's columns of one 128-row tile
        // are one contiguous block)
        auto prefetch_terms = [&](int t) {
          if ((long long)t * 256 + rank * kCM >= a.M) return;
          for (int l = 0; l < a.n_layers - 1; ++l) {
            const CondLayerDev& L = a.L[l];
            if (L.term_mode != FC_COND_TERM_NONE)
              bulk_prefetch_l2(L.terms + (long long)(2 * t + rank) * L.term_tile, (uint32_t)(L.n_tiles * L.bn * kCM * 4));
          }
        };
        if constexpr (CTX) prefetch_terms(cl0);
        for (int tile = cl0; tile < a.num_tiles; tile += cl_step) {
          if constexpr (CTX) {
            if (tile + cl_step < a.num_tiles) prefetch_terms(tile + cl_step);
          }
          for (int l = 0; l < a.n_layers; ++l) {
            const CondLayerDev& L = a.L[l];
            const unsigned char* src = a.weights + ((size_t)L.w_off16 << 4) + (size_t)rank * L.cta_bytes;
            const int n_slots = L.n_tiles * L.k_chunks;
            for (int i = 0; i < n_slots; ++i) {
              if (!cond_wait_cluster(empty_bar(s), ph ^ 1u, abort_s)) COND_FAIL(1);
              mbar_expect_tx(full_bar(s), L.cta_bytes);
              bulk_load_1d(base + (uint32_t)(s * kSlotBytes), src, L.cta_bytes, full_bar(s));
              src += 2 * (size_t)L.cta_bytes;
              if (++s == kCondStages) {
                s = 0;
                ph ^= 1u;
              }
            }
          }
          // next row tile's conditioner input -> L2 while this one is computed (contiguous rows only)
          const int nxt = tile + cl_step;
          if (nxt < a.num_tiles && a.lda == a.k_in) {
            const long long r0 = (long long)nxt * 256 + rank * kCM;
            long long rows = a.M - r0;
            rows = rows > kCM ? kCM : rows;
            if (rows > 0) bulk_prefetch_l2(a.a + r0 * a.lda, (uint32_t)(rows * a.lda * 4));
          }
        }
      }
    } else if (warp == 3) {
      // ---------------------------------------------------------------- relay: this CTA's half of a slot has landed
      if (lane == 0) {
        int s = 0;
        uint32_t ph = 0;
        for (int tile = cl0; tile < a.num_tiles; tile += cl_step) {
          for (int i = 0; i < a.slots_per_tile; ++i) {
            if (!cond_wait(full_bar(s), ph, abort_s)) COND_FAIL(2);
            if (rank == 0) {
              mbar_arrive(ready_bar(s));
            } else {
              mbar_arrive_remote_relaxed(ready_bar(s), 0);
            }
            if (++s == kCondStages) {
              s = 0;
              ph ^= 1u;
            }
          }
        }
      }
    } else if (warp == 1 && rank == 0) {
      // ---------------------------------------------------------------- MMA issuer (whole warp walks, one lane issues)
      int s = 0, acc = 0;
      uint32_t ph = 0, aph = 0, lcount = 0;
      const uint64_t b0 = make_smem_desc(base, 128);
      CPROF_DECL(m_opnd);
      CPROF_DECL(m_tempty);
      CPROF_DECL(m_ready);
      CPROF_DECL(m_chunks);
      CPROF_T0(m_begin);
      for (int tile = cl0; tile < a.num_tiles; tile += cl_step) {
        for (int l = 0; l < a.n_layers; ++l, ++lcount) {
          const CondLayerDev& L = a.L[l];
          const uint32_t idesc = make_idesc_f16(2 * kCM, L.bn);
          const uint64_t lo_off = (uint64_t)((L.cta_bytes >> 1) >> 4);
          for (int nt = 0; nt < L.n_tiles; ++nt) {
            for (int c = 0; c < L.k_chunks; ++c) {
              {
                CPROF_T0(t0);
                if (nt == 0 && (c & 1) == 0) {  // operand chunks c, c + 1 written (by both CTAs)
                  if (!cond_wait_cluster(opnd_bar(c >> 1), lcount & 1u, abort_s)) COND_FAIL(3);
                }
                CPROF_ADD(m_opnd, t0);
              }
              {
                CPROF_T0(t0);
                if (!cond_wait_cluster(tempty_bar(acc), aph ^ 1u, abort_s)) COND_FAIL(4);
                CPROF_ADD(m_tempty, t0);
              }
              {
                CPROF_T0(t0);
                if (!cond_wait_cluster(ready_bar(s), ph, abort_s)) COND_FAIL(5);
                CPROF_ADD(m_ready, t0);
              }
#if FC_COND_PROFILE
              ++m_chunks;
#endif
              tc_fence_after();
              const int steps = (c == L.k_chunks - 1) ? L.k_steps_last : 4;
              const uint64_t b_hi = b0 + (uint64_t)((uint32_t)s * (uint32_t)(kSlotBytes >> 4)), b_lo = b_hi + lo_off;
              const uint32_t d = tmem_base + kTmemAcc + (uint32_t)(acc * 128);
              const uint32_t a_hi = tmem_base + kTmemA + (uint32_t)(c * 32), a_lo = a_hi + 128u;
              if (elect_one()) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                  if (kk < steps) {
                    const uint64_t o = (uint64_t)(kk * 2);  // 16 fp16 = 32 bytes inside the swizzle span
                    // small terms first
                    umma_f16_ts_pair(d, a_lo + (uint32_t)(kk * 8), b_hi + o, idesc, kk > 0 ? 1u : 0u);
                    umma_f16_ts_pair(d, a_hi + (uint32_t)(kk * 8), b_lo + o, idesc, 1u);
                    umma_f16_ts_pair(d, a_hi + (uint32_t)(kk * 8), b_hi + o, idesc, 1u);
                  }
                }
                umma_commit_pair(empty_bar(s), 3);
                umma_commit_pair(tfull_bar(acc), 3);
              }
              __syncwarp();
              if (++s == kCondStages) {
                s = 0;
                ph ^= 1u;
              }
              if (++acc == 2) {
                acc = 0;
                aph ^= 1u;
              }
            }
          }
        }
      }
#if FC_COND_PROFILE
      if (blockIdx.x == 0 && lane == 0) {
        g_cond_prof[0] = (unsigned long long)(clock64() - m_begin);
        g_cond_prof[1] = (unsigned long long)m_opnd;
        g_cond_prof[2] = (unsigned long long)m_tempty;
        g_cond_prof[3] = (unsigned long long)m_ready;
        g_cond_prof[4] = (unsigned long long)m_chunks;
      }
#endif
    }
  } else if (warp < 4 + kRowWarps) {
    // ------------------------------------------------------------------ row threads, two per row
    cond_set_max_regs_inc<184>();
    const int q = warp & 3, half = (warp - 4) >> 2;
    const int rl = q * 32 + lane;  // row inside the CTA's tile = TMEM lane
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    int acc_i = 0;
    uint32_t aph = 0, lcount = 0, pt = 0, tcount = 0;  // pt: parameter tiles handed to the bijection warps so far
    unsigned status = 0;
    // pending bijection work: this thread's own feature of the last finished final-layer N tile
    float pp[PPAD];
    float pxv = 0.f, lad_acc = 0.f;
    float pxg[G > 1 ? G : 1];  // grouped features (G > 1): the slot's inputs; their columns are re-derived from pxc = slot index
    int pxc = -1;
    long long prow = 0;
#pragma unroll
    for (int g = 0; g < (G > 1 ? G : 1); ++g) pxg[g] = 0.f;
    bool pvalid = false, pending = false, tile_open = false;  // tile_open: the row tile's log-det share is not handed over yet
#pragma unroll
    for (int j = 0; j < PPAD; ++j) pp[j] = 0.f;
    CPROF_DECL(r_spline);
    CPROF_DECL(r_l0);
    CPROF_DECL(r_wait_h);
    CPROF_DECL(r_drain_h);
    CPROF_DECL(r_final_h);
    CPROF_DECL(r_prod_h);
    CPROF_DECL(r_wait_f);
    CPROF_DECL(r_drain_f);
    CPROF_DECL(r_hand);
    CPROF_T0(r_begin);

    auto signal_operand = [&]() {
      tmem_wait_st();
      __threadfence_block();  // the scale words written next to the operand
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_remote_relaxed(opnd_bar(0), 0);
        mbar_arrive_remote_relaxed(opnd_bar(1), 0);
      }
    };
    auto signal_group = [&](int g) {
      tmem_wait_st();
      __threadfence_block();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_relaxed(opnd_bar(g), 0);
    };
    auto spline = [&]() {
      if constexpr (G == 1) {
        if (pxc >= 0) {
          float yv, lv;
          Bij::eval(a, pxv, pp, yv, lv, status);
          if (pvalid) a.y[prow * a.ldy + pxc] = yv;
          lad_acc += lv;
        }
      } else {
        if (pxc >= 0) {  // pxc: the slot; its features pxc * G ..
#pragma unroll
          for (int g = 0; g < G; ++g) {
            const int f = pxc * G + g;
            if (f < a.D_t) {
              float yv, lv;
              Bij::eval_g(a, g, pxg[g], pp, yv, lv);
              if (pvalid) a.y[prow * a.ldy + (a.tcols ? __ldg(a.tcols + f) : f)] = yv;
              lad_acc += lv;
            }
          }
        }
      }
      pending = false;
    };
    // this thread's share of the row tile's log|det J| goes to the row's bijection thread, which sums and stores it
    auto finish_tile = [&]() {
      ladx[((tcount & 1u) * 2 + half) * kCM + rl] = lad_acc;
      __syncwarp();
      if (lane == 0) mbar_arrive(lad_bar);  // release: orders the warp's stores above
      lad_acc = 0.f;
      ++tcount;
    };

    for (int tile = cl0; tile < a.num_tiles; tile += cl_step) {
      const long long row = (long long)tile * 256 + rank * kCM + rl;
      const bool valid = row < a.M;
      // ---- operand of the initial layer: this row of the conditioner input, chunks half, half + 2
      {
        CPROF_T0(t_l0);
        const CondLayerDev& L0 = a.L[0];
        float* sc_next = scs + (lcount & 1u) * (4 * kCM);
        for (int c = half; c < L0.k_chunks; c += 2) {
          float v[64];
          const float* src = a.a + row * a.lda + c * 64;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid && c * 64 + 4 * j < a.k_in) t = __ldg(reinterpret_cast<const float4*>(src) + j);
            v[4 * j + 0] = t.x;
            v[4 * j + 1] = t.y;
            v[4 * j + 2] = t.z;
            v[4 * j + 3] = t.w;
          }
          sc_next[c * kCM + rl] = produce_chunk(v, tmem_base + lane_sel + kTmemA + (uint32_t)(c * 32));
        }
        signal_operand();
        CPROF_ADD(r_l0, t_l0);
      }
      // ---- finish the previous row tile while the initial layer's MMAs run
      if (tile_open) {
        CPROF_T0(t_s);
        if (pending) spline();
        finish_tile();
        tile_open = false;
        CPROF_ADD(r_spline, t_s);
      }
      // ---- hidden layers
      for (int l = 0; l < a.n_layers - 1; ++l, ++lcount) {
        const CondLayerDev& L = a.L[l];
        const float* sc_cur = scs + (lcount & 1u) * (4 * kCM);
        float* sc_next = scs + ((lcount + 1u) & 1u) * (4 * kCM);
        float av[NT * 64];
        uint32_t pw[64];
        float pre_inv = 0.f;
        const float winv_l = vwinv[l];
        if (l == 0 && pt > 0) {
          // the residual stream's space still holds the previous row tile's last parameter tiles: wait until the bijection
          // warps have consumed both buffers (as if about to write each of them again)
          const uint32_t n0w = (pt + 1u) >> 1, n1w = pt >> 1;  // writes so far to buffer 0 / 1
          if (!cond_wait(pempty_bar(0), (n0w & 1u) ^ 1u, abort_s)) COND_FAIL(8);
          if (n1w > 0 && !cond_wait(pempty_bar(1), (n1w & 1u) ^ 1u, abort_s)) COND_FAIL(9);
        }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
          const int n0 = nt * 128 + half * 64;
          float* hcol = hs + n0 * kCM + rl;
          // this row's context terms of the 64 columns (T128: the warp's 32 rows read 512 contiguous bytes per float4)
          const float4* g4 = nullptr;
          if (CTX && L.term_mode != FC_COND_TERM_NONE && valid)
            g4 = reinterpret_cast<const float4*>(L.terms + (long long)(2 * tile + rank) * L.term_tile) + (n0 >> 2) * kCM + rl;
          {
            // the register accumulators start from the bias (all lanes read the same words: broadcast) plus, in the second
            // layer of a block, the skip connection (resnet.py:56 / made.py:181: inputs + temps) — fetched while the
            // first partial sums are still being computed; with context terms (MADE) + g or + relu(g), fetched the same way
            const float4* b4 = reinterpret_cast<const float4*>(vbias + L.col0 + n0);
            const bool add_h = L.kind == FC_COND_BLOCK_SECOND && !(CTX && L.term_mode == FC_COND_TERM_GATE);
#pragma unroll
            for (int j4 = 0; j4 < 16; ++j4) {
              const float4 b = b4[j4];
              av[nt * 64 + 4 * j4 + 0] = b.x;
              av[nt * 64 + 4 * j4 + 1] = b.y;
              av[nt * 64 + 4 * j4 + 2] = b.z;
              av[nt * 64 + 4 * j4 + 3] = b.w;
            }
            if (add_h) {
#pragma unroll
              for (int j = 0; j < 64; j += 2) {
                const float2 r = __fadd2_rn(make_float2(av[nt * 64 + j], av[nt * 64 + j + 1]),
                                            make_float2(hcol[j * kCM], hcol[(j + 1) * kCM]));
                av[nt * 64 + j] = r.x;
                av[nt * 64 + j + 1] = r.y;
              }
            }
            if (CTX && g4 != nullptr && L.term_mode != FC_COND_TERM_GATE) {
              const bool rl_g = L.term_mode == FC_COND_TERM_ADD_RELU;
#pragma unroll
              for (int j4 = 0; j4 < 16; ++j4) {
                float4 g = __ldg(g4 + j4 * kCM);
                if (rl_g) {
                  g.x = fmaxf(g.x, 0.f);
                  g.y = fmaxf(g.y, 0.f);
                  g.z = fmaxf(g.z, 0.f);
                  g.w = fmaxf(g.w, 0.f);
                }
                av[nt * 64 + 4 * j4 + 0] += g.x;
                av[nt * 64 + 4 * j4 + 1] += g.y;
                av[nt * 64 + 4 * j4 + 2] += g.z;
                av[nt * 64 + 4 * j4 + 3] += g.w;
              }
            }
          }
          for (int c = 0; c < L.k_chunks; ++c) {
            CPROF_T0(t_w);
            if (!cond_wait_cluster(tfull_bar(acc_i), aph, abort_s)) COND_FAIL(6);
            CPROF_ADD(r_wait_h, t_w);
            CPROF_T0(t_d);
            tc_fence_after();
            const float inv_s = sc_cur[c * kCM + rl] * winv_l;  // both exact powers of two
            if (NT == 2 && nt == 1 && c == L.k_chunks - 1) {
              // every MMA of this layer has completed: the operand in tensor memory may be overwritten.  Chunks 0 / 1 of
              // the next operand were converted while the second N tile ran; hand them over first, so that the next
              // layer's MMAs start while this thread finishes the second N tile
              store_chunk(pw, tmem_base + lane_sel + kTmemA + (uint32_t)(half * 32));
              sc_next[half * kCM + rl] = pre_inv;
              signal_group(0);
            }
            drain_scaled<64>(tmem_base + lane_sel + kTmemAcc + (uint32_t)(acc_i * 128 + half * 64), inv_s, av + nt * 64);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote_relaxed(tempty_bar(acc_i), 0);
            if (++acc_i == 2) {
              acc_i = 0;
              aph ^= 1u;
            }
            CPROF_ADD(r_drain_h, t_d);
          }
          CPROF_T0(t_f);
          if (CTX && L.term_mode == FC_COND_TERM_GATE) {
            // ResidualNet block with context (resnet.py:45-52): h + t * sigmoid(g), F.glu of [t | g]
#pragma unroll
            for (int j4 = 0; j4 < 16; ++j4) {
              const float4 g = g4 != nullptr ? __ldg(g4 + j4 * kCM) : make_float4(0.f, 0.f, 0.f, 0.f);
              const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int j = 4 * j4 + i;
                av[nt * 64 + j] = fmaf(av[nt * 64 + j], fc_sigmoid(gv[i]), hcol[j * kCM]);
              }
            }
          }
          // residual stream, ReLU
          if (L.kind == FC_COND_INITIAL || (L.kind == FC_COND_BLOCK_SECOND && L.relu_next)) {
            // (after the last block nothing reads the residual stream again)
#pragma unroll
            for (int j = 0; j < 64; ++j) hcol[j * kCM] = av[nt * 64 + j];
          }
          if (L.relu_next) {
#pragma unroll
            for (int j = 0; j < 64; ++j) av[nt * 64 + j] = fmaxf(av[nt * 64 + j], 0.f);
          }
          CPROF_ADD(r_final_h, t_f);
          if (NT == 2 && nt == 0) {
            // this half of operand chunks 0 / 1 is final: convert now, while the second N tile is being computed
            pre_inv = convert_chunk(av, pw);
          }
        }
        CPROF_T0(t_p);
        // every MMA of this layer has completed (its last partial accumulator has been drained)
        {
          const int cidx = (NT - 1) * 2 + half;
          sc_next[cidx * kCM + rl] =
              produce_chunk(av + (NT - 1) * 64, tmem_base + lane_sel + kTmemA + (uint32_t)(cidx * 32));
        }
        if (NT == 2) {
          signal_group(1);
        } else {
          signal_operand();
        }
        CPROF_ADD(r_prod_h, t_p);
      }
      // ---- final layer: N tiles of 96 parameter columns.  Of the features whose parameters it accumulates, a row thread
      // evaluates one itself — the spline of N tile j - 1 between the drains of N tile j — and hands the other to the row's
      // bijection thread through one of two parameter tiles in the (now dead) residual stream's space
      {
        const CondLayerDev& L = a.L[a.n_layers - 1];
        const float* sc_cur = scs + (lcount & 1u) * (4 * kCM);
        const float winv_f = vwinv[a.n_layers - 1];
        for (int nt = 0; nt < L.n_tiles; ++nt) {
          float pv[NF * PPAD];
          const int fg = nt * FEATS + half * NF;  // this thread's own feature (G > 1: slot of G features)
          const bool live = fg * G < a.D_t;
          int xc = -1;
          float xv = 0.f;
          float xg[G > 1 ? G : 1];
          if constexpr (Bij::kStore) {
            xc = live ? fg : -1;  // nothing to read
          } else if constexpr (G == 1) {
            xc = live ? (a.tcols ? __ldg(a.tcols + fg) : fg) : -1;
            xv = (valid && live) ? __ldg(a.x + row * a.ldx + xc) : 0.f;
          } else {
            xc = live ? fg : -1;
#pragma unroll
            for (int g = 0; g < G; ++g) {
              const int f = fg * G + g;
              xg[g] = (valid && f < a.D_t) ? __ldg(a.x + row * a.ldx + (a.tcols ? __ldg(a.tcols + f) : f)) : 0.f;
            }
          }
          const int n0 = nt * 96 + half * (NF * PPAD);
          {
            const float4* b4 = reinterpret_cast<const float4*>(vbias + L.col0 + n0);
#pragma unroll
            for (int j4 = 0; j4 < NF * PPAD / 4; ++j4) {
              const float4 b = b4[j4];
              pv[4 * j4 + 0] = b.x;
              pv[4 * j4 + 1] = b.y;
              pv[4 * j4 + 2] = b.z;
              pv[4 * j4 + 3] = b.w;
            }
          }
#pragma unroll
          for (int c = 0; c < KCH; ++c) {
            if constexpr (NT == 1) {
              if (c >= L.k_chunks) break;  // a net of <= 64 units zero-padded to 128 has one real chunk, not two
            }
            CPROF_T0(t_w);
            if (!cond_wait_cluster(tfull_bar(acc_i), aph, abort_s)) COND_FAIL(7);
            CPROF_ADD(r_wait_f, t_w);
            CPROF_T0(t_d);
            tc_fence_after();
            const float inv_s = sc_cur[c * kCM + rl] * winv_f;
            drain_scaled<NF * PPAD>(tmem_base + lane_sel + kTmemAcc + (uint32_t)(acc_i * 128 + half * (NF * PPAD)), inv_s, pv);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote_relaxed(tempty_bar(acc_i), 0);
            if (++acc_i == 2) {
              acc_i = 0;
              aph ^= 1u;
            }
            CPROF_ADD(r_drain_f, t_d);
            if (c == 0 && pending) {
              CPROF_T0(t_s);
              spline();
              CPROF_ADD(r_spline, t_s);
            }
          }
          const int nown = tile_own(nt), nhand = NF - nown;
          if (nhand > 0) {
            CPROF_T0(t_h);
            const uint32_t b = pt & 1u, nw = pt >> 1;  // buffer, and how often it has been written before
            if (!cond_wait(pempty_bar(b), (nw & 1u) ^ 1u, abort_s)) COND_FAIL(10);
            float* pcol = hs + (b * (2 * NF * PPAD) + half * (NF * PPAD)) * kPS + rl;
#pragma unroll
            for (int j = 0; j < NF * PPAD; ++j) {
              if (j >= nown * PPAD) pcol[(j - nown * PPAD) * kPS] = pv[j];
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(pfull_bar(b));  // release: orders the warp's stores above
            ++pt;
            CPROF_ADD(r_hand, t_h);
          }
          if (nown > 0) {
#pragma unroll
            for (int j = 0; j < PPAD; ++j) pp[j] = pv[j];
            pxv = xv;
            pxc = xc;
            if constexpr (G > 1) {
#pragma unroll
              for (int g = 0; g < G; ++g) pxg[g] = xg[g];
            }
            prow = row;
            pvalid = valid;
            pending = true;
          }
        }
        ++lcount;
        tile_open = true;
      }
    }
    if (tile_open) {
      if (pending) spline();
      finish_tile();
    }
    if (status != 0 && a.status) atomicOr(a.status, (int)status);
#if FC_COND_PROFILE
    if (blockIdx.x == 0 && warp == 4 && lane == 0) {
      g_cond_prof[8] = (unsigned long long)(clock64() - r_begin);
      g_cond_prof[9] = (unsigned long long)r_l0;
      g_cond_prof[11] = (unsigned long long)r_wait_h;
      g_cond_prof[12] = (unsigned long long)r_drain_h;
      g_cond_prof[13] = (unsigned long long)r_final_h;
      g_cond_prof[14] = (unsigned long long)r_prod_h;
      g_cond_prof[15] = (unsigned long long)r_wait_f;
      g_cond_prof[16] = (unsigned long long)r_drain_f;
      g_cond_prof[10] = (unsigned long long)r_hand;
      g_cond_prof[17] = (unsigned long long)r_spline;
    }
#endif
  } else {
    // ------------------------------------------------------------------ bijection threads, one per row
    cond_set_max_regs_dec<104>();
    const int r = threadIdx.x - 32 * (4 + kRowWarps);  // row inside the CTA's tile
    unsigned status = 0;
    uint32_t pt = 0, tcount = 0;
    CPROF_DECL(b_wait);
    CPROF_DECL(b_work);
    CPROF_T0(b_begin);
    const int n_final = a.L[a.n_layers - 1].n_tiles;
    for (int tile = cl0; tile < a.num_tiles; tile += cl_step) {
      const long long row = (long long)tile * 256 + rank * kCM + r;
      const bool valid = row < a.M;
      // identity columns (coupling.py:96-98) when the layer does not work in place: each warp copies its 32 rows, one row
      // per step (coalesced)
      if (a.n_copy > 0 && a.y != a.x) {
        const long long row0 = (long long)tile * 256 + rank * kCM + (r & ~31);
        for (int i0 = 0; i0 < a.n_copy; i0 += 32) {
          const int cc = (i0 + lane < a.n_copy) ? __ldg(a.ccols + i0 + lane) : -1;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) {
            if (cc >= 0 && row0 + rr < a.M) a.y[(row0 + rr) * a.ldy + cc] = __ldg(a.x + (row0 + rr) * a.ldx + cc);
          }
        }
      }
      float lad_acc = 0.f;
      for (int nt = 0; nt < n_final; ++nt) {
        const int nown = tile_own(nt), nhand = NF - nown;
        if (nhand == 0) continue;
        if constexpr (Bij::kStore) {
          // the whole 96-column tile of this warp's 32 rows, row by row: lanes on consecutive outputs
          const uint32_t b = pt & 1u;
          {
            CPROF_T0(t_w);
            if (!cond_wait(pfull_bar(b), (pt >> 1) & 1u, abort_s)) COND_FAIL(11);
            CPROF_ADD(b_wait, t_w);
          }
          CPROF_T0(t_s);
          const int rl0 = r & ~31;
          const long long grow0 = row - (r & 31);
          const int nrows = (int)min((long long)32, a.M - grow0);  // rows of this warp inside the batch (<= 0: none)
          const float* tile_s = hs + (b * (2 * NF * PPAD)) * kPS + rl0;
#pragma unroll
          for (int cc = 0; cc < 2 * NF * PPAD; cc += 32) {
            const int c = cc + lane;
            const int col = nt * (2 * NF * PPAD) + c;
            const bool live = col < a.store_n;
            float* out = a.params_out + grow0 * a.ldp + col;
            const float* src = tile_s + c * kPS;
            // eight shared-memory loads in flight, then eight predicated stores (a loop of guarded load-store pairs compiles to
            // one branch region per element with the load latency exposed every time: 120 cycles per element)
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
              float v[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) v[u] = src[r0 + u];
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                if (live && r0 + u < nrows) out[0] = v[u];
                out += a.ldp;
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(pempty_bar(b));
          ++pt;
          CPROF_ADD(b_work, t_s);
          continue;
        }
        // the features the two row threads of this row hand over: the last nhand of each half of the N tile
        float xv[2 * NF * G];
        int xc[2 * NF];  // G == 1: the column; G > 1: the slot
#pragma unroll
        for (int f = 0; f < 2 * NF; ++f) {  // inputs first: their latency hides behind the wait for the parameters
          const int h = f / NF, sl = f % NF;
          const int fg = nt * FEATS + h * NF + nown + sl;
          const bool live = sl < nhand && fg * G < a.D_t;
          if constexpr (G == 1) {
            xc[f] = live ? (a.tcols ? __ldg(a.tcols + fg) : fg) : -1;
            xv[f] = (valid && live) ? __ldg(a.x + row * a.ldx + xc[f]) : 0.f;
          } else {
            xc[f] = live ? fg : -1;
#pragma unroll
            for (int g = 0; g < G; ++g) {
              const int ff = fg * G + g;
              xv[f * G + g] = (valid && live && ff < a.D_t) ? __ldg(a.x + row * a.ldx + (a.tcols ? __ldg(a.tcols + ff) : ff)) : 0.f;
            }
          }
        }
        const uint32_t b = pt & 1u;
        {
          CPROF_T0(t_w);
          if (!cond_wait(pfull_bar(b), (pt >> 1) & 1u, abort_s)) COND_FAIL(11);
          CPROF_ADD(b_wait, t_w);
        }
        CPROF_T0(t_s);
        const float* pcol = hs + (b * (2 * NF * PPAD)) * kCM + r;
#pragma unroll
        for (int f = 0; f < 2 * NF; ++f) {
          const int h = f / NF, sl = f % NF;
          if (sl < nhand) {
            float p[PPAD];
#pragma unroll
            for (int j = 0; j < PPAD; ++j) p[j] = pcol[((h * NF + sl) * PPAD + j) * kCM];
            if constexpr (G == 1) {
              float yv, lv;
              Bij::eval(a, xv[f], p, yv, lv, status);
              if (xc[f] >= 0) {
                if (valid) a.y[row * a.ldy + xc[f]] = yv;
                lad_acc += lv;
              }
            } else {
              if (xc[f] >= 0) {
#pragma unroll
                for (int g = 0; g < G; ++g) {
                  const int ff = xc[f] * G + g;
                  if (ff < a.D_t) {
                    float yv, lv;
                    Bij::eval_g(a, g, xv[f * G + g], p, yv, lv);
                    if (valid) a.y[row * a.ldy + (a.tcols ? __ldg(a.tcols + ff) : ff)] = yv;
                    lad_acc += lv;
                  }
                }
              }
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(pempty_bar(b));
        ++pt;
        CPROF_ADD(b_work, t_s);
      }
      // per-sample log|det J| (sum_except_batch, utils/torchutils.py:25-30): the row's three evaluating threads summed their
      // features in order; the partial sums are combined in a fixed order
      if (!cond_wait(lad_bar, tcount & 1u, abort_s)) COND_FAIL(12);
      {
        const float* lx = ladx + (tcount & 1u) * (2 * kCM);
        const float tot = (lx[r] + lx[kCM + r]) + lad_acc;
        if constexpr (!Bij::kStore) {
          if (valid) a.lad[row] = a.accumulate ? a.lad[row] + tot : tot;
        }
      }
      ++tcount;
    }
    if (status != 0 && a.status) atomicOr(a.status, (int)status);
#if FC_COND_PROFILE
    if (blockIdx.x == 0 && warp == 4 + kRowWarps && lane == 0) {
      g_cond_prof[16 + 2] = (unsigned long long)(clock64() - b_begin);
      g_cond_prof[16 + 3] = (unsigned long long)b_wait;
      g_cond_prof[16 + 4] = (unsigned long long)b_work;
    }
#endif
  }

teardown:
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();  // no CTA leaves (or frees tensor memory) while its partner can still signal it
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
#undef COND_FAIL
}

// ------------------------------------------------------------------------------------------------------------
// Packing: one nn.Linear / MaskedLinear -> ring slots of fp16 (hi, lo) planes in the shared-memory image the MMA reads
// (K-major rows of 64 fp16 = 128 bytes, 16-byte chunks XOR-swizzled with the row index: the 128-byte swizzle), one
// slot per (N tile, 64-value chunk), each slot [rank 0: hi | lo][rank 1: hi | lo].
// ------------------------------------------------------------------------------------------------------------
__global__ void cond_pack_init_kernel(float* bias_out, float* winv_out, int n_pad) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += gridDim.x * blockDim.x) bias_out[i] = 0.f;
  if (blockIdx.x == 0 && threadIdx.x == 0) *winv_out = 0.f;  // holds max |w| (as ordered bits) until the pack kernel ran
}

// largest magnitude of the (masked) weight matrix: non-negative floats order like their bit patterns
__global__ void __launch_bounds__(128) cond_pack_max_kernel(const float* __restrict__ W, int64_t ldw,
                                                            const float* __restrict__ mask, int64_t ldm, int K,
                                                            float* __restrict__ max_out) {
  const int n = blockIdx.x;
  float m = 0.f;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float w = W[n * ldw + k];
    if (mask) w *= mask[n * ldm + k];  // MaskedLinear: weight * mask (made.py:72)
    m = fmaxf(m, fabsf(w));
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m > 0.f && m < 1e30f) atomicMax(reinterpret_cast<unsigned int*>(max_out), __float_as_uint(m));
}

// one block per source weight row; the last block to finish replaces max |w| by 1 / scale
__global__ void __launch_bounds__(128) cond_pack_kernel(const float* __restrict__ W, int64_t ldw, const float* __restrict__ mask,
                                                        int64_t ldm, const float* __restrict__ bias,
                                                        const int32_t* __restrict__ row_map,
                                                        const int32_t* __restrict__ col_map, int N, int K, int bn,
                                                        int k_chunks, unsigned char* __restrict__ out,
                                                        float* __restrict__ bias_out, const float* __restrict__ max_in,
                                                        float* __restrict__ scale_out) {
  const int n = blockIdx.x;
  const float m = *max_in;
  float s = 1.f, inv_s = 1.f;
  if (m > 1e-30f) {
    const uint32_t E = __float_as_uint(m) >> 23;
    s = __uint_as_float((267u - E) << 23);       // the largest weight lands in [2^13, 2^14)
    inv_s = __uint_as_float((E - 13u) << 23);
  }
  const int rn = row_map ? row_map[n] : n;
  const int bnh = bn >> 1;
  const int nt = rn / bn, r_in = rn % bn, rank = r_in / bnh, r = r_in % bnh;
  const size_t cta_bytes = (size_t)2 * bnh * 128;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float w = W[n * ldw + k];
    if (mask) w *= mask[n * ldm + k];
    w *= s;
    const __half hi = __float2half_rn(w);
    const __half lo = __float2half_rn(w - __half2float(hi));
    const int ck = col_map ? col_map[k] : k;
    const int c = ck >> 6, kk = ck & 63;
    const size_t slot = ((size_t)(nt * k_chunks + c) * 2 + rank) * cta_bytes;
    const size_t off = (size_t)r * 128 + (size_t)((((kk >> 3) ^ (r & 7)) << 4) + (kk & 7) * 2);
    *reinterpret_cast<__half*>(out + slot + off) = hi;
    *reinterpret_cast<__half*>(out + slot + (size_t)bnh * 128 + off) = lo;
  }
  if (threadIdx.x == 0) {
    bias_out[rn] = bias ? bias[n] : 0.f;
    if (n == 0) *scale_out = inv_s;
  }
}

template <class Bij, int PPAD, int NT, bool HAND, bool CTX>
static int launch_conditioner_t(const CondArgs& args, cudaStream_t stream) {
  auto kern = conditioner_f16x3_kernel<Bij, PPAD, NT, HAND, CTX>;
  static_assert(CondSmem::TOTAL <= 232448, "shared memory per CTA");
  static std::atomic<uint64_t> configured{0};
  int dev_id = 0;
  cudaGetDevice(&dev_id);
  const uint64_t dev_bit = 1ull << (dev_id & 63);
  if (!(configured.load(std::memory_order_acquire) & dev_bit)) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CondSmem::TOTAL) != cudaSuccess)
      return FC_ERR_CUDA;
    configured.fetch_or(dev_bit, std::memory_order_release);
  }
  const int max_pairs = device_info().sm_count / 2;
  const int pairs = args.num_tiles < max_pairs ? args.num_tiles : max_pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * pairs));
  cfg.blockDim = dim3(kCondThreads);
  cfg.dynamicSmemBytes = CondSmem::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, kern, args) != cudaSuccess) return FC_ERR_CUDA;
  FC_CHECK_LAUNCH();
  return FC_OK;
}
template <class Bij, int PPAD, int NT, bool HAND = false>
static int launch_conditioner(const CondArgs& args, cudaStream_t stream) {
  return args.has_terms ? launch_conditioner_t<Bij, PPAD, NT, HAND, true>(args, stream)
                        : launch_conditioner_t<Bij, PPAD, NT, HAND, false>(args, stream);
}

}  // namespace fc

using namespace fc;

extern "C" int64_t fc_conditioner_layer_bytes(int32_t n_pad, int32_t k_pad, int32_t bn) {
  if (n_pad <= 0 || k_pad <= 0 || (bn != 128 && bn != 96) || n_pad % bn != 0 || k_pad % 64 != 0) return FC_ERR_INVALID_ARGUMENT;
  return (int64_t)(n_pad / bn) * (k_pad / 64) * 2 * (2 * (bn / 2) * 128);
}

extern "C" int fc_conditioner_pack_layer(const float* W, int64_t w_row_stride, const float* mask, int64_t mask_row_stride,
                                         const float* bias, int32_t N, int32_t K, const int32_t* row_map,
                                         const int32_t* col_map, int32_t n_pad, int32_t k_pad, int32_t bn, void* w_packed,
                                         float* bias_packed, float* winv_packed, void* stream) {
  if (!W || !w_packed || !bias_packed || !winv_packed || N <= 0 || K <= 0 || n_pad < N || k_pad < K)
    return FC_ERR_INVALID_ARGUMENT;
  const int64_t bytes = fc_conditioner_layer_bytes(n_pad, k_pad, bn);
  if (bytes < 0) return (int)bytes;
  if (reinterpret_cast<uintptr_t>(w_packed) & 15) return FC_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(w_packed, 0, (size_t)bytes, st) != cudaSuccess) return FC_ERR_CUDA;
  // winv_packed[1] holds max |w| until the pack kernel has read it, winv_packed[0] receives 1 / scale
  cond_pack_init_kernel<<<(n_pad + 255) / 256, 256, 0, st>>>(bias_packed, winv_packed + 1, n_pad);
  cond_pack_max_kernel<<<N, 128, 0, st>>>(W, w_row_stride, mask, mask_row_stride, K, winv_packed + 1);
  cond_pack_kernel<<<N, 128, 0, st>>>(W, w_row_stride, mask, mask_row_stride, bias, row_map, col_map, N, K, bn, k_pad / 64,
                                      reinterpret_cast<unsigned char*>(w_packed), bias_packed, winv_packed + 1, winv_packed);
  FC_CHECK_LAUNCH();
  return FC_OK;
}

extern "C" int fc_conditioner_profile(unsigned long long* out32) {
  if (!out32) return FC_ERR_INVALID_ARGUMENT;
  if (cudaMemcpyFromSymbol(out32, g_cond_prof, sizeof(unsigned long long) * 32) != cudaSuccess) return FC_ERR_CUDA;
  return FC_OK;
}

extern "C" int fc_conditioner_error(int32_t* out) {
  if (!out) return FC_ERR_INVALID_ARGUMENT;
  if (cudaMemcpyFromSymbol(out, g_cond_error, sizeof(int32_t)) != cudaSuccess) return FC_ERR_CUDA;
  return FC_OK;
}

// Argument checks and the layer table shared by the fc_conditioner_*_apply entry points.  ppad: accumulator columns per
// feature of the final layer's 96-column N tiles.
static int cond_build_args(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                           int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                           int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols, int ppad, int hand_default,
                           int32_t* status, CondArgs& args, int group = 1, bool store = false) {
  if (!net || !net->weights || net->n_layers < 2 || net->n_layers > kMaxCondLayers) return FC_ERR_INVALID_ARGUMENT;
  if (B < 0 || D_t <= 0) return FC_ERR_INVALID_ARGUMENT;
  if (B > 0 && (!a || (!store && (!x || !y || !logabsdet)))) return FC_ERR_INVALID_ARGUMENT;
  if (B >= ((int64_t)1 << 31)) return FC_ERR_UNSUPPORTED;
  if (tcols.idx && tcols.n != D_t) return FC_ERR_INVALID_ARGUMENT;
  if (net->hidden != 128 && net->hidden != 256) return FC_ERR_UNSUPPORTED;
  if (net->k_in <= 0 || net->k_in > 256 || (net->k_in & 3) || (lda & 3) || lda < net->k_in ||
      (reinterpret_cast<uintptr_t>(a) & 15) || (reinterpret_cast<uintptr_t>(net->weights) & 15))
    return FC_ERR_UNSUPPORTED;
  const int kch = net->hidden / 64;
  const int hidden_k = (net->hidden_k > 0 && net->hidden == 128) ? net->hidden_k : net->hidden;
  if (hidden_k > net->hidden || (hidden_k & 3)) return FC_ERR_INVALID_ARGUMENT;
  args.weights = reinterpret_cast<const unsigned char*>(net->weights);
  args.a = a;
  args.lda = lda;
  args.k_in = net->k_in;
  args.M = B;
  args.num_tiles = (int)((B + 255) / 256);
  args.n_layers = net->n_layers;
  args.slots_per_tile = 0;
  for (int l = 0; l < net->n_layers; ++l) {
    const fc_conditioner_layer& s = net->layers[l];
    CondLayerDev& d = args.L[l];
    const bool last = l == net->n_layers - 1;
    if (!s.bias || !s.winv || s.n_tiles <= 0 || s.w_offset < 0 || (s.w_offset & 15)) return FC_ERR_INVALID_ARGUMENT;
    if (last != (s.kind == FC_COND_FINAL) || (l == 0) != (s.kind == FC_COND_INITIAL)) return FC_ERR_INVALID_ARGUMENT;
    if ((reinterpret_cast<uintptr_t>(s.bias) & 3) || (reinterpret_cast<uintptr_t>(s.winv) & 3)) return FC_ERR_UNSUPPORTED;
    d.n_tiles = s.n_tiles;
    d.bn = last ? 96 : 128;
    // reduction length: the input width, then the REAL hidden width (a narrower net zero-padded to 128 multiplies only its
    // real k-values: the padding chunks are never staged, issued or drained)
    const int k = l == 0 ? net->k_in : hidden_k;
    d.k_chunks = (k + 63) / 64;
    d.k_steps_last = ((k - (d.k_chunks - 1) * 64) + 15) / 16;
    if (!last && s.n_tiles != net->hidden / 128) return FC_ERR_INVALID_ARGUMENT;
    if (last && (int64_t)s.n_tiles * (96 / ppad) * group < D_t) return FC_ERR_INVALID_ARGUMENT;
    // (chunks are skipped only in the 128-wide kernel; the 256-wide one multiplies all four)
    if (l > 0 && (d.k_chunks > kch || (net->hidden == 256 && d.k_chunks != kch))) return FC_ERR_INVALID_ARGUMENT;
    d.kind = s.kind;
    d.relu_next = s.relu_next;
    d.w_off16 = (unsigned)(s.w_offset >> 4);
    d.cta_bytes = (unsigned)(2 * (d.bn / 2) * 128);
    d.bias = s.bias;
    d.winv = s.winv;
    // context terms: each mode belongs to one layer kind (header: FC_COND_TERM_*)
    if (s.term_mode < FC_COND_TERM_NONE || s.term_mode > FC_COND_TERM_GATE) return FC_ERR_INVALID_ARGUMENT;
    static const int kTermKind[4] = {-1, FC_COND_BLOCK_FIRST, FC_COND_INITIAL, FC_COND_BLOCK_SECOND};
    d.term_mode = s.term_mode;
    d.terms = nullptr;
    d.term_tile = 0;
    if (s.term_mode != FC_COND_TERM_NONE) {
      if (s.kind != kTermKind[s.term_mode] || (B > 0 && !s.terms)) return FC_ERR_INVALID_ARGUMENT;
      if ((reinterpret_cast<uintptr_t>(s.terms) & 15) || s.term_width < (int64_t)s.n_tiles * 128 || (s.term_width & 15))
        return FC_ERR_UNSUPPORTED;
      d.terms = s.terms;
      d.term_tile = 128 * s.term_width;
      args.has_terms = 1;
    }
    d.col0 = args.total_cols;
    args.total_cols += d.n_tiles * d.bn;
    args.slots_per_tile += d.n_tiles * d.k_chunks;
  }
  if (args.total_cols * 4 + 4 * kMaxCondLayers > kVecBytes) return FC_ERR_UNSUPPORTED;  // biases must fit in shared memory
  args.x = x;
  args.ldx = x_row_stride;
  args.y = y;
  args.ldy = y_row_stride;
  args.lad = logabsdet;
  args.accumulate = accumulate_logabsdet;
  args.tcols = tcols.idx;
  args.ccols = ccols.idx;
  args.n_copy = ccols.n;
  args.D_t = D_t;
  args.status = status;
  // Measured: with two features per row thread and tile (8 bins) handing more to the bijection warps does not pay
  // (cfg 2: 24.4 ms never, 24.9 every 2nd, 26.4 always), nor with 16-bin splines (cfg 3 D-pass inverse 9.4 -> 10.8 ms
  // at every 3rd tile); for the sum of sigmoids (one feature per thread and tile, the bijection warps would otherwise
  // idle) every 3rd tile is best (cfg 4: 2.00 -> 1.90 ms).
  args.hand_period = hand_default;
  void* err_ptr = nullptr;
  if (cudaGetSymbolAddress(&err_ptr, g_cond_error) != cudaSuccess) return FC_ERR_CUDA;
  args.error = reinterpret_cast<int32_t*>(err_ptr);
  return FC_OK;
}

extern "C" int fc_conditioner_rqs_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                                        int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                                        int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols,
                                        const fc_rqs_config* cfg, int32_t* status, void* stream) {
  RqsParams c;
  int rc = make_rqs_params(cfg, c);
  if (rc != FC_OK) return rc;
  // bins with a register-resident instantiation; P = 3K - 1 (linear tails) or 3K + 1 parameters in 24 or 48 columns
  if ((c.K != 8 && c.K != 10 && c.K != 16) || c.P > 48) return FC_ERR_UNSUPPORTED;
  const int ppad = c.P <= 24 ? 24 : 48;
  CondArgs args{};
  rc = cond_build_args(net, a, lda, B, x, x_row_stride, y, y_row_stride, logabsdet, accumulate_logabsdet, D_t, tcols, ccols,
                       ppad, 0, status, args);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  args.c = c;
  cudaStream_t st = (cudaStream_t)stream;
  const bool wide = net->hidden == 256;
#define FC_COND_LAUNCH(KC, PP) (wide ? launch_conditioner<CondRqs<KC>, PP, 2>(args, st) : launch_conditioner<CondRqs<KC>, PP, 1>(args, st))
  if (c.K == 8) return ppad == 24 ? FC_COND_LAUNCH(8, 24) : FC_COND_LAUNCH(8, 48);
  if (c.K == 10) return FC_COND_LAUNCH(10, 48);
  return FC_COND_LAUNCH(16, 48);
#undef FC_COND_LAUNCH
}

extern "C" int fc_conditioner_affine_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                                           int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                                           int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols,
                                           int32_t activation, int32_t inverse, void* stream) {
  if (activation < FC_SCALE_SIGMOID2 || activation > FC_SCALE_SOFTPLUS_EPS) return FC_ERR_INVALID_ARGUMENT;
  CondArgs args{};
  int rc = cond_build_args(net, a, lda, B, x, x_row_stride, y, y_row_stride, logabsdet, accumulate_logabsdet, D_t, tcols,
                           ccols, 24, 0, nullptr, args, CondAffine::G);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  args.affine_activation = activation;
  args.affine_inverse = inverse != 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (net->hidden == 256) return launch_conditioner<CondAffine, 24, 2>(args, st);
  return launch_conditioner<CondAffine, 24, 1>(args, st);
}

extern "C" int fc_conditioner_store_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, float* params,
                                          int64_t params_row_stride, int32_t n_out, void* stream) {
  if (n_out <= 0) return FC_ERR_INVALID_ARGUMENT;
  if (B > 0 && !params) return FC_ERR_INVALID_ARGUMENT;
  if (params_row_stride < n_out) return FC_ERR_INVALID_ARGUMENT;
  CondArgs args{};
  fc_cols none{nullptr, 0};
  int rc = cond_build_args(net, a, lda, B, nullptr, 0, nullptr, 0, nullptr, 0, (n_out + 47) / 48, none, none, 48, 1, nullptr, args,
                           1, true);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  args.hand_period = 1;  // every tile leaves through the shared-memory parameter tile
  args.params_out = params;
  args.ldp = params_row_stride;
  args.store_n = n_out;
  cudaStream_t st = (cudaStream_t)stream;
  if (net->hidden == 256) return launch_conditioner<CondStore, 48, 2, true>(args, st);
  return launch_conditioner<CondStore, 48, 1, true>(args, st);
}

extern "C" int fc_conditioner_sos_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                                        int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                                        int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols,
                                        int32_t n_sigmoids, float offset, void* stream) {
  if (n_sigmoids < 1) return FC_ERR_INVALID_ARGUMENT;
  if (n_sigmoids != 10) return FC_ERR_UNSUPPORTED;  // the unrolled, MUFU-lean form (conditional.py:746 default)
  CondArgs args{};
  int rc = cond_build_args(net, a, lda, B, x, x_row_stride, y, y_row_stride, logabsdet, accumulate_logabsdet, D_t, tcols,
                           ccols, 48, 3, nullptr, args);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  args.sos_offset = offset;
  cudaStream_t st = (cudaStream_t)stream;
  if (net->hidden == 256) return launch_conditioner<CondSos<10>, 48, 2, true>(args, st);
  return launch_conditioner<CondSos<10>, 48, 1, true>(args, st);
}
