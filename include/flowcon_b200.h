/*
 * flowcon_b200.h — C ABI of libflowcon_b200.so: sm_100a kernels for FlowConductor's element-wise
 * bijection hot path (rational-quadratic splines, affine, sum-of-sigmoids) with the per-sample
 * log|det J| reduction, coupling column split/scatter and the final-conditioner GEMM fused in.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller; fp32 unless stated; row-major.
 *  - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it, stateless and
 *    re-entrant.  Return value: 0, or a negative FC_ERR_* code (never throws, never syncs).
 *  - matrices are described by (base, row_stride in ELEMENTS, optional int32 column list).  A NULL
 *    column list means columns 0..D_t-1.  This is how the coupling split / scatter of the reference
 *    (flowcon/transforms/coupling.py:82-83,96-98) is folded into the kernels.
 *  - `params` is the conditioner output [B, D_t * P] exactly as the reference lays it out
 *    (feature-major; coupling.py:289, autoregressive.py:581-583): P consecutive floats per feature.
 *  - domain violations that the reference reports by raising after a host sync
 *    (InputOutsideDomain rational_quadratic.py:81-82, discriminant assert :142) are OR-ed into the
 *    caller's `status` word (FC_STATUS_*); pass NULL to ignore.
 *
 * The reference is pure Python: there is no existing FFI.  Each entry point below names the
 * reference function (file:line under /root/reference) it replaces; INTEGRATION.md shows the ctypes
 * binding and the monkey-patch a maintainer would add on the reference side.
 */
#ifndef FLOWCON_B200_H
#define FLOWCON_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FC_OK 0
#define FC_ERR_INVALID_ARGUMENT (-1)
#define FC_ERR_UNSUPPORTED (-2)
#define FC_ERR_CUDA (-3)

#define FC_STATUS_INPUT_OUTSIDE_DOMAIN 1 /* rational_quadratic.py:81-82 */
#define FC_STATUS_NEGATIVE_DISCRIMINANT 2 /* rational_quadratic.py:142 */
#define FC_STATUS_NONFINITE 4

#define FC_TAILS_NONE 0   /* constrained spline on [left,right] -> [bottom,top] */
#define FC_TAILS_LINEAR 1 /* identity outside [-tail_bound, tail_bound]; P = 3K-1 */

/* Spline hyper-parameters: arguments of rational_quadratic_spline /
 * unconstrained_rational_quadratic_spline (flowcon/transforms/splines/rational_quadratic.py:13-25,66-80). */
typedef struct fc_rqs_config {
  int32_t num_bins;      /* K; P = 3K-1 (linear tails) or 3K+1 (none) */
  int32_t tails;         /* FC_TAILS_* */
  int32_t identity_init; /* enable_identity_init: softplus beta = ln2 / (1 - min_derivative) */
  int32_t inverse;       /* 0 forward, 1 inverse */
  float left, right, bottom, top; /* linear tails: -tail_bound, tail_bound, -tail_bound, tail_bound */
  float min_bin_width, min_bin_height, min_derivative;
  float wh_scale; /* raw widths/heights are multiplied by this: 1/sqrt(hidden_features) where the
                     reference divides in place (coupling.py:554-556, conditional.py:711-713), else 1 */
} fc_rqs_config;

/* A [B, *] fp32 matrix seen through an optional column list. */
typedef struct fc_cols {
  const int32_t* idx; /* device int32[n], or NULL for 0..n-1 */
  int32_t n;
} fc_cols;

/*
 * RQ-spline layer, forward or inverse (cfg->inverse):   replaces
 *   unconstrained_rational_quadratic_spline / rational_quadratic_spline (rational_quadratic.py:13-181),
 *   searchsorted (utils/torchutils.py:147-149), sum_except_batch (utils/torchutils.py:25-30) and the
 *   column split/scatter of CouplingTransform.forward/inverse (coupling.py:82-83,96-98).
 * For r < B, j < D_t:  y[r, tcols[j]] = spline(x[r, tcols[j]]; params[r, j*P .. j*P+P-1])
 *                      y[r, ccols[i]] = x[r, ccols[i]]            (identity columns; ccols.n may be 0)
 *                      logabsdet[r]   = (accumulate ? logabsdet[r] : 0) + sum_j log|dy/dx|
 */
int fc_rqs_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                 float* y, int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet,
                 int64_t B, int32_t D_t, fc_cols tcols, fc_cols ccols, const fc_rqs_config* cfg,
                 int32_t* status, void* stream);

/* Debugging / test aid: which kernel skeleton the calling thread's last element-wise layer call (fc_*_apply,
 * fc_*_backward) launched: 0 general strides (staged), 1 per-warp TMA ring, 2 CTA-level tile ring; -1 none yet. */
int fc_elementwise_last_path(void);

/*
 * Parity aid (not on the data path): the bin index the kernels' own arithmetic selects for every transformed element
 * — what searchsorted (utils/torchutils.py:147-149) returns inside rational_quadratic_spline (:115-118) — and
 * optionally the element's distance to the nearest knot of the searched axis in units of the interval length.
 * bins / knot_dist: [B, D_t] row-major; bin -1 = outside the linear tails (identity).  The north-star criterion "bin
 * indices identical except for inputs within 1e-6 of a knot" is asserted with this on the GPU.
 */
int fc_rqs_bins(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride, int64_t B,
                int32_t D_t, fc_cols tcols, const fc_rqs_config* cfg, int32_t* bins, float* knot_dist, void* stream);

/*
 * Backward of fc_rqs_apply (the reference differentiates its op chain with autograd; SURVEY App. B).
 * grad_params is written densely ([B, D_t*P], zero where the reference's gradient is zero).
 *   grad_x[r, tcols[j]] = grad_y[r, tcols[j]] * dy/dx + grad_logabsdet[r] * d lad/dx
 *   grad_x[r, ccols[i]] = grad_y[r, ccols[i]]
 */
int fc_rqs_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                    const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet,
                    float* grad_x, int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride,
                    int64_t B, int32_t D_t, fc_cols tcols, fc_cols ccols, const fc_rqs_config* cfg,
                    void* stream);

/*
 * Piecewise-linear spline layer (SURVEY 8f n3): replaces linear_spline / unconstrained_linear_spline
 * (flowcon/transforms/splines/linear.py:9-105) as called by PiecewiseLinearCouplingTransform._piecewise_cdf
 * (coupling.py:340-352), MaskedPiecewiseLinearAutoregressiveTransform._elementwise (autoregressive.py:355-366) and
 * PiecewiseLinearCDF._spline (nonlinearities.py:263-277).  params[r] = per transformed feature num_bins raw bin
 * probabilities (P = num_bins).  tails = FC_TAILS_LINEAR: identity outside [left, right] (= [-tail_bound, tail_bound],
 * bottom/top equal left/right); FC_TAILS_NONE: inputs outside the domain set FC_STATUS_INPUT_OUTSIDE_DOMAIN (the
 * reference raises, linear.py:45-46).  Column lists, strides, logabsdet accumulation and status as for fc_rqs_apply.
 */
int fc_linspline_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride, float* y,
                       int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int32_t D_t,
                       fc_cols tcols, fc_cols ccols, int32_t num_bins, int32_t tails, float left, float right,
                       float bottom, float top, int32_t inverse, int32_t* status, void* stream);
/* adjoint of fc_linspline_apply (either direction): grad_x [B, *] and grad_params [B, D_t * num_bins] */
int fc_linspline_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                          const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet, float* grad_x,
                          int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride, int64_t B, int32_t D_t,
                          fc_cols tcols, fc_cols ccols, int32_t num_bins, int32_t tails, float left, float right,
                          float bottom, float top, int32_t inverse, void* stream);

/*
 * Piecewise-quadratic spline layer (SURVEY 8f n3): replaces quadratic_spline / unconstrained_quadratic_spline
 * (flowcon/transforms/splines/quadratic.py:11-159) as called by PiecewiseQuadraticCouplingTransform._piecewise_cdf
 * (coupling.py:403-427), MaskedPiecewiseQuadraticAutoregressiveTransform._elementwise (autoregressive.py) and
 * PiecewiseQuadraticCDF._spline (nonlinearities.py:309-334).  params[r] = per transformed feature
 * [num_bins raw widths ; raw knot heights], num_bins + 1 heights without tails (P = 2K+1), num_bins - 1 with linear tails
 * (P = 2K-1, the two boundary heights are derived, quadratic.py:87-101).  Raw widths AND heights are multiplied by
 * wh_scale (1/sqrt(hidden) when the conditioner exposes hidden_features, coupling.py:409-411; else 1).
 */
typedef struct fc_quadspline_config {
  int32_t num_bins;
  int32_t tails;   /* FC_TAILS_* */
  int32_t inverse; /* 0 forward, 1 inverse */
  float left, right, bottom, top;
  float min_bin_width, min_bin_height; /* quadratic.py:7-8 defaults 1e-3 */
  float wh_scale;
} fc_quadspline_config;

int fc_quadspline_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride, float* y,
                        int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int32_t D_t,
                        fc_cols tcols, fc_cols ccols, const fc_quadspline_config* cfg, int32_t* status, void* stream);
/* adjoint of fc_quadspline_apply (either direction): grad_x [B, *] and grad_params [B, D_t * P] */
int fc_quadspline_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                           const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet, float* grad_x,
                           int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride, int64_t B, int32_t D_t,
                           fc_cols tcols, fc_cols ccols, const fc_quadspline_config* cfg, void* stream);

/*
 * Cubic spline layer (SURVEY 8f n3): replaces cubic_spline / unconstrained_cubic_spline
 * (flowcon/transforms/splines/cubic.py:15-267) as called by PiecewiseCubicCouplingTransform._piecewise_cdf
 * (coupling.py:468-500), MaskedPiecewiseCubicAutoregressiveTransform._elementwise (autoregressive.py:491-517) and
 * PiecewiseCubicCDF._spline (nonlinearities.py:363-398).  params[r] = per transformed feature
 * [num_bins raw widths ; num_bins raw heights ; raw left derivative ; raw right derivative] (P = 2K+2); raw widths and
 * heights are multiplied by cfg->wh_scale.  The configuration struct is the quadratic layer's.  The inverse solves the
 * bin's monotone cubic by a safeguarded Newton iteration (the reference: closed form after Blinn 2007).
 */
int fc_cubicspline_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride, float* y,
                         int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int32_t D_t,
                         fc_cols tcols, fc_cols ccols, const fc_quadspline_config* cfg, int32_t* status, void* stream);
int fc_cubicspline_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                            const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet, float* grad_x,
                            int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride, int64_t B, int32_t D_t,
                            fc_cols tcols, fc_cols ccols, const fc_quadspline_config* cfg, void* stream);

/* Affine element-wise transforms. */
#define FC_AFFINE_BLOCKED 0     /* params[r] = [shift(D_t) | raw_scale(D_t)]      coupling.py:234-238 */
#define FC_AFFINE_INTERLEAVED 1 /* params[r] = [raw_scale_0, shift_0, raw_scale_1, ...] autoregressive.py:124-129 */
#define FC_SCALE_SIGMOID2 0       /* sigmoid(u + 2) + 1e-3                 coupling.py:224 */
#define FC_SCALE_SOFTPLUS_CLAMP3 1 /* clamp(softplus(u) + 1e-3, 0, 3)       coupling.py:225 */
#define FC_SCALE_SOFTPLUS_EPS 2    /* softplus(u) + 1e-3                    autoregressive.py:102 */

/* replaces AffineCouplingTransform._coupling_transform_forward/_inverse (coupling.py:240-252) and
 * MaskedAffineAutoregressiveTransform._elementwise_forward/_inverse (autoregressive.py:97-117). */
int fc_affine_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                    float* y, int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet,
                    int64_t B, int32_t D_t, fc_cols tcols, fc_cols ccols, int32_t layout, int32_t activation,
                    int32_t inverse, void* stream);

int fc_affine_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                       const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet,
                       float* grad_x, int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride,
                       int64_t B, int32_t D_t, fc_cols tcols, fc_cols ccols, int32_t layout, int32_t activation,
                       int32_t inverse, void* stream);

/*
 * Sum-of-sigmoids + extended softplus (adaptive_sigmoids.py:111-142, nonlinearities.py:519-552).
 * params[r, j*(3n+1) ..] = [shift_raw(n) | log_scale_raw(n) | softmax_raw(n) | esp_shift_raw].
 * `offset` is added to the forward output / subtracted from the inverse input
 * (MaskedSumOfSigmoidsTransform uses -0.5, autoregressive.py:309,313; the conditional wrapper 0).
 * inverse != 0: per-element bracketed bisection (`bisection_iterations`, initial bracket +-`lim`,
 * replaces MonotonicTransform.bisection_inverse no_analytic_inv/base.py:36-83) followed by two Newton
 * steps with the analytic derivative (replaces newton_inverse :23-34); logabsdet is negated.
 */
int fc_sos_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                 float* y, int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet,
                 int64_t B, int32_t D, int32_t n_sigmoids, float offset, int32_t inverse,
                 int32_t bisection_iterations, float lim, void* stream);

int fc_sos_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                    const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet,
                    float* grad_x, int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride,
                    int64_t B, int32_t D, int32_t n_sigmoids, void* stream);

/*
 * Adjoint of the numerical inverse (fc_sos_apply with inverse = 1).  x is the inverse's OUTPUT; grad_y and
 * grad_logabsdet (may be NULL) are the gradients of that output and of the inverse's logabsdet.  Writes the gradient of
 * the inverse's input (grad_x) and of the raw parameters.  Arguments and validation as fc_sos_backward; the offset,
 * the iteration count and the bracket do not enter.
 */
int fc_sos_inverse_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                            const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet,
                            float* grad_x, int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride,
                            int64_t B, int32_t D, int32_t n_sigmoids, void* stream);

/* Base density tail: out[r] = -0.5 * sum_j z[r,j]^2 - 0.5*D*ln(2*pi) + logabsdet[r]
 * (StandardNormal._log_prob distributions/normal.py:23-33 + flows/base.py:48). logabsdet may be NULL. */
int fc_stdnormal_log_prob(const float* z, int64_t z_row_stride, const float* logabsdet, float* out,
                          int64_t B, int32_t D, void* stream);

/*
 * Conditioner dense layers on the tensor cores (tcgen05 / TMEM / TMA), fp32-faithful "3xTF32" arithmetic.
 *
 * fc_linear_weights is the packed form of one nn.Linear / MaskedLinear (flowcon/nn/nets/resnet.py:26-28,69-91,
 * flowcon/transforms/made.py:15-72): two K-major [n_pad, k_pad] planes (tf32 "hi", then tf32 "lo" = W - hi) and a
 * padded bias.  fc_linear_pack builds it:  packed row row_map[n] (default n), packed column col_map[k] (default
 * k) <- W[n, k] * mask[n, k];  everything else is zero.  row_map is how the final layer's per-feature parameter
 * groups are padded (P -> P_pad accumulator columns per feature: 24 for K = 8 bins, 48 for K = 16) and how the
 * blocked affine layout is interleaved; col_map is how the coupling layer's identity-column gather
 * (coupling.py:82-86) is folded into the first layer (the GEMM then reads the full-width inputs).
 * k_pad must be a multiple of 32, n_pad a multiple of the kernel's N tile (256 for fc_linear_apply, 192 for
 * fc_linear_rqs_apply).
 */
typedef struct fc_linear_weights {
  const float* w;    /* device [2][n_pad][k_pad] */
  const float* bias; /* device [n_pad] */
  int32_t n_pad, k_pad;
} fc_linear_weights;

int fc_linear_pack(const float* W, int64_t w_row_stride, const float* mask, int64_t mask_row_stride,
                   const float* bias, int32_t N, int32_t K, const int32_t* row_map, const int32_t* col_map,
                   int32_t n_pad, int32_t k_pad, float* w_packed, float* bias_packed, void* stream);

/*
 * out[M, n_out] = act_out( act_in(A[M, K]) * W^T + bias (+ residual) ),  act = ReLU when the flag is set.
 * Replaces F.linear in ResidualNet / ResidualBlock / MADE hidden layers (resnet.py:39-56,93-99,
 * made.py:71-72,96-124,152-181): relu_in is the pre-activation of the residual blocks, `residual` their skip
 * connection.  A, out, residual: 16-byte aligned, row strides multiples of 4 floats; n_out a multiple of 4.
 *
 * `layouts` (FC_LINEAR_A_T128 | FC_LINEAR_OUT_T128): activations between the conditioner's own layers are kept in the
 * "T128" layout instead of row-major: 128-row tiles, and inside a tile the 16-byte column groups are the slow index,
 *     element (r, c) of a [M, W] matrix  ->  float offset  (r/128)*128*W + ((c/4)*128 + r%128)*4 + c%4,
 * W a multiple of 16, buffer size T*128*W floats with T = ceil(M/128) ROUNDED UP TO AN EVEN NUMBER: the kernels work on
 * CTA pairs (256 rows = two tiles) and a pair stores / loads both tiles of its last unit (tail rows and the tail tile are
 * written, never read back as results).  One epilogue thread owns one row, so with T128 the 32 threads of a warp store (and re-read as
 * the skip connection) 512 contiguous bytes per instruction instead of 32 scattered 16-byte pieces, and the next
 * layer's TMA box of BK k-values is BK/4 contiguous 2 KB runs.  For a T128 operand its stride argument (lda / ldo /
 * ldr) is W.  The residual always has the layout of `out`.
 */
#define FC_LINEAR_A_T128 1
#define FC_LINEAR_OUT_T128 2
/* `residual` gates instead of being added: out = residual > 0 ? (A W^T + bias) : 0 — the ReLU backward of an
 * input-gradient product, `residual` being the saved pre-activation (autograd of resnet.py:26-28: F.relu then Linear) */
#define FC_LINEAR_RESIDUAL_GATES 4
int fc_linear_apply(const float* A, int64_t lda, int64_t M, int32_t K, const fc_linear_weights* w, int32_t relu_in,
                    float* out, int64_t ldo, int32_t n_out, int32_t relu_out, const float* residual, int64_t ldr,
                    int32_t layouts, void* stream);

/*
 * Split-K form for products whose reduction is long and whose output is small — the weight gradient of a dense
 * layer, grad_W[N, K_in] = grad_y^T[N, B] * x[B, K_in]^T-packed, reduces over the whole batch (autograd of
 * resnet.py:26-28 / made.py:71-72; the reference leaves it to torch.mm).  The A operand is given TRANSPOSED: At is
 * [K, M] row-major with row stride ldat — for a weight gradient simply grad_y [B, N] as the backward pass holds it, so
 * no transposed copy of grad_y is written.  The reduction range [0, K) is cut into k_slices ranges, every (row tile,
 * range) pair is one work unit, and range s writes its partial product to rows [s * slice_rows, s * slice_rows + M) of
 * the row-major matrix `partials` ([k_slices * slice_rows, ldo]); the caller sums the k_slices partial results.
 * slice_rows >= M must be a multiple of 256 (rows M.. of a range are scratch).  `w` is x packed by
 * fc_linear_pack_transposed (zero bias).  colsum: NULL, or [k_slices][slice_rows]
 * floats that receive, per range, the column sums of At (entry s * slice_rows + m = sum over the range's rows k of
 * At[k][m]); their sum over s is grad_y.sum(0), the bias gradient, for free.
 */
int fc_linear_splitk_t_apply(const float* At, int64_t ldat, int64_t M, int64_t K, const fc_linear_weights* w,
                             int32_t k_slices, float* partials, int64_t slice_rows, int64_t ldo, int32_t n_out,
                             float* colsum, void* stream);

/* Weight operand for fc_linear_splitk_t_apply (the batch has to be its contiguous reduction axis): the packed hi / lo
 * planes of X^T (zero bias): packed row c = column c of X. */
int fc_linear_pack_transposed(const float* X, int64_t x_row_stride, int64_t B, int32_t K, int32_t n_pad, int32_t k_pad,
                              int32_t relu /* pack max(X, 0): the layer's input went through F.relu */,
                              float* w_packed, float* bias_packed, void* stream);

/*
 * Final conditioner layer with the rational-quadratic spline in the GEMM epilogue (SURVEY a15 + a1-a6):
 *   params[r, :] = act_in(hidden[r, :H]) * W^T + bias      (never written to memory)
 *   y[r, tcols[j]] = spline(x[r, tcols[j]]; params[r, j*P .. j*P+P-1]),   y[r, ccols[i]] = x[r, ccols[i]],
 *   logabsdet[r] = (accumulate ? logabsdet[r] : 0) + sum_j log|dy/dx|
 * i.e. final_layer (resnet.py:99 / made.py:266-272) + fc_rqs_apply in one kernel.  `w` must have been packed with
 * row_map[j*P + i] = j*P_pad + i.  Supported: linear tails, num_bins 8 or 16 (else FC_ERR_UNSUPPORTED: run
 * fc_linear_apply + fc_rqs_apply).  y may alias x.  layouts: FC_LINEAR_A_T128 if `hidden` is a T128 buffer (ldh = H).
 */
int fc_linear_rqs_apply(const float* hidden, int64_t ldh, int64_t B, int32_t H, const fc_linear_weights* w,
                        int32_t relu_in, const float* x, int64_t x_row_stride, float* y, int64_t y_row_stride,
                        float* logabsdet, int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols,
                        const fc_rqs_config* cfg, int32_t* status, int32_t layouts, void* stream);

/*
 * Final conditioner layer with the AFFINE transform in the GEMM epilogue (SURVEY a15 + a7 / a9): final_layer +
 * fc_affine_apply in one kernel.  `w` must have been packed so that packed row 2j is feature j's raw scale and row
 * 2j+1 its shift (row_map: blocked coupling layout [shift | raw_scale] -> shift_j at 2j+1, raw_scale_j at 2j; the
 * autoregressive layout is already interleaved), n_pad a multiple of 64.  activation: FC_SCALE_*.
 */
int fc_linear_affine_apply(const float* hidden, int64_t ldh, int64_t B, int32_t H, const fc_linear_weights* w,
                           int32_t relu_in, const float* x, int64_t x_row_stride, float* y, int64_t y_row_stride,
                           float* logabsdet, int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols,
                           int32_t activation, int32_t inverse, int32_t layouts, void* stream);

/*
 * Debugging aid: in a library built with -DFC_LINEAR_PROFILE=1 and with FC_LINEAR_DEBUG=4 in the environment, the last
 * fc_linear_* launch records, for CTA 0, the cycles its MMA-issuing warp spent waiting on each barrier ([0] total,
 * [1] accumulator free, [3] operand landed and converted, [5] ring slots processed) and one epilogue warp's split
 * ([8] total, [9] tile set-up, [10] waiting for a partial accumulator, [11] draining it) and one converter warp's
 * ([12] waiting for the TMA boxes, [13] converting); all zero otherwise.
 * Synchronises the device.  Not part of the data path.
 */
int fc_linear_debug_profile(unsigned long long* out16);

/*
 * A WHOLE conditioner network + the rational-quadratic spline it parameterises in one persistent kernel
 * (csrc/fc_conditioner.cu; SURVEY 8(f) n1).  Replaces ResidualNet.forward (flowcon/nn/nets/resnet.py:92-100) or the
 * residual MADE.forward (flowcon/transforms/made.py:274-283) followed by the spline of coupling.py:549-582 /
 * autoregressive.py:578-615: the [B, hidden] activations and the [B, D_t * P] parameters never exist in memory.
 * Arithmetic: "3xFP16" — every fp32 product as three fp16 tensor-core products of exactly scaled (hi, lo) splits,
 * partial sums drained into fp32 registers every 64 k-values (same error as an fp32 FMA chain; DESIGN.md 4.12).
 *
 * Layers: [initial] ([block first] [block second])* [final].  Each layer's weights are packed by
 * fc_conditioner_pack_layer into one contiguous buffer (`weights` + w_offset; size fc_conditioner_layer_bytes):
 * bn = 128 columns per N tile for every layer but the final one (bn = 96: 4 features x 24 padded parameters for 8
 * bins, 2 x 48 for 16 bins — row_map[j*P + i] = j*P_pad + i as for fc_linear_rqs_apply), k_pad = the layer's input width
 * rounded up to 64, n_pad = n_tiles * bn; row_map / col_map / mask as for fc_linear_pack.  The packer also writes bias
 * ([n_pad] floats) and winv (2 floats: [0] = the exact power of two that undoes the layer's fp16 weight scaling, [1]
 * scratch).
 * Supported: hidden width 128 or 256, input width k_in <= 256 (a multiple of 4), at most FC_COND_MAX_LAYERS layers,
 * 8, 10 or 16 bins with at most 48 parameters per feature (linear tails: all three; no tails: 8 and 10 bins) — the final layer
 * is packed with 24 accumulator columns per feature when P <= 24, else 48; everything else FC_ERR_UNSUPPORTED (run the
 * per-layer fc_linear_* kernels).
 */
#define FC_COND_MAX_LAYERS 10
#define FC_COND_INITIAL 0      /* h = W a + b */
#define FC_COND_BLOCK_FIRST 1  /* t = W relu(h) + b            (resnet.py:41-44) */
#define FC_COND_BLOCK_SECOND 2 /* h = h + W relu(t) + b        (resnet.py:45-56) */
#define FC_COND_FINAL 3        /* params = W h + b             (resnet.py:99, no activation in front) */
/* Context terms (conditional nets, inference): a hidden layer may consume g = Wc ctx + bc, precomputed for the whole batch
 * ([B, T] in the T128 layout, see FC_LINEAR_A_T128; fc_context_terms or fc_linear_apply with FC_LINEAR_OUT_T128).
 * `terms` points at the layer's first column of that matrix (base + 128 * column floats, 16-byte aligned), `term_width`
 * is T (a multiple of 16); column j of the layer's output consumes column j of `terms`.
 *   ADD       block first of a residual MADE      t = W relu(h) + b + g                (made.py:170-181)
 *   ADD_RELU  initial layer of a MADE             h = W x + b + relu(g)                (made.py:274-279)
 *   GATE      block second of a ResidualNet       h = h + (W relu(t) + b) * sigmoid(g) (resnet.py:45-52: F.glu)
 * A mode on another layer kind is FC_ERR_INVALID_ARGUMENT, a misaligned `terms` / term_width FC_ERR_UNSUPPORTED. */
#define FC_COND_TERM_NONE 0
#define FC_COND_TERM_ADD 1
#define FC_COND_TERM_ADD_RELU 2
#define FC_COND_TERM_GATE 3
typedef struct fc_conditioner_layer {
  int32_t kind;      /* FC_COND_* */
  int32_t n_tiles;   /* N tiles: hidden / 128, or ceil(D_t / features per 96-column tile) for the final layer */
  int32_t relu_next; /* the following layer multiplies relu(result) */
  int32_t term_mode; /* FC_COND_TERM_* (0 for a net without context) */
  int64_t w_offset;  /* byte offset of the layer's packed weights inside `weights` (a multiple of 16) */
  const float* bias; /* device [n_tiles * bn] */
  const float* winv; /* device [2], see above */
  const float* terms; /* device, T128 [B, term_width] from the layer's first column on; null with FC_COND_TERM_NONE */
  int64_t term_width;
} fc_conditioner_layer;
typedef struct fc_conditioner {
  const void* weights; /* device, 16-byte aligned */
  int32_t n_layers, hidden, k_in;
  int32_t hidden_k; /* 0, or the real hidden width of a narrower net zero-padded to `hidden`: the layers after the first are
                       then packed with k_pad = hidden_k rounded up to 64 and only those k-values are multiplied */
  fc_conditioner_layer layers[FC_COND_MAX_LAYERS];
} fc_conditioner;

int64_t fc_conditioner_layer_bytes(int32_t n_pad, int32_t k_pad, int32_t bn);
int fc_conditioner_pack_layer(const float* W, int64_t w_row_stride, const float* mask, int64_t mask_row_stride,
                              const float* bias, int32_t N, int32_t K, const int32_t* row_map, const int32_t* col_map,
                              int32_t n_pad, int32_t k_pad, int32_t bn, void* w_packed, float* bias_packed,
                              float* winv_packed, void* stream);
/* a: the matrix the initial layer multiplies ([B, k_in], row stride lda; for a coupling layer the full-width inputs
 * with the identity-column gather folded into col_map, for a MADE the inputs; for a conditional ResidualNet the context
 * columns follow, [x | ctx]).  x / y / logabsdet / tcols / ccols / cfg / status exactly as for fc_linear_rqs_apply; y may
 * alias x.  A conditional net (every fc_conditioner_*_apply): the layers with a term_mode read the context terms of this
 * call (FC_COND_TERM_*, [B, T] in T128 from fc_context_terms or fc_linear_apply), bound in the layer table. */
int fc_conditioner_rqs_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                             int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                             int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols,
                             const fc_rqs_config* cfg, int32_t* status, void* stream);
/* Same kernel with the sum-of-sigmoids bijection (flowcon/transforms/adaptive_sigmoids.py:111-142 + ExtendedSoftplus,
 * nonlinearities.py:543-552) in the forward direction: replaces ConditionalSumOfSigmoidsTransform.forward
 * (flowcon/transforms/conditional.py:746-787: ResidualNet on the context, then SumOfSigmoids) and the forward of
 * MaskedSumOfSigmoidsTransform (autoregressive.py:266-318, offset = -0.5); the [B, D_t * (3 n + 1)] parameter tensor is never
 * materialised.  The final layer is packed with 48 accumulator columns per feature (row_map[j*P + i] = j*48 + i, two features
 * per 96-column tile).  n_sigmoids = 10 only (FC_ERR_UNSUPPORTED otherwise: materialise the parameters, fc_sos_apply). */
int fc_conditioner_sos_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                             int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                             int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols, int32_t n_sigmoids,
                             float offset, void* stream);
/* Same kernel with the affine bijection (AffineCouplingTransform, flowcon/transforms/coupling.py:212-252, and the forward of
 * MaskedAffineAutoregressiveTransform, autoregressive.py:97-129): the final layer is packed so that feature j's (raw scale,
 * shift) sit in rows (2j, 2j + 1) — row_map as for fc_linear_affine_apply, 48 features per 96-column tile.  `activation`
 * FC_SCALE_*; inverse != 0: y = (x - shift) / scale. */
int fc_conditioner_affine_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, const float* x,
                                int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                                int32_t accumulate_logabsdet, int32_t D_t, fc_cols tcols, fc_cols ccols, int32_t activation,
                                int32_t inverse, void* stream);
/* Same kernel without a bijection: the conditioner's outputs (ResidualNet.forward, flowcon/nn/nets/resnet.py:92-100 /
 * MADE.forward, flowcon/transforms/made.py:274-283) are written to params[B][n_out] (row stride in floats) in ONE launch, for
 * the bijections that run as element-wise kernels afterwards (fc_linspline_apply, fc_quadspline_apply, fc_cubicspline_apply,
 * fc_sos_apply ...).  The final layer is packed without a row map (packed row j <- output j), n_out padded to a multiple of
 * 96 columns. */
int fc_conditioner_store_apply(const fc_conditioner* net, const float* a, int64_t lda, int64_t B, float* params,
                               int64_t params_row_stride, int32_t n_out, void* stream);
/* The context terms of a conditional conditioner for narrow contexts (C <= 64, below the tensor-core GEMM's minimum
 * reduction): out = ctx W^T + bias as [B, T] in the T128 layout (buffer of an even number of 128-row tiles; the rows
 * beyond B of the last tiles are not written), fp32 FMA chains in k order.  ctx [B, C] (row stride ldc), W [T, C]
 * row-major, bias [T]; T a multiple of 16. */
int fc_context_terms(const float* ctx, int64_t ldc, int64_t B, int32_t C, const float* W, const float* bias, int32_t T,
                     float* out, void* stream);
/* Debugging aid: every barrier wait inside the kernel is bounded; if one ever times out the kernel ends early and leaves
 * a non-zero code (wait site + 100 * warp) here.  Synchronises the device.  Not part of the data path. */
int fc_conditioner_error(int32_t* out);
/* Debugging aid (library built with -DFC_COND_PROFILE=1, else all zero): cycles CTA 0's MMA-issuing warp ([0] total, [1]
 * waiting for the operand, [2] for a free partial accumulator, [3] for a weight slot, [4] slots) and its first row warp
 * ([8] total, [9] initial operand, [10] parameter hand-off, [11]/[12]/[13]/[14] hidden layers: waiting for a partial
 * accumulator / draining / skip-ReLU / converting the next operand, [15]/[16] final layer: waiting / draining) and its
 * first bijection warp ([18] total, [19] waiting for parameters, [20] evaluating) spent in the last fc_conditioner_*
 * launch.  Synchronises the device. */
int fc_conditioner_profile(unsigned long long* out32);

/*
 * The INVERSE of a masked autoregressive layer in one kernel, MADE evaluated incrementally (csrc/fc_made_inverse.cu;
 * SURVEY 8(f) n2).  Replaces AutoregressiveTransform.inverse (flowcon/transforms/autoregressive/autoregressive.py:44-53:
 * D passes of the whole conditioner, flowcon/transforms/made.py:274-283, each followed by the element-wise inverse) for
 * a residual MADE, with or without context layers: pass f computes only the hidden units that become valid with feature
 * f - 1 and the parameters of feature f.  The caller (flowconductor_b200/made_inverse.py) compiles the network into a program of
 * PHASES; a phase is a [rows x width] fp32 weight matrix at `weights + 4 * w_off4 + FC_MADE_RECORD_FLOATS` (row-major, masked,
 * zero-padded; the FC_MADE_RECORD_FLOATS words in front of it are a bit copy of the phase's own record, which the kernel
 * receives through its weight ring instead of reading `phases` on the serial chain; width <= 1920) whose
 * column groups are up to FC_MADE_TASKS tasks that run concurrently (one per warp):
 *
 *   task:  units [j0, j0 + nj) of `out_array`  =  (bias[b_off ...] if FC_MADE_INIT_BIAS else their stored partial sums)
 *                                                 + W[0 .. kn)[c0 .. c0 + nj) . act(`in_array`[k0 .. k0 + kn))  (+ `res_array`[j0 ...])
 *
 * Arrays: 0 = the features (inputs of the MADE: inverted so far), 1 .. n_arrays = hidden-layer outputs in an order of the
 * units in which every masked weight row is a prefix of its input (sorted by degree, made.py:28-51); out_array 0 = the
 * parameter tile of the feature being inverted (j0 = offset inside its P parameters).  act = ReLU with FC_MADE_RELU_IN.
 * c0 and width are multiples of 4, nj <= FC_MADE_MAX_NJ, kn <= rows; nj = 0 marks an unused task slot.  After a phase with
 * feature >= 0 the bijection's inverse of that feature is evaluated from the parameter tile.  Shared memory bounds the
 * network: fc_made_inverse_smem_bytes(...) must not exceed the device's opt-in limit (FC_ERR_UNSUPPORTED otherwise: run the
 * D-pass inverse).
 *
 * Context (a MADE with context_features): the context terms do not depend on x, so they are computed for the whole batch
 * first — `terms` is this call's [B, term_width] matrix g = Wc ctx + bc in the T128 layout (fc_context_terms or
 * fc_linear_apply with FC_LINEAR_OUT_T128).  Each of the n_term_arrays entries names a hidden array whose units start
 * every row tile from bias[b_off + j] + act(terms[row][column + j]) instead of being written with FC_MADE_INIT_BIAS:
 *   relu = 1  MADE initial layer             h = W x + b + relu(Wc ctx + bc)      (made.py:138-140)
 *   relu = 0  first layer of a residual block t = W0 relu(h) + b0 + Wc ctx + bc  (made.py:100-102)
 * so the tasks that write such an array must not set FC_MADE_INIT_BIAS.  term_width is a multiple of 16, column a multiple
 * of 4 with column + hidden <= term_width, b_off + hidden <= n_bias, each array 1 .. n_arrays at most once, `terms`
 * 16-byte aligned; anything else is FC_ERR_INVALID_ARGUMENT.  n_term_arrays = 0 (terms NULL): a MADE without context.
 */
#define FC_MADE_MAX_NJ 24
#define FC_MADE_TASKS 8
#define FC_MADE_RECORD_FLOATS 128 /* the phase's record, struct fc_made_phase padded to 512 bytes, precedes its matrix in `weights` */
#define FC_MADE_RELU_IN 1
#define FC_MADE_INIT_BIAS 2
#define FC_MADE_MAX_TERM_ARRAYS 8
typedef struct fc_made_task {
  int32_t in_array, out_array, k0, kn;
  int32_t j0, nj, c0, flags;
  int32_t res_array, b_off, reserved0, reserved1;
} fc_made_task;
typedef struct fc_made_phase {
  int32_t rows, width, w_off4, feature;
  fc_made_task tasks[FC_MADE_TASKS];
} fc_made_phase;
typedef struct fc_made_term_array {
  int32_t array;  /* hidden array 1 .. n_arrays whose units start from bias + act(term) */
  int32_t column; /* first column of its units in `terms` (a multiple of 4): unit j reads column + j */
  int32_t b_off;  /* the layer's bias inside `bias` */
  int32_t relu;   /* 1: act = ReLU (MADE initial layer), 0: identity (first layer of a block) */
} fc_made_term_array;
typedef struct fc_made_program {
  const fc_made_phase* phases; /* device, 16-byte aligned */
  const float* weights;        /* device, 16-byte aligned */
  const float* bias;           /* device */
  int32_t n_phases, features, params_per_feature, n_arrays, hidden;
  int32_t n_bias;              /* floats in `bias` (staged in shared memory) */
  const float* terms;          /* device, this call's context terms [B, term_width] in T128; NULL when n_term_arrays == 0 */
  int32_t term_width, n_term_arrays;
  fc_made_term_array term_arrays[FC_MADE_MAX_TERM_ARRAYS];
} fc_made_program;
/* Debugging aid (library built with -DFC_MADE_PROFILE=1, else all zero): cycles warp 0 ([0..6]) and warp 5 ([8..14]) of CTA 0
 * spent in the last fc_made_inverse_* launch: [0] reading phase records, [1] waiting for weight slots, [2] multiplying,
 * [3] storing units, [4] phase barriers, [5] inverting features (+ barrier), [6] total.  Synchronises the device. */
int fc_made_inverse_profile(unsigned long long* out32);
/* shared memory the kernel needs with its smallest weight ring (it takes more stages when there is room) */
int64_t fc_made_inverse_smem_bytes(int32_t features, int32_t params_per_feature, int32_t n_arrays, int32_t hidden,
                                   int32_t n_bias);
/* z: the layer's inputs in the inverse direction [B, features]; x: outputs (may alias z); logabsdet [B] as the reference's
 * inverse returns it (the negated forward log-determinant at x).  cfg->inverse must be 1. */
int fc_made_inverse_rqs(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x, int64_t x_row_stride,
                        float* logabsdet, int32_t accumulate_logabsdet, int64_t B, const fc_rqs_config* cfg,
                        int32_t* status, void* stream);
/* The other autoregressive layers through the same kernel: MaskedSumOfSigmoidsTransform (autoregressive.py:266-318, offset
 * -0.5: numerical inverse as fc_sos_apply), MaskedPiecewiseLinear / Quadratic / CubicAutoregressiveTransform
 * (autoregressive.py:321-523; arguments as fc_linspline_apply / fc_quadspline_apply / fc_cubicspline_apply with inverse = 1). */
int fc_made_inverse_sos(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x, int64_t x_row_stride,
                        float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int32_t n_sigmoids, float offset,
                        int32_t bisection_iterations, float lim, void* stream);
int fc_made_inverse_linspline(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x,
                              int64_t x_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B,
                              int32_t num_bins, int32_t tails, float left, float right, float bottom, float top,
                              int32_t* status, void* stream);
int fc_made_inverse_quadspline(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x,
                               int64_t x_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B,
                               const fc_quadspline_config* cfg, int32_t* status, void* stream);
int fc_made_inverse_cubicspline(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x,
                                int64_t x_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B,
                                const fc_quadspline_config* cfg, int32_t* status, void* stream);
/* interleaved (raw scale, shift) parameters, autoregressive.py:97-129 */
int fc_made_inverse_affine(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x,
                           int64_t x_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B,
                           int32_t activation, void* stream);

/*
 * Activation normalisation (csrc/fc_actnorm.cu; SURVEY 8(f) n4): ActNorm.forward / inverse for 2-D inputs,
 * flowcon/transforms/normalization.py:144-218 —  forward y = exp(log_scale) * x + shift, logabsdet = sum(log_scale);
 * inverse y = (x - shift) / exp(log_scale), logabsdet = -sum(log_scale).  log_scale, shift: device [D].  y may alias x.
 * The backward writes grad_x and the per-feature parameter gradients (reductions over the batch, summed in a fixed order:
 * deterministic); grad_logabsdet may be null; workspace: fc_actnorm_workspace_floats(B, D) floats of device scratch.
 */
int fc_actnorm_apply(const float* x, int64_t x_row_stride, const float* log_scale, const float* shift, float* y,
                     int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int32_t D,
                     int32_t inverse, void* stream);
int64_t fc_actnorm_workspace_floats(int64_t B, int32_t D);
int fc_actnorm_backward(const float* x, int64_t x_row_stride, const float* log_scale, const float* shift, const float* grad_y,
                        int64_t gy_row_stride, const float* grad_logabsdet, float* grad_x, int64_t gx_row_stride,
                        float* grad_log_scale, float* grad_shift, float* workspace, int64_t B, int32_t D, int32_t inverse,
                        void* stream);

/*
 * Dense D x D row map of the LU-factorised linear layer (csrc/fc_lulinear.cu; LULinear, flowcon/transforms/lu.py on top of
 * flowcon/transforms/linear.py) for 1 <= D <= 63:  y = x · Mᵀ + c,  logabsdet[b] = *logdet (written, or added to with
 * accumulate_logabsdet).  M: device [D, D] row-major, c: device [D], logdet: device scalar — the caller composes them from
 * the LU factors (forward M = L U, c = bias; inverse M = U⁻¹ L⁻¹, c = -M bias), so nothing is read back to the host and
 * the call can be captured into a CUDA graph.  x and y are [B, D] with their own row strides (>= D), so column slices of
 * wider tensors work; any B.  D outside [1, 63] returns FC_ERR_INVALID_ARGUMENT (wider maps are tensor-core GEMMs).
 * The backward reads (x, grad_y) once and writes grad_x = grad_y · M, grad_M = grad_yᵀ · x and grad_c = Σ_b grad_y[b]
 * (per-CTA partial sums summed in a fixed order: deterministic); workspace: fc_lulinear_workspace_floats(B, D) floats of
 * device scratch.  grad_logdet = Σ_b grad_logabsdet[b] is left to the caller.
 */
int fc_lulinear_apply(const float* x, int64_t x_row_stride, const float* M, const float* c, const float* logdet, float* y,
                      int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B, int32_t D,
                      void* stream);
int64_t fc_lulinear_workspace_floats(int64_t B, int32_t D);
int fc_lulinear_backward(const float* x, int64_t x_row_stride, const float* M, const float* grad_y, int64_t gy_row_stride,
                         float* grad_x, int64_t gx_row_stride, float* grad_M, float* grad_c, float* workspace, int64_t B,
                         int32_t D, void* stream);

/*
 * Batch normalisation as a flow layer (csrc/fc_batchnorm.cu; BatchNorm, flowcon/transforms/normalization.py, 2-D inputs)
 * for 1 <= D <= 4096 in every entry (wider: FC_ERR_UNSUPPORTED).  With w = softplus(unconstrained_weight) + eps and
 * σ = sqrt(var + eps) per feature:
 *   forward  y = w · ((x − mean) / σ) + bias,     logabsdet[b] = Σ_d (log w_d − ½ log(var_d + eps))
 *   inverse  y = σ · ((x − bias) / w) + mean,     logabsdet[b] = −Σ_d (log w_d − ½ log(var_d + eps))
 * The mean is subtracted (the bias, inverse) before the scale is applied, never folded into one shift.  mean, var,
 * unconstrained_weight, bias: device [D], read by the kernels (a captured graph sees later updates of them).
 * fc_batchnorm_stats writes the batch mean and the UNBIASED variance (B - 1; NaN for B = 1, as torch.var) of x [B, D],
 * B >= 1: Welford per thread, Chan merges in a fixed order, no atomics — two calls are bitwise equal.
 * fc_batchnorm_backward, mode FC_BATCHNORM_TRAIN (mean / var are the batch statistics of x, differentiated through),
 * FC_BATCHNORM_EVAL_FORWARD or FC_BATCHNORM_EVAL_INVERSE (running buffers, constants): grad_x, and the gradients of
 * unconstrained_weight and bias (deterministic, per-CTA partial sums summed in a fixed order); grad_logabsdet may be
 * null.  Training mode reads x and grad_y twice (column sums, then grad_x: three launches), eval mode once (two).
 * workspace: fc_batchnorm_workspace_floats(B, D) floats of device scratch, for the statistics and the backward.
 * x, y and the gradients are [B, D] with their own row strides (>= D); any B >= 0 (stats: B >= 1).
 */
#define FC_BATCHNORM_TRAIN 0
#define FC_BATCHNORM_EVAL_FORWARD 1
#define FC_BATCHNORM_EVAL_INVERSE 2
int64_t fc_batchnorm_workspace_floats(int64_t B, int32_t D);
int fc_batchnorm_stats(const float* x, int64_t x_row_stride, float* mean, float* var, float* workspace, int64_t B,
                       int32_t D, void* stream);
int fc_batchnorm_apply(const float* x, int64_t x_row_stride, const float* mean, const float* var,
                       const float* unconstrained_weight, const float* bias, float eps, float* y, int64_t y_row_stride,
                       float* logabsdet, int64_t B, int32_t D, int32_t inverse, void* stream);
int fc_batchnorm_backward(const float* x, int64_t x_row_stride, const float* mean, const float* var,
                          const float* unconstrained_weight, const float* bias, float eps, const float* grad_y,
                          int64_t gy_row_stride, const float* grad_logabsdet, float* grad_x, int64_t gx_row_stride,
                          float* grad_unconstrained_weight, float* grad_bias, float* workspace, int64_t B, int32_t D,
                          int32_t mode, void* stream);

/*
 * Diagonal Gaussian base densities (csrc/fc_diagnormal.cu; DiagonalNormal and ConditionalDiagonalNormal,
 * flowcon/distributions/normal.py), any D >= 1.  The parameters are params [C, 2D] row-major (row stride >= 2D; ignored
 * when one row serves every data row): means in columns [0, D), log standard deviations s in columns [D, 2D), so a
 * context encoder's output is read in place.  Data row r uses parameter row r / group (C = ceil(R / group)):
 * group 1 for a conditional log-density, n for n draws per context row, R for one shared row.
 *   fc_diagnormal_log_prob   out[r] = −½ Σ_d z² − Σ_d s − ½ D ln 2π (+ logabsdet[r]),  z = (x − m) · e^{−s};
 *                            logabsdet may be NULL
 *   fc_diagnormal_sample     samples[r] = m + e^{s} · noise[r]
 * The backward entries write grad_params [C, 2D] (dense): for the log-density, grad_x = −g z e^{−s} and the group sums
 * of g z e^{−s} (means) and g (z² − 1) (log standard deviations), g = grad_out [R]; for sampling, the group sums of
 * grad_samples (means) and grad_samples · e^{s} · noise (log standard deviations).  The sums are taken in a fixed
 * order (deterministic); workspace: fc_diagnormal_workspace_floats(R, D, group) floats of device scratch (may be NULL
 * when that is 0).  x, noise, samples and the gradients are [R, D] with their own row strides (>= D); any R >= 0.
 */
int fc_diagnormal_log_prob(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                           const float* logabsdet, float* out, int64_t R, int32_t D, int64_t group, void* stream);
int fc_diagnormal_log_prob_backward(const float* x, int64_t x_row_stride, const float* params,
                                    int64_t params_row_stride, const float* grad_out, float* grad_x,
                                    int64_t gx_row_stride, float* grad_params, float* workspace, int64_t R, int32_t D,
                                    int64_t group, void* stream);
int fc_diagnormal_sample(const float* noise, int64_t noise_row_stride, const float* params, int64_t params_row_stride,
                         float* samples, int64_t samples_row_stride, int64_t R, int32_t D, int64_t group, void* stream);
int fc_diagnormal_sample_backward(const float* noise, int64_t noise_row_stride, const float* params,
                                  int64_t params_row_stride, const float* grad_samples, int64_t gs_row_stride,
                                  float* grad_params, float* workspace, int64_t R, int32_t D, int64_t group,
                                  void* stream);
int64_t fc_diagnormal_workspace_floats(int64_t R, int32_t D, int64_t group);

/*
 * Element-wise squashing layers (csrc/fc_pointwise.cu; Sigmoid / Logit, Tanh, LeakyReLU, Exp, CauchyCDF,
 * flowcon/transforms/nonlinearities.py) on x [B, D], any B >= 0, D >= 1, row strides >= D:
 *   op                         forward y, log-det term                      inverse x, log-det term
 *   FC_POINTWISE_SIGMOID       σ(T x), log T − softplus(−T x) − softplus(T x)  logit(clamp(y, eps, 1 − eps)) / T, minus it
 *   FC_POINTWISE_TANH          tanh x, log(1 − tanh² x)                      atanh y, −log(1 − y²)
 *   FC_POINTWISE_LEAKY_RELU    leaky_relu(x, slope), log slope · [x < 0]      leaky_relu(y, 1 / slope), −log slope · [y < 0]
 *   FC_POINTWISE_EXP           eˣ, x                                         log y, −log y
 *   FC_POINTWISE_CAUCHY_CDF    atan(x) / π + ½, −log π − log(1 + x²)         tan(π (y − ½)), log π + log(1 + x²)
 * logabsdet[b] = (accumulate ? logabsdet[b] : 0) + Σ_d (log-det term).  `temperature` is a device pointer to T (one
 * float, read by the kernels: a captured graph sees later updates; Sigmoid only).  The directions in which the
 * reference raises InputOutsideDomain (the inverses of Sigmoid, Tanh, Exp and CauchyCDF) OR
 * FC_STATUS_INPUT_OUTSIDE_DOMAIN into *status (may be NULL) for inputs outside [0, 1], outside (−1, 1), <= 0 and
 * outside [0, 1] respectively, and compute on.
 * fc_pointwise_backward reads the layer's input x once and writes grad_x = grad_y · dy/dx + grad_logabsdet[b] ·
 * d(log-det term)/dx (grad_y and grad_logabsdet may be NULL: zero).  With grad_temperature non-NULL (Sigmoid) it also
 * writes ∂/∂T of the same objective, summed over every element through per-CTA partials in a fixed order and a finish
 * kernel: two calls are bitwise equal.  workspace: fc_pointwise_workspace_floats(B, D) floats of device scratch.
 */
#define FC_POINTWISE_SIGMOID 0
#define FC_POINTWISE_TANH 1
#define FC_POINTWISE_LEAKY_RELU 2
#define FC_POINTWISE_EXP 3
#define FC_POINTWISE_CAUCHY_CDF 4
typedef struct fc_pointwise_config {
  int32_t op;                /* FC_POINTWISE_* */
  int32_t inverse;           /* 0 forward, 1 inverse */
  float slope;               /* LeakyReLU: the layer's negative slope (> 0) */
  float eps;                 /* Sigmoid: the inverse's clamp */
  const float* temperature;  /* Sigmoid: device [1] */
} fc_pointwise_config;
int fc_pointwise_apply(const float* x, int64_t x_row_stride, float* y, int64_t y_row_stride, float* logabsdet,
                       int32_t accumulate_logabsdet, int64_t B, int64_t D, const fc_pointwise_config* cfg,
                       int32_t* status, void* stream);
int64_t fc_pointwise_workspace_floats(int64_t B, int64_t D);
int fc_pointwise_backward(const float* x, int64_t x_row_stride, const float* grad_y, int64_t gy_row_stride,
                          const float* grad_logabsdet, float* grad_x, int64_t gx_row_stride, float* grad_temperature,
                          float* workspace, int64_t B, int64_t D, const fc_pointwise_config* cfg, void* stream);

/* Library / build info (also used by the loader test). */
const char* fc_version(void);
int fc_built_for_sm(void); /* 100 */

#ifdef __cplusplus
}
#endif
#endif /* FLOWCON_B200_H */
