// fc_sos.cu — sum-of-sigmoids + extended-softplus element-wise transform for sm_100a.
//
// Replaces SumOfSigmoids.forward / sum_of_sigmoids / get_params (flowcon/transforms/adaptive_sigmoids.py
// :111-142), ExtendedSoftplus.forward (flowcon/transforms/nonlinearities.py:519-552) and, for the
// inverse, MonotonicTransform.newton_inverse / bisection_inverse (no_analytic_inv/base.py:23-83) — the
// reference builds an nn.Module per call and runs ~35 pointwise passes over [B, D, n] (forward) or ~55
// full forward passes plus two autograd passes with host syncs (inverse).
// Kernel skeleton: fc_staged.cuh; element math: fc_math.cuh.
#include "fc_pipeline.cuh"
#include "fc_made_inverse.cuh"

namespace fc {

template <int kMB>
struct SosOpT {
  static constexpr int kTileBwdWarps = 8, kTileBwdMaxWarps = 16;  // the adjoint wants 128 registers (fc_pipeline.cuh)
  static constexpr int kMinBlocks = kMB;
  int n;
  float offset;
  __device__ __forceinline__ int P() const { return 3 * n + 1; }
  __device__ __forceinline__ void eval(float x, const float* p, float& y, float& lad, unsigned& status) const {
    float lj;
    if (n == 10) {  // the default of ConditionalSumOfSigmoidsTransform (conditional.py:746): fully unrolled
      sos_eval_t<10>(x, p, n, y, lj);
    } else {
      sos_eval_t<0>(x, p, n, y, lj);
    }
    y += offset;
    lad = lj;
    (void)status;
  }
  __device__ __forceinline__ void backward(float x, const float* p, float gy, float gl, float& gx, float* gp) const {
    // gp may alias p (in-place tile): sos_backward_elem finishes every read of slot j / n+j / 2n+j before it
    // writes that slot, and reads the whole softmax block (normaliser, dot product) before the first write.
    if (n == 10) {
      sos_backward_elem_t<10>(x, p, n, gy, gl, gx, gp);
    } else {
      sos_backward_elem_t<0>(x, p, n, gy, gl, gx, gp);
    }
  }
};

using SosOp = SosOpT<0>;

// adjoint of the numerical inverse: x is the inverse's output (sos_backward_elem_t<NC, true>)
struct SosInverseAdjointOp {
  static constexpr int kTileBwdWarps = 8, kTileBwdMaxWarps = 16;
  int n;
  __device__ __forceinline__ int P() const { return 3 * n + 1; }
  __device__ __forceinline__ void backward(float x, const float* p, float gy, float gl, float& gx, float* gp) const {
    // gp may alias p: the same read-before-write order as SosOpT::backward
    if (n == 10) {
      sos_backward_elem_t<10, true>(x, p, n, gy, gl, gx, gp);
    } else {
      sos_backward_elem_t<0, true>(x, p, n, gy, gl, gx, gp);
    }
  }
};

// the numerical inverse is its own kernel instantiation: its register-resident constants must not raise the
// register count of the forward kernel
struct SosInverseOp {
  int n;
  float offset;
  int iters;
  float lim;
  __device__ __forceinline__ int P() const { return 3 * n + 1; }
  __device__ __forceinline__ void eval(float x, const float* p, float& y, float& lad, unsigned& status) const {
    float lj;
    if (n == 10) {
      sos_invert_t<10>(x - offset, p, n, iters, lim, y, lj);
    } else {
      sos_invert_t<0>(x - offset, p, n, iters, lim, y, lj);
    }
    lad = -lj;
    (void)status;
  }
};

// incremental autoregressive inverse (fc_made_inverse.cuh): the numerical inverse of one feature
template <int NC>
struct MadeSosOp {
  int n;
  float offset;
  int iters;
  float lim;
  __device__ __forceinline__ void eval(float z, const float* pc, float& x, float& lad, unsigned&) const {
    float p[3 * (NC ? NC : FC_SOS_MAX_SIGMOIDS) + 1];
    made_load_params(pc, 3 * n + 1, p);
    float lj;
    sos_invert_t<NC>(z - offset, p, n, iters, lim, x, lj);
    lad = -lj;
  }
};

}  // namespace fc

using namespace fc;

extern "C" int fc_made_inverse_sos(const fc_made_program* prog, const float* z, int64_t z_row_stride, float* x,
                                   int64_t x_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B,
                                   int32_t n_sigmoids, float offset, int32_t bisection_iterations, float lim, void* stream) {
  if (n_sigmoids < 1) return FC_ERR_INVALID_ARGUMENT;
  if (n_sigmoids > FC_SOS_MAX_SIGMOIDS) return FC_ERR_UNSUPPORTED;
  MadeArgs a{};
  int rc = made_check(prog, z, z_row_stride, x, x_row_stride, logabsdet, B, 3 * n_sigmoids + 1, a);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  a.accumulate = accumulate_logabsdet;
  a.status = nullptr;
  if (n_sigmoids == 10) {
    MadeSosOp<10> op{n_sigmoids, offset, bisection_iterations, lim};
    return launch_made(a, op, (cudaStream_t)stream);
  }
  MadeSosOp<0> op{n_sigmoids, offset, bisection_iterations, lim};
  return launch_made(a, op, (cudaStream_t)stream);
}

extern "C" int fc_sos_apply(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                            float* y, int64_t y_row_stride, float* logabsdet, int32_t accumulate_logabsdet, int64_t B,
                            int32_t D, int32_t n_sigmoids, float offset, int32_t inverse, int32_t bisection_iterations,
                            float lim, void* stream) {
  fc_cols none = {nullptr, 0};
  int rc = check_layer_args(x, params, y, B, D, none, none);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  if (!logabsdet) return FC_ERR_INVALID_ARGUMENT;
  if (n_sigmoids < 1) return FC_ERR_INVALID_ARGUMENT;
  if (n_sigmoids > FC_SOS_MAX_SIGMOIDS) return FC_ERR_UNSUPPORTED;
  if (B == 0) return FC_OK;
  LayerArgs a;
  a.x = x; a.params = params; a.y = y; a.lad = logabsdet; a.status = nullptr;
  a.x_stride = x_row_stride; a.p_stride = params_row_stride; a.y_stride = y_row_stride;
  a.B = B; a.D_t = D; a.n_copy = 0; a.tcols = nullptr; a.ccols = nullptr;
  a.accumulate = accumulate_logabsdet;
  const size_t smem = plan_tiles(a, 3 * n_sigmoids + 1);
  if (inverse) {
    SosInverseOp op;
    op.n = n_sigmoids; op.offset = offset; op.iters = bisection_iterations; op.lim = lim;
    const int piped = try_launch_pipelined(a, op, 3 * n_sigmoids + 1, (int)x_row_stride, (cudaStream_t)stream);
    if (piped != 0) return piped < 0 ? piped : FC_OK;
    return launch_apply(a, op, smem, (cudaStream_t)stream);
  }
  static const bool full_regs = env_int("FC_SOS_FULLREGS", 1) != 0;
  if (full_regs) {  // 128 registers, one CTA per SM: no spills (the kernel is bound by the special-function unit)
    SosOpT<1> op1;
    op1.n = n_sigmoids; op1.offset = offset;
    const int piped1 = try_launch_pipelined(a, op1, 3 * n_sigmoids + 1, (int)x_row_stride, (cudaStream_t)stream);
    if (piped1 != 0) return piped1 < 0 ? piped1 : FC_OK;
  }
  SosOp op;
  op.n = n_sigmoids; op.offset = offset;
  const int piped = try_launch_pipelined(a, op, 3 * n_sigmoids + 1, (int)x_row_stride, (cudaStream_t)stream);
  if (piped != 0) return piped < 0 ? piped : FC_OK;
  return launch_apply(a, op, smem, (cudaStream_t)stream);
}

template <class Op>
static int sos_backward_launch(const Op& op, const float* x, int64_t x_row_stride, const float* params,
                               int64_t params_row_stride, const float* grad_y, int64_t gy_row_stride,
                               const float* grad_logabsdet, float* grad_x, int64_t gx_row_stride, float* grad_params,
                               int64_t gp_row_stride, int64_t B, int32_t D, int32_t n_sigmoids, void* stream) {
  fc_cols none = {nullptr, 0};
  int rc = check_layer_args(x, params, grad_x, B, D, none, none);
  if (rc != FC_OK) return rc;
  if (B == 0) return FC_OK;
  if (!grad_y || !grad_params) return FC_ERR_INVALID_ARGUMENT;
  if (n_sigmoids < 1) return FC_ERR_INVALID_ARGUMENT;
  if (n_sigmoids > FC_SOS_MAX_SIGMOIDS) return FC_ERR_UNSUPPORTED;
  LayerBwdArgs a;
  a.x = x; a.params = params; a.gy = grad_y; a.gl = grad_logabsdet; a.gx = grad_x; a.gp = grad_params;
  a.x_stride = x_row_stride; a.p_stride = params_row_stride; a.gy_stride = gy_row_stride;
  a.gx_stride = gx_row_stride; a.gp_stride = gp_row_stride;
  a.B = B; a.D_t = D; a.n_copy = 0; a.tcols = nullptr; a.ccols = nullptr;
  const size_t smem = plan_tiles(a, 3 * n_sigmoids + 1);
  const int piped = try_launch_pipelined_backward(a, op, 3 * n_sigmoids + 1, (int)x_row_stride, (cudaStream_t)stream);
  if (piped != 0) return piped < 0 ? piped : FC_OK;
  return launch_backward(a, op, smem, (cudaStream_t)stream);
}

extern "C" int fc_sos_backward(const float* x, int64_t x_row_stride, const float* params, int64_t params_row_stride,
                               const float* grad_y, int64_t gy_row_stride, const float* grad_logabsdet, float* grad_x,
                               int64_t gx_row_stride, float* grad_params, int64_t gp_row_stride, int64_t B, int32_t D,
                               int32_t n_sigmoids, void* stream) {
  SosOp op;
  op.n = n_sigmoids; op.offset = 0.f;
  return sos_backward_launch(op, x, x_row_stride, params, params_row_stride, grad_y, gy_row_stride, grad_logabsdet,
                             grad_x, gx_row_stride, grad_params, gp_row_stride, B, D, n_sigmoids, stream);
}

extern "C" int fc_sos_inverse_backward(const float* x, int64_t x_row_stride, const float* params,
                                       int64_t params_row_stride, const float* grad_y, int64_t gy_row_stride,
                                       const float* grad_logabsdet, float* grad_x, int64_t gx_row_stride,
                                       float* grad_params, int64_t gp_row_stride, int64_t B, int32_t D,
                                       int32_t n_sigmoids, void* stream) {
  SosInverseAdjointOp op;
  op.n = n_sigmoids;
  return sos_backward_launch(op, x, x_row_stride, params, params_row_stride, grad_y, gy_row_stride, grad_logabsdet,
                             grad_x, gx_row_stride, grad_params, gp_row_stride, B, D, n_sigmoids, stream);
}
