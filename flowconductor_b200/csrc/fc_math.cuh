// fc_math.cuh — per-element arithmetic of the bijections, shared by every kernel in this directory.
//
// All functions are __host__ __device__ so that the exact statements the GPU executes can also be
// compiled with g++ into a test-only shim (tests/hostmath) and checked against the oracle on a box
// without a GPU.  The product never calls the host instantiation.
//
// Arithmetic follows the reference's operation order where fp32 parity depends on it (citations are
// file:line under /root/reference):
//   knots:   softmax -> min + (1-min*K)*p -> running sum -> (hi-lo)*cum + lo -> forced end knots ->
//            bin sizes from knot differences          splines/rational_quadratic.py:91-98,106-113
//   bin:     largest i with knot_i <= x  (== count(knots <= x) - 1 for sorted knots, last knot + 1e-6)
//                                                      utils/torchutils.py:147-149
//   forward: rational_quadratic.py:162-181     inverse: rational_quadratic.py:132-160
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/flowcon_b200.h"

#if defined(__CUDACC__)
#define FC_HD __host__ __device__ __forceinline__
#else
#define FC_HD inline
#endif

// Un-contracted fp32 primitives for the knot pipeline: eager PyTorch rounds after every op, and the bin
// an input lands in depends on the knot bits.  (The closed forms below may use FMA: more accurate.)
#if defined(__CUDA_ARCH__)
#define FC_MUL(a, b) __fmul_rn((a), (b))
#define FC_ADD(a, b) __fadd_rn((a), (b))
#define FC_SUB(a, b) __fsub_rn((a), (b))
#else
#define FC_MUL(a, b) ((a) * (b))  // host shim is built with -ffp-contract=off
#define FC_ADD(a, b) ((a) + (b))
#define FC_SUB(a, b) ((a) - (b))
#endif

// Fast primitives (DESIGN.md "arithmetic budget"): the layer kernels are instruction-issue bound with IEEE
// division / full-range expf, so the hot path uses the SFU approximations where the error analysis allows:
//   fc_exp2: ex2.approx (~1-2 ulp).  Used for softmax numerators 2^(t - max), t <= max: the absolute error of a
//            softmax term is <= e^-|x| |x| 6e-8 <= 2.2e-8, below the fp32 rounding of the term itself.
//   fc_rcp : rcp.approx + one Newton step (<= 1 ulp), a*fc_rcp(b) replaces a/b (<= 1.5 ulp vs 0.5 ulp).
//   fc_sqrt: sqrt.approx (max rel. error 2^-23).
// Host builds (test shim) use the libm equivalents.
#if defined(__CUDA_ARCH__)
#define FC_DEVICE_MATH 1
#else
#define FC_DEVICE_MATH 0
#endif

#define FC_LOG2E 1.4426950408889634f

#define FC_MAX_BINS_GENERIC 64  // runtime-K instantiation keeps its arrays in local memory up to this

namespace fc {

FC_HD float fc_exp2(float x) {
#if FC_DEVICE_MATH
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return exp2f(x);
#endif
}

FC_HD float fc_rcp(float x) {
#if FC_DEVICE_MATH
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return fmaf(r, fmaf(-x, r, 1.f), r);
#else
  return 1.f / x;
#endif
}

FC_HD float fc_sqrt(float x) {
#if FC_DEVICE_MATH
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return sqrtf(x);
#endif
}

// a / b to <= 0.5 ulp + epsilon: approximate reciprocal, then one residual correction of the QUOTIENT.
FC_HD float fc_div(float a, float b) {
#if FC_DEVICE_MATH
  const float r = fc_rcp(b);
  const float q = a * r;
  return fmaf(fmaf(-b, q, a), r, q);
#else
  return a / b;
#endif
}

// exp(x) for the softplus argument (|x| <= 20): relative error <= |x| 6e-8 + ~2 ulp
FC_HD float fc_exp(float x) { return fc_exp2(x * FC_LOG2E); }

// Device-side copy of fc_rqs_config plus host-precomputed constants.
struct RqsParams {
  int K, tails, identity_init, inverse;
  float left, right, bottom, top;
  float min_w, min_h, min_d, wh_scale;
  float wh_scale_l2e;    // wh_scale * log2(e): the softmax is evaluated in base 2
  float beta, inv_beta;  // softplus beta (rational_quadratic.py:100-103)
  float pad_deriv;       // derivative at the two padded boundary knots, linear tails (:33-36 then :104)
  float coef_w, coef_h;  // 1 - min*K (:92, :107)
  int P;                 // params per feature
};

// log1p(E) for E in [0, 1]:  2 atanh(E / (2 + E)) = 2 s (1 + s^2/3 + s^4/5 + ... + s^12/13), s <= 1/3
// (truncation < 1.5e-8 relative).  Branch-free, no integer ops; ~12 instructions.
FC_HD float fc_log1p_unit_r(float E, float r /* = 1 / (2 + E) */) {
  const float sv = E * r, s2 = sv * sv;
  float poly = fmaf(s2, 2.f / 13.f, 2.f / 11.f);
  poly = fmaf(s2, poly, 2.f / 9.f);
  poly = fmaf(s2, poly, 2.f / 7.f);
  poly = fmaf(s2, poly, 2.f / 5.f);
  poly = fmaf(s2, poly, 2.f / 3.f);
  poly = fmaf(s2, poly, 2.f);
  return sv * poly;
}
FC_HD float fc_log1p_unit(float E) {
#if FC_DEVICE_MATH
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(2.f + E));
#else
  const float r = 1.f / (2.f + E);
#endif
  const float sv = E * r, s2 = sv * sv;
  float poly = fmaf(s2, 2.f / 13.f, 2.f / 11.f);
  poly = fmaf(s2, poly, 2.f / 9.f);
  poly = fmaf(s2, poly, 2.f / 7.f);
  poly = fmaf(s2, poly, 2.f / 5.f);
  poly = fmaf(s2, poly, 2.f / 3.f);
  poly = fmaf(s2, poly, 2.f);
  return sv * poly;
}

// torch.nn.functional.softplus(x, beta, threshold=20) = log1p(exp(beta x)) / beta (x itself above the
// threshold), evaluated as (max(z,0) + log1p(exp(-|z|))) / beta with z = beta x: one formula for the whole
// range (for z > 20 the correction is < 2.1e-9 and vanishes in fp32, which reproduces the threshold rule).
FC_HD float softplus_beta(float x, float beta, float inv_beta) {
  const float z = x * beta;
  const float E = fc_exp2(-fabsf(z) * FC_LOG2E);
  return (fmaxf(z, 0.f) + fc_log1p_unit(E)) * inv_beta;
}

FC_HD float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

FC_HD float softplus1(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// derivative of softplus_beta w.r.t. x
FC_HD float softplus_beta_grad(float x, float beta) {
  const float bx = x * beta;
  return bx > 20.f ? 1.f : sigmoidf_(bx);
}

// Host side: validate an fc_rqs_config and derive the constants the kernels use.
inline int make_rqs_params(const fc_rqs_config* cfg, RqsParams& c) {
  if (!cfg) return FC_ERR_INVALID_ARGUMENT;
  if (cfg->num_bins < 1) return FC_ERR_INVALID_ARGUMENT;
  if (cfg->num_bins > FC_MAX_BINS_GENERIC) return FC_ERR_UNSUPPORTED;
  if (cfg->tails != FC_TAILS_NONE && cfg->tails != FC_TAILS_LINEAR) return FC_ERR_INVALID_ARGUMENT;
  // rational_quadratic.py:86-89 raises ValueError for these
  if (cfg->min_bin_width * cfg->num_bins > 1.0f || cfg->min_bin_height * cfg->num_bins > 1.0f)
    return FC_ERR_INVALID_ARGUMENT;
  c.K = cfg->num_bins;
  c.tails = cfg->tails;
  c.identity_init = cfg->identity_init;
  c.inverse = cfg->inverse;
  c.left = cfg->left;
  c.right = cfg->right;
  c.bottom = cfg->bottom;
  c.top = cfg->top;
  c.min_w = cfg->min_bin_width;
  c.min_h = cfg->min_bin_height;
  c.min_d = cfg->min_derivative;
  c.wh_scale = cfg->wh_scale;
  c.wh_scale_l2e = (float)((double)cfg->wh_scale * 1.4426950408889634);
  const double beta = cfg->identity_init ? log(2.0) / (1.0 - (double)cfg->min_derivative) : 1.0;
  c.beta = (float)beta;
  c.inv_beta = (float)(1.0 / beta);
  // rational_quadratic.py:34: constant = log(exp(1 - min_derivative) - 1), stored into an fp32 tensor
  const float pad_raw = (float)log(exp(1.0 - (double)cfg->min_derivative) - 1.0);
  c.pad_deriv = c.min_d + softplus_beta(pad_raw, c.beta, c.inv_beta);
  // (1 - min * K) is evaluated in Python doubles in the reference, then multiplies an fp32 tensor
  c.coef_w = (float)(1.0 - (double)cfg->min_bin_width * cfg->num_bins);
  c.coef_h = (float)(1.0 - (double)cfg->min_bin_height * cfg->num_bins);
  c.P = cfg->tails == FC_TAILS_LINEAR ? 3 * c.K - 1 : 3 * c.K + 1;
  return FC_OK;
}

// derivative value at knot j (0..K).  `pd` points at the raw derivative block of this feature.  Branch-free:
// with linear tails the two boundary knots take the padded constant (rational_quadratic.py:33-36).
FC_HD float knot_derivative(const RqsParams& c, int K, const float* pd, int j) {
  const bool lin = c.tails == FC_TAILS_LINEAR;
  const bool padded = lin && (j == 0 || j == K);
  const int idx = padded ? 0 : (lin ? j - 1 : j);
  const float d = c.min_d + softplus_beta(pd[idx], c.beta, c.inv_beta);
  return padded ? c.pad_deriv : d;
}

// Register-resident variant for the fused kernels: `pd` is a register array, so the raw derivative is picked with a
// select chain over compile-time indices instead of a dynamic index (which would push the array to local memory).  Same
// arithmetic as knot_derivative: K - 1 raw derivatives with linear tails (padded boundary knots), K + 1 without.
// NPD: entries of `pd` the caller's array really has (KC - 1: linear tails only; KC + 1: both).
template <int KC, int NPD>
FC_HD float knot_derivative_regs(const RqsParams& c, const float* pd, int j) {
  static_assert(NPD >= KC - 1 && NPD <= KC + 1, "raw derivatives per feature");
  const bool lin = NPD < KC + 1 || c.tails == FC_TAILS_LINEAR;
  const bool padded = lin && (j == 0 || j == KC);
  const int idx = padded ? 0 : (lin ? j - 1 : j);
  float raw = pd[0];
#pragma unroll
  for (int i = 1; i < NPD; ++i) raw = (i == idx) ? pd[i] : raw;
  const float d = c.min_d + softplus_beta(raw, c.beta, c.inv_beta);
  return padded ? c.pad_deriv : d;
}

// softmax numerators e[i] = 2^(scale_l2e*u[i] - max) == exp(scale*u[i] - max'); returns their sum.
template <int KC>
FC_HD float softmax_numerators(const float* u, int K, float scale_l2e, float* e) {
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < (KC ? KC : K); ++i) {
    e[i] = u[i] * scale_l2e;
    m = fmaxf(m, e[i]);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < (KC ? KC : K); ++i) {
    e[i] = fc_exp2(e[i] - m);
    s += e[i];
  }
  return s;
}

// One running-sum step of the knot pipeline.  torch.cumsum on CPU accumulates fp32 inputs in double
// (acc_type<float,false>), so for more than 8 bins a plain fp32 running sum is measurably worse than the
// reference; Kahan compensation is used there.
template <bool kCompensated>
FC_HD void knot_accumulate(float size, float& cum, float& comp) {
  if (kCompensated) {
    const float yv = FC_SUB(size, comp);
    const float t = FC_ADD(cum, yv);
    comp = FC_SUB(FC_SUB(t, cum), yv);
    cum = t;
  } else {
    cum = FC_ADD(cum, size);
  }
}

// Walk the knots of BOTH axes in one pass.  The "search" axis (widths for the forward map, heights for the
// inverse) locates the bin: k = largest i with knot_i <= x.  Knots are increasing, so the predicates
// p_i = (x >= knot_i) are a run of trues followed by falses and "last true wins" selects bin k on both axes with
// the same predicates.  size_i = min + (1 - min K) softmax_i is one FMA per bin (g = (1 - min K) / sum(e) is
// computed to full precision by the caller: an error in g would move every knot coherently).
// Outputs: k, [s_lo, s_hi] = knots k, k+1 of the search axis, [o_lo, o_hi] the same for the other axis.
template <int KC>
FC_HD void knot_scan2(const float* es, float gs, float lo_s, float hi_s, float min_s, const float* eo, float go,
                      float lo_o, float hi_o, float min_o, int K, float x, int& k, float& s_lo, float& s_hi,
                      float& o_lo, float& o_hi) {
  constexpr bool kCompensated = (KC == 0 || KC > 8);
  const float span_s = hi_s - lo_s, span_o = hi_o - lo_o;
  float cum_s = 0.f, comp_s = 0.f, prev_s = lo_s;
  float cum_o = 0.f, comp_o = 0.f, prev_o = lo_o;
  k = 0;
  s_lo = lo_s;
  s_hi = hi_s;
  o_lo = lo_o;
  o_hi = hi_o;
#pragma unroll
  for (int i = 0; i < (KC ? KC : K); ++i) {
    knot_accumulate<kCompensated>(fmaf(es[i], gs, min_s), cum_s, comp_s);
    knot_accumulate<kCompensated>(fmaf(eo[i], go, min_o), cum_o, comp_o);
    const bool last = (i == K - 1);
    const float next_s = last ? hi_s : fmaf(span_s, cum_s, lo_s);
    const float next_o = last ? hi_o : fmaf(span_o, cum_o, lo_o);
    if (x >= prev_s) {
      k = i;
      s_lo = prev_s;
      s_hi = next_s;
      o_lo = prev_o;
      o_hi = next_o;
    }
    prev_s = next_s;
    prev_o = next_o;
  }
}

// Everything the closed forms need about the selected bin.
struct RqsBin {
  int k;
  float cw, w;   // left width knot, bin width
  float ch, h;   // bottom height knot, bin height
  float inv_w;   // 1 / w
  float delta, d0, d1;
};

// Shared front half of forward / inverse / backward: inside test, softmax, knots, bin, derivatives.
// ew / eh receive the softmax numerators (needed again by the backward); inv_w / inv_h their 1/sum.
template <int KC, bool kRegs = false, int NPD = (KC > 1 ? KC - 1 : 1)>
FC_HD void rqs_locate(const RqsParams& c, int K, float x, const float* p, RqsBin& bin, float* ew, float* eh,
                      float& inv_w, float& inv_h) {
  const float sum_w = softmax_numerators<KC>(p, K, c.wh_scale_l2e, ew);
  const float sum_h = softmax_numerators<KC>(p + K, K, c.wh_scale_l2e, eh);
  inv_w = fc_rcp(sum_w);
  inv_h = fc_rcp(sum_h);
  const float gw = fc_div(c.coef_w, sum_w), gh = fc_div(c.coef_h, sum_h);
  float a, b, a2, b2;
  if (!c.inverse) {
    knot_scan2<KC>(ew, gw, c.left, c.right, c.min_w, eh, gh, c.bottom, c.top, c.min_h, K, x, bin.k, a, b, a2, b2);
    bin.cw = a;
    bin.w = FC_SUB(b, a);
    bin.ch = a2;
    bin.h = FC_SUB(b2, a2);
  } else {
    knot_scan2<KC>(eh, gh, c.bottom, c.top, c.min_h, ew, gw, c.left, c.right, c.min_w, K, x, bin.k, a, b, a2, b2);
    bin.ch = a;
    bin.h = FC_SUB(b, a);
    bin.cw = a2;
    bin.w = FC_SUB(b2, a2);
  }
  bin.inv_w = fc_rcp(bin.w);
  bin.delta = bin.h * bin.inv_w;
  const float* pd = p + 2 * K;
  if (kRegs && KC > 1) {
    bin.d0 = knot_derivative_regs<(KC > 1 ? KC : 2), (KC > 1 ? NPD : 1)>(c, pd, bin.k);
    bin.d1 = knot_derivative_regs<(KC > 1 ? KC : 2), (KC > 1 ? NPD : 1)>(c, pd, bin.k + 1);
  } else {
    bin.d0 = knot_derivative(c, K, pd, bin.k);
    bin.d1 = knot_derivative(c, K, pd, bin.k + 1);
  }
}

// Domain handling shared by all entry points.  Returns true if the element takes the spline branch;
// `xs` is the value fed to the spline (clamped into the domain when the reference would have raised).
FC_HD bool rqs_domain(const RqsParams& c, float x, float& xs, unsigned& status) {
  const float lo = c.inverse ? c.bottom : c.left;
  const float hi = c.inverse ? c.top : c.right;
  if (c.tails == FC_TAILS_LINEAR) {
    const bool inside = (x >= lo) && (x <= hi);  // rational_quadratic.py:26 (both ends inclusive)
    xs = inside ? x : 0.f;
    return inside;
  }
  xs = x;
  if (!(x >= lo && x <= hi)) {  // rational_quadratic.py:81-82 raises InputOutsideDomain
    status |= FC_STATUS_INPUT_OUTSIDE_DOMAIN;
    xs = fminf(fmaxf(x, lo), hi);
    if (!(xs == xs)) xs = lo;
  }
  return true;
}

// Inverse closed form: root theta of the quadratic (rational_quadratic.py:132-146).
FC_HD float rqs_inverse_root(const RqsBin& b, float x, unsigned& status) {
  const float u = x - b.ch;
  const float s = b.d0 + b.d1 - 2.f * b.delta;
  const float qa = u * s + b.h * (b.delta - b.d0);
  const float qb = b.h * b.d0 - u * s;
  const float qc = -b.delta * u;
  float disc = qb * qb - 4.f * qa * qc;
  if (!(disc >= 0.f)) {
    status |= FC_STATUS_NEGATIVE_DISCRIMINANT;
    disc = 0.f;
  }
  return (2.f * qc) * fc_rcp(-qb - fc_sqrt(disc));
}

// log(v) for the derivative value v of the spline (1e-4 .. 1e4): lg2.approx (absolute error 2^-22 for v in
// (0.5, 2), relative 2^-22 elsewhere) times ln 2 — the same size as the fp32 rounding of the reference's
// log(numerator) - 2 log(denominator) (rational_quadratic.py:158,179), at 2 instructions instead of ~45.
FC_HD float fc_log_deriv(float v) {
#if FC_DEVICE_MATH
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(v));
  return y * 0.6931471805599453f;
#else
  return logf(v);
#endif
}

// log|dy/dx| of the forward spline at theta (rational_quadratic.py:148-158 / :173-179); also returns
// 1/denominator, which the forward output needs.
FC_HD float rqs_logdet_at(const RqsBin& b, float theta, float& inv_den) {
  const float t1mt = theta * (1.f - theta);
  const float den = b.delta + (b.d0 + b.d1 - 2.f * b.delta) * t1mt;
  const float omt = 1.f - theta;
  const float dnum = (b.delta * b.delta) * (b.d1 * (theta * theta) + 2.f * b.delta * t1mt + b.d0 * (omt * omt));
  inv_den = fc_rcp(den);
  return fc_log_deriv(dnum * inv_den * inv_den);
}

// One element, forward or inverse (c.inverse).  p -> this feature's P raw parameters.
// Branch-free over the tails: outside elements evaluate the spline on a clamped input and are then replaced
// by the identity (rational_quadratic.py:38-39), so a warp never diverges on the inside test.
// NPD (register-resident arrays only): raw derivative entries the array holds — KC - 1 restricts the instantiation to
// linear tails, KC + 1 serves both.
template <int KC, bool kRegs = false, int NPD = (KC > 1 ? KC - 1 : 1)>
FC_HD void rqs_eval(const RqsParams& c, float x, const float* p, float& y, float& lad, unsigned& status) {
  const int K = KC ? KC : c.K;
  float xs;
  const bool inside = rqs_domain(c, x, xs, status);
  float ew[KC ? KC : FC_MAX_BINS_GENERIC], eh[KC ? KC : FC_MAX_BINS_GENERIC];
  float inv_w, inv_h;
  RqsBin b;
  rqs_locate<KC, kRegs, NPD>(c, K, xs, p, b, ew, eh, inv_w, inv_h);
  float inv_den, ys, ls;
  if (c.inverse) {
    const float root = rqs_inverse_root(b, xs, status);
    ys = root * b.w + b.cw;
    ls = -rqs_logdet_at(b, root, inv_den);
  } else {
    const float theta = (xs - b.cw) * b.inv_w;
    const float t1mt = theta * (1.f - theta);
    const float num = b.h * (b.delta * (theta * theta) + b.d0 * t1mt);
    ls = rqs_logdet_at(b, theta, inv_den);
    ys = b.ch + num * inv_den;
  }
  y = inside ? ys : x;
  lad = inside ? ls : 0.f;
}

// Backward of rqs_eval for one element.  Upstream: gy = dL/dy, gl = dL/d(lad).  Writes dL/dx and the P
// parameter gradients to gp[0..P-1] (zeros where the reference's autograd gives zero).  SURVEY.md App. B.
//
// Forward direction.  With a,b the width knots of the bin, cc,ee the height knots:
//   W=b-a, H=ee-cc, theta=(x-a)/W, delta=H/W, s=d0+d1-2delta, t=theta(1-theta),
//   N=H(delta theta^2 + d0 t), D=delta+s t, y=cc+N/D, Q=d1 theta^2+2 delta t+d0(1-theta)^2,
//   lad=2 log delta + log Q - 2 log D.
// Inverse direction: out=g^{-1}(x), lad=-ladf(out); implicit differentiation through the same adjoint
//   with  gy' = -dL/dx  (dL/dx = (gy - gl * d ladf/d out)/g'(out)),  gl' = -gl.
template <int KC>
FC_HD void rqs_backward_elem(const RqsParams& c, float x, const float* p, float gy, float gl, float& gx,
                             float* gp) {
  const int K = KC ? KC : c.K;
  const int P = c.P;
  float xs;
  unsigned status = 0;
  if (!rqs_domain(c, x, xs, status)) {
    gx = gy;
    for (int i = 0; i < P; ++i) gp[i] = 0.f;
    return;
  }
  float ew[KC ? KC : FC_MAX_BINS_GENERIC], eh[KC ? KC : FC_MAX_BINS_GENERIC];
  float inv_w, inv_h;
  RqsBin b;
  rqs_locate<KC>(c, K, xs, p, b, ew, eh, inv_w, inv_h);

  const float W = b.w, H = b.h, delta = b.delta, d0 = b.d0, d1 = b.d1;
  const float s = d0 + d1 - 2.f * delta;
  float theta;
  if (c.inverse) {
    theta = rqs_inverse_root(b, xs, status);
  } else {
    theta = (xs - b.cw) * b.inv_w;
  }
  const float omt = 1.f - theta;
  const float t = theta * omt;
  const float M = delta * theta * theta + d0 * t;
  const float N = H * M;
  const float D = delta + s * t;
  const float Q = d1 * theta * theta + 2.f * delta * t + d0 * omt * omt;
  const float invD = fc_rcp(D), invQ = fc_rcp(Q), invW = b.inv_w;

  float gyf = gy, glf = gl;  // upstream of the FORWARD map evaluated at theta
  float gx_inverse = 0.f;
  if (c.inverse) {
    // d ladf / d theta, and g'(out) = delta^2 Q / D^2
    const float dQ = 2.f * d1 * theta - 2.f * d0 * omt;
    const float dt = 1.f - 2.f * theta;
    const float dlad_dtheta = invQ * (dQ + 2.f * delta * dt) - 2.f * invD * s * dt;
    const float gprime = delta * delta * Q * invD * invD;
    glf = -gl;
    gx_inverse = (gy + glf * dlad_dtheta * invW) * fc_rcp(gprime);
    gyf = -gx_inverse;
  }
  // adjoints
  const float Nb = gyf * invD;
  float Db = -gyf * N * invD * invD - 2.f * glf * invD;
  const float Qb = glf * invQ;
  float deltab = 2.f * glf * fc_rcp(delta) + Qb * 2.f * t + Db;
  float tb = Qb * 2.f * delta + Db * s;
  float d0b = Qb * omt * omt;
  float d1b = Qb * theta * theta;
  float thetab = Qb * (2.f * d1 * theta - 2.f * d0 * omt);
  const float sb = Db * t;
  float Hb = Nb * M;
  const float Mb = Nb * H;
  deltab += Mb * theta * theta;
  thetab += Mb * 2.f * delta * theta;
  d0b += Mb * t + sb;
  tb += Mb * d0;
  d1b += sb;
  deltab -= 2.f * sb;
  thetab += tb * (1.f - 2.f * theta);
  Hb += deltab * invW;
  float Wb = -deltab * delta * invW;
  const float xb = thetab * invW;   // d/dx of theta=(x-a)/W
  float ab = -xb;                    // knot a (left width knot)
  Wb -= thetab * theta * invW;
  const float bb = Wb;               // knot b = a + W
  ab -= Wb;
  const float eb = Hb;               // top height knot
  const float cb = gyf - Hb;         // bottom height knot (y = cc + ...)
  gx = c.inverse ? gx_inverse : xb;

  const int k = b.k;
  // ---- widths: knot_m = left + span * sum_{i<m} w_i for interior m; w_i = min + coef * softmax_i
  {
    const float span = c.right - c.left;
    const float GA = (k >= 1) ? ab * span * c.coef_w : 0.f;
    const float GB = (k + 1 <= K - 1) ? bb * span * c.coef_w : 0.f;
    float dot = 0.f;  // sum_j p_j * pbar_j
#pragma unroll
    for (int i = 0; i < (KC ? KC : K); ++i) {
      const float pi = ew[i] * inv_w;
      const float pb = (i < k ? GA : 0.f) + (i <= k ? GB : 0.f);
      dot += pi * pb;
    }
#pragma unroll
    for (int i = 0; i < (KC ? KC : K); ++i) {
      const float pi = ew[i] * inv_w;
      const float pb = (i < k ? GA : 0.f) + (i <= k ? GB : 0.f);
      gp[i] = c.wh_scale * pi * (pb - dot);
    }
  }
  // ---- heights
  {
    const float span = c.top - c.bottom;
    const float GA = (k >= 1) ? cb * span * c.coef_h : 0.f;
    const float GB = (k + 1 <= K - 1) ? eb * span * c.coef_h : 0.f;
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < (KC ? KC : K); ++i) {
      const float pi = eh[i] * inv_h;
      const float pb = (i < k ? GA : 0.f) + (i <= k ? GB : 0.f);
      dot += pi * pb;
    }
#pragma unroll
    for (int i = 0; i < (KC ? KC : K); ++i) {
      const float pi = eh[i] * inv_h;
      const float pb = (i < k ? GA : 0.f) + (i <= k ? GB : 0.f);
      gp[K + i] = c.wh_scale * pi * (pb - dot);
    }
  }
  // ---- derivatives: only the two knots of the bin, through softplus' = sigmoid(beta * raw)
  {
    // (gp may alias p — the kernels overwrite the staged tile in place — so read before writing)
    const float* pd = p + 2 * K;
    float* gd = gp + 2 * K;
    const int nd = P - 2 * K;
    const int off = (c.tails == FC_TAILS_LINEAR) ? -1 : 0;  // knot j <-> raw index j + off
    const int j0 = k + off, j1 = k + 1 + off;
    const bool has0 = j0 >= 0 && j0 < nd, has1 = j1 >= 0 && j1 < nd;
    const float g0 = has0 ? d0b * softplus_beta_grad(pd[j0], c.beta) : 0.f;
    const float g1 = has1 ? d1b * softplus_beta_grad(pd[j1], c.beta) : 0.f;
    for (int i = 0; i < nd; ++i) gd[i] = 0.f;
    if (has0) gd[j0] = g0;
    if (has1) gd[j1] = g1;
  }
}

// ------------------------------------------------------------------------------------------------
// affine (coupling.py:224-252, autoregressive.py:97-129)
// ------------------------------------------------------------------------------------------------
FC_HD float affine_scale(float u, int activation) {
  if (activation == FC_SCALE_SIGMOID2) return sigmoidf_(u + 2.f) + 1e-3f;
  const float sp = softplus1(u) + 1e-3f;
  if (activation == FC_SCALE_SOFTPLUS_CLAMP3) return fminf(fmaxf(sp, 0.f), 3.f);
  return sp;
}

// d scale / d u
FC_HD float affine_scale_grad(float u, int activation) {
  if (activation == FC_SCALE_SIGMOID2) {
    const float sg = sigmoidf_(u + 2.f);
    return sg * (1.f - sg);
  }
  const float g = u > 20.f ? 1.f : sigmoidf_(u);
  if (activation == FC_SCALE_SOFTPLUS_CLAMP3) {
    const float sp = softplus1(u) + 1e-3f;
    return (sp > 3.f || sp < 0.f) ? 0.f : g;  // torch.clamp backward: gradient passes where min <= x <= max
  }
  return g;
}

FC_HD void affine_eval(float x, float raw_scale, float shift, int activation, int inverse, float& y, float& lad) {
  const float scale = affine_scale(raw_scale, activation);
  const float ls = logf(scale);
  if (inverse) {
    y = (x - shift) / scale;
    lad = -ls;
  } else {
    y = x * scale + shift;
    lad = ls;
  }
}

FC_HD void affine_backward_elem(float x, float raw_scale, float shift, int activation, int inverse, float gy,
                                float gl, float& gx, float& g_raw, float& g_shift) {
  const float scale = affine_scale(raw_scale, activation);
  const float ds = affine_scale_grad(raw_scale, activation);
  if (inverse) {
    const float inv = 1.f / scale;
    gx = gy * inv;
    g_shift = -gy * inv;
    const float y = (x - shift) * inv;
    g_raw = (-gy * y * inv - gl * inv) * ds;
  } else {
    gx = gy * scale;
    g_shift = gy;
    g_raw = (gy * x + gl / scale) * ds;
  }
}

// ------------------------------------------------------------------------------------------------
// piecewise-linear spline (flowcon/transforms/splines/linear.py:9-105; Mueller et al. 2018): K equal-width bins, the
// per-feature parameters are the K unnormalised bin probabilities
// ------------------------------------------------------------------------------------------------
struct LinSplineParams {
  int K, tails, inverse;
  float left, right, bottom, top;
  float log_k;          // log(K): logabsdet = log(pdf) - log(1/K) (linear.py:94-95)
  float inv_w, inv_h;   // 1 / (right - left), 1 / (top - bottom): the normalisations :49-51 as multiplications
};

// The K raw values of one feature -> registers.  Neighbouring lanes own neighbouring features, K words apart: with
// scalar loads K = 8 is an 8-way shared-memory bank conflict (K = 23 / 31 / 47 of the other layers are odd, hence
// conflict-free).  K = 8: two 16-byte loads whose order alternates every 4 lanes (lanes l and l + 4 would hit the same
// banks); K = 10: five 8-byte loads (10 l mod 32 is distinct over a half warp).  Falls back to scalar loads when the
// block is not aligned (general strides).
template <int KC>
FC_HD void linspline_load(int K, const float* u, float* raw) {
#if FC_DEVICE_MATH
  if (KC == 8 && (reinterpret_cast<uintptr_t>(u) & 15) == 0) {
    const bool sw = ((threadIdx.x >> 2) & 1) != 0;
    const float4 a = *reinterpret_cast<const float4*>(u + (sw ? 4 : 0));
    const float4 b = *reinterpret_cast<const float4*>(u + (sw ? 0 : 4));
    raw[0] = sw ? b.x : a.x; raw[1] = sw ? b.y : a.y; raw[2] = sw ? b.z : a.z; raw[3] = sw ? b.w : a.w;
    raw[4] = sw ? a.x : b.x; raw[5] = sw ? a.y : b.y; raw[6] = sw ? a.z : b.z; raw[7] = sw ? a.w : b.w;
    return;
  }
  if (KC == 10 && (reinterpret_cast<uintptr_t>(u) & 7) == 0) {
#pragma unroll
    for (int h = 0; h < 5; ++h) {
      const float2 v = *reinterpret_cast<const float2*>(u + 2 * h);
      raw[2 * h] = v.x;
      raw[2 * h + 1] = v.y;
    }
    return;
  }
#endif
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) raw[j] = u[j];
}

// the mirror image for the K parameter gradients
template <int KC>
FC_HD void linspline_store(int K, float* gu, const float* v) {
#if FC_DEVICE_MATH
  if (KC == 8 && (reinterpret_cast<uintptr_t>(gu) & 15) == 0) {
    const bool sw = ((threadIdx.x >> 2) & 1) != 0;
    const float4 lo = make_float4(v[0], v[1], v[2], v[3]), hi = make_float4(v[4], v[5], v[6], v[7]);
    *reinterpret_cast<float4*>(gu + (sw ? 4 : 0)) = sw ? hi : lo;
    *reinterpret_cast<float4*>(gu + (sw ? 0 : 4)) = sw ? lo : hi;
    return;
  }
  if (KC == 10 && (reinterpret_cast<uintptr_t>(gu) & 7) == 0) {
#pragma unroll
    for (int h = 0; h < 5; ++h) *reinterpret_cast<float2*>(gu + 2 * h) = make_float2(v[2 * h], v[2 * h + 1]);
    return;
  }
#endif
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) gu[j] = v[j];
}

// softmax of the K raw values (linear.py:53) into p[]; max-subtracted like torch.softmax
template <int KC>
FC_HD void linspline_pdf(int K, const float* u, float* p) {
  linspline_load<KC>(K, u, p);
  float m = -INFINITY;
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) m = fmaxf(m, p[j]);
  const float ml2 = m * FC_LOG2E;
  float se = 0.f;
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) {
    p[j] = fc_exp2(fmaf(p[j], FC_LOG2E, -ml2));
    se += p[j];
  }
  const float inv = fc_rcp(se);
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) p[j] *= inv;
}

// domain handling as in rqs_domain: linear tails -> identity outside [-b, b] (linear.py:12-22, both ends inclusive);
// no tails -> the reference raises InputOutsideDomain (linear.py:45-46): flag + clamp
FC_HD bool linspline_domain(const LinSplineParams& c, float x, float& xs, unsigned& status) {
  const float lo = c.inverse ? c.bottom : c.left;
  const float hi = c.inverse ? c.top : c.right;
  if (c.tails == FC_TAILS_LINEAR) {
    const bool inside = (x >= lo) && (x <= hi);
    xs = inside ? x : lo;
    return inside;
  }
  xs = x;
  if (!(x >= lo && x <= hi)) {
    status |= FC_STATUS_INPUT_OUTSIDE_DOMAIN;
    xs = fminf(fmaxf(x, lo), hi);
    if (!(xs == xs)) xs = lo;
  }
  return true;
}

// forward pieces at a normalised position xn in [0, 1]: bin, position inside it, cdf at the bin's left edge
template <int KC>
FC_HD void linspline_forward_bin(int K, float xn, const float* p, int& idx, float& alpha, float& cdf_lo) {
  const float bin_pos = xn * (float)K;               // linear.py:84
  idx = (int)floorf(bin_pos);
  idx = idx >= K ? K - 1 : (idx < 0 ? 0 : idx);      // :86-87
  alpha = bin_pos - (float)idx;                      // :89
  cdf_lo = 0.f;                                      // running sum = torch.cumsum (:55), cdf[idx] of the padded cdf (:57)
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) cdf_lo += j < idx ? p[j] : 0.f;
}

// One element, forward or inverse (c.inverse).  u -> this feature's K raw parameters.
template <int KC>
FC_HD void linspline_eval(const LinSplineParams& c, float x, const float* u, float& y, float& lad, unsigned& status) {
  const int K = KC ? KC : c.K;
  float p[KC ? KC : FC_MAX_BINS_GENERIC];
  float xs;
  const bool inside = linspline_domain(c, x, xs, status);
  linspline_pdf<KC>(K, u, p);
  float ys, ls;
  if (!c.inverse) {
    const float xn = (xs - c.left) * c.inv_w;  // :51
    int idx;
    float alpha, cdf_lo;
    linspline_forward_bin<KC>(K, xn, p, idx, alpha, cdf_lo);
    float pi = 0.f;  // p[idx] as a masked sum (a select chain becomes an indexed load and pushes p[] to local memory)
#pragma unroll(KC ? KC : 4)
    for (int j = 0; j < K; ++j) pi = fmaf(j == idx ? 1.f : 0.f, p[j], pi);
    float o = cdf_lo + alpha * pi;                       // :93-94
    o = fminf(fmaxf(o, 0.f), 1.f);                       // :95
    ls = fc_log_deriv(pi) + c.log_k;                     // :97-98
    ys = o * (c.top - c.bottom) + c.bottom;              // :103
  } else {
    const float yn = (xs - c.bottom) * c.inv_h;  // :49
    // knots c_0 = 0, c_m = p_0 + .. + p_{m-1}, c_K = 1 (forced, :56) + 1e-6 (searchsorted bumps the last knot IN PLACE,
    // torchutils.py:147-149, before the slopes are taken, linear.py:60-71: the last bin's slope sees the bump)
    int idx = -1;
    float run = 0.f, c_lo = 0.f, c_hi = 0.f;
#pragma unroll(KC ? KC + 1 : 4)  // K + 1 trips: a partial unroll would index p[] dynamically and push it to local memory
    for (int m = 0; m <= K; ++m) {
      const float knot = m == K ? 1.f + 1e-6f : run;
      if (yn >= knot) {
        idx = m;
        c_lo = knot;
      }
      if (m < K) run += p[m];
    }
    idx = idx < 0 ? 0 : (idx > K - 1 ? K - 1 : idx);
    // upper knot of the bin (second pass keeps the loop branch-free for the unrolled instantiations)
    run = 0.f;
    c_lo = 0.f;
#pragma unroll(KC ? KC : 4)
    for (int m = 0; m < K; ++m) {
      c_lo = m == idx ? run : c_lo;
      run += p[m];
      c_hi = m == idx ? (m == K - 1 ? 1.f + 1e-6f : run) : c_hi;
    }
    // bin boundaries torch.linspace(0, 1, K + 1): b_m = m / K, so the slope's denominator :66-68 is 1 / K (the
    // reference's fp32 difference of two linspace values carries a rounding error the fp64 reference does not have)
    const float b_hi = (float)(idx + 1) * fc_rcp((float)K);
    const float slope = (c_hi - c_lo) * (float)K;
    const float offset = c_hi - slope * b_hi;                                      // :69
    float o = fc_div(yn - offset, slope);                                          // :75
    o = fminf(fmaxf(o, 0.f), 1.f);                                                 // :76
    ls = -fc_log_deriv(slope);                                                     // :78
    ys = o * (c.right - c.left) + c.left;                                          // :101
  }
  y = inside ? ys : x;
  lad = inside ? ls : 0.f;
}

// Backward of linspline_eval for one element (the reference differentiates the op chain; closed form here).
// Forward direction, inside the domain, S = top - bottom, W = right - left, i = bin, a = position in the bin:
//   y = S (sum_{j<i} p_j + a p_i) + bottom,  lad = log p_i + log K,  dy/dx = S K p_i / W
//   dL/dp_j = gy S ([j<i] + a [j=i]) + gl [j=i] / p_i ;   dL/du_j = p_j (dL/dp_j - sum_k p_k dL/dp_k)  (softmax)
// Inverse direction: out = f^-1(v), lad = -ladf(out); implicit differentiation through the same adjoint:
//   dL/dv = gy / f'(out) =: g;  parameter gradients = forward adjoint at out with upstream (-g, -gl).
template <int KC>
FC_HD void linspline_backward_elem(const LinSplineParams& c, float x, const float* u, float gy, float gl, float& gx,
                                   float* gu) {
  const int K = KC ? KC : c.K;
  float p[KC ? KC : FC_MAX_BINS_GENERIC];
  float xs;
  unsigned status = 0;
  const bool inside = linspline_domain(c, x, xs, status);
  if (!inside) {  // identity outside the tails: no parameter dependence
    gx = gy;
#pragma unroll(KC ? KC : 4)
    for (int j = 0; j < K; ++j) p[j] = 0.f;
    linspline_store<KC>(K, gu, p);
    return;
  }
  linspline_pdf<KC>(K, u, p);
  const float S = c.top - c.bottom;
  float pos = xs;  // forward-direction input at which the adjoint is evaluated
  if (c.inverse) {
    LinSplineParams ci = c;
    float out, unused;
    linspline_eval<KC>(ci, x, u, out, unused, status);
    pos = out;
  }
  const float xn = (pos - c.left) * c.inv_w;
  int idx;
  float alpha, cdf_lo;
  linspline_forward_bin<KC>(K, xn, p, idx, alpha, cdf_lo);
  float pi = 0.f;
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) pi = fmaf(j == idx ? 1.f : 0.f, p[j], pi);
  const float dydx = S * (float)K * pi * c.inv_w;
  float gyf = gy, glf = gl;
  if (c.inverse) {
    // the reference's inverse takes the last bin's slope from the bumped end knot (1 + 1e-6 - c_{K-1}, see
    // linspline_eval): visible in d out / d v when that bin's probability is small
    const float mass = idx == K - 1 ? (1.f + 1e-6f) - cdf_lo : pi;
    const float g = fc_div(gy, S * (float)K * mass * c.inv_w);
    gx = g;
    gyf = -g;
    glf = -gl;
  } else {
    gx = gy * dydx;
  }
  const float gi = fc_div(glf, pi);
  float dot = 0.f;
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) {
    const float gp = gyf * S * (j < idx ? 1.f : (j == idx ? alpha : 0.f)) + (j == idx ? gi : 0.f);
    dot += p[j] * gp;
  }
#pragma unroll(KC ? KC : 4)
  for (int j = 0; j < K; ++j) {
    const float gp = gyf * S * (j < idx ? 1.f : (j == idx ? alpha : 0.f)) + (j == idx ? gi : 0.f);
    p[j] = p[j] * (gp - dot);
  }
  linspline_store<KC>(K, gu, p);  // (gu may alias u: everything was read before the first write)
}

// ------------------------------------------------------------------------------------------------
// sum of sigmoids + extended softplus (adaptive_sigmoids.py:111-142, nonlinearities.py:519-552)
// ------------------------------------------------------------------------------------------------
#define FC_SOS_MAX_SIGMOIDS 64

FC_HD float logaddexpf_(float a, float b) {
  const float m = fmaxf(a, b);
  if (m == -INFINITY) return -INFINITY;
  return m + log1pf(expf(-fabsf(a - b)));
}

// Fast building blocks of the sum-of-sigmoids hot path.  With full-range expf / tanhf / IEEE divisions one element
// (n = 10) costs ~2000 instructions and the kernel sits at 29 % of the HBM roofline; these keep it near 600.
//   fc_sigmoid_parts: E = 2^(-|z| log2e) (ex2.approx), r = 1/(1+E): sigma(z), sigma'(z) = E r^2.  The argument
//     rounding (|z| 1.44 * 2^-24) is a RELATIVE error |z| 8.6e-8 of E, i.e. an absolute error of sigma below
//     |z| e^-|z| 8.6e-8 <= 3.2e-8.
//   fc_tanh: sign(t) (1-E)/(1+E), E = e^(-2|t|), switched to the odd Taylor polynomial below |t| = 0.3 where 1-E
//     would cancel (5 terms: truncation < 2e-8 relative at 0.3).
FC_HD void fc_sigmoid_parts(float z, float& sig, float& dsig) {
  const float E = fc_exp2(-fabsf(z) * FC_LOG2E);
  const float r = fc_rcp(1.f + E);
  const float Er = E * r;
  sig = z >= 0.f ? r : Er;
  dsig = Er * r;
}

// sigma(z) alone, same arithmetic (the context gate of a conditional ResidualNet block, F.glu)
FC_HD float fc_sigmoid(float z) {
  const float E = fc_exp2(-fabsf(z) * FC_LOG2E);
  const float r = fc_rcp(1.f + E);
  return z >= 0.f ? r : E * r;
}

FC_HD float fc_tanh(float t) {
  const float at = fabsf(t);
  const float E = fc_exp2(at * (-2.f * FC_LOG2E));
  const float big = (1.f - E) * fc_rcp(1.f + E);
  const float t2 = t * t;
  float poly = fmaf(t2, 62.f / 2835.f, -17.f / 315.f);
  poly = fmaf(t2, poly, 2.f / 15.f);
  poly = fmaf(t2, poly, -1.f / 3.f);
  poly = fmaf(t2 * at, poly, at);  // |t| (1 - t^2/3 + 2 t^4/15 - 17 t^6/315 + 62 t^8/2835)
  const float m = at < 0.3f ? poly : big;
  return t < 0.f ? -m : m;
}

// softplus(z) = max(z, 0) + log1p(e^-|z|)   (torch threshold rule reproduced as in softplus_beta)
FC_HD float fc_softplus1(float z) { return fmaxf(z, 0.f) + fc_log1p_unit(fc_exp2(-fabsf(z) * FC_LOG2E)); }

// --- MUFU-lean forms (compile-time sigmoid count).  The sum-of-sigmoids kernels are bound by the special-function
// unit (16 results / clk / SM), not by HBM: one element of the n = 10 forward issued ~105 MUFU ops.  Two rules bring
// that to ~65: (1) softmax numerators are kept in registers instead of being recomputed per pass, (2) reciprocals
// come in pairs, 1/a and 1/b from ONE rcp of the product (a, b in [1, 3] here, so a b cannot overflow).
FC_HD void fc_rcp2(float a, float b, float& ra, float& rb) {
  const float r = fc_rcp(a * b);
  ra = r * b;
  rb = r * a;
}
// E = e^-|z| of a sigmoid argument
FC_HD float fc_sig_E(float z) { return fc_exp2(-fabsf(z) * FC_LOG2E); }
// sigma(z), sigma'(z) [and 1 - sigma(z)] from E and r = 1/(1+E)
FC_HD void fc_sig_finish(float z, float E, float r, float& sig, float& dsig) {
  const float Er = E * r;
  sig = z >= 0.f ? r : Er;
  dsig = Er * r;
}
FC_HD void fc_sig_finish3(float z, float E, float r, float& sig, float& omsig, float& dsig) {
  const float Er = E * r;
  sig = z >= 0.f ? r : Er;
  omsig = z >= 0.f ? Er : r;
  dsig = Er * r;
}
// two sigmoids, one reciprocal
FC_HD void fc_sigmoid_pair(float z0, float z1, float& s0, float& d0, float& s1, float& d1) {
  const float E0 = fc_sig_E(z0), E1 = fc_sig_E(z1);
  float r0, r1;
  fc_rcp2(1.f + E0, 1.f + E1, r0, r1);
  fc_sig_finish(z0, E0, r0, s0, d0);
  fc_sig_finish(z1, E1, r1, s1, d1);
}
FC_HD void fc_sigmoid_pair3(float z0, float z1, float& s0, float& o0, float& d0, float& s1, float& o1, float& d1) {
  const float E0 = fc_sig_E(z0), E1 = fc_sig_E(z1);
  float r0, r1;
  fc_rcp2(1.f + E0, 1.f + E1, r0, r1);
  fc_sig_finish3(z0, E0, r0, s0, o0, d0);
  fc_sig_finish3(z1, E1, r1, s1, o1, d1);
}
// tanh(t) from E = e^(-2|t|) and r = 1/(1+E) (same switch to the Taylor polynomial as fc_tanh); sech^2 = 4 E r^2
FC_HD float fc_tanh_finish(float t, float E, float r) {
  const float at = fabsf(t);
  const float big = (1.f - E) * r;
  const float t2 = t * t;
  float poly = fmaf(t2, 62.f / 2835.f, -17.f / 315.f);
  poly = fmaf(t2, poly, 2.f / 15.f);
  poly = fmaf(t2, poly, -1.f / 3.f);
  poly = fmaf(t2 * at, poly, at);
  const float m = at < 0.3f ? poly : big;
  return t < 0.f ? -m : m;
}
// slope a = 0.1 + 9.9 sigma(raw_scale) and shift sh = 10 tanh(raw_shift) of one sigmoid (adaptive_sigmoids.py
// :137-140) with one reciprocal; optionally d a / d raw_scale / 9.9 = sigma' and sech^2(raw_shift)
FC_HD void sos_slope_shift(float raw_shift, float raw_scale, float& a, float& sh, float& dsa, float& sech2) {
  const float Ea = fc_sig_E(raw_scale);
  const float Et = fc_exp2(fabsf(raw_shift) * (-2.f * FC_LOG2E));
  float ra, rt;
  fc_rcp2(1.f + Ea, 1.f + Et, ra, rt);
  float sa;
  fc_sig_finish(raw_scale, Ea, ra, sa, dsa);
  a = fmaf(sa, 10.f - 0.1f, 0.1f);
  sh = fc_tanh_finish(raw_shift, Et, rt) * 10.f;
  sech2 = 4.f * Et * rt * rt;
}
// extended softplus (nonlinearities.py:519-552) value and derivative at x for offset s:
//   y = softplus(x - s) - softplus(-(x + s)),  dy/dx = sigma(x - s) + sigma(-(x + s));  4 MUFU ops
FC_HD void fc_ext_softplus(float x, float s, float& y, float& dy) {
  const float z1 = x - s, z2 = -(x + s);
  const float E1 = fc_sig_E(z1), E2 = fc_sig_E(z2);
  float r1, r2, q1, q2;
  fc_rcp2(1.f + E1, 1.f + E2, r1, r2);
  fc_rcp2(2.f + E1, 2.f + E2, q1, q2);
  float s1, s2, unused;
  fc_sig_finish(z1, E1, r1, s1, unused);
  fc_sig_finish(z2, E2, r2, s2, unused);
  const float l1 = fc_log1p_unit_r(E1, q1), l2 = fc_log1p_unit_r(E2, q2);
  y = (fmaxf(z1, 0.f) + l1) - (fmaxf(z2, 0.f) + l2);
  dy = s1 + s2;
}

// Forward for one element.  raw -> [shift_raw(n) | log_scale_raw(n) | softmax_raw(n) | esp_raw].
// Returns y (without wrapper offset) and the per-element log-derivative.
// The Jacobian is accumulated in the LINEAR domain,  J = sum_j w_j a_j sigma'(pre_j) + sigma(x - s) + sigma(-x - s)
// (the derivative of the extended softplus written out), and logj = log J; the reference's log-domain composition
// (logsumexp :124-130, logaddexp :116, nonlinearities.py:543-552) is the same number and is only used as the fallback
// when J underflows.
// NC > 0: compile-time sigmoid count (loops fully unrolled, parameter reads at immediate offsets); NC = 0: runtime n.
// log-domain Jacobian for a fully saturated element (J underflows in the linear domain): the reduction exactly as
// the reference composes it (logsumexp :124-130, logaddexp :116, nonlinearities.py:543-552).  Rare; libm arithmetic.
FC_HD float sos_logj_saturated(float x, const float* raw, int n) {
  const float* sm = raw + 2 * n;
  float m = -INFINITY;
  for (int j = 0; j < n; ++j) m = fmaxf(m, sm[j]);
  float se = 0.f;
  for (int j = 0; j < n; ++j) se += expf(sm[j] - m);
  const float inv_se = 1.f / se;
  float wsum = 0.f;
  for (int j = 0; j < n; ++j) wsum += expf(sm[j] - m) * inv_se + 1e-6f;
  const float inv_wsum = 1.f / wsum;
  const float s = softplus1(raw[3 * n]) + 0.1f;
  const float lj_esp = logaddexpf_(x - logaddexpf_(s, x), -softplus1(s + x));
  float acc = 0.f;
  float mx = -INFINITY;
  for (int j = 0; j < n; ++j) {
    const float w = (expf(sm[j] - m) * inv_se + 1e-6f) * inv_wsum;
    const float a = sigmoidf_(raw[n + j]) * (10.f - 0.1f) + 0.1f;
    const float pre = a * (x - tanhf(raw[j]) * 10.f);
    const float term = logf(w) + logf(a) + (pre - 2.f * softplus1(pre));
    mx = fmaxf(mx, term);
  }
  for (int j = 0; j < n; ++j) {
    const float w = (expf(sm[j] - m) * inv_se + 1e-6f) * inv_wsum;
    const float a = sigmoidf_(raw[n + j]) * (10.f - 0.1f) + 0.1f;
    const float pre = a * (x - tanhf(raw[j]) * 10.f);
    const float term = logf(w) + logf(a) + (pre - 2.f * softplus1(pre));
    acc += expf(term - mx);
  }
  return logaddexpf_(mx + logf(acc), lj_esp);  // :116
}

// softmax numerators e_j = 2^((t_j - max) log2 e) kept in registers, 1 / sum e_j and 1 / sum (softmax_j + eps)
// (adaptive_sigmoids.py:133-135)
template <int NC>
FC_HD void sos_softmax_numerators(const float* sm, float (&e)[NC], float& inv_se, float& inv_wsum) {
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < NC; ++j) m = fmaxf(m, sm[j]);
  const float ml2 = m * FC_LOG2E;
  float se = 0.f;
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    e[j] = fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2));
    se += e[j];
  }
  inv_se = fc_rcp(se);
  float wsum = 0.f;
#pragma unroll
  for (int j = 0; j < NC; ++j) wsum += fmaf(e[j], inv_se, 1e-6f);
  inv_wsum = fc_rcp(wsum);
}

template <int NC>
FC_HD void sos_eval_t(float x, const float* raw, int n_runtime, float& y, float& logj) {
  if constexpr (NC > 0) {
    // MUFU-lean path (see fc_rcp2): ~65 special-function ops for NC = 10
    float e[NC], inv_se, inv_wsum;
    sos_softmax_numerators<NC>(raw + 2 * NC, e, inv_se, inv_wsum);
    float ysum = 0.f, wtot = 0.f, jac = 0.f;
#pragma unroll
    for (int j = 0; j + 1 < NC; j += 2) {
      float a0, sh0, a1, sh1, u0, u1;
      sos_slope_shift(raw[j], raw[NC + j], a0, sh0, u0, u1);
      sos_slope_shift(raw[j + 1], raw[NC + j + 1], a1, sh1, u0, u1);
      const float w0 = fmaf(e[j], inv_se, 1e-6f) * inv_wsum, w1 = fmaf(e[j + 1], inv_se, 1e-6f) * inv_wsum;
      float sig0, d0, sig1, d1;
      fc_sigmoid_pair(a0 * (x - sh0), a1 * (x - sh1), sig0, d0, sig1, d1);
      ysum = fmaf(w0, sig0, ysum);
      wtot += w0;
      jac = fmaf(w0 * a0, d0, jac);
      ysum = fmaf(w1, sig1, ysum);
      wtot += w1;
      jac = fmaf(w1 * a1, d1, jac);
    }
    if constexpr (NC & 1) {
      constexpr int j = NC - 1;
      float a0, sh0, u0, u1, sig0, d0;
      sos_slope_shift(raw[j], raw[NC + j], a0, sh0, u0, u1);
      const float w0 = fmaf(e[j], inv_se, 1e-6f) * inv_wsum;
      fc_sigmoid_parts(a0 * (x - sh0), sig0, d0);
      ysum = fmaf(w0, sig0, ysum);
      wtot += w0;
      jac = fmaf(w0 * a0, d0, jac);
    }
    const float s = fc_softplus1(raw[3 * NC]) + 0.1f;
    float y_esp, j_esp;
    fc_ext_softplus(x, s, y_esp, j_esp);
    y = ysum * fc_rcp(wtot) + y_esp;  // :127
    const float J = jac + j_esp;
    logj = J > 1e-30f ? fc_log_deriv(J) : sos_logj_saturated(x, raw, NC);
    return;
  }
  const int n = NC ? NC : n_runtime;
  // softmax weights + eps, renormalised (adaptive_sigmoids.py:133-135); the numerators are cheap enough (one FMA +
  // one ex2) to be recomputed per pass instead of kept in a register array of runtime length
  const float* sm = raw + 2 * n;
  float m = -INFINITY;
#pragma unroll(NC ? NC : 4)
  for (int j = 0; j < n; ++j) m = fmaxf(m, sm[j]);
  const float ml2 = m * FC_LOG2E;
  float se = 0.f;
#pragma unroll(NC ? NC : 4)
  for (int j = 0; j < n; ++j) se += fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2));
  const float inv_se = fc_rcp(se);
  float wsum = 0.f;
#pragma unroll(NC ? NC : 4)
  for (int j = 0; j < n; ++j) wsum += fmaf(fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2)), inv_se, 1e-6f);
  const float inv_wsum = fc_rcp(wsum);

  float ysum = 0.f, wtot = 0.f, jac = 0.f;
#pragma unroll(NC ? NC : 2)
  for (int j = 0; j < n; ++j) {  // several sigmoids in flight: the chain ex2 -> rcp -> ... of one is ~100 cycles long
    const float w = fmaf(fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2)), inv_se, 1e-6f) * inv_wsum;
    float sa, dsa;
    fc_sigmoid_parts(raw[n + j], sa, dsa);
    const float a = fmaf(sa, 10.f - 0.1f, 0.1f);  // :137-138
    const float sh = fc_tanh(raw[j]) * 10.f;      // :140
    const float pre = a * (x - sh);
    float sig, dsig;
    fc_sigmoid_parts(pre, sig, dsig);
    ysum = fmaf(w, sig, ysum);
    wtot += w;
    jac = fmaf(w * a, dsig, jac);
  }
  const float y_sig = ysum * fc_rcp(wtot);  // :127
  // extended softplus (nonlinearities.py:519-520, 543-552)
  const float s = fc_softplus1(raw[3 * n]) + 0.1f;
  const float y_esp = fc_softplus1(x - s) - fc_softplus1(-(x + s));
  float s1, s2, unused;
  fc_sigmoid_parts(x - s, s1, unused);
  fc_sigmoid_parts(-(x + s), s2, unused);
  y = y_sig + y_esp;
  const float J = jac + (s1 + s2);
  if (J > 1e-30f) {
    logj = fc_log_deriv(J);
    return;
  }
  logj = sos_logj_saturated(x, raw, n);  // everything is saturated
}

FC_HD void sos_eval(float x, const float* raw, int n, float& y, float& logj) { sos_eval_t<0>(x, raw, n, y, logj); }

// sigmoid(x), 1 - sigmoid(x) and sigmoid'(x) without cancellation for saturated arguments.
FC_HD void sigmoid_parts(float x, float& sig, float& omsig, float& dsig) {
  const float E = expf(-fabsf(x));
  const float r = 1.f / (1.f + E);
  const float big = r, small = E * r;
  sig = x >= 0.f ? big : small;
  omsig = x >= 0.f ? small : big;
  dsig = E * r * r;
}

// 1 - tanh(x)^2 = 4 e^{-2|x|} / (1 + e^{-2|x|})^2
FC_HD float sech2f_(float x) {
  const float E = expf(-2.f * fabsf(x));
  const float r = 1.f / (1.f + E);
  return 4.f * E * r * r;
}

// Backward for one element: upstream gy (on y) and gl (on the per-element log-derivative).
// Linear-domain derivation: J = J_sig + J_esp, logj = log J with
//   J_sig = sum_j w_j a_j sig'_j   (the reference's logsumexp, adaptive_sigmoids.py:124-130, exponentiated)
//   y_sig = sum_j w_j sig_j / sum_j w_j.
// sigma(z), 1 - sigma(z), sigma'(z) on SFU arithmetic (see fc_sigmoid_parts); 1 - tanh^2 the same way
FC_HD void fc_sigmoid_parts3(float z, float& sig, float& omsig, float& dsig) {
  const float E = fc_exp2(-fabsf(z) * FC_LOG2E);
  const float r = fc_rcp(1.f + E);
  const float Er = E * r;
  sig = z >= 0.f ? r : Er;
  omsig = z >= 0.f ? Er : r;
  dsig = Er * r;
}
FC_HD float fc_sech2(float t) {
  const float E = fc_exp2(fabsf(t) * (-2.f * FC_LOG2E));
  const float r = fc_rcp(1.f + E);
  return 4.f * E * r * r;
}

// extended-softplus pieces of the backward: j = dy/dx, dj/dx, dy/ds, dj/ds at x, and softplus'(raw offset)
FC_HD void sos_backward_esp(float x, float er, float& j_esp, float& dj_dx, float& dy_ds, float& dj_ds,
                            float& dsoftplus) {
  const float Ee = fc_sig_E(er);
  float re, qe;
  fc_rcp2(1.f + Ee, 2.f + Ee, re, qe);
  const float s = (fmaxf(er, 0.f) + fc_log1p_unit_r(Ee, qe)) + 0.1f;
  float unused;
  fc_sig_finish(er, Ee, re, dsoftplus, unused);  // softplus' (1 above the threshold to fp32 precision)
  float sp, omsp, dsp, sn, omsn, dsn;
  fc_sigmoid_pair3(x - s, -(x + s), sp, omsp, dsp, sn, omsn, dsn);
  j_esp = sp + sn;
  dj_dx = dsp - dsn;
  dy_ds = -sp + sn;
  dj_ds = -dsp - dsn;
}

// kInverse: the adjoint of the numerical inverse (fc_sos_inverse_backward).  x is then the inverse's output, z = f(x),
// gy and gl are the upstream gradients of x and of the inverse's log-derivative -log J(x).  With J_x = d log J / dx,
//   dL/dz = (gy - gl J_x) / J,
// and since dx/dtheta = -(df/dtheta) / J, the raw-parameter gradient is the forward adjoint at x with upstream
// (gy, gl) := (-dL/dz, -gl).  Pass 1 (the totals) does not depend on the upstream gradients, so the swap happens
// between the two passes; gx receives dL/dz.
template <int NC, bool kInverse = false>
FC_HD void sos_backward_elem_t(float x, const float* raw, int n_runtime, float gy, float gl, float& gx, float* graw) {
  if constexpr (NC > 0 && (NC % 2 == 0)) {
    // MUFU-lean path: two passes instead of three (the softmax dot product sum_j p_j dL/dw_j is linear in the
    // pass-1 totals: dot = [gy (S1 - ysum P) + gJ S2] / wsum with S1 = sum p_j sig_j, S2 = sum p_j a_j sig'_j,
    // P = sum p_j), softmax numerators in registers, paired reciprocals: ~110 MUFU ops for NC = 10 instead of ~240.
    float e[NC], inv_se, inv_wsum_unused;
    sos_softmax_numerators<NC>(raw + 2 * NC, e, inv_se, inv_wsum_unused);
    const float inv_wsum = fc_rcp(1.f + 1e-6f * (float)NC);  // sum_j (softmax_j + eps)
    float ysum = 0.f, jac = 0.f, djac_dx = 0.f, S1 = 0.f, S2 = 0.f, P = 0.f;
#pragma unroll
    for (int j = 0; j < NC; j += 2) {
      float a0, sh0, a1, sh1, u0, u1;
      sos_slope_shift(raw[j], raw[NC + j], a0, sh0, u0, u1);
      sos_slope_shift(raw[j + 1], raw[NC + j + 1], a1, sh1, u0, u1);
      float sig0, om0, ds0, sig1, om1, ds1;
      fc_sigmoid_pair3(a0 * (x - sh0), a1 * (x - sh1), sig0, om0, ds0, sig1, om1, ds1);
      const float p0 = e[j] * inv_se, p1 = e[j + 1] * inv_se;
      const float w0 = (p0 + 1e-6f) * inv_wsum, w1 = (p1 + 1e-6f) * inv_wsum;
      ysum += w0 * sig0;
      jac += w0 * a0 * ds0;
      djac_dx += w0 * a0 * a0 * ds0 * (om0 - sig0);
      S1 = fmaf(p0, sig0, S1);
      S2 = fmaf(p0 * a0, ds0, S2);
      P += p0;
      ysum += w1 * sig1;
      jac += w1 * a1 * ds1;
      djac_dx += w1 * a1 * a1 * ds1 * (om1 - sig1);
      S1 = fmaf(p1, sig1, S1);
      S2 = fmaf(p1 * a1, ds1, S2);
      P += p1;
    }
    float j_esp, dj_esp_dx, dy_esp_ds, dj_esp_ds, ds_der;
    sos_backward_esp(x, raw[3 * NC], j_esp, dj_esp_dx, dy_esp_ds, dj_esp_ds, ds_der);
    const float J = fmaxf(jac + j_esp, 1e-37f);
    float gJ = gl * fc_rcp(J);
    if constexpr (kInverse) {  // see the comment above sos_backward_elem_t
      gx = (gy - gJ * (djac_dx + dj_esp_dx)) * fc_rcp(J);
      gy = -gx;
      gJ = -gJ;
    } else {
      gx = gy * (jac + j_esp) + gJ * (djac_dx + dj_esp_dx);
    }
    graw[3 * NC] = (gy * dy_esp_ds + gJ * dj_esp_ds) * ds_der;
    const float dot = (gy * (S1 - ysum * P) + gJ * S2) * inv_wsum;
#pragma unroll
    for (int j = 0; j < NC; j += 2) {
      float a0, sh0, dl0, sc0, a1, sh1, dl1, sc1;
      sos_slope_shift(raw[j], raw[NC + j], a0, sh0, dl0, sc0);
      sos_slope_shift(raw[j + 1], raw[NC + j + 1], a1, sh1, dl1, sc1);
      float sig0, om0, ds0, sig1, om1, ds1;
      fc_sigmoid_pair3(a0 * (x - sh0), a1 * (x - sh1), sig0, om0, ds0, sig1, om1, ds1);
      const float p0 = e[j] * inv_se, p1 = e[j + 1] * inv_se;
      const float w0 = (p0 + 1e-6f) * inv_wsum, w1 = (p1 + 1e-6f) * inv_wsum;
      const float gw0 = gy * (sig0 - ysum) + gJ * a0 * ds0, gw1 = gy * (sig1 - ysum) + gJ * a1 * ds1;
      // pre = a (x - sh):  d/d pre of [gy w sig + gJ w a ds] = gy w ds + gJ w a dds,  dds = ds (1 - 2 sig)
      const float gpre0 = gy * w0 * ds0 + gJ * w0 * a0 * (ds0 * (om0 - sig0));
      const float gpre1 = gy * w1 * ds1 + gJ * w1 * a1 * (ds1 * (om1 - sig1));
      const float ga0 = gpre0 * (x - sh0) + gJ * w0 * ds0, ga1 = gpre1 * (x - sh1) + gJ * w1 * ds1;
      // (graw may alias raw: every read of the slots of this pair is done, and the softmax block was read in pass 1)
      graw[2 * NC + j] = p0 * (gw0 * inv_wsum - dot);
      graw[2 * NC + j + 1] = p1 * (gw1 * inv_wsum - dot);
      graw[NC + j] = ga0 * 9.9f * dl0;
      graw[NC + j + 1] = ga1 * 9.9f * dl1;
      graw[j] = -gpre0 * a0 * 10.f * sc0;
      graw[j + 1] = -gpre1 * a1 * 10.f * sc1;
    }
    return;
  }
  const int n = NC ? NC : n_runtime;
  const float* sm = raw + 2 * n;
  float m = -INFINITY;
#pragma unroll(NC ? NC : 4)
  for (int j = 0; j < n; ++j) m = fmaxf(m, sm[j]);
  float se = 0.f;
  const float ml2 = m * FC_LOG2E;
#pragma unroll(NC ? NC : 4)
  for (int j = 0; j < n; ++j) se += fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2));
  const float inv_se = fc_rcp(se);
  const float wsum = 1.f + 1e-6f * (float)n;  // sum_j (softmax_j + eps)
  const float inv_wsum = fc_rcp(wsum);

  // pass 1: totals
  float ysum = 0.f, jac = 0.f, djac_dx = 0.f;
#pragma unroll(NC ? NC : 2)
  for (int j = 0; j < n; ++j) {
    const float w = fmaf(fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2)), inv_se, 1e-6f) * inv_wsum;
    float lsg0, omlsg0, dlsg0;
    fc_sigmoid_parts3(raw[n + j], lsg0, omlsg0, dlsg0);
    const float a = fmaf(lsg0, 9.9f, 0.1f);
    const float sh = fc_tanh(raw[j]) * 10.f;
    float sig, omsig, ds;
    fc_sigmoid_parts3(a * (x - sh), sig, omsig, ds);
    ysum += w * sig;
    jac += w * a * ds;
    djac_dx += w * a * a * ds * (omsig - sig);
  }
  // extended softplus pieces
  const float er = raw[3 * n];
  const float s = fc_softplus1(er) + 0.1f;
  float ds_der, ds_om, ds_d;
  fc_sigmoid_parts3(er, ds_der, ds_om, ds_d);  // softplus' (1 above the threshold to fp32 precision)
  float sp, omsp, dsp, sn, omsn, dsn;
  fc_sigmoid_parts3(x - s, sp, omsp, dsp);       // d softplus(x-s)/dx and its derivative
  fc_sigmoid_parts3(-(x + s), sn, omsn, dsn);    // d (-softplus(-(x+s)))/dx
  const float j_esp = sp + sn;
  const float dj_esp_dx = dsp - dsn;
  const float dy_esp_ds = -sp + sn;
  const float dj_esp_ds = -dsp - dsn;
  const float J = fmaxf(jac + j_esp, 1e-37f);  // total derivative
  float gJ = gl * fc_rcp(J);
  if constexpr (kInverse) {
    gx = (gy - gJ * (djac_dx + dj_esp_dx)) * fc_rcp(J);
    gy = -gx;
    gJ = -gJ;
  } else {
    gx = gy * (jac + j_esp) + gJ * (djac_dx + dj_esp_dx);
  }
  graw[3 * n] = (gy * dy_esp_ds + gJ * dj_esp_ds) * ds_der;

  // pass 2: per-sigmoid parameter gradients
  // softmax path: w_j = (p_j + eps)/wsum ; dL/dw_j = gy * (sig_j - ysum) + gJ * a_j ds_j
  float dot = 0.f;  // sum_j p_j * dL/dp_j
#pragma unroll(NC ? NC : 2)
  for (int j = 0; j < n; ++j) {
    const float pj = fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2)) * inv_se;
    float lsg0, omlsg0, dlsg0;
    fc_sigmoid_parts3(raw[n + j], lsg0, omlsg0, dlsg0);
    const float a = fmaf(lsg0, 9.9f, 0.1f);
    float sig, omsig, ds;
    fc_sigmoid_parts3(a * (x - fc_tanh(raw[j]) * 10.f), sig, omsig, ds);
    const float gw = gy * (sig - ysum) + gJ * a * ds;
    dot += pj * gw * inv_wsum;
  }
#pragma unroll(NC ? NC : 2)
  for (int j = 0; j < n; ++j) {
    const float pj = fc_exp2(fmaf(sm[j], FC_LOG2E, -ml2)) * inv_se;
    const float w = (pj + 1e-6f) * inv_wsum;
    float lsg, omlsg, dlsg;
    fc_sigmoid_parts3(raw[n + j], lsg, omlsg, dlsg);
    const float a = fmaf(lsg, 9.9f, 0.1f);
    const float th = fc_tanh(raw[j]);
    const float sh = th * 10.f;
    float sig, omsig, ds;
    fc_sigmoid_parts3(a * (x - sh), sig, omsig, ds);
    const float dds = ds * (omsig - sig);
    const float gw = gy * (sig - ysum) + gJ * a * ds;
    // pre = a (x - sh):  d/d pre of [gy w sig + gJ w a ds] = gy w ds + gJ w a dds
    const float gpre = gy * w * ds + gJ * w * a * dds;
    const float ga = gpre * (x - sh) + gJ * w * ds;
    const float gsh = -gpre * a;
    // (graw may alias raw: all reads of slot j / n+j / 2n+j of this iteration are done)
    graw[2 * n + j] = pj * (gw * inv_wsum - dot);
    graw[n + j] = ga * 9.9f * dlsg;
    graw[j] = gsh * 10.f * fc_sech2(raw[j]);
  }
}

FC_HD void sos_backward_elem(float x, const float* raw, int n, float gy, float gl, float& gx, float* graw) {
  sos_backward_elem_t<0>(x, raw, n, gy, gl, gx, graw);
}

// x-independent part of the transform, kept in registers across the evaluations of the numerical inverse:
// mixture weights w_j and the reciprocal of their total, slopes a_j, shifts sh_j and the softplus offset s.
// Same arithmetic, in the same order, as sos_eval_t, so forward and inverse see the same function.
template <int NC>
struct SosConsts {
  float w[NC], a[NC], sh[NC];
  float s, inv_wtot;
};

template <int NC>
FC_HD void sos_precompute(const float* raw, SosConsts<NC>& k) {
  float e[NC], inv_se, inv_wsum;
  sos_softmax_numerators<NC>(raw + 2 * NC, e, inv_se, inv_wsum);
  float wtot = 0.f;
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    k.w[j] = fmaf(e[j], inv_se, 1e-6f) * inv_wsum;
    wtot += k.w[j];
    float u0, u1;
    sos_slope_shift(raw[j], raw[NC + j], k.a[j], k.sh[j], u0, u1);
  }
  k.inv_wtot = fc_rcp(wtot);
  k.s = fc_softplus1(raw[3 * NC]) + 0.1f;
}

// value and (linear-domain) derivative from the precomputed constants: ~1.5 MUFU ops per sigmoid
template <int NC>
FC_HD void sos_eval_pre(float x, const SosConsts<NC>& k, float& y, float& J) {
  float ysum = 0.f, jac = 0.f;
#pragma unroll
  for (int j = 0; j + 1 < NC; j += 2) {
    float sig0, d0, sig1, d1;
    fc_sigmoid_pair(k.a[j] * (x - k.sh[j]), k.a[j + 1] * (x - k.sh[j + 1]), sig0, d0, sig1, d1);
    ysum = fmaf(k.w[j], sig0, ysum);
    jac = fmaf(k.w[j] * k.a[j], d0, jac);
    ysum = fmaf(k.w[j + 1], sig1, ysum);
    jac = fmaf(k.w[j + 1] * k.a[j + 1], d1, jac);
  }
  if constexpr (NC & 1) {
    constexpr int j = NC - 1;
    float sig0, d0;
    fc_sigmoid_parts(k.a[j] * (x - k.sh[j]), sig0, d0);
    ysum = fmaf(k.w[j], sig0, ysum);
    jac = fmaf(k.w[j] * k.a[j], d0, jac);
  }
  float y_esp, j_esp;
  fc_ext_softplus(x, k.s, y_esp, j_esp);
  y = ysum * k.inv_wtot + y_esp;
  J = jac + j_esp;
}

// Numerical inverse for one element: find x with sos(x) = z.
// The reference grows a batch-global bracket [-lim, lim] until it holds every root (no_analytic_inv/base.py
// :48-60), halves it `iters` times (:67-79) and polishes with two damped Newton steps (:23-33): ~55 full-batch
// forward passes.  Here each element keeps its own bracket and runs a safeguarded Newton iteration (a Newton step
// when it lands inside the bracket and at least halves the previous step, a bisection step otherwise), which reaches
// the same fp32 root in 4-8 evaluations; `iters` caps the iteration count, and the reference's two damped Newton
// steps close the solve.  Eval(x, y, J) returns the value and the derivative.
template <class Eval>
FC_HD float sos_solve(float z, int iters, float lim, const Eval& eval) {
  float hi = lim, lo = -lim, y, J;
  for (int g = 0; g < 64; ++g) {
    eval(hi, y, J);
    if (!(z > y)) break;
    hi *= 1.5f;
  }
  hi += 1.f;
  for (int g = 0; g < 64; ++g) {
    eval(lo, y, J);
    if (!(z < y)) break;
    lo *= 1.5f;
  }
  lo -= 1.f;
  // the transform is x + O(1) in its linear tails: z itself is a good first iterate
  float x = fminf(fmaxf(z, lo), hi);
  float dxold = hi - lo, dx = dxold;
  const float ftol = 2.4e-7f * fmaxf(1.f, fabsf(z));
  eval(x, y, J);
  float f = y - z;
  for (int i = 0; i < iters; ++i) {
    if (f < 0.f) lo = x; else hi = x;
    const bool inside = ((x - hi) * J - f) * ((x - lo) * J - f) < 0.f;
    const bool shrinking = fabsf(2.f * f) <= fabsf(dxold * J);
    dxold = dx;
    float xn;
    if (inside && shrinking) {
      dx = f * fc_rcp(J);
      xn = x - dx;
    } else {
      dx = 0.5f * (hi - lo);
      xn = lo + dx;
    }
    if (xn == x || !(hi > lo)) break;  // fp32 resolution reached
    const bool last = fabsf(xn - x) <= 1.2e-7f * fabsf(x);  // a sub-ulp step: the polish below finishes it
    x = xn;
    if (last) break;
    eval(x, y, J);
    f = y - z;
    if (fabsf(f) <= ftol) break;  // residual at the rounding noise of y: the polish below finishes
  }
  for (int i = 0; i < 2; ++i) {  // base.py:30-33
    eval(x, y, J);
    x = x - (y - z) / (J + 1e-7f);
  }
  return x;
}

template <int NC>
FC_HD void sos_invert_t(float z, const float* raw, int n, int iters, float lim, float& x, float& logj) {
  if constexpr (NC > 0) {
    SosConsts<NC> k;
    sos_precompute<NC>(raw, k);
    x = sos_solve(z, iters, lim, [&](float xx, float& y, float& J) { sos_eval_pre<NC>(xx, k, y, J); });
  } else {
    x = sos_solve(z, iters, lim, [&](float xx, float& y, float& J) {
      float lj;
      sos_eval_t<0>(xx, raw, n, y, lj);
      J = expf(lj);
    });
  }
  float y;
  sos_eval_t<NC>(x, raw, n, y, logj);
}

FC_HD void sos_invert(float z, const float* raw, int n, int iters, float lim, float& x, float& logj) {
  sos_invert_t<0>(z, raw, n, iters, lim, x, logj);
}

// ------------------------------------------------------------------------------------------------
// piecewise-quadratic spline (flowcon/transforms/splines/quadratic.py:11-159): a piecewise-linear pdf over K bins
// (K widths, K+1 knot heights) integrated to a piecewise-quadratic cdf.  Per-feature parameters: K raw widths, then
// K+1 raw heights (no tails) or K-1 (linear tails: the two boundary heights are derived, :87-101).
// ------------------------------------------------------------------------------------------------
struct QuadSplineParams {
  int K, tails, inverse;
  float left, right, bottom, top, inv_w, inv_h;
  float min_w, min_h, wh_scale;
};

#define FC_QK(KC) ((KC) ? (KC) : FC_MAX_BINS_GENERIC)

// normalised bin widths w[K], un-normalised knot heights E[K+1], their area, normalised heights H[K+1]; sm[] keeps the
// softmax for the backward; for linear tails cst = boundary constant and den its denominator
template <int KC>
struct QuadKnots {
  float sm[FC_QK(KC)], w[FC_QK(KC)], E[FC_QK(KC) + 1], H[FC_QK(KC) + 1];
  float area, cst, den;
};

template <int KC>
FC_HD void quad_prepare(const QuadSplineParams& c, const float* u, QuadKnots<KC>& q) {
  const int K = KC ? KC : c.K;
  const float s = c.wh_scale;  // coupling.py:409-411: raw widths and heights divided by sqrt(hidden)
  float m = -INFINITY;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) m = fmaxf(m, u[j]);
  const float sl2 = s * FC_LOG2E, ml2 = m * sl2;
  float se = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) {
    q.sm[j] = fc_exp2(fmaf(u[j], sl2, -ml2));
    se += q.sm[j];
  }
  const float inv = fc_rcp(se), coef = 1.f - c.min_w * (float)K;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) {
    q.sm[j] *= inv;
    q.w[j] = fmaf(coef, q.sm[j], c.min_w);  // quadratic.py:81-82
  }
  const float* uh = u + K;
  if (c.tails == FC_TAILS_LINEAR) {  // K-1 raw heights -> E[1..K-1]; E[0] = E[K] = constant (:87-101)
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int j = 0; j < K - 1; ++j) q.E[j + 1] = fc_softplus1(uh[j] * s) + 1e-3f;  // :84
    float num = 0.25f * q.w[0] * q.E[1] + 0.25f * q.w[K - 1] * q.E[K - 1];
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int i = 0; i + 2 < K; ++i) num = fmaf(0.5f * (q.E[i + 1] + q.E[i + 2]), q.w[i + 1], num);
    q.den = 1.f - 0.25f * q.w[0] - 0.25f * q.w[K - 1];
    q.cst = fc_div(num, q.den);
    q.E[0] = q.cst;
    q.E[K] = q.cst;
  } else {
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int j = 0; j <= K; ++j) q.E[j] = fc_softplus1(uh[j] * s) + 1e-3f;
    q.cst = 0.f;
    q.den = 1.f;
  }
  float area = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) area = fmaf(0.5f * (q.E[i] + q.E[i + 1]), q.w[i], area);  // :103-106
  q.area = area;
  const float ia = fc_rcp(area) * (1.f - c.min_h);
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j <= K; ++j) q.H[j] = fmaf(q.E[j], ia, c.min_h);  // :107-108
}

// the bin of a normalised position: by location (forward) or by left-cdf (inverse); both knot vectors have their last
// knot forced to 1 and bumped by 1e-6 for the comparison (:110-123, torchutils.py:147-149).  Returns the bin's left
// location, width, left cdf and the two knot heights.
template <int KC>
FC_HD void quad_locate(int K, const QuadKnots<KC>& q, float pos, bool by_cdf, int& idx, float& loc, float& bw,
                       float& lcdf, float& hl, float& hr) {
  // One pass, "last true wins": bin m is taken when pos >= its left knot (bin 0 always).  The knots are running sums of
  // positive terms, hence monotone, so this is the count of knots <= pos that searchsorted returns; a position beyond the
  // bumped last knot (1 + 1e-6) lands in bin K - 1 either way.  The selects depend on a comparison of values, not of the
  // loop index, so the knot arrays stay in registers.
  idx = 0;
  loc = 0.f;
  lcdf = 0.f;
  bw = q.w[0];
  hl = q.H[0];
  hr = q.H[1];
  float rl = 0.f, rc = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int m = 0; m < K; ++m) {
    if (m > 0) {
      const bool ge = pos >= (by_cdf ? rc : rl);
      idx = ge ? m : idx;
      loc = ge ? rl : loc;
      lcdf = ge ? rc : lcdf;
      bw = ge ? q.w[m] : bw;
      hl = ge ? q.H[m] : hl;
      hr = ge ? q.H[m + 1] : hr;
    }
    rl += q.w[m];
    rc = fmaf(0.5f * (q.H[m] + q.H[m + 1]), q.w[m], rc);
  }
}

FC_HD bool quad_domain(const QuadSplineParams& c, float x, float& xs, unsigned& status) {
  const float lo = c.inverse ? c.bottom : c.left;
  const float hi = c.inverse ? c.top : c.right;
  if (c.tails == FC_TAILS_LINEAR) {
    const bool inside = (x >= lo) && (x <= hi);  // quadratic.py:22
    xs = inside ? x : lo;
    return inside;
  }
  xs = x;
  if (!(x >= lo && x <= hi)) {  // :67-68 raises InputOutsideDomain
    status |= FC_STATUS_INPUT_OUTSIDE_DOMAIN;
    xs = fminf(fmaxf(x, lo), hi);
    if (!(xs == xs)) xs = lo;
  }
  return true;
}

template <int KC>
FC_HD void quadspline_eval(const QuadSplineParams& c, float x, const float* u, float& y, float& lad, unsigned& status) {
  const int K = KC ? KC : c.K;
  float xs;
  const bool inside = quad_domain(c, x, xs, status);
  QuadKnots<KC> q;
  quad_prepare<KC>(c, u, q);
  int idx;
  float loc, bw, lcdf, hl, hr, ys, ls;
  if (!c.inverse) {
    const float xn = (xs - c.left) * c.inv_w;
    quad_locate<KC>(K, q, xn, false, idx, loc, bw, lcdf, hl, hr);
    const float alpha = fc_div(xn - loc, bw);                                  // :144
    const float a = 0.5f * (hr - hl) * bw, b = hl * bw;                        // :130-132
    float o = fmaf(fmaf(a, alpha, b), alpha, lcdf);                            // :145
    o = fminf(fmaxf(o, 0.f), 1.f);
    ls = fc_log_deriv(fmaf(alpha, hr - hl, hl));                               // :147-149
    ys = o * (c.top - c.bottom) + c.bottom;
  } else {
    const float yn = (xs - c.bottom) * c.inv_h;
    quad_locate<KC>(K, q, yn, true, idx, loc, bw, lcdf, hl, hr);
    const float a = 0.5f * (hr - hl) * bw, b = hl * bw, r = yn - lcdf;
    // root of a alpha^2 + b alpha - r = 0 (:134-136) in the cancellation-free form 2 r / (b + sqrt(b^2 + 4 a r)):
    // identical to (-b + sqrt(b^2 - 4 a c_)) / (2 a), and finite when the two knot heights coincide (a = 0)
    const float disc = fmaxf(fmaf(4.f * a, r, b * b), 0.f);
    const float alpha = fc_div(2.f * r, b + fc_sqrt(disc));
    float o = fmaf(alpha, bw, loc);                                            // :137
    o = fminf(fmaxf(o, 0.f), 1.f);
    ls = -fc_log_deriv(fmaf(alpha, hr - hl, hl));                              // :139-141
    ys = o * (c.right - c.left) + c.left;
  }
  y = inside ? ys : x;
  lad = inside ? ls : 0.f;
}

// Backward of quadspline_eval for one element: closed-form reverse pass through bin quantities -> normalised heights ->
// area normalisation (-> boundary constant with linear tails) -> softplus / softmax.  The inverse direction by implicit
// differentiation through the forward adjoint at out = f^-1(v) (as rqs_backward_elem).  gu may alias u.
template <int KC>
FC_HD void quadspline_backward_elem(const QuadSplineParams& c, float x, const float* u, float gy, float gl, float& gx,
                                    float* gu) {
  const int K = KC ? KC : c.K;
  const int NH = c.tails == FC_TAILS_LINEAR ? K - 1 : K + 1;
  float xs;
  unsigned status = 0;
  const bool inside = quad_domain(c, x, xs, status);
  if (!inside) {
    gx = gy;
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int j = 0; j < 2 * K + 1; ++j)
      if (j < K + NH) gu[j] = 0.f;
    return;
  }
  QuadKnots<KC> q;
  quad_prepare<KC>(c, u, q);
  float pos = xs;
  if (c.inverse) {
    float out, unused;
    quadspline_eval<KC>(c, x, u, out, unused, status);
    pos = out;
  }
  const float S = c.top - c.bottom;
  const float xn = (pos - c.left) * c.inv_w;
  int idx;
  float loc, bw, lcdf, hl, hr;
  quad_locate<KC>(K, q, xn, false, idx, loc, bw, lcdf, hl, hr);
  const float alpha = fc_div(xn - loc, bw);
  const float d = hr - hl, Dv = fmaf(alpha, d, hl), inv_bw = fc_rcp(bw), inv_D = fc_rcp(Dv);
  float gyS, glf;
  if (c.inverse) {
    // dL/dv = (g_out - gl * d ladf/d out) / f'(out),  f' = S D inv_w,  d ladf / d out = d / (D bw) inv_w
    const float g = fc_div(gy - gl * d * inv_D * inv_bw * c.inv_w, S * Dv * c.inv_w);
    gx = g;
    gyS = -g * S;
    glf = -gl;
  } else {
    gx = (gy * S * Dv + gl * d * inv_D * inv_bw) * c.inv_w;
    gyS = gy * S;
    glf = gl;
  }
  const float g_alpha = gyS * bw * Dv + glf * d * inv_D;
  const float g_bw = gyS * (0.5f * d * alpha * alpha + hl * alpha) - g_alpha * alpha * inv_bw;
  const float g_hr = gyS * 0.5f * bw * alpha * alpha + glf * alpha * inv_D;
  const float g_hl = gyS * (bw * alpha - 0.5f * bw * alpha * alpha) + glf * (1.f - alpha) * inv_D;
  const float g_loc = -g_alpha * inv_bw;
  float gw[FC_QK(KC)], gH[FC_QK(KC) + 1];
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j <= K; ++j) gH[j] = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) {
    const bool below = i < idx;
    gw[i] = below ? g_loc + gyS * 0.5f * (q.H[i] + q.H[i + 1]) : (i == idx ? g_bw : 0.f);
    const float t = below ? gyS * 0.5f * q.w[i] : 0.f;
    gH[i] += t + (i == idx ? g_hl : 0.f);
    gH[i + 1] += t + (i == idx ? g_hr : 0.f);
  }
  // H = min_h + (1 - min_h) E / area
  const float ia = fc_rcp(q.area), k1 = (1.f - c.min_h) * ia;
  float dotE = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j <= K; ++j) dotE = fmaf(gH[j], q.E[j], dotE);
  const float g_area = -k1 * ia * dotE;
  float gE[FC_QK(KC) + 1];
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j <= K; ++j) {
    const float wl = j > 0 ? q.w[j - 1] : 0.f, wr = j < K ? q.w[j] : 0.f;
    gE[j] = fmaf(k1, gH[j], g_area * 0.5f * (wl + wr));
  }
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) gw[i] = fmaf(g_area * 0.5f, q.E[i] + q.E[i + 1], gw[i]);
  const float s = c.wh_scale;
  const float* uh = u + K;
  float gh[FC_QK(KC) + 1];  // raw-height gradients (NH of them)
  if (c.tails == FC_TAILS_LINEAR) {
    const float gC = gE[0] + gE[K];
    const float g_num = fc_div(gC, q.den), g_den = -g_num * q.cst;
    // e_j = E[j+1], j = 0..K-2
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int j = 0; j < K - 1; ++j) {
      float dn = 0.f;
      if (j >= 1) dn += 0.5f * q.w[j];
      if (j + 3 <= K) dn += 0.5f * q.w[j + 1];
      if (j == 0) dn += 0.25f * q.w[0];
      if (j == K - 2) dn += 0.25f * q.w[K - 1];
      float sg, unused;
      fc_sigmoid_parts(uh[j] * s, sg, unused);
      gh[j] = (gE[j + 1] + g_num * dn) * sg * s;
    }
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int mI = 0; mI < K; ++mI) {
      float dn;
      if (mI == 0) dn = 0.25f * q.E[1];
      else if (mI == K - 1) dn = 0.25f * q.E[K - 1];
      else dn = 0.5f * (q.E[mI] + q.E[mI + 1]);
      const float dd = (mI == 0 || mI == K - 1) ? -0.25f : 0.f;
      gw[mI] += g_num * dn + g_den * dd;
    }
  } else {
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int j = 0; j <= K; ++j) {
      float sg, unused;
      fc_sigmoid_parts(uh[j] * s, sg, unused);
      gh[j] = gE[j] * sg * s;
    }
  }
  // w = min_w + (1 - min_w K) softmax(s uw)
  const float coef = 1.f - c.min_w * (float)K;
  float dot = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) dot = fmaf(q.sm[i], gw[i] * coef, dot);
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) gu[i] = s * q.sm[i] * (gw[i] * coef - dot);
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j <= K; ++j)
    if (j < NH) gu[K + j] = gh[j];
}

// ------------------------------------------------------------------------------------------------
// cubic spline (flowcon/transforms/splines/cubic.py:15-267) — element math only, host-validated against the reference's
// golden vectors (tests/test_kernel_math_host.py); the kernel wiring is the next step (DESIGN.md section 7).
// Per-feature parameters: K raw widths, K raw heights, raw left / right boundary derivative (P = 2K + 2).
// ------------------------------------------------------------------------------------------------
struct CubicSplineParams {
  int K, tails, inverse;
  float left, right, bottom, top, inv_w, inv_h;
  float min_w, min_h, wh_scale;
};

template <int KC>
struct CubicKnots {
  float smw[FC_QK(KC)], smh[FC_QK(KC)], w[FC_QK(KC)], h[FC_QK(KC)], s[FC_QK(KC)], dv[FC_QK(KC) + 1];
  float sig_l, sig_r;
};

template <int KC>
FC_HD void cubic_softmax_floor(int K, const float* u, float scale, float floor_v, float* sm, float* out) {
  float m = -INFINITY;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) m = fmaxf(m, u[j]);
  const float sl2 = scale * FC_LOG2E, ml2 = m * sl2;
  float se = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) {
    sm[j] = fc_exp2(fmaf(u[j], sl2, -ml2));
    se += sm[j];
  }
  const float inv = fc_rcp(se), coef = 1.f - floor_v * (float)K;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) {
    sm[j] *= inv;
    out[j] = fmaf(coef, sm[j], floor_v);
  }
}

// widths, heights, bin slopes and the K+1 knot derivatives (cubic.py:98-132): boundary knots sigmoid(raw) * 3 * slope,
// interior knots the monotone rule min(min(s_l, s_r), weighted mean) * (sign s_l + sign s_r) = 2 min(...) (slopes > 0)
template <int KC>
FC_HD void cubic_prepare(const CubicSplineParams& c, const float* u, CubicKnots<KC>& q) {
  const int K = KC ? KC : c.K;
  cubic_softmax_floor<KC>(K, u, c.wh_scale, c.min_w, q.smw, q.w);
  cubic_softmax_floor<KC>(K, u + K, c.wh_scale, c.min_h, q.smh, q.h);
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j < K; ++j) q.s[j] = fc_div(q.h[j], q.w[j]);
  float unused;
  fc_sigmoid_parts(u[2 * K], q.sig_l, unused);
  fc_sigmoid_parts(u[2 * K + 1], q.sig_r, unused);
  q.dv[0] = q.sig_l * 3.f * q.s[0];
  q.dv[K] = q.sig_r * 3.f * q.s[K - 1];
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 1; j < K; ++j) {
    const float m1 = fminf(q.s[j - 1], q.s[j]);
    const float m2 = fc_div(0.5f * (q.w[j] * q.s[j - 1] + q.w[j - 1] * q.s[j]), q.w[j - 1] + q.w[j]);
    q.dv[j] = 2.f * fminf(m1, m2);
  }
}

// bin of a normalised position (by cumulative width forward, cumulative height inverse; last knot forced to 1 and
// bumped for the comparison) and its quantities, gathered with masked sums (see quad_locate)
template <int KC>
FC_HD void cubic_locate(int K, const CubicKnots<KC>& q, float pos, bool by_height, int& idx, float& x_lo, float& y_lo,
                        float& w, float& s, float& d0, float& d1) {
  // one pass, "last true wins" (see quad_locate)
  idx = 0;
  x_lo = 0.f;
  y_lo = 0.f;
  w = q.w[0];
  s = q.s[0];
  d0 = q.dv[0];
  d1 = q.dv[1];
  float rw = 0.f, rh = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int m = 0; m < K; ++m) {
    if (m > 0) {
      const bool ge = pos >= (by_height ? rh : rw);
      idx = ge ? m : idx;
      x_lo = ge ? rw : x_lo;
      y_lo = ge ? rh : y_lo;
      w = ge ? q.w[m] : w;
      s = ge ? q.s[m] : s;
      d0 = ge ? q.dv[m] : d0;
      d1 = ge ? q.dv[m + 1] : d1;
    }
    rw += q.w[m];
    rh += q.h[m];
  }
}

FC_HD bool cubic_domain(const CubicSplineParams& c, float x, float& xs, unsigned& status) {
  const float lo = c.inverse ? c.bottom : c.left;
  const float hi = c.inverse ? c.top : c.right;
  if (c.tails == FC_TAILS_LINEAR) {
    const bool inside = (x >= lo) && (x <= hi);  // cubic.py:30
    xs = inside ? x : lo;
    return inside;
  }
  xs = x;
  if (!(x >= lo && x <= hi)) {  // :84-85 raises InputOutsideDomain
    status |= FC_STATUS_INPUT_OUTSIDE_DOMAIN;
    xs = fminf(fmaxf(x, lo), hi);
    if (!(xs == xs)) xs = lo;
  }
  return true;
}

template <int KC>
FC_HD void cubicspline_eval(const CubicSplineParams& c, float x, const float* u, float& y, float& lad,
                            unsigned& status) {
  const int K = KC ? KC : c.K;
  float xs;
  const bool inside = cubic_domain(c, x, xs, status);
  CubicKnots<KC> q;
  cubic_prepare<KC>(c, u, q);
  int idx;
  float x_lo, y_lo, w, s, d0, d1, ys, ls;
  const float pos = c.inverse ? (xs - c.bottom) * c.inv_h : (xs - c.left) * c.inv_w;
  cubic_locate<KC>(K, q, pos, c.inverse != 0, idx, x_lo, y_lo, w, s, d0, d1);
  const float iw = fc_rcp(w);
  const float a = (d0 + d1 - 2.f * s) * iw * iw;   // cubic.py:134-137
  const float b = (3.f * s - 2.f * d0 - d1) * iw;
  if (!c.inverse) {
    const float t = pos - x_lo;
    const float o = fmaf(fmaf(fmaf(a, t, b), t, d0), t, y_lo);          // :241-247
    ls = fc_log_deriv(fmaf(fmaf(3.f * a, t, 2.f * b), t, d0));          // :249-255
    ys = o * (c.top - c.bottom) + c.bottom;
  } else {
    // The reference solves the cubic in closed form (Blinn 2007, :152-237).  The polynomial is monotone on its bin by
    // construction of the knot derivatives, so a safeguarded Newton iteration on [0, w] finds the same root, needs no
    // case analysis (one / three real roots / nearly quadratic), and has no a -> 0 singularity.
    const float r = pos - y_lo;
    float lo = 0.f, hi = w;
    float t = fminf(fmaxf(fc_div(r, s), 0.f), w);  // the chord's root as first iterate
    for (int it = 0; it < 24; ++it) {
      const float f = fmaf(fmaf(fmaf(a, t, b), t, d0), t, -r);
      const float fp = fmaf(fmaf(3.f * a, t, 2.f * b), t, d0);
      if (f > 0.f) hi = t; else lo = t;
      float tn = t - fc_div(f, fp);
      if (!(tn > lo && tn < hi)) tn = 0.5f * (lo + hi);
      if (tn == t) break;
      t = tn;
    }
    ls = -fc_log_deriv(fmaf(fmaf(3.f * a, t, 2.f * b), t, d0));         // :229-235
    ys = (t + x_lo) * (c.right - c.left) + c.left;
  }
  y = inside ? ys : x;
  lad = inside ? ls : 0.f;
}

// Backward: closed-form reverse pass (bin polynomial -> knot derivatives (min rule: the gradient follows the active
// branch) -> slopes -> floored softmaxes); inverse direction by implicit differentiation at out = f^-1(v).
template <int KC>
FC_HD void cubicspline_backward_elem(const CubicSplineParams& c, float x, const float* u, float gy, float gl, float& gx,
                                     float* gu) {
  const int K = KC ? KC : c.K;
  float xs;
  unsigned status = 0;
  const bool inside = cubic_domain(c, x, xs, status);
  if (!inside) {
    gx = gy;
#pragma unroll(KC ? 2 * KC + 2 : 4)
    for (int j = 0; j < 2 * K + 2; ++j) gu[j] = 0.f;
    return;
  }
  CubicKnots<KC> q;
  cubic_prepare<KC>(c, u, q);
  float posx = xs;
  if (c.inverse) {
    float out, unused;
    cubicspline_eval<KC>(c, x, u, out, unused, status);
    posx = out;
  }
  const float S = c.top - c.bottom;
  const float un = (posx - c.left) * c.inv_w;
  int idx;
  float x_lo, y_lo, w, s, d0, d1;
  cubic_locate<KC>(K, q, un, false, idx, x_lo, y_lo, w, s, d0, d1);
  const float iw = fc_rcp(w);
  const float a = (d0 + d1 - 2.f * s) * iw * iw, b = (3.f * s - 2.f * d0 - d1) * iw;
  const float t = un - x_lo;
  const float Dv = fmaf(fmaf(3.f * a, t, 2.f * b), t, d0), iD = fc_rcp(Dv);
  const float D2 = fmaf(6.f * a, t, 2.f * b);  // P''(t)
  float gyS, glf;
  if (c.inverse) {
    const float g = fc_div(gy - gl * D2 * iD * c.inv_w, S * Dv * c.inv_w);
    gx = g;
    gyS = -g * S;
    glf = -gl;
  } else {
    gx = (gy * S * Dv + gl * D2 * iD) * c.inv_w;
    gyS = gy * S;
    glf = gl;
  }
  const float g_t = gyS * Dv + glf * D2 * iD;
  const float g_a = gyS * t * t * t + glf * 3.f * t * t * iD;
  const float g_b = gyS * t * t + glf * 2.f * t * iD;
  const float g_c = gyS * t + glf * iD;
  // a, b, c -> d0, d1, s, w of the bin
  const float g_d0 = g_a * iw * iw - 2.f * g_b * iw + g_c;
  const float g_d1 = g_a * iw * iw - g_b * iw;
  const float g_s = -2.f * g_a * iw * iw + 3.f * g_b * iw;
  const float g_wb = -(2.f * a * g_a + b * g_b) * iw;
  float gw[FC_QK(KC)], gh[FC_QK(KC)], gs[FC_QK(KC)];
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) {
    const bool below = i < idx;
    gw[i] = (below ? -g_t : 0.f) + (i == idx ? g_wb : 0.f);  // x_lo = sum_{j<idx} w_j
    gh[i] = below ? gyS : 0.f;                               // y_lo = sum_{j<idx} h_j
    gs[i] = i == idx ? g_s : 0.f;
  }
  // knot derivatives idx and idx + 1
  float g_dl = 0.f, g_dr = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int j = 0; j <= K; ++j) {
    const float g = (j == idx ? g_d0 : 0.f) + (j == idx + 1 ? g_d1 : 0.f);
    if (j == 0) {
      g_dl = g * 3.f * q.s[0] * q.sig_l * (1.f - q.sig_l);
      gs[0] += g * 3.f * q.sig_l;
    } else if (j == K) {
      g_dr = g * 3.f * q.s[K - 1] * q.sig_r * (1.f - q.sig_r);
      gs[K - 1] += g * 3.f * q.sig_r;
    } else {
      const float sl = q.s[j - 1], sr = q.s[j], wl = q.w[j - 1], wr = q.w[j];
      const float m1 = fminf(sl, sr);
      const float N = wr * sl + wl * sr, Dn = wl + wr, iDn = fc_rcp(Dn);
      const float m2 = 0.5f * N * iDn;
      if (m1 <= m2) {  // min over the two slopes is active
        gs[j - 1] += sl <= sr ? 2.f * g : 0.f;
        gs[j] += sl <= sr ? 0.f : 2.f * g;
      } else {         // the weighted mean is active: dv = N / Dn
        const float gN = g * iDn, gDn = -g * N * iDn * iDn;
        gs[j - 1] += gN * wr;
        gs[j] += gN * wl;
        gw[j] += gN * sl + gDn;
        gw[j - 1] += gN * sr + gDn;
      }
    }
  }
  // s = h / w
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) {
    const float iwi = fc_rcp(q.w[i]);
    gh[i] += gs[i] * iwi;
    gw[i] -= gs[i] * q.s[i] * iwi;
  }
  // floored softmaxes of the scaled raw values
  const float sc = c.wh_scale, cw = 1.f - c.min_w * (float)K, ch = 1.f - c.min_h * (float)K;
  float dotw = 0.f, doth = 0.f;
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) {
    dotw = fmaf(q.smw[i], gw[i] * cw, dotw);
    doth = fmaf(q.smh[i], gh[i] * ch, doth);
  }
#pragma unroll(KC ? 2 * KC + 2 : 4)
  for (int i = 0; i < K; ++i) {
    gu[i] = sc * q.smw[i] * (gw[i] * cw - dotw);
    gu[K + i] = sc * q.smh[i] * (gh[i] * ch - doth);
  }
  gu[2 * K] = g_dl;
  gu[2 * K + 1] = g_dr;
}

}  // namespace fc
