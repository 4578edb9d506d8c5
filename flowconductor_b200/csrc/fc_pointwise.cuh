// fc_pointwise.cuh — per-element arithmetic of the element-wise squashing layers (Sigmoid / Logit, Tanh, LeakyReLU, Exp,
// CauchyCDF, flowcon/transforms/nonlinearities.py), shared by csrc/fc_pointwise.cu and the g++ test shim
// tests/hostmath/pointwise.cpp (FC_HD: __host__ __device__ under nvcc, inline under g++).
//
// pw_eval:  the map of one element in either direction and its log|dy/dx| term.
// pw_grad:  the derivatives the backward needs at the same (layer-input) element: dy/dx, d(log-det)/dx and, for
//           Sigmoid, the derivatives of both with respect to the temperature.
// Deviations from the reference's literal fp32 formulas, all toward the exact value:
//   Tanh forward log-det  2 (log 2 − |x| − softplus(−2|x|)) instead of log(1 − tanh² x): finite where tanh x rounds to
//                         ±1 (|x| ≳ 9), where the reference returns −inf;
//   Tanh inverse          atanh(y) and −(log1p(y) + log1p(−y)) instead of ½ log((1+y)/(1−y)) and −log(1 − y²);
//   Sigmoid               σ(u) and softplus(±u) from e^{−|u|}; the inverse log-det from the clamped input,
//                         −log T − log y' − log1p(−y'), which is the reference's −(log T − softplus(−Tx) − softplus(Tx))
//                         at x = logit(y') / T without the round trip;
//   CauchyCDF             log(1 + x²) as 2 log|x| + log1p(x⁻²) for |x| > 1, finite where x² overflows.
#pragma once
#include "fc_math.cuh"

namespace fc {

constexpr float kPwPi = 3.14159265358979323846f;
constexpr float kPwLogPi = 1.14472988584940017414f;
constexpr float kPwLog2 = 0.69314718055994530942f;

// Everything the element math reads besides the element: the temperature T (Sigmoid), the active slope s (LeakyReLU:
// the layer's slope forward, its reciprocal inverse), log_s = log of the layer's slope (the reference's fp32
// log_negative_slope) and the clamp eps (Sigmoid inverse).
struct PwScalars {
  float T, log_T, s, log_s, eps;
};

// log(1 + x²) without overflow
FC_HD float pw_log1p_sq(float x) {
  const float ax = fabsf(x);
  if (ax > 1.f) {
    const float r = 1.f / ax;
    return 2.f * logf(ax) + log1pf(r * r);
  }
  return log1pf(ax * ax);
}

// y and the element's log-det term; `bad` is set where the reference raises InputOutsideDomain
template <int OP, bool INV>
FC_HD void pw_eval(float x, const PwScalars& c, float& y, float& lad, bool& bad) {
  if constexpr (OP == FC_POINTWISE_SIGMOID) {
    if constexpr (!INV) {
      const float u = c.T * x;
      const float e = expf(-fabsf(u));
      const float r = 1.f / (1.f + e);
      y = u >= 0.f ? r : e * r;
      lad = (c.log_T - fabsf(u)) - 2.f * log1pf(e);
    } else {
      bad |= (x < 0.f) || (x > 1.f);
      const float yc = fminf(fmaxf(x, c.eps), 1.f - c.eps);
      const float lg = logf(yc), l1 = log1pf(-yc);
      y = (lg - l1) / c.T;
      lad = (-c.log_T - lg) - l1;
    }
  } else if constexpr (OP == FC_POINTWISE_TANH) {
    if constexpr (!INV) {
      const float a = fabsf(x);
      y = tanhf(x);
      lad = 2.f * ((kPwLog2 - a) - log1pf(expf(-2.f * a)));
    } else {
      bad |= (x <= -1.f) || (x >= 1.f);
      y = atanhf(x);
      lad = -(log1pf(x) + log1pf(-x));
    }
  } else if constexpr (OP == FC_POINTWISE_LEAKY_RELU) {
    y = x > 0.f ? x : c.s * x;
    lad = x < 0.f ? (INV ? -c.log_s : c.log_s) : 0.f;
  } else if constexpr (OP == FC_POINTWISE_EXP) {
    if constexpr (!INV) {
      y = expf(x);
      lad = x;
    } else {
      bad |= x <= 0.f;
      y = logf(x);
      lad = -y;
    }
  } else {  // FC_POINTWISE_CAUCHY_CDF
    if constexpr (!INV) {
      y = atanf(x) * (1.f / kPwPi) + 0.5f;
      lad = -kPwLogPi - pw_log1p_sq(x);
    } else {
      bad |= (x < 0.f) || (x > 1.f);
      y = tanf(kPwPi * (x - 0.5f));
      lad = kPwLogPi + pw_log1p_sq(y);
    }
  }
}

// dy/dx (dy), d(log-det)/dx (dl) and, for Sigmoid, dy/dT (dyT) and d(log-det)/dT (dlT) at input x
template <int OP, bool INV>
FC_HD void pw_grad(float x, const PwScalars& c, float& dy, float& dl, float& dyT, float& dlT) {
  dyT = 0.f, dlT = 0.f;
  if constexpr (OP == FC_POINTWISE_SIGMOID) {
    if constexpr (!INV) {
      const float u = c.T * x;
      const float e = expf(-fabsf(u));
      const float r = 1.f / (1.f + e);
      const float sd = e * r * r;                          // σ(u) σ(−u)
      const float one_m_2s = u >= 0.f ? (e - 1.f) * r : (1.f - e) * r;  // 1 − 2σ(u)
      dy = c.T * sd;
      dl = c.T * one_m_2s;
      dyT = x * sd;
      dlT = 1.f / c.T + x * one_m_2s;
    } else {
      // torch.clamp passes the gradient on [eps, 1 − eps] (bounds included) and nowhere else
      const bool in = x >= c.eps && x <= 1.f - c.eps;
      const float yc = fminf(fmaxf(x, c.eps), 1.f - c.eps);
      const float q = 1.f / (yc * (1.f - yc));
      dy = in ? q / c.T : 0.f;
      dl = in ? (2.f * yc - 1.f) * q : 0.f;
      const float xo = (logf(yc) - log1pf(-yc)) / c.T;
      dyT = -xo / c.T;
      dlT = -1.f / c.T;  // T x = logit(y') does not depend on T
    }
  } else if constexpr (OP == FC_POINTWISE_TANH) {
    if constexpr (!INV) {
      const float e = expf(-2.f * fabsf(x));
      const float r = 1.f / (1.f + e);
      dy = 4.f * e * r * r;  // 1 − tanh² x
      dl = -2.f * tanhf(x);
    } else {
      const float q = 1.f / ((1.f - x) * (1.f + x));
      dy = q;
      dl = 2.f * x * q;
    }
  } else if constexpr (OP == FC_POINTWISE_LEAKY_RELU) {
    dy = x > 0.f ? 1.f : c.s;
    dl = 0.f;
  } else if constexpr (OP == FC_POINTWISE_EXP) {
    if constexpr (!INV) {
      dy = expf(x);
      dl = 1.f;
    } else {
      dy = 1.f / x;
      dl = -dy;
    }
  } else {  // FC_POINTWISE_CAUCHY_CDF
    if constexpr (!INV) {
      const float q = 1.f / (1.f + x * x);
      dy = q * (1.f / kPwPi);
      dl = -2.f * x * q;
    } else {
      const float t = tanf(kPwPi * (x - 0.5f));
      dy = kPwPi * fmaf(t, t, 1.f);
      dl = 2.f * kPwPi * t;
    }
  }
}

}  // namespace fc
