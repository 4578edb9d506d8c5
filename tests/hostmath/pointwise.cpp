// TEST INFRASTRUCTURE ONLY — the element math of the squashing layers (flowconductor_b200/csrc/fc_pointwise.cuh: pw_eval,
// pw_grad, what fc_pointwise_apply / fc_pointwise_backward run per element) compiled with g++ so that
// tests/test_pointwise_host.py can check it against fp64 formulas without a GPU.  Never loaded by the product package.
#include "../../flowconductor_b200/csrc/fc_pointwise.cuh"

using namespace fc;

template <int OP, bool INV>
static void eval_n(const float* x, long n, const PwScalars& c, float* y, float* lad, int* bad) {
  for (long i = 0; i < n; ++i) {
    bool b = false;
    pw_eval<OP, INV>(x[i], c, y[i], lad[i], b);
    bad[i] = b;
  }
}

template <int OP, bool INV>
static void grad_n(const float* x, long n, const PwScalars& c, float* dy, float* dl, float* dyT, float* dlT) {
  for (long i = 0; i < n; ++i) pw_grad<OP, INV>(x[i], c, dy[i], dl[i], dyT[i], dlT[i]);
}

#define HM_PW_SWITCH(FN, ...)                                       \
  switch (op * 2 + (inverse ? 1 : 0)) {                             \
    case 0: FN<FC_POINTWISE_SIGMOID, false>(__VA_ARGS__); break;    \
    case 1: FN<FC_POINTWISE_SIGMOID, true>(__VA_ARGS__); break;     \
    case 2: FN<FC_POINTWISE_TANH, false>(__VA_ARGS__); break;       \
    case 3: FN<FC_POINTWISE_TANH, true>(__VA_ARGS__); break;        \
    case 4: FN<FC_POINTWISE_LEAKY_RELU, false>(__VA_ARGS__); break; \
    case 5: FN<FC_POINTWISE_LEAKY_RELU, true>(__VA_ARGS__); break;  \
    case 6: FN<FC_POINTWISE_EXP, false>(__VA_ARGS__); break;        \
    case 7: FN<FC_POINTWISE_EXP, true>(__VA_ARGS__); break;         \
    case 8: FN<FC_POINTWISE_CAUCHY_CDF, false>(__VA_ARGS__); break; \
    case 9: FN<FC_POINTWISE_CAUCHY_CDF, true>(__VA_ARGS__); break;  \
  }

// the scalars as fc_pointwise.cu sets them up: T and log T, the active slope (reciprocal for the inverse), log slope
static PwScalars scalars(int inverse, float T, float slope, float eps) {
  PwScalars c;
  c.T = T, c.log_T = logf(T), c.eps = eps, c.log_s = logf(slope);
  c.s = inverse ? (float)(1.0 / (double)slope) : slope;
  return c;
}

extern "C" {

void hm_pw_eval(int op, int inverse, const float* x, long n, float T, float slope, float eps, float* y, float* lad,
                int* bad) {
  const PwScalars c = scalars(inverse, T, slope, eps);
  HM_PW_SWITCH(eval_n, x, n, c, y, lad, bad)
}

void hm_pw_grad(int op, int inverse, const float* x, long n, float T, float slope, float eps, float* dy, float* dl,
                float* dyT, float* dlT) {
  const PwScalars c = scalars(inverse, T, slope, eps);
  HM_PW_SWITCH(grad_n, x, n, c, dy, dl, dyT, dlT)
}
}
