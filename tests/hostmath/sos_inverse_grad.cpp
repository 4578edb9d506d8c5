// TEST INFRASTRUCTURE ONLY — the sum-of-sigmoids inverse adjoint of flowconductor_b200/csrc/fc_math.cuh
// (sos_backward_elem_t<NC, true>, what fc_sos_inverse_backward runs per element) compiled with g++ so that
// tests/test_sos_inverse_grad_host.py can check it against the oracle without a GPU.  Never loaded by the product package.
#include "../../flowconductor_b200/csrc/fc_math.cuh"

using namespace fc;

extern "C" {

// x is the inverse's output; gx receives the gradient of the inverse's input
void hm_sos_inverse_backward(const float* x, const float* params, const float* gy, const float* gl, float* gx, float* gp,
                             long n, int n_sigmoids) {
  const int P = 3 * n_sigmoids + 1;
  for (long i = 0; i < n; ++i)
    sos_backward_elem_t<0, true>(x[i], params + i * P, n_sigmoids, gy[i], gl[i], gx[i], gp + i * P);
}

// the compile-time n = 10 instantiation the kernels run for the default sigmoid count
void hm_sos_inverse_backward_n10(const float* x, const float* params, const float* gy, const float* gl, float* gx,
                                 float* gp, long n) {
  for (long i = 0; i < n; ++i)
    sos_backward_elem_t<10, true>(x[i], params + i * 31, 10, gy[i], gl[i], gx[i], gp + i * 31);
}
}
