"""CPU checks of the sum-of-sigmoids inverse adjoint (sos_backward_elem_t<NC, true>, fc_sos_inverse_backward).

The element math is compiled with g++ (tests/hostmath/sos_inverse_grad.cpp, into a temporary directory) and compared
with autograd through the reference's numerical inverse (`restated.sos_inverse`: bisection, then two Newton steps with
`create_graph=True`), in fp32 and fp64, on the golden sum-of-sigmoids cases.  The C entry's argument checks run before any CUDA call, so they are tested here too."""
import ctypes
import os
import subprocess

import pytest
import torch

from flowconductor_b200 import _cabi
from oracle import restated
from tests.helpers import ROOT, assert_parity, load_golden
from tests.test_kernel_math_host import fptr, hm  # noqa: F401  (hm: the host-math library fixture, for the inverse)

SRC = os.path.join(ROOT, "tests", "hostmath", "sos_inverse_grad.cpp")


@pytest.fixture(scope="module")
def adj(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("hostmath") / "libsos_inverse_grad.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-x", "c++", SRC,
                           "-o", lib])
    return ctypes.CDLL(lib)


@pytest.fixture(scope="module")
def gold():
    return load_golden("functions")


def reference_inverse_grads(z, params, ns, gy, gl, dtype):
    """Gradients of <gy, x> + <gl, lad> through the reference's inverse, x, lad = sos_inverse(z, params)."""
    z = z.to(dtype).requires_grad_(True)
    p = params.to(dtype).requires_grad_(True)
    x, lad = restated.sos_inverse(z, p, ns)
    loss = (gy.to(dtype) * x).sum() + (gl.to(dtype) * lad).sum()
    gz, gp = torch.autograd.grad(loss, [z, p])
    return gz, gp


@pytest.mark.parametrize("name", ["sos_n10", "sos_n3_wide"])
def test_inverse_adjoint_matches_autograd_through_the_reference_inverse(hm, adj, gold, name):  # noqa: F811
    ns = int(gold[name + "/meta"][0])
    p = gold[name + "/params"].contiguous()
    z = gold[name + "/y32"].contiguous()
    n, d = z.shape
    x, lj = torch.empty_like(z), torch.empty_like(z)
    hm.hm_sos_invert(fptr(z), fptr(p), fptr(x), fptr(lj), ctypes.c_long(z.numel()), ns, 50, ctypes.c_float(120.0))
    gy = gold[name + "/gy"].contiguous()
    gl_row = gold[name + "/gl"]
    gl = gl_row[:, None].expand(n, d).contiguous()
    gz32, gp32 = reference_inverse_grads(z, p, ns, gy, gl_row, torch.float32)
    gz64, gp64 = reference_inverse_grads(z, p, ns, gy, gl_row, torch.float64)

    variants = [("generic", lambda gz, gp: adj.hm_sos_inverse_backward(
        fptr(x), fptr(p), fptr(gy), fptr(gl), fptr(gz), fptr(gp), ctypes.c_long(z.numel()), ns))]
    if ns == 10:  # the unrolled two-pass instantiation the n = 10 kernels run
        variants.append(("n10", lambda gz, gp: adj.hm_sos_inverse_backward_n10(
            fptr(x), fptr(p), fptr(gy), fptr(gl), fptr(gz), fptr(gp), ctypes.c_long(z.numel()))))
    for what, run in variants:
        gz, gp = torch.empty_like(z), torch.empty_like(p)
        run(gz, gp)
        s = max(1e-2, gz64.abs().mean().item())
        assert_parity(gz, gz32, gz64, 1e-4, s, "{} grad z ({})".format(name, what))
        s = max(1e-2, gp64.abs().mean().item())
        assert_parity(gp, gp32, gp64, 1e-4, s, "{} grad params ({})".format(name, what))


@pytest.mark.parametrize("name", ["sos_n10", "sos_n3_wide"])
def test_inverse_adjoint_without_logdet_gradient(hm, adj, gold, name):  # noqa: F811
    """gl = 0 (the kernels' reading of a NULL grad_logabsdet): grad z is gy / f'(x) alone."""
    ns = int(gold[name + "/meta"][0])
    p = gold[name + "/params"].contiguous()
    z = gold[name + "/y32"].contiguous()
    x, lj = torch.empty_like(z), torch.empty_like(z)
    hm.hm_sos_invert(fptr(z), fptr(p), fptr(x), fptr(lj), ctypes.c_long(z.numel()), ns, 50, ctypes.c_float(120.0))
    gy = gold[name + "/gy"].contiguous()
    zeros = torch.zeros_like(z)
    gz, gp = torch.empty_like(z), torch.empty_like(p)
    adj.hm_sos_inverse_backward(fptr(x), fptr(p), fptr(gy), fptr(zeros), fptr(gz), fptr(gp), ctypes.c_long(z.numel()), ns)
    gz64, gp64 = reference_inverse_grads(z, p, ns, gy, torch.zeros(z.shape[0]), torch.float64)
    gz32, gp32 = reference_inverse_grads(z, p, ns, gy, torch.zeros(z.shape[0]), torch.float32)
    assert_parity(gz, gz32, gz64, 1e-4, max(1e-2, gz64.abs().mean().item()), name + " grad z (gl = 0)")
    assert_parity(gp, gp32, gp64, 1e-4, max(1e-2, gp64.abs().mean().item()), name + " grad params (gl = 0)")
    # the forward derivative at x is exp(logj): grad z = gy exp(-logj)
    assert torch.allclose(gz.double(), gy.double() * torch.exp(-lj.double()), rtol=1e-5, atol=0)


def test_inverse_backward_entry_rejects_bad_arguments_without_a_gpu():
    lib = _cabi.lib()
    f = lib.fc_sos_inverse_backward
    buf = (ctypes.c_float * 1024)()
    q = ctypes.addressof(buf)
    B, D = 4, 2

    def call(x=q, params=q, gy=q, gl=None, gx=q, gp=q, b=B, n=10):
        P = D * (3 * n + 1)
        return f(x, D, params, P, gy, D, gl, gx, D, gp, P, b, D, n, None)

    assert call(n=0) == -1  # FC_ERR_INVALID_ARGUMENT
    assert call(n=65) == -2  # FC_ERR_UNSUPPORTED: more sigmoids than FC_SOS_MAX_SIGMOIDS
    assert call(gy=None) == -1
    assert call(gp=None) == -1
    assert call(gx=None) == -1
    assert call(x=None) == -1
    assert call(params=None) == -1
    assert f(None, 0, None, 0, None, 0, None, None, 0, None, 0, 0, D, 10, None) == 0  # an empty batch is a no-op
