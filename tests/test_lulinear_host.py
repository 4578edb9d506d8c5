"""LULinear without a GPU: constructor, parameters and init, state_dict, the restated oracle against independent fp64
math, and argument validation of the C entries (no launch happens on an invalid argument)."""
import numpy as np
import pytest
import torch

from flowconductor_b200 import _cabi, ops, transforms, workloads
from tests import lu_oracle

INVALID = -1


@pytest.mark.parametrize("features", [0, -3, 2.5, "4", True, None])
def test_constructor_rejects_non_positive_int(features):
    with pytest.raises(TypeError, match="Number of features must be a positive integer."):
        transforms.LULinear(features)


@pytest.mark.parametrize("D", [1, 2, 7, 64])
def test_parameters_and_identity_init(D):
    layer = transforms.LULinear(D)
    n = D * (D - 1) // 2
    assert list(layer.state_dict().keys()) == ["bias", "lower_entries", "upper_entries", "unconstrained_upper_diag"]
    assert [tuple(p.shape) for _, p in layer.named_parameters()] == [(D,), (n,), (n,), (D,)]
    assert not list(layer.buffers())  # the index arrays are plain attributes
    assert np.array_equal(layer.lower_indices[0], np.tril_indices(D, -1)[0])
    assert torch.count_nonzero(layer.bias) == 0 and torch.count_nonzero(layer.lower_entries) == 0
    assert torch.count_nonzero(layer.upper_entries) == 0
    assert torch.allclose(layer.unconstrained_upper_diag, torch.full((D,), float(np.log(np.exp(1 - 1e-3) - 1))))
    assert torch.allclose(layer.weight(), torch.eye(D), atol=1e-6)
    assert torch.allclose(layer.weight_inverse(), torch.eye(D), atol=1e-6)
    assert abs(float(layer.logabsdet().detach())) < 1e-5 * D
    lower, upper = layer._create_lower_upper()
    assert torch.equal(torch.diagonal(lower), torch.ones(D)) and torch.equal(torch.diagonal(upper), layer.upper_diag)


def test_random_init_scale():
    torch.manual_seed(0)
    D = 50
    layer = transforms.LULinear(D, identity_init=False, eps=1e-2)
    bound = 1.0 / np.sqrt(D)
    assert torch.count_nonzero(layer.bias) == 0
    for p in (layer.lower_entries, layer.upper_entries, layer.unconstrained_upper_diag):
        assert float(p.abs().max()) <= bound and float(p.abs().max()) > 0.8 * bound
    assert torch.allclose(layer.upper_diag, torch.nn.functional.softplus(layer.unconstrained_upper_diag) + 1e-2)
    W = layer.weight().double()
    assert torch.allclose(layer.weight_inverse().double() @ W, torch.eye(D, dtype=torch.float64), atol=1e-5)
    assert abs(float(layer.logabsdet()) - float(torch.linalg.slogdet(W)[1])) < 1e-4


def test_use_cache_and_train():
    layer = transforms.LULinear(3, using_cache=True)
    assert layer.using_cache
    layer.use_cache(False)
    assert not layer.using_cache
    with pytest.raises(TypeError, match="Mode must be boolean."):
        layer.use_cache(1)
    assert layer.train() is layer and layer.eval() is layer


def test_state_dict_round_trip():
    a, b = transforms.LULinear(5, identity_init=False), transforms.LULinear(5)
    b.load_state_dict(a.state_dict(), strict=True)
    assert torch.equal(a.weight(), b.weight())


def _state64(D, seed):
    layer = transforms.LULinear(D, identity_init=False)
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(v.shape, generator=g, dtype=torch.float64) * 0.5 for k, v in layer.state_dict().items()}


@pytest.mark.parametrize("D", [1, 2, 5, 12])
def test_lu_oracle_against_fp64_math(D):
    """The literal restatement (two F.linear, two triangular solves) against W built independently, its slogdet, its
    inverse and the log-determinant of the autograd Jacobian."""
    state = _state64(D, D)
    spec = {"kind": "lu_linear", "prefix": ""}
    lower = torch.eye(D, dtype=torch.float64)
    upper = torch.zeros(D, D, dtype=torch.float64)
    k = 0
    for i in range(D):
        for j in range(i):
            lower[i, j] = state["lower_entries"][k]
            k += 1
    k = 0
    for i in range(D):
        for j in range(i + 1, D):
            upper[i, j] = state["upper_entries"][k]
            k += 1
    diag = torch.log1p(torch.exp(state["unconstrained_upper_diag"])) + 1e-3
    upper += torch.diag(diag)
    W = lower @ upper
    x = torch.randn(9, D, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    y, lad = lu_oracle.apply_layer(state, spec, x)
    assert torch.allclose(y, x @ W.T + state["bias"], atol=1e-12, rtol=1e-12)
    sign, logdet = torch.linalg.slogdet(W)
    assert torch.allclose(lad, logdet.expand(9), atol=1e-12)
    jac = torch.autograd.functional.jacobian(lambda v: lu_oracle.apply_layer(state, spec, v.view(1, D))[0].view(D), x[0])
    assert abs(float(torch.linalg.slogdet(jac)[1] - lad[0])) < 1e-10
    xi, lad_inv = lu_oracle.apply_layer(state, spec, y, inverse=True)
    assert torch.allclose(xi, (y - state["bias"]) @ torch.linalg.inv(W).T, atol=1e-10)
    assert torch.allclose(xi, x, atol=1e-10)
    assert torch.allclose(lad_inv, -lad, atol=0)


def test_composed_operands_match_the_factors():
    """The fp64 composition the kernel consumes: forward (L U, bias, Σ log d), inverse (U⁻¹ L⁻¹, -M bias, -Σ log d)."""
    torch.manual_seed(3)
    layer = transforms.LULinear(9, identity_init=False)
    with torch.no_grad():
        layer.bias.uniform_(-1, 1)
        M, c, ld = layer._compose(False)
        Mi, ci, ldi = layer._compose(True)
    W = layer.weight().double()
    assert M.dtype == torch.float32 and torch.allclose(M.double(), W, atol=1e-6)
    assert torch.equal(c, layer.bias.detach())
    assert torch.allclose(Mi.double(), torch.linalg.inv(W), atol=1e-5)
    assert torch.allclose(ci.double(), -torch.linalg.inv(W) @ layer.bias.double(), atol=1e-5)
    assert torch.allclose(ld.double(), torch.linalg.slogdet(W)[1], atol=1e-5) and float(ldi) == -float(ld)


def test_workloads_with_lu_layers():
    for name, d in (("nsf_lu_small", 6), ("nsf_lu", 32)):
        wl = workloads.get_workload(name)
        assert wl["features"] == d
        kinds = [layer["kind"] for layer in wl["layers"]]
        assert kinds[1::2] == ["lu_linear"] * (len(kinds) // 2) and set(kinds[0::2]) == {"prq_coupling"}
    wl = workloads.get_workload("nsf_lu_small")
    flow = workloads.build_flow(wl)
    assert isinstance(flow._transform._transforms[1], transforms.LULinear)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    lu = state[workloads.layer_prefix(1) + "lower_entries"]
    assert float(lu.abs().max()) <= 1 / np.sqrt(6) and torch.count_nonzero(lu) == lu.numel()
    x = torch.randn(5, 6, generator=torch.Generator().manual_seed(0))
    lp = lu_oracle.flow_log_prob(state, workloads.oracle_specs(wl), x)
    assert lp.shape == (5,) and torch.isfinite(lp).all()


def test_inputs_must_be_2d_cuda_fp32():
    layer = transforms.LULinear(4)
    with pytest.raises(NotImplementedError):
        layer(torch.randn(2, 4, 3, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        layer(torch.randn(3, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        layer.inverse(torch.randn(3, 4, dtype=torch.float64))
    with pytest.raises(RuntimeError, match="CUDA"):
        transforms.LULinear(80)(torch.randn(3, 80))  # the tensor-core side does not fall back to the CPU either
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.lulinear_layer(torch.randn(3, 4), torch.eye(4), torch.zeros(4), torch.zeros(()))


def test_c_entries_reject_invalid_arguments():
    """Every check runs before a launch: null pointers are never dereferenced."""
    L = _cabi.lib()
    dummy = 256  # never dereferenced: the call must fail validation first

    def apply(x=dummy, xs=8, M=dummy, c=dummy, ld=dummy, y=dummy, ys=8, lad=dummy, B=4, D=8):
        return L.fc_lulinear_apply(x, xs, M, c, ld, y, ys, lad, 0, B, D, None)

    for kw in ({"D": 0}, {"D": 64}, {"D": -1}, {"B": -1}, {"M": None}, {"c": None}, {"ld": None}, {"x": None},
               {"y": None}, {"lad": None}, {"xs": 7}, {"ys": 7}):
        assert apply(**kw) == INVALID, kw
    assert apply(B=0, x=None, y=None, lad=None) == 0  # an empty batch launches nothing

    def backward(x=dummy, xs=8, M=dummy, gy=dummy, gys=8, gx=dummy, gxs=8, gM=dummy, gc=dummy, ws=dummy, B=4, D=8):
        return L.fc_lulinear_backward(x, xs, M, gy, gys, gx, gxs, gM, gc, ws, B, D, None)

    for kw in ({"D": 0}, {"D": 64}, {"B": -1}, {"M": None}, {"gM": None}, {"gc": None}, {"x": None}, {"gy": None},
               {"gx": None}, {"ws": None}, {"xs": 3}, {"gys": 3}, {"gxs": 3}):
        assert backward(**kw) == INVALID, kw
    for B, D in ((-1, 8), (4, 0), (4, 64)):
        assert L.fc_lulinear_workspace_floats(B, D) == INVALID
