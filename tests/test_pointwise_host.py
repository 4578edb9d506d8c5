"""The element-wise squashing layers without a GPU: constructors, parameters and state_dict keys, the reference's errors,
the CPU refusal, the C entries' argument checks (which run before any CUDA call), the bounded_maf workloads, and the
per-element math of csrc/fc_pointwise.cuh compiled with g++ (tests/hostmath/pointwise.cpp, into a temporary directory)
against fp64 formulas: values, log-dets and every derivative the backward uses, including the stable Tanh log-det at |x|
up to 50."""
import ctypes
import math
import os
import subprocess

import pytest
import torch

from flowconductor_b200 import _cabi, ops, transforms, workloads
from oracle import locate
from tests import pointwise_oracle as pwo
from tests.helpers import ROOT

SRC = os.path.join(ROOT, "tests", "hostmath", "pointwise.cpp")
INVALID = -1
OPS = {"sigmoid": _cabi.POINTWISE_SIGMOID, "tanh": _cabi.POINTWISE_TANH, "leaky_relu": _cabi.POINTWISE_LEAKY_RELU,
       "exp": _cabi.POINTWISE_EXP, "cauchy": _cabi.POINTWISE_CAUCHY_CDF}


@pytest.fixture(scope="module")
def pw(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("hostmath") / "libpointwise.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-x", "c++", SRC,
                           "-o", lib])
    return ctypes.CDLL(lib)


def fptr(t):
    return ctypes.cast(t.data_ptr(), ctypes.c_void_p)


def host_eval(pw, op, inverse, x, T=1.0, slope=1e-2, eps=1e-6):
    x = x.float().contiguous()
    y, lad, bad = torch.empty_like(x), torch.empty_like(x), torch.empty(x.shape, dtype=torch.int32)
    pw.hm_pw_eval(OPS[op], int(inverse), fptr(x), ctypes.c_long(x.numel()), ctypes.c_float(T), ctypes.c_float(slope),
                  ctypes.c_float(eps), fptr(y), fptr(lad), fptr(bad))
    return y, lad, bad.bool()


def host_grad(pw, op, inverse, x, T=1.0, slope=1e-2, eps=1e-6):
    x = x.float().contiguous()
    out = [torch.empty_like(x) for _ in range(4)]
    pw.hm_pw_grad(OPS[op], int(inverse), fptr(x), ctypes.c_long(x.numel()), ctypes.c_float(T), ctypes.c_float(slope),
                  ctypes.c_float(eps), *(fptr(t) for t in out))
    return out


def elementwise(op, inverse, x, T, slope=1e-2, eps=1e-6):
    """The oracle per element (x [n] as [n, 1] rows), in x's dtype: (y, per-element log-det)."""
    x2 = x.reshape(-1, 1)
    if op == "sigmoid":
        y, lad = pwo.sigmoid(x2, T, eps, inverse)
    elif op == "tanh":
        y, lad = pwo.tanh(x2, inverse)
        if not inverse:
            lad = pwo.tanh_stable_logdet(x2)
    elif op == "leaky_relu":
        y, lad = pwo.leaky_relu(x2, slope, inverse)
    elif op == "exp":
        y, lad = pwo.exp(x2, inverse)
    else:
        y, lad = pwo.cauchy_cdf(x2, inverse)
    return y.reshape(-1), lad


def inputs_for(op, inverse, n=4000, seed=0):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(n, generator=g, dtype=torch.float64)
    if not inverse or op == "leaky_relu":
        return torch.cat([z, 10 * z[: n // 4], torch.tensor([0.0, -0.0, 1e-30, -1e-30])]).float()
    if op == "exp":
        return torch.exp(2 * z).float()
    if op == "tanh":
        return torch.tanh(z).float().clamp(-0.9999, 0.9999)
    u = torch.sigmoid(2 * z).float().clamp(1e-4, 1 - 1e-4)
    if op == "sigmoid":
        u = torch.cat([u, torch.tensor([0.0, 1.0, 1e-6, 1 - 1e-6, 1e-7, 1 - 1e-7])])
    return u


CASES = [(op, inv) for op in OPS for inv in (False, True)]


@pytest.mark.parametrize("op,inverse", CASES)
def test_element_math_against_fp64(pw, op, inverse):
    T = 1.7 if op == "sigmoid" else 1.0
    x = inputs_for(op, inverse)
    y, lad, bad = host_eval(pw, op, inverse, x, T=T, slope=0.03)
    assert not bad.any()
    y64, lad64 = elementwise(op, inverse, x.double(), torch.tensor([T], dtype=torch.float32).double(), 0.03)
    assert torch.isfinite(y).all() and torch.isfinite(lad).all()
    # a few fp32 ulps of the value, and of the inputs' conditioning on the inverses
    cond = 1.0
    if inverse and op in ("sigmoid", "tanh", "cauchy"):
        a = x.double().abs().clamp(1e-6, 1 - 1e-6)  # the clamp's bound itself differs between fp32 and fp64
        cond = 1.0 / torch.minimum(a, 1 - a)
    tol = 4e-7 * cond * (1 + x.double().abs())
    assert ((y.double() - y64).abs() <= tol * y64.abs().clamp_min(1e-6 if op == "sigmoid" and not inverse else 1.0)).all(), op
    assert ((lad.double() - lad64).abs() <= tol * lad64.abs().clamp_min(1.0)).all(), op


def test_tanh_stable_logdet_up_to_50(pw):
    x = torch.linspace(-50, 50, 20001)
    _, lad, _ = host_eval(pw, "tanh", False, x)
    x64 = x.double()
    want = math.log(4) - 2 * x64.abs() - 2 * torch.log1p(torch.exp(-2 * x64.abs()))
    assert torch.isfinite(lad).all()
    assert ((lad.double() - want).abs() <= 1e-6 * want.abs().clamp_min(1.0)).all()
    ref32 = torch.log(1 - torch.tanh(x) ** 2)  # the reference's fp32 formula: −inf from |x| ≈ 9 on
    assert not torch.isfinite(ref32[x.abs() > 10]).any()


@pytest.mark.parametrize("op,inverse", CASES)
def test_derivatives_against_fp64_autograd(pw, op, inverse):
    T = 0.8 if op == "sigmoid" else 1.0
    x = inputs_for(op, inverse, n=1000, seed=1)
    if op == "exp" and not inverse:
        x = x.clamp(-60, 60)
    if op == "sigmoid" and inverse:  # fp32 and fp64 place the clamp's bounds apart (test_sigmoid_inverse_clamp_gradient)
        x = x[(x > 2e-6) & (x < 1 - 2e-6)]
    dy, dl, dyT, dlT = host_grad(pw, op, inverse, x, T=T, slope=0.2)
    x64 = x.double().requires_grad_(True)
    t64 = torch.tensor([T], dtype=torch.float32).double().requires_grad_(True)
    y, lad = elementwise(op, inverse, x64, t64, 0.2)
    want = {}
    for name, f in (("y", y), ("lad", lad)):
        if not f.requires_grad:  # LeakyReLU's log-det is piecewise constant
            want[name] = (torch.zeros_like(x64), None)
            continue
        gx, gt = torch.autograd.grad(f.sum(), (x64, t64), retain_graph=True, allow_unused=True)
        want[name] = (torch.zeros_like(x64) if gx is None else gx, gt)
    # per-element temperature derivatives, from the summed autograd one (each element's y depends on T alone)
    for got, name in ((dy, "y"), (dl, "lad")):
        ref = want[name][0]
        xs = x
        scale = ref.abs().clamp_min(1.0)
        if inverse and op in ("sigmoid", "tanh", "cauchy"):
            scale = scale / torch.minimum(xs.double().abs(), 1 - xs.double().abs()).clamp_min(1e-6)
        assert ((got.double() - ref).abs() <= 2e-6 * scale).all(), (op, inverse, name)
    if op == "sigmoid":
        for got, name in ((dyT, "y"), (dlT, "lad")):
            ref = want[name][1]
            assert abs(float(got.double().sum()) - float(ref)) <= 1e-5 * max(1.0, float(got.double().abs().sum())), name
    else:
        assert not dyT.any() and not dlT.any()


def test_sigmoid_inverse_clamp_gradient(pw):
    """torch.clamp semantics: the gradient passes on [eps, 1 − eps], bounds included, and is zero strictly outside."""
    eps = 1e-6
    x = torch.tensor([0.0, eps / 2, eps, 0.5, 1 - eps, 1 - eps / 4, 1.0])
    dy, dl, dyT, _ = host_grad(pw, "sigmoid", True, x, T=1.0, eps=eps)
    lo, hi = torch.tensor(eps, dtype=torch.float32), 1 - torch.tensor(eps, dtype=torch.float32)
    inside = (x >= lo) & (x <= hi)
    assert torch.equal(dy != 0, inside) and (dl[~inside] == 0).all()
    assert torch.isfinite(dyT).all() and (dyT[:3] > 0).all()  # x = logit(y') / T still moves with T out there


def test_domain_flags(pw):
    for op, x, want in (("sigmoid", [-1e-7, 0.0, 1.0, 1.0000001], [1, 0, 0, 1]),
                        ("tanh", [-1.0, -0.999, 0.999, 1.0], [1, 0, 0, 1]),
                        ("exp", [-1.0, 0.0, 1e-38, 2.0], [1, 1, 0, 0]),
                        ("cauchy", [-1e-7, 0.0, 1.0, 1.0000001], [1, 0, 0, 1])):
        _, _, bad = host_eval(pw, op, True, torch.tensor(x))
        assert bad.int().tolist() == want, op
        _, _, bad = host_eval(pw, op, False, torch.tensor(x))
        assert not bad.any(), op


def test_constructors_and_state_dicts():
    s = transforms.Sigmoid()
    assert list(s.state_dict()) == ["temperature"] and list(s.parameters()) == []
    assert s.temperature.shape == (1,) and float(s.temperature) == 1.0 and s.eps == 1e-6
    s = transforms.Sigmoid(temperature=2.5, eps=1e-5, learn_temperature=True)
    assert [n for n, _ in s.named_parameters()] == ["temperature"] and float(s.temperature) == 2.5 and s.eps == 1e-5
    lg = transforms.Logit(temperature=0.5)
    assert list(lg.state_dict()) == ["_transform.temperature"] and float(lg._transform.temperature) == 0.5
    assert isinstance(lg, transforms.InverseTransform) and list(lg.parameters()) == []
    for cls in (transforms.Tanh, transforms.Exp, transforms.CauchyCDF, transforms.CauchyCDFInverse):
        assert list(cls().state_dict()) == []
    assert isinstance(transforms.CauchyCDF(location=1.0, scale=2.0, features=3), transforms.CauchyCDF)
    assert isinstance(transforms.CauchyCDFInverse()._transform, transforms.CauchyCDF)
    lr = transforms.LeakyReLU(0.2)
    assert lr.negative_slope == 0.2 and float(lr.log_negative_slope) == pytest.approx(math.log(0.2), rel=1e-6)
    assert list(lr.state_dict()) == []
    sq = transforms.Sigmoid(learn_temperature=True)
    cdf = transforms.CompositeCDFTransform(sq, transforms.PiecewiseRationalQuadraticCDF([4], 8))
    assert list(cdf.state_dict()) == ["_transforms.0.temperature", "_transforms.1.unnormalized_widths",
                                      "_transforms.1.unnormalized_heights", "_transforms.1.unnormalized_derivatives",
                                      "_transforms.2._transform.temperature"]
    assert cdf._transforms[2]._transform is sq and len(list(cdf.parameters())) == 4


def test_reference_errors():
    for bad in (0.0, -0.1):
        with pytest.raises(ValueError, match="Slope must be positive"):
            transforms.LeakyReLU(bad)


def test_cpu_tensors_are_refused():
    x = torch.rand(4, 3)
    for layer in (transforms.Sigmoid(), transforms.Logit(), transforms.Tanh(), transforms.LeakyReLU(), transforms.Exp(),
                  transforms.CauchyCDF(), transforms.CauchyCDFInverse()):
        for call in (layer.forward, layer.inverse):
            with pytest.raises(RuntimeError, match="CUDA"):
                call(x)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.pointwise_layer(x, None, _cabi.POINTWISE_TANH, False, 0.0, 0.0)


def test_c_abi_rejects_invalid_arguments():
    L = _cabi.lib()
    fake = ctypes.c_void_p(256)  # never dereferenced: the checks return before any CUDA call

    def apply(x=fake, xs=4, y=fake, ys=4, lad=fake, B=8, D=4, cfg=None):
        return L.fc_pointwise_apply(x, xs, y, ys, lad, 0, B, D, None if cfg is None else ctypes.byref(cfg), None, None)

    def backward(x=fake, xs=4, gx=fake, gxs=4, gt=None, ws=None, B=8, D=4, cfg=None):
        return L.fc_pointwise_backward(x, xs, None, 4, None, gx, gxs, gt, ws, B, D,
                                       None if cfg is None else ctypes.byref(cfg), None)

    tanh = _cabi.PointwiseConfig(_cabi.POINTWISE_TANH, 0, 0.0, 0.0, None)
    assert apply(cfg=None) == INVALID
    assert apply(cfg=_cabi.PointwiseConfig(5, 0, 0.0, 0.0, None)) == INVALID
    assert apply(cfg=_cabi.PointwiseConfig(-1, 0, 0.0, 0.0, None)) == INVALID
    assert apply(cfg=_cabi.PointwiseConfig(_cabi.POINTWISE_SIGMOID, 0, 0.0, 1e-6, None)) == INVALID
    assert apply(cfg=_cabi.PointwiseConfig(_cabi.POINTWISE_LEAKY_RELU, 0, 0.0, 0.0, None)) == INVALID
    assert apply(B=-1, cfg=tanh) == INVALID
    assert apply(D=0, cfg=tanh) == INVALID
    assert apply(xs=3, cfg=tanh) == INVALID and apply(ys=3, cfg=tanh) == INVALID
    assert apply(x=None, cfg=tanh) == INVALID and apply(y=None, cfg=tanh) == INVALID
    assert apply(lad=None, cfg=tanh) == INVALID
    assert apply(B=0, cfg=tanh) == 0  # nothing to do, nothing launched
    assert backward(cfg=None) == INVALID
    assert backward(x=None, cfg=tanh) == INVALID and backward(gx=None, cfg=tanh) == INVALID
    assert backward(xs=3, cfg=tanh) == INVALID and backward(gxs=3, cfg=tanh) == INVALID
    assert backward(gt=fake, ws=fake, cfg=tanh) == INVALID  # a temperature gradient exists for Sigmoid only
    sig = _cabi.PointwiseConfig(_cabi.POINTWISE_SIGMOID, 1, 0.0, 1e-6, fake)
    assert backward(gt=fake, ws=None, cfg=sig) == INVALID
    assert backward(B=0, cfg=sig) == 0
    assert L.fc_pointwise_workspace_floats(-1, 4) == INVALID and L.fc_pointwise_workspace_floats(8, 0) == INVALID
    assert L.fc_pointwise_workspace_floats(0, 4) == 1 and L.fc_pointwise_workspace_floats(1 << 30, 4) == 2048


def test_bounded_workloads():
    wl = workloads.get_workload("bounded_maf")
    assert (wl["features"], wl["batch"]) == (16, 262144)
    kinds = [layer["kind"] for layer in wl["layers"]]
    assert kinds[:4] == ["logit", "permutation", "maf_prq", "composite_cdf"] and kinds.count("maf_prq") == 5
    flow = workloads.build_flow(wl)
    layers = flow._transform._transforms
    assert type(layers[0]) is transforms.Logit
    cdf = layers[3]
    assert type(cdf) is transforms.CompositeCDFTransform
    assert isinstance(cdf._transforms[0].temperature, torch.nn.Parameter)
    assert type(cdf._transforms[1]) is transforms.PiecewiseRationalQuadraticCDF and cdf._transforms[1].tails is None
    small = workloads.get_workload("bounded_maf_small")
    assert (small["features"], small["batch"]) == (6, 128)
    flow = workloads.build_flow(small)
    assert isinstance(flow._transform._transforms[0]._transform.temperature, torch.nn.Parameter)
    x = workloads.sample_data(small, 4096, seed=3)
    assert x.shape == (4096, 6) and bool((x > 0).all()) and bool((x < 1).all())
    assert torch.equal(x, workloads.sample_data(small, 4096, seed=3))
    state = workloads.trained_like_(dict(workloads.build_flow(wl).state_dict()), wl)
    a, b = state["_transform._transforms.3._transforms.0.temperature"], state[
        "_transform._transforms.3._transforms.2._transform.temperature"]
    assert torch.equal(a, b) and float(a) != 1.0
    flow = workloads.build_flow(wl)
    flow.load_state_dict(state)  # the shared squashing layer takes one value
    assert float(flow._transform._transforms[3]._transforms[2]._transform.temperature) == float(a)
    assert float(state["_transform._transforms.0._transform.temperature"]) == 1.0  # Logit's buffer stays


@pytest.mark.skipif(not locate.have_reference(), reason="the FlowConductor reference tree is not available")
def test_oracle_against_the_reference_classes():
    nl = locate.import_reference().transforms.nonlinearities
    g = torch.Generator().manual_seed(0)
    x = torch.randn(64, 5, generator=g)
    u = torch.rand(64, 5, generator=g) * 0.98 + 0.01
    T = torch.tensor([1.3])
    for ref, fwd, inv, xin, uin in (
            (nl.Sigmoid(temperature=1.3), lambda v: pwo.sigmoid(v, T), lambda v: pwo.sigmoid(v, T, inverse=True), x, u),
            (nl.Tanh(), pwo.tanh, lambda v: pwo.tanh(v, True), x, 2 * u - 1),
            (nl.Exp(), pwo.exp, lambda v: pwo.exp(v, True), x, u),
            (nl.CauchyCDF(), pwo.cauchy_cdf, lambda v: pwo.cauchy_cdf(v, True), x, u)):
        for got, want in ((fwd(xin), ref(xin)), (inv(uin), ref.inverse(uin))):
            assert torch.allclose(got[0], want[0]) and torch.allclose(got[1], want[1], atol=1e-5)
