"""BatchNorm and the packaged flows without a GPU: constructor, parameters, buffers and init, state_dict, the flows' layer
structure, the restated oracle against hand-written fp64 formulas and autograd (the gradient formulas the kernels use),
and argument validation of the C entries (no launch happens on an invalid argument)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from flowconductor_b200 import _cabi, flows, ops, transforms, workloads
from tests import bn_oracle

INVALID, UNSUPPORTED = -1, -2


@pytest.mark.parametrize("features", [0, -3, 2.5, "4", True, None])
def test_constructor_rejects_non_positive_int(features):
    with pytest.raises(TypeError, match="Number of features must be a positive integer."):
        transforms.BatchNorm(features)


@pytest.mark.parametrize("D", [1, 6, 43])
def test_parameters_buffers_and_init(D):
    layer = transforms.BatchNorm(D)
    assert list(layer.state_dict().keys()) == ["unconstrained_weight", "bias", "running_mean", "running_var"]
    assert [n for n, _ in layer.named_parameters()] == ["unconstrained_weight", "bias"]
    assert [n for n, _ in layer.named_buffers()] == ["running_mean", "running_var"]
    assert layer.eps == 1e-5 and layer.momentum == 0.1
    assert torch.allclose(layer.weight, torch.ones(D), atol=1e-7, rtol=0)
    assert torch.count_nonzero(layer.bias) == 0
    assert torch.count_nonzero(layer.running_mean) == 0 and torch.count_nonzero(layer.running_var) == 0
    other = transforms.BatchNorm(D, eps=1e-3, momentum=0.3, affine=False)
    assert torch.allclose(other.weight, torch.ones(D), atol=1e-6, rtol=0) and other.momentum == 0.3


def test_state_dict_round_trip():
    a, b = transforms.BatchNorm(5), transforms.BatchNorm(5)
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for t in list(a.parameters()) + list(a.buffers()):
            t.copy_(torch.randn(t.shape, generator=g))
    b.load_state_dict(a.state_dict(), strict=True)
    for k, v in a.state_dict().items():
        assert torch.equal(v, b.state_dict()[k]), k


def test_inputs_must_be_2d_cuda_fp32():
    layer = transforms.BatchNorm(4)
    with pytest.raises(ValueError, match="Expected 2-dim inputs"):
        layer(torch.randn(2, 4, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        layer(torch.randn(3, 4))
    layer.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        layer(torch.randn(3, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        layer.inverse(torch.randn(3, 4))
    layer.train()
    with pytest.raises(transforms.InverseNotAvailable, match="only available in eval mode"):
        layer.inverse(torch.randn(3, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.batchnorm_train(torch.randn(3, 4), torch.zeros(4), torch.zeros(4), 1e-5)


def test_masked_autoregressive_flow_structure():
    flow = flows.MaskedAutoregressiveFlow(6, 16, 2, 2, batch_norm_between_layers=True)
    kinds = [type(t).__name__ for t in flow._transform._transforms]
    assert kinds == ["ReversePermutation", "MaskedAffineAutoregressiveTransform", "BatchNorm"] * 2
    plain = flows.MaskedAutoregressiveFlow(5, 8, 3, 1, use_random_permutations=True)
    kinds = [type(t).__name__ for t in plain._transform._transforms]
    assert kinds == ["RandomPermutation", "MaskedAffineAutoregressiveTransform"] * 3
    assert type(flow._distribution).__name__ == "StandardNormal"
    wl = workloads.get_workload("maf_bn_small")
    assert list(flow.state_dict().keys()) == list(workloads.build_flow(wl).state_dict().keys())
    assert [k for k in flow.state_dict() if "autoregressive_net.blocks.2" in k] == []


def test_simple_realnvp_structure():
    flow = flows.SimpleRealNVP(6, 16, 2, 2, batch_norm_between_layers=True)
    layers = flow._transform._transforms
    assert [type(t).__name__ for t in layers] == ["AffineCouplingTransform", "BatchNorm"] * 2
    # mask = ones; mask[::2] = -1; negated after every layer: odd features first, then even ones
    assert layers[0].transform_features.tolist() == [1, 3, 5] and layers[2].transform_features.tolist() == [0, 2, 4]
    assert layers[0].transform_net.hidden_features == 16 and len(layers[0].transform_net.blocks) == 2
    vp = flows.SimpleRealNVP(5, 8, 3, 1, use_volume_preserving=True)
    assert [type(t).__name__ for t in vp._transform._transforms] == ["AdditiveCouplingTransform"] * 3
    wl = workloads.get_workload("realnvp_bn_small")
    ours = workloads.build_flow(wl).state_dict()
    assert list(flow.state_dict().keys()) == list(ours.keys())
    for k, v in flow.state_dict().items():
        assert v.shape == ours[k].shape, k
        if k.endswith("_features"):
            assert torch.equal(v, ours[k]), k


def test_workloads_with_batchnorm():
    for name, d, n_bn in (("maf_bn_small", 6, 2), ("realnvp_bn_small", 6, 2), ("maf_bn", 43, 5)):
        wl = workloads.get_workload(name)
        assert wl["features"] == d and [layer["kind"] for layer in wl["layers"]].count("batchnorm") == n_bn
    wl = workloads.get_workload("maf_bn")
    assert wl["batch"] == 262144 and {layer.get("hidden_features") for layer in wl["layers"]} == {None, 256}
    wl = workloads.get_workload("maf_bn_small")
    flow = workloads.build_flow(wl)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    p = workloads.layer_prefix(2)
    assert (state[p + "running_var"] > 0).all() and torch.count_nonzero(state[p + "running_mean"]) == 6
    assert not torch.allclose(F.softplus(state[p + "unconstrained_weight"]), torch.ones(6), atol=0.05)
    x = torch.randn(5, 6, generator=torch.Generator().manual_seed(0))
    specs = workloads.oracle_specs(wl)
    for training in (False, True):
        lp = bn_oracle.flow_log_prob(state, specs, x, training=training)
        assert lp.shape == (5,) and torch.isfinite(lp).all()


def _state64(D, seed):
    g = torch.Generator().manual_seed(seed)
    return {"unconstrained_weight": torch.randn(D, generator=g, dtype=torch.float64) * 0.5,
            "bias": torch.randn(D, generator=g, dtype=torch.float64),
            "running_mean": torch.randn(D, generator=g, dtype=torch.float64),
            "running_var": torch.exp(torch.randn(D, generator=g, dtype=torch.float64))}


@pytest.mark.parametrize("D", [1, 3, 7])
def test_oracle_against_fp64_formulas(D):
    """The literal restatement against element-by-element fp64 formulas, the Jacobian's log-determinant, and the
    inverse identity."""
    eps = 1e-5
    state = _state64(D, D)
    x = torch.randn(9, D, dtype=torch.float64, generator=torch.Generator().manual_seed(1)) * 2 + 3
    w = np.log1p(np.exp(state["unconstrained_weight"].numpy())) + eps
    b = state["bias"].numpy()
    xn = x.numpy()
    mu, var = xn.mean(0), ((xn - xn.mean(0)) ** 2).sum(0) / (xn.shape[0] - 1)
    y, lad = bn_oracle.batch_norm(state, "", x, training=True)
    assert np.allclose(y.numpy(), w * (xn - mu) / np.sqrt(var + eps) + b, atol=1e-12, rtol=1e-12)
    assert np.allclose(lad.numpy(), np.sum(np.log(w) - 0.5 * np.log(var + eps)), atol=1e-12)
    rm, rv = state["running_mean"].numpy(), state["running_var"].numpy()
    y, lad = bn_oracle.batch_norm(state, "", x)
    assert np.allclose(y.numpy(), w * (xn - rm) / np.sqrt(rv + eps) + b, atol=1e-12, rtol=1e-12)
    jac = torch.autograd.functional.jacobian(lambda v: bn_oracle.batch_norm(state, "", v.view(1, D))[0].view(D), x[0])
    assert abs(float(torch.linalg.slogdet(jac)[1] - lad[0])) < 1e-10
    xi, lad_inv = bn_oracle.batch_norm(state, "", y, inverse=True)
    assert torch.allclose(xi, x, atol=1e-10) and torch.allclose(lad_inv, -lad, atol=1e-12)
    s = dict(state)
    bn_oracle.update_running(s, "", x)
    assert np.allclose(s["running_mean"].numpy(), 0.9 * rm + 0.1 * mu) and np.allclose(s["running_var"].numpy(),
                                                                                     0.9 * rv + 0.1 * var)


@pytest.mark.parametrize("mode", ["train", "eval_forward", "eval_inverse"])
@pytest.mark.parametrize("D", [1, 4])
def test_gradient_formulas_against_autograd(mode, D):
    """The closed forms the backward kernels evaluate (include/flowcon_b200.h, DESIGN §4.17) against fp64 autograd of
    the oracle, with both upstream gradients and each one alone."""
    eps = 1e-5
    B = 11
    gen = torch.Generator().manual_seed(D)
    state = _state64(D, 7)
    x0 = torch.randn(B, D, dtype=torch.float64, generator=gen) * 3 + 5
    gys = torch.randn(B, D, dtype=torch.float64, generator=gen)
    gls = torch.randn(B, dtype=torch.float64, generator=gen)
    for gy, gl in ((gys, gls), (gys, torch.zeros_like(gls)), (torch.zeros_like(gys), gls)):
        uw = state["unconstrained_weight"].clone().requires_grad_(True)
        bias = state["bias"].clone().requires_grad_(True)
        x = x0.clone().requires_grad_(True)
        st = dict(state, unconstrained_weight=uw, bias=bias)
        y, lad = bn_oracle.batch_norm(st, "", x, inverse=mode == "eval_inverse", training=mode == "train")
        ((y * gy).sum() + (lad * gl).sum()).backward()
        with torch.no_grad():
            w = F.softplus(state["unconstrained_weight"]) + eps
            b = state["bias"]
            G = gl.sum()
            if mode == "train":
                mu, v = x0.mean(0), x0.var(0)
            else:
                mu, v = state["running_mean"], state["running_var"]
            s = torch.sqrt(v + eps)
            if mode == "eval_inverse":
                gx = gy * s / w
                gb = -(gy * s / w).sum(0)
                gw = -(gy * s * (x0 - b) / w ** 2).sum(0) - G / w
            else:
                xh = (x0 - mu) / s
                gb = gy.sum(0)
                gw = (gy * xh).sum(0) + G / w
                if mode == "train":
                    gx = (w / s) * (gy - gy.mean(0) - xh * (gy * xh).sum(0) / (B - 1)) - G * xh / ((B - 1) * s)
                else:
                    gx = gy * w / s
            guw = gw * torch.sigmoid(state["unconstrained_weight"])
        assert torch.allclose(x.grad, gx, atol=1e-12, rtol=1e-10)
        assert torch.allclose(bias.grad, gb, atol=1e-12, rtol=1e-10)
        assert torch.allclose(uw.grad, guw, atol=1e-12, rtol=1e-10)


def test_c_entries_reject_invalid_arguments():
    """Every check runs before a launch: null pointers are never dereferenced."""
    L = _cabi.lib()
    dummy = 256  # never dereferenced: the call must fail validation first

    def stats(x=dummy, xs=8, m=dummy, v=dummy, ws=dummy, B=4, D=8):
        return L.fc_batchnorm_stats(x, xs, m, v, ws, B, D, None)

    for kw in ({"D": 0}, {"D": -1}, {"B": 0}, {"B": -1}, {"x": None}, {"m": None}, {"v": None}, {"ws": None},
               {"xs": 7}):
        assert stats(**kw) == INVALID, kw
    assert stats(D=4097, xs=4097) == UNSUPPORTED

    def apply(x=dummy, xs=8, m=dummy, v=dummy, uw=dummy, b=dummy, y=dummy, ys=8, lad=dummy, B=4, D=8):
        return L.fc_batchnorm_apply(x, xs, m, v, uw, b, 1e-5, y, ys, lad, B, D, 0, None)

    for kw in ({"D": 0}, {"B": -1}, {"m": None}, {"v": None}, {"uw": None}, {"b": None}, {"x": None}, {"y": None},
               {"lad": None}, {"xs": 7}, {"ys": 7}):
        assert apply(**kw) == INVALID, kw
    assert apply(D=4097, xs=4097, ys=4097) == UNSUPPORTED
    assert apply(B=0, x=None, y=None, lad=None) == 0  # an empty batch launches nothing

    def backward(x=dummy, xs=8, m=dummy, v=dummy, uw=dummy, b=dummy, gy=dummy, gys=8, gl=dummy, gx=dummy, gxs=8,
                 guw=dummy, gb=dummy, ws=dummy, B=4, D=8, mode=0):
        return L.fc_batchnorm_backward(x, xs, m, v, uw, b, 1e-5, gy, gys, gl, gx, gxs, guw, gb, ws, B, D, mode, None)

    for kw in ({"D": 0}, {"B": -1}, {"mode": 3}, {"mode": -1}, {"m": None}, {"v": None}, {"uw": None}, {"b": None},
               {"guw": None}, {"gb": None}, {"x": None}, {"gy": None}, {"gx": None}, {"ws": None}, {"xs": 7},
               {"gys": 7}, {"gxs": 7}):
        assert backward(**kw) == INVALID, kw
    assert backward(D=4097, xs=4097, gys=4097, gxs=4097) == UNSUPPORTED
    for B, D in ((-1, 8), (4, 0)):
        assert L.fc_batchnorm_workspace_floats(B, D) == INVALID
    assert L.fc_batchnorm_workspace_floats(4, 4097) == UNSUPPORTED
    assert L.fc_batchnorm_workspace_floats(4, 4096) >= 3 * 4096
