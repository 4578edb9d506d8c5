"""DiagonalNormal and ConditionalDiagonalNormal without a GPU: constructors, parameters and state_dict keys, every error
the reference raises, the CPU refusal, the workloads with a learned base, the restated oracle against fp64 formulas and
the closed-form gradients the kernels evaluate, argument validation of the C entries, and the oracle against the live
reference classes where the reference tree is available."""
import math

import pytest
import torch
from torch import nn

from flowconductor_b200 import _cabi, distributions, flows, ops, transforms, workloads
from oracle import locate
from tests import diagnormal_oracle as dno

INVALID = -1


@pytest.mark.parametrize("shape", [[1], [6], [3, 4]])
def test_diagonal_normal_constructor_and_state_dict(shape):
    dist = distributions.DiagonalNormal(shape)
    D = math.prod(shape)
    assert list(dist.state_dict().keys()) == ["mean_", "log_std_"]
    assert [n for n, _ in dist.named_parameters()] == ["mean_", "log_std_"]
    assert dist.mean_.shape == (1, D) and dist.log_std_.shape == (1, D)
    assert torch.count_nonzero(dist.mean_) == 0 and torch.count_nonzero(dist.log_std_) == 0
    assert dist._log_z.dtype == torch.float64 and dist._log_z.dim() == 0
    assert float(dist._log_z) == pytest.approx(0.5 * D * math.log(2 * math.pi), rel=1e-15)


def test_conditional_diagonal_normal_constructor_and_state_dict():
    dist = distributions.ConditionalDiagonalNormal([6], context_encoder=nn.Linear(4, 12))
    assert list(dist.state_dict().keys()) == ["_context_encoder.weight", "_context_encoder.bias"]
    assert float(dist._log_z) == pytest.approx(3 * math.log(2 * math.pi), rel=1e-15)
    bare = distributions.ConditionalDiagonalNormal([3])
    assert list(bare.state_dict().keys()) == []
    ctx = torch.randn(5, 6)
    means, log_stds = bare._compute_params(ctx)
    assert torch.equal(means, ctx[:, :3]) and torch.equal(log_stds, ctx[:, 3:])
    assert means.data_ptr() == ctx.data_ptr()  # views of the encoder output, the blocked layout
    assert torch.equal(bare.mean(ctx), ctx[:, :3])


def test_reference_errors():
    dist = distributions.ConditionalDiagonalNormal([3])
    with pytest.raises(ValueError, match="Context can't be None."):
        dist.log_prob(torch.randn(4, 3))
    with pytest.raises(ValueError, match="Context can't be None."):
        dist.sample(2)
    with pytest.raises(RuntimeError, match="even"):
        dist._compute_params(torch.randn(4, 5))
    odd = distributions.ConditionalDiagonalNormal([3], context_encoder=nn.Linear(2, 7))
    with pytest.raises(RuntimeError, match="even"):
        odd.log_prob(torch.randn(4, 3), torch.randn(4, 2))
    flat = distributions.ConditionalDiagonalNormal([3], context_encoder=lambda c: c.reshape(-1, 12))
    with pytest.raises(RuntimeError, match="batch dimension"):
        flat.log_prob(torch.randn(4, 3), torch.randn(4, 6))
    with pytest.raises(ValueError, match="Expected input of shape"):
        dist.log_prob(torch.randn(4, 2), torch.randn(4, 6))
    with pytest.raises(ValueError, match="Number of input items"):
        dist.log_prob(torch.randn(4, 3), torch.randn(5, 6))
    with pytest.raises(ValueError, match="Expected input of shape"):
        distributions.DiagonalNormal([3]).log_prob(torch.randn(4, 4))


def test_cpu_tensors_are_refused():
    for call in (lambda: distributions.DiagonalNormal([3]).log_prob(torch.randn(4, 3)),
                 lambda: distributions.DiagonalNormal([3]).sample(4),
                 lambda: distributions.ConditionalDiagonalNormal([3]).log_prob(torch.randn(4, 3), torch.randn(4, 6)),
                 lambda: distributions.ConditionalDiagonalNormal([3]).sample(2, torch.randn(4, 6)),
                 lambda: ops.diagnormal_log_prob(torch.randn(4, 3), torch.randn(4, 6), 1, None),
                 lambda: ops.diagnormal_sample(torch.randn(4, 3), torch.randn(1, 6), 4)):
        with pytest.raises(RuntimeError, match="CUDA"):
            call()


def test_workloads_with_a_learned_base():
    for name, kind, keys in (("cond_prq_diag_small", "ConditionalDiagonalNormal",
                              ["_distribution._context_encoder.weight", "_distribution._context_encoder.bias"]),
                             ("maf_diag_small", "DiagonalNormal", ["_distribution.mean_", "_distribution.log_std_"]),
                             ("cond_sos_diag", "ConditionalDiagonalNormal",
                              ["_distribution._context_encoder.weight", "_distribution._context_encoder.bias"])):
        wl = workloads.get_workload(name)
        flow = workloads.build_flow(wl)
        assert type(flow._distribution).__name__ == kind and flow._context_used_in_base
        assert [k for k in flow.state_dict() if k.startswith("_distribution.")] == keys
    wl = workloads.get_workload("cond_sos_diag")
    assert (wl["features"], wl["context_features"], wl["batch"]) == (32, 8, 262144)
    assert workloads.build_flow(wl)._distribution._context_encoder.weight.shape == (64, 8)
    # the layers are initialised as without the base: only the encoder draws after them
    plain = workloads.build_flow(workloads.get_workload("cond_prq_small")).state_dict()
    diag = workloads.build_flow(workloads.get_workload("cond_prq_diag_small")).state_dict()
    for k, v in plain.items():
        assert torch.equal(v, diag[k]), k
    wl = workloads.get_workload("maf_diag_small")
    state = workloads.trained_like_(dict(workloads.build_flow(wl).state_dict()), wl)
    assert torch.count_nonzero(state["_distribution.mean_"]) == 6 and torch.count_nonzero(state["_distribution.log_std_"]) == 6


@pytest.mark.parametrize("D", [1, 3, 7])
def test_oracle_against_fp64_formulas(D):
    g = torch.Generator().manual_seed(D)
    x = torch.randn(9, D, dtype=torch.float64, generator=g)
    m = torch.randn(9, D, dtype=torch.float64, generator=g)
    s = 0.5 * torch.randn(9, D, dtype=torch.float64, generator=g)
    lp = dno.normal_log_prob(x, m, s)
    want = torch.distributions.Normal(m, torch.exp(s)).log_prob(x).sum(1)
    assert torch.allclose(lp, want, atol=1e-12, rtol=1e-12)
    lp1 = dno.normal_log_prob(x, m[:1], s[:1])  # one shared row broadcasts
    assert torch.allclose(lp1, torch.distributions.Normal(m[:1], torch.exp(s[:1])).log_prob(x).sum(1), atol=1e-12)
    eps = torch.randn(9 * 4, D, dtype=torch.float64, generator=g)
    y = dno.sample_from_noise(m, s, eps, 4)
    assert y.shape == (9, 4, D)
    assert torch.allclose(y[2, 3], m[2] + torch.exp(s[2]) * eps[2 * 4 + 3], atol=1e-15)


def test_gradient_formulas_against_autograd():
    """The closed forms of the backward kernels (include/flowcon_b200.h) against fp64 autograd of the oracle, for
    G = 1, G = n and one shared row."""
    g = torch.Generator().manual_seed(3)
    D, C, n = 5, 4, 3
    for group in (1, n, C * n):
        R = C * n
        P = -(-R // group)
        params = torch.randn(P, 2 * D, dtype=torch.float64, generator=g).requires_grad_(True)
        x = torch.randn(R, D, dtype=torch.float64, generator=g).requires_grad_(True)
        w = torch.randn(R, dtype=torch.float64, generator=g)
        m, s = dno.params_from(params, D)
        rep = torch.arange(R) // group
        (dno.normal_log_prob(x, m[rep], s[rep]) * w).sum().backward()
        with torch.no_grad():
            m0, s0 = m[rep], s[rep]
            e = torch.exp(-s0)
            z = (x - m0) * e
            gz = w[:, None] * z * e
            assert torch.allclose(x.grad, -gz, atol=1e-12)
            gm = torch.zeros(P, D, dtype=torch.float64).index_add_(0, rep, gz)
            gs = torch.zeros(P, D, dtype=torch.float64).index_add_(0, rep, w[:, None] * (z * z - 1))
            assert torch.allclose(params.grad, torch.cat([gm, gs], 1), atol=1e-12)
        params.grad = None
        eps = torch.randn(R, D, dtype=torch.float64, generator=g)
        gy = torch.randn(R, D, dtype=torch.float64, generator=g)
        m, s = dno.params_from(params, D)
        (dno.sample_from_noise(m, s, eps, group).reshape(-1, D)[:R] * gy).sum().backward() if group != R else \
            ((m + torch.exp(s) * eps) * gy).sum().backward()
        with torch.no_grad():
            gm = torch.zeros(P, D, dtype=torch.float64).index_add_(0, rep, gy)
            gs = torch.zeros(P, D, dtype=torch.float64).index_add_(0, rep, gy * torch.exp(s[rep]) * eps)
            assert torch.allclose(params.grad, torch.cat([gm, gs], 1), atol=1e-12)


def test_c_entries_reject_invalid_arguments():
    """Every check runs before a launch: null pointers are never dereferenced."""
    L = _cabi.lib()
    dummy = 256  # never dereferenced: the call must fail validation first

    def lp(x=dummy, xs=8, p=dummy, ps=16, out=dummy, R=4, D=8, G=1):
        return L.fc_diagnormal_log_prob(x, xs, p, ps, None, out, R, D, G, None)

    for kw in ({"D": 0}, {"R": -1}, {"G": 0}, {"x": None}, {"p": None}, {"out": None}, {"xs": 7}, {"ps": 15}):
        assert lp(**kw) == INVALID, kw
    assert lp(R=0, x=None, out=None) == 0  # an empty batch launches nothing

    def sample(e=dummy, es=8, p=dummy, ps=16, y=dummy, ys=8, R=4, D=8, G=2):
        return L.fc_diagnormal_sample(e, es, p, ps, y, ys, R, D, G, None)

    for kw in ({"D": 0}, {"R": -1}, {"G": 0}, {"e": None}, {"p": None}, {"y": None}, {"es": 7}, {"ys": 7},
               {"ps": 15}):
        assert sample(**kw) == INVALID, kw

    def lp_bwd(x=dummy, xs=8, p=dummy, ps=16, g=dummy, gx=dummy, gxs=8, gp=dummy, ws=dummy, R=4, D=8, G=1):
        return L.fc_diagnormal_log_prob_backward(x, xs, p, ps, g, gx, gxs, gp, ws, R, D, G, None)

    for kw in ({"D": 0}, {"R": -1}, {"G": 0}, {"x": None}, {"p": None}, {"g": None}, {"gx": None}, {"gp": None},
               {"xs": 7}, {"gxs": 7}, {"ps": 15}):
        assert lp_bwd(**kw) == INVALID, kw

    def s_bwd(e=dummy, es=8, p=dummy, ps=16, gy=dummy, gys=8, gp=dummy, ws=dummy, R=4, D=8, G=2):
        return L.fc_diagnormal_sample_backward(e, es, p, ps, gy, gys, gp, ws, R, D, G, None)

    for kw in ({"D": 0}, {"R": -1}, {"G": 0}, {"e": None}, {"p": None}, {"gy": None}, {"gp": None}, {"es": 7},
               {"gys": 7}, {"ps": 15}):
        assert s_bwd(**kw) == INVALID, kw
    for R, D, G in ((-1, 8, 1), (4, 0, 1), (4, 8, 0)):
        assert L.fc_diagnormal_workspace_floats(R, D, G) == INVALID
    assert L.fc_diagnormal_workspace_floats(1 << 20, 8, 1) == 0  # per-row gradients need no scratch
    assert L.fc_diagnormal_workspace_floats(16, 8, 16) == 0


@pytest.mark.skipif(not locate.have_reference(), reason="reference tree not found")
def test_oracle_against_live_reference():
    locate.import_reference()
    from flowcon.distributions.normal import ConditionalDiagonalNormal as RefCond
    from flowcon.distributions.normal import DiagonalNormal as RefDiag

    torch.manual_seed(5)
    D, C = 6, 7
    enc = nn.Linear(4, 2 * D)
    ref = RefCond([D], context_encoder=enc)
    ours = distributions.ConditionalDiagonalNormal([D], context_encoder=nn.Linear(4, 2 * D))
    assert list(ref.state_dict().keys()) == list(ours.state_dict().keys())
    assert [k for k, _ in ref.named_buffers()] == [k for k, _ in ours.named_buffers()]
    ours.load_state_dict(ref.state_dict(), strict=True)
    ctx = torch.randn(C, 4)
    x = torch.randn(C, D)
    state = {"_distribution." + k: v for k, v in ref.state_dict().items()}
    with torch.no_grad():
        want = ref.log_prob(x, ctx)
        got = dno.base_log_prob(state, {"kind": "conditional_diagonal_normal"}, x, ctx)
        assert torch.allclose(got, want, atol=1e-5, rtol=1e-6)
        got64 = dno.base_log_prob({k: v.double() for k, v in state.items()}, {"kind": "conditional_diagonal_normal"},
                                  x.double(), ctx)
        assert torch.allclose(got64.float(), want, atol=1e-4, rtol=1e-5)
        torch.manual_seed(9)
        want = ref.sample(5, ctx)
        torch.manual_seed(9)
        noise = torch.randn(C * 5, D)
        m, s = dno.params_from(enc(ctx), D)
        assert torch.equal(dno.sample_from_noise(m, s, noise, 5), want)
        assert torch.equal(ref.mean(ctx), m)
    for bad, err in ((None, ValueError), (torch.randn(C, 3), RuntimeError)):
        with pytest.raises(err):
            RefCond([D]).log_prob(x, bad) if bad is None else RefCond([D])._compute_params(bad)
    diag = RefDiag([D])
    assert list(diag.state_dict().keys()) == ["mean_", "log_std_"] and diag.mean_.shape == (1, D)
    with torch.no_grad():
        diag.mean_.normal_()
        diag.log_std_.normal_(0.0, 0.3)
        state = {"_distribution." + k: v for k, v in diag.state_dict().items()}
        assert torch.allclose(dno.base_log_prob(state, {"kind": "diagonal_normal"}, x), diag.log_prob(x), atol=1e-5)
    with pytest.raises(NotImplementedError):
        diag.sample(3)
    assert "_log_z" not in diag.state_dict()
    ref_flow_keys = flows.Flow(transforms.CompositeTransform([transforms.ReversePermutation(D)]),
                               RefCond([D], context_encoder=nn.Linear(4, 2 * D))).state_dict().keys()
    assert list(ref_flow_keys)[-2:] == ["_distribution._context_encoder.weight", "_distribution._context_encoder.bias"]
