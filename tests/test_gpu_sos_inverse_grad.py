"""Gradients through the numerical sum-of-sigmoids inverse (ops.sos_layer_inverse_backward -> fc_sos_inverse_backward):
the op against autograd through the reference's inverse (bisection + two Newton steps with create_graph), the tile ring
against the general-strides kernel, identities of forward o inverse at full size, the layers and flows that end in the
op (SumOfSigmoids, MaskedSumOfSigmoidsTransform, ConditionalSumOfSigmoidsTransform, Flow.sample_and_log_prob), CUDA
graph capture of a reverse-KL training step, guard bands, and a short reverse-KL fit."""
import math

import pytest
import torch

from flowconductor_b200 import _cabi, flows, graphs, ops, transforms, workloads
from flowconductor_b200.distributions.normal import StandardNormal
from oracle import restated
from tests.helpers import assert_parity, golden_state, load_golden
from tests.test_gpu_guard import GuardedAllocations
from tests.test_gpu_tile_ring import STAGED, TILE_RING, _env

pytestmark = pytest.mark.gpu
GRAD_TOL = 1e-4
INV_GRAD_TOL = 1e-3  # numerical and D-pass inverses (the rule of test_gpu_parity.test_flow_matches_reference)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _inputs(B, D, n, seed, big=False):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, D, generator=g) * 3
    if big:  # adaptive_sigmoid_test.py:64-79: |x| up to ~200
        z[: B // 4] = (torch.rand(B // 4, D, generator=g) * 2 - 1) * 200
    p = torch.randn(B, D * (3 * n + 1), generator=g)
    gy = torch.randn(B, D, generator=g)
    gl = torch.randn(B, generator=g)
    return z, p, gy, gl


def _oracle_grads(z, p, n, offset, gy, gl, dtype):
    z = z.to(dtype).requires_grad_(True)
    p = p.to(dtype).requires_grad_(True)
    x, lad = restated.sos_inverse(z, p, n, offset=offset)
    loss = (gy.to(dtype) * x).sum() + ((gl.to(dtype) * lad).sum() if gl is not None else 0)
    return torch.autograd.grad(loss, [z, p])


@pytest.mark.parametrize("with_lad", [True, False])
@pytest.mark.parametrize("offset", [0.0, -0.5])
@pytest.mark.parametrize("n", [10, 3, 30, 64])
def test_inverse_gradients_match_the_reference_inverse(dev, n, offset, with_lad):
    B, D = 64, 5
    z, p, gy, gl = _inputs(B, D, n, seed=n * 7 + int(with_lad), big=True)
    gl = gl if with_lad else None
    zd = z.to(dev).requires_grad_(True)
    pd = p.to(dev).requires_grad_(True)
    x, lad = ops.sos_layer(zd, pd, n, offset, True, 50, 120.0)
    loss = (gy.to(dev) * x).sum() + ((gl.to(dev) * lad).sum() if gl is not None else 0)
    gz, gp = torch.autograd.grad(loss, [zd, pd])
    r32 = _oracle_grads(z, p, n, offset, gy, gl, torch.float32)
    r64 = _oracle_grads(z, p, n, offset, gy, gl, torch.float64)
    what = "n=%d offset=%g lad=%s" % (n, offset, with_lad)
    assert_parity(gz, r32[0], r64[0], GRAD_TOL, max(1e-2, r64[0].abs().mean().item()), what + " grad z")
    assert_parity(gp, r32[1], r64[1], GRAD_TOL, max(1e-2, r64[1].abs().mean().item()), what + " grad params")


@pytest.mark.parametrize("n", [10, 3])
@pytest.mark.parametrize("D", [16, 21, 64])
@pytest.mark.parametrize("B", [1, 37, 4099])
def test_inverse_adjoint_tile_ring_matches_the_general_kernel_bit_for_bit(dev, B, D, n):
    lib = _cabi.lib()
    g = torch.Generator(device=dev).manual_seed(B * 131 + D + n)
    x = torch.randn(B, D, generator=g, device=dev)
    p = torch.randn(B, D * (3 * n + 1), generator=g, device=dev)
    gy, gl = torch.randn(B, D, generator=g, device=dev), torch.randn(B, generator=g, device=dev)
    try:
        for lad in (gl, None):
            _env()
            got = ops.sos_layer_inverse_backward(x, p, gy, lad, n)
            assert lib.fc_elementwise_last_path() == TILE_RING
            _env(FC_TILE=0, FC_PIPE=0)
            want = ops.sos_layer_inverse_backward(x, p, gy, lad, n)
            assert lib.fc_elementwise_last_path() == STAGED
            for u, v in zip(got, want):
                assert torch.equal(u, v), (B, D, n, lad is None)
    finally:
        _env()


def _split_terms(x, p, n, gy_f, gl_f, gl_i):
    """The separate adjoint terms of y = forward(inverse(z)): the forward adjoint at x, and the inverse adjoint fed with
    its x-gradient (and with the inverse log-det gradient gl_i on its own)."""
    gx_f, gp_f = ops.sos_layer_backward(x, p, gy_f, gl_f, n)
    gz_y, gp_y = ops.sos_layer_inverse_backward(x, p, gx_f, None, n)
    if gl_i is None:
        return gz_y.abs(), gp_f.abs() + gp_y.abs()
    gz_l, gp_l = ops.sos_layer_inverse_backward(x, p, torch.zeros_like(x), gl_i, n)
    return gz_y.abs() + gz_l.abs(), gp_f.abs() + gp_y.abs() + gp_l.abs()


def _cancelled(total, scale):
    ok = total.abs() <= GRAD_TOL * (scale + scale.mean())
    return bool(ok.all()), float((total.abs() / (scale + scale.mean())).max())


def test_forward_of_inverse_is_the_identity_at_full_size(dev):
    """cfg 4 shapes (262 144 x 32, n = 10), through the inverse and the forward kernel under autograd:
    y = forward(inverse(z)) = z gives d<g, y>/dz = g and no parameter gradient; lad_fwd(x) + lad_inv(z) = 0 gives no
    gradient at all.  The residuals are judged against the size of the terms that cancel, with their mean as a floor: a
    softmax-weight gradient p_j (g_j - sum_k p_k g_k) is itself a difference, rounded relative to its parts."""
    B, D, n = 262144, 32, 10
    g0 = torch.Generator(device=dev).manual_seed(4)
    z = (torch.randn(B, D, generator=g0, device=dev) * 3).requires_grad_(True)
    p = torch.randn(B, D * (3 * n + 1), generator=g0, device=dev).requires_grad_(True)
    g = torch.randn(B, D, generator=g0, device=dev)
    x, lad_i = ops.sos_layer(z, p, n, 0.0, True, 50, 120.0)
    y, lad_f = ops.sos_layer(x, p, n, 0.0, False, 50, 120.0)
    gz, gp = torch.autograd.grad((g * y).sum(), [z, p], retain_graph=True)
    with torch.no_grad():
        sz, sp = _split_terms(x.detach(), p.detach(), n, g, None, None)
        assert ((gz - g).abs() <= 1e-5 * g.abs() + 1e-30).all()
        assert torch.allclose(sz, g.abs(), rtol=1e-5, atol=0)
        ok, worst = _cancelled(gp, sp)
        assert ok, worst
    gz, gp = torch.autograd.grad((lad_f + lad_i).sum(), [z, p])
    with torch.no_grad():
        ones = torch.ones(B, device=dev)
        sz, sp = _split_terms(x.detach(), p.detach(), n, torch.zeros_like(g), ones, ones)
        for total, scale in ((gz, sz), (gp, sp)):
            ok, worst = _cancelled(total, scale)
            assert ok, worst


def _scaled_parity(ours, r32, r64, what):
    scale = max(1e-6, r64.abs().max().item())
    assert_parity(ours / scale, r32 / scale, r64 / scale, INV_GRAD_TOL, 1.0, what)


def test_sum_of_sigmoids_module_parameter_gradients(dev):
    torch.manual_seed(11)
    F, n, B = 5, 10, 96
    t = transforms.SumOfSigmoids(features=F, n_sigmoids=n)
    with torch.no_grad():
        t.log_scale_preact.normal_()
        t.raw_softmax.normal_()
        t.extended_softplus.shift.normal_()
    t = t.to(dev)
    g = torch.Generator().manual_seed(12)
    z = torch.randn(B, F, generator=g) * 3
    gy, gl = torch.randn(B, F, generator=g), torch.randn(B, generator=g)
    names = ["shift_preact", "log_scale_preact", "raw_softmax", "extended_softplus.shift"]
    params = dict(t.named_parameters())
    zd = z.to(dev).requires_grad_(True)
    x, lad = t.inverse(zd)
    ours = torch.autograd.grad((gy.to(dev) * x).sum() + (gl.to(dev) * lad).sum(), [zd] + [params[k] for k in names])
    refs = []
    for dtype in (torch.float32, torch.float64):
        leaves = [params[k].detach().cpu().to(dtype).requires_grad_(True) for k in names]
        raw = torch.cat(leaves[:3] + [leaves[3].reshape(1, F, 1)], dim=-1).expand(B, -1, -1).reshape(B, -1)
        zr = z.to(dtype).requires_grad_(True)
        xr, ladr = restated.sos_inverse(zr, raw, n)
        refs.append(torch.autograd.grad((gy.to(dtype) * xr).sum() + (gl.to(dtype) * ladr).sum(), [zr] + leaves))
    for i, what in enumerate(["inputs"] + names):
        _scaled_parity(ours[i], refs[0][i], refs[1][i], "SumOfSigmoids grad " + what)


def _load(name, dev):
    gold = load_golden(name)
    wl = workloads.get_workload(name)
    flow = workloads.build_flow(wl)
    flow.load_state_dict(golden_state(gold), strict=True)
    return gold, wl, flow.to(dev)


def _oracle_state(gold, names, dtype):
    state = golden_state(gold, dtype)
    for k in names:
        state[k] = state[k].requires_grad_(True)
    return state


@pytest.mark.parametrize("name", ["maf_sos_small", "cfg4_small"])
def test_golden_models_inverse_vjp(dev, name):
    """VJP of (inverse outputs, inverse logabsdet) with random cotangents at the golden noise / context."""
    gold, wl, flow = _load(name, dev)
    specs = workloads.oracle_specs(wl)
    noise = gold["noise"]
    ctx = gold["context"] if "context" in gold else None
    g = torch.Generator().manual_seed(3)
    gy, gl = torch.randn(noise.shape, generator=g), torch.randn(noise.shape[0], generator=g)
    named = [(k, v) for k, v in flow.named_parameters() if v.requires_grad]
    names = [k for k, _ in named]

    inputs = [noise.to(dev).requires_grad_(True)] + ([ctx.to(dev).requires_grad_(True)] if ctx is not None else [])
    x, lad = flow._transform.inverse(inputs[0], context=inputs[1] if ctx is not None else None)
    ours = torch.autograd.grad((gy.to(dev) * x).sum() + (gl.to(dev) * lad).sum(), inputs + [v for _, v in named])
    refs = []
    for dtype in (torch.float32, torch.float64):
        state = _oracle_state(gold, names, dtype)
        rin = [noise.to(dtype).requires_grad_(True)] + ([ctx.to(dtype).requires_grad_(True)] if ctx is not None else [])
        xr, ladr = restated.composite(state, specs, rin[0], rin[1] if ctx is not None else None, inverse=True)
        refs.append(torch.autograd.grad((gy.to(dtype) * xr).sum() + (gl.to(dtype) * ladr).sum(),
                                        rin + [state[k] for k in names]))
    labels = ["noise"] + (["context"] if ctx is not None else []) + names
    for i, what in enumerate(labels):
        _scaled_parity(ours[i], refs[0][i], refs[1][i], name + " grad " + what)


def _target_log_prob(x, mean, prec_chol):
    """log N(x; mean, cov) with cov^-1 = L L^T (a fixed correlated Gaussian)."""
    u = (x - mean) @ prec_chol
    d = x.shape[-1]
    return -0.5 * (u ** 2).sum(-1) - 0.5 * d * math.log(2 * math.pi) + torch.log(torch.diagonal(prec_chol)).sum()


def _gaussian(d, rho, dtype=torch.float32, device=None):
    cov = torch.full((d, d), rho, dtype=torch.float64) + (1 - rho) * torch.eye(d, dtype=torch.float64)
    mean = torch.linspace(-0.5, 0.5, d, dtype=torch.float64)
    prec_chol = torch.linalg.cholesky(torch.linalg.inv(cov))
    return mean.to(dtype=dtype, device=device), prec_chol.to(dtype=dtype, device=device)


@pytest.mark.parametrize("name", ["maf_sos_small", "cfg4_small"])
def test_reverse_kl_through_sample_and_log_prob(dev, name):
    """(log q(x) - log p(x)).mean() with x, log q(x) from Flow.sample_and_log_prob; gradients against the reference
    algorithm on the same noise."""
    gold, wl, flow = _load(name, dev)
    specs = workloads.oracle_specs(wl)
    D = wl["features"]
    ctx = gold["context"][:8] if "context" in gold else None
    num = 64 if ctx is None else 8
    named = [(k, v) for k, v in flow.named_parameters() if v.requires_grad]
    names = [k for k, _ in named]
    mean, L = _gaussian(D, 0.6, device=dev)
    torch.manual_seed(21)
    x, lq = flow.sample_and_log_prob(num, context=ctx.to(dev) if ctx is not None else None)
    loss = (lq - _target_log_prob(x, mean, L)).mean()
    loss.backward()
    ours = [v.grad if v.grad is not None else torch.zeros_like(v) for _, v in named]
    assert all(torch.isfinite(gv).all() for gv in ours)
    torch.manual_seed(21)
    noise = flow._distribution.sample(num, context=ctx.to(dev) if ctx is not None else None).reshape(-1, D).cpu()
    crep = ctx.repeat_interleave(num, dim=0) if ctx is not None else None
    refs = []
    for dtype in (torch.float32, torch.float64):
        state = _oracle_state(gold, names, dtype)
        xr, ladr = restated.composite(state, specs, noise.to(dtype), crep.to(dtype) if ctx is not None else None,
                                      inverse=True)
        lqr = restated.standard_normal_log_prob(noise.to(dtype)) - ladr
        m, Lr = _gaussian(D, 0.6, dtype)
        loss_r = (lqr - _target_log_prob(xr, m, Lr)).mean()
        refs.append(torch.autograd.grad(loss_r, [state[k] for k in names], allow_unused=True))
    assert abs(loss.item() - float(loss_r)) <= 1e-3 * max(1.0, abs(float(loss_r)))
    for i, k in enumerate(names):
        r32 = refs[0][i] if refs[0][i] is not None else torch.zeros_like(refs[1][i])
        r64 = refs[1][i] if refs[1][i] is not None else torch.zeros(ours[i].shape, dtype=torch.float64)
        _scaled_parity(ours[i], r32, r64, name + " reverse-KL grad " + k)


def test_cuda_graph_reverse_kl_step_matches_eager(dev):
    """graphs.GraphedTrainStep over a reverse-KL step of a conditional sum-of-sigmoids flow (noise and context are the
    static inputs): three replays leave exactly the parameters three eager steps leave, so the path is capturable (no host
    synchronisation) and deterministic."""
    wl = workloads.get_workload("cfg4_small")
    D = wl["features"]
    fl = [workloads.build_flow(wl, seed=5).to(dev) for _ in range(2)]
    fl[1].load_state_dict(fl[0].state_dict())
    opts = [torch.optim.Adam(f.parameters(), lr=1e-3, capturable=True) for f in fl]
    mean, L = _gaussian(D, 0.6, device=dev)

    def loss_fn(flow):
        def f(noise, ctx):
            x, lad = flow._transform.inverse(noise, context=ctx)
            lq = flow._distribution.log_prob(noise) - lad
            return (lq - _target_log_prob(x, mean, L)).mean()
        return f

    g = torch.Generator().manual_seed(9)
    batches = [(torch.randn(256, D, generator=g).to(dev), torch.randn(256, wl["context_features"], generator=g).to(dev))
               for _ in range(3)]
    stepper = graphs.GraphedTrainStep(fl[1], opts[1], loss_fn(fl[1]), *batches[0])
    for noise, ctx in batches:
        opts[0].zero_grad(set_to_none=True)
        loss = loss_fn(fl[0])(noise, ctx)
        loss.backward()
        opts[0].step()
        assert loss.item() == stepper.step(noise, ctx).item()
    for pe, pg in zip(fl[0].parameters(), fl[1].parameters()):
        assert torch.equal(pe, pg)


def test_outputs_under_autograd_are_unchanged(dev):
    g = torch.Generator(device=dev).manual_seed(2)
    for n, offset in ((10, 0.0), (3, -0.5)):
        z = torch.randn(4099, 21, generator=g, device=dev) * 3
        p = torch.randn(4099, 21 * (3 * n + 1), generator=g, device=dev)
        with torch.no_grad():
            want = ops.sos_layer(z, p, n, offset, True, 50, 120.0)
        got = ops.sos_layer(z.requires_grad_(True), p.requires_grad_(True), n, offset, True, 50, 120.0)
        assert got[0].requires_grad
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    t = transforms.SumOfSigmoids(features=7, n_sigmoids=10).to(dev)
    z = torch.randn(300, 7, generator=g, device=dev)
    with torch.no_grad():
        want = t.inverse(z)
    got = t.inverse(z)
    assert got[0].requires_grad and torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


@pytest.mark.parametrize("rows", [1, 37, 1500, 4099])
@pytest.mark.parametrize("D,n", [(21, 10), (64, 3)])
def test_inverse_adjoint_stays_inside_its_buffers(dev, rows, D, n):
    g0 = torch.Generator(device=dev).manual_seed(rows + D)
    x = torch.randn(rows, D, generator=g0, device=dev)
    p = torch.randn(rows, D * (3 * n + 1), generator=g0, device=dev)
    gy, gl = torch.randn(rows, D, generator=g0, device=dev), torch.randn(rows, generator=g0, device=dev)
    with torch.no_grad(), GuardedAllocations() as g:
        gz, gp = ops.sos_layer_inverse_backward(x, p, gy, gl, n)
        assert _cabi.lib().fc_elementwise_last_path() == TILE_RING
    g.check("sum-of-sigmoids inverse adjoint rows=%d D=%d n=%d" % (rows, D, n))
    assert torch.isfinite(gz).all() and torch.isfinite(gp).all()


def test_reverse_kl_training_halves_the_kl(dev):
    """A 2-D MAF of sum-of-sigmoids layers fitted by sampling (reverse KL) to a fixed correlated Gaussian."""
    torch.manual_seed(0)
    D = 2
    flow = flows.Flow(transforms.CompositeTransform([
        transforms.MaskedSumOfSigmoidsTransform(D, 32, n_sigmoids=10),
        transforms.ReversePermutation(D),
        transforms.MaskedSumOfSigmoidsTransform(D, 32, n_sigmoids=10)]), StandardNormal([D])).to(dev)
    mean, L = _gaussian(D, 0.8, device=dev)
    opt = torch.optim.Adam(flow.parameters(), lr=3e-3)
    fixed = torch.randn(8192, D, generator=torch.Generator().manual_seed(1)).to(dev)

    def kl_estimate():
        with torch.no_grad():
            x, lad = flow._transform.inverse(fixed)
            return float((flow._distribution.log_prob(fixed) - lad - _target_log_prob(x, mean, L)).mean())

    kl0 = kl_estimate()
    for _ in range(200):
        opt.zero_grad(set_to_none=True)
        x, lq = flow.sample_and_log_prob(1024)
        loss = (lq - _target_log_prob(x, mean, L)).mean()
        loss.backward()
        opt.step()
    kl1 = kl_estimate()
    assert math.isfinite(kl1) and kl1 <= 0.5 * kl0, (kl0, kl1)
