"""DiagonalNormal and ConditionalDiagonalNormal on the B200 (csrc/fc_diagnormal.cu) against the fp64 oracle: the
log-density with and without logabsdet, parameters read from a strided encoder output, one shared parameter row, all
gradients (encoder weights included), seeded sampling against the reference's composition, determinism of the
reductions, guard bands, and the flows cond_prq_diag_small / maf_diag_small (log_prob, sampling, CUDA graphs, graphed
training steps)."""
import pytest
import torch
from torch import nn

from flowconductor_b200 import _cabi, distributions, graphs, ops, workloads
from tests import diagnormal_oracle as dno
from tests.helpers import assert_parity
from tests.test_gpu_guard import GuardedAllocations

pytestmark = pytest.mark.gpu
DS = [1, 3, 6, 21, 64, 257, 4096]
BS = [1, 129, 4099, 1 << 20]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _params(rows, D, dev, seed, strided):
    """[rows, 2D] parameters; strided: a column slice of a wider encoder output (row stride 2D + 5, base offset 3)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    wide = torch.randn(rows, 2 * D + 5, generator=g, device=dev) * 0.5
    p = wide[:, 3:3 + 2 * D] if strided else wide[:, :2 * D].contiguous()
    return p


def _sizes():
    for D in DS:
        for B in BS:
            if B * D <= (1 << 24):
                yield D, B


@pytest.mark.parametrize("D,B", list(_sizes()))
def test_log_prob_parity(dev, D, B):
    g = torch.Generator(device=dev).manual_seed(D + B)
    x = torch.randn(B, D, generator=g, device=dev) * 1.5
    lad = torch.randn(B, generator=g, device=dev)
    for strided in (False, True):
        params = _params(B, D, dev, 1, strided)
        m, s = params[:, :D], params[:, D:]
        for with_lad in (False, True):
            got = ops.diagnormal_log_prob(x, params, 1, lad if with_lad else None)
            want32 = dno.normal_log_prob(x, m, s).cpu()
            want64 = dno.normal_log_prob(x.double(), m.double(), s.double()).cpu()
            if with_lad:
                want32, want64 = want32 + lad.cpu(), want64 + lad.double().cpu()
            assert_parity(got, want32, want64, 1e-5, 1.0, "D={} B={} strided={} lad={}".format(D, B, strided, with_lad))
    shared = _params(1, D, dev, 2, False)
    got = ops.diagnormal_log_prob(x, shared, B, None)
    want32 = dno.normal_log_prob(x, shared[:, :D], shared[:, D:]).cpu()
    want64 = dno.normal_log_prob(x.double(), shared[:, :D].double(), shared[:, D:].double()).cpu()
    assert_parity(got, want32, want64, 1e-5, 1.0, "shared D={} B={}".format(D, B))


def _check_grad(got, want, what, rtol=2e-4):
    got = got.double().cpu()
    err = (got - want).abs().max().item()
    assert err <= rtol * max(1.0, want.abs().max().item()), (what, err, want.abs().max().item())


@pytest.mark.parametrize("D", DS)
def test_log_prob_gradients_through_encoder(dev, D):
    """ConditionalDiagonalNormal with a linear encoder (G = 1) and DiagonalNormal (G = R): gradients of the inputs, the
    encoder weights / the base parameters and logabsdet against fp64 autograd of the oracle."""
    B = 4099 if D <= 257 else 129
    torch.manual_seed(D)
    enc = nn.Linear(5, 2 * D)
    cond = distributions.ConditionalDiagonalNormal([D], context_encoder=enc).to(dev)
    diag = distributions.DiagonalNormal([D]).to(dev)
    with torch.no_grad():
        enc.weight.mul_(0.5)
        diag.mean_.normal_()
        diag.log_std_.normal_(0.0, 0.3)
    g = torch.Generator().manual_seed(D)
    x0, ctx = torch.randn(B, D, generator=g), torch.randn(B, 5, generator=g)
    lad0, w = torch.randn(B, generator=g), torch.randn(B, generator=g)
    for dist in (cond, diag):
        dist.zero_grad(set_to_none=True)
        x = x0.to(dev).requires_grad_(True)
        lad = lad0.to(dev).requires_grad_(True)
        _cabi.STATS.reset()
        lp = dist.log_prob_plus(x, lad, context=ctx.to(dev))
        (lp * w.to(dev)).sum().backward()
        assert _cabi.STATS.counts.get("fc_diagnormal_log_prob_backward") == 1
        state = {"_distribution." + k: v.detach().double().cpu().requires_grad_(True) for k, v in dist.state_dict().items()}
        x64, lad64 = x0.double().requires_grad_(True), lad0.double().requires_grad_(True)
        kind = "diagonal_normal" if dist is diag else "conditional_diagonal_normal"
        lp64 = dno.base_log_prob(state, {"kind": kind}, x64, ctx.double()) + lad64
        (lp64 * w.double()).sum().backward()
        state32 = {k: v.detach().float() for k, v in state.items()}
        lp32 = dno.base_log_prob(state32, {"kind": kind}, x0, ctx) + lad0
        assert_parity(lp.detach(), lp32, lp64.detach(), 1e-5, 1.0, kind + " D=%d" % D)
        _check_grad(x.grad, x64.grad, "x")
        _check_grad(lad.grad, lad64.grad, "logabsdet")
        for k, p in dist.named_parameters():
            _check_grad(p.grad, state["_distribution." + k].grad, "%s D=%d %s" % (kind, D, k))


@pytest.mark.parametrize("D", [1, 6, 64, 257])
@pytest.mark.parametrize("n", [1, 7, 1024])
def test_sampling_matches_reference_composition(dev, D, n):
    """Seeded samples against the reference's `_sample` (same torch.randn draw, repeat_rows, multiply-add), their
    gradients through the encoder, and sample_and_log_prob."""
    C = 3 if n == 1024 else 129
    torch.manual_seed(n)
    enc = nn.Linear(4, 2 * D).to(dev)
    cond = distributions.ConditionalDiagonalNormal([D], context_encoder=enc)
    ctx = torch.randn(C, 4, device=dev)
    torch.manual_seed(11)
    got = cond.sample(n, ctx)
    torch.manual_seed(11)
    with torch.no_grad():
        m, s = dno.params_from(enc(ctx), D)
    noise = torch.randn(C * n, D, device=dev)
    want32 = dno.sample_from_noise(m, s, noise, n).cpu()
    want64 = dno.sample_from_noise(m.double(), s.double(), noise.double(), n).cpu()
    assert got.shape == (C, n, D)
    assert_parity(got, want32, want64, 1e-5, 1.0, "sample D={} n={}".format(D, n))
    # gradients of a loss on the samples, through the encoder (the noise gets none)
    gy = torch.randn(C, n, D, device=dev)
    enc.zero_grad(set_to_none=True)
    torch.manual_seed(11)
    (cond.sample(n, ctx) * gy).sum().backward()
    w64 = enc.weight.detach().double().requires_grad_(True)
    b64 = enc.bias.detach().double().requires_grad_(True)
    m64, s64 = dno.params_from(torch.nn.functional.linear(ctx.double(), w64, b64), D)
    (dno.sample_from_noise(m64, s64, noise.double(), n) * gy.double()).sum().backward()
    _check_grad(enc.weight.grad, w64.grad.cpu(), "encoder weight")
    _check_grad(enc.bias.grad, b64.grad.cpu(), "encoder bias")
    with torch.no_grad():
        torch.manual_seed(12)
        samples, lp = cond.sample_and_log_prob(n, ctx)
        torch.manual_seed(12)
        assert torch.equal(samples, cond.sample(n, ctx))
        rows = samples.reshape(-1, D)
        reps = torch.repeat_interleave(ctx, n, dim=0)
        want = cond.log_prob(rows, reps).reshape(C, n)
        assert torch.equal(lp, want)
        m, s = dno.params_from(enc(reps).double(), D)
        assert_parity(lp, want, dno.normal_log_prob(rows.double(), m, s).reshape(C, n), 1e-5, 1.0, "sample_and_log_prob")


def test_diagonal_normal_sampling(dev):
    diag = distributions.DiagonalNormal([5]).to(dev)
    with torch.no_grad():
        diag.mean_.normal_()
        diag.log_std_.normal_(0.0, 0.3)
    torch.manual_seed(3)
    got = diag.sample(4099)
    torch.manual_seed(3)
    noise = torch.randn(4099, 5, device=dev)
    with torch.no_grad():
        want = (diag.mean_ + torch.exp(diag.log_std_) * noise).cpu()
        want64 = (diag.mean_.double() + torch.exp(diag.log_std_.double()) * noise.double()).cpu()
    assert got.shape == (4099, 5)
    assert_parity(got.detach(), want, want64, 1e-5, 1.0, "DiagonalNormal.sample")
    assert diag.sample(6, torch.zeros(3, 2, device=dev)).shape == (3, 6, 5)
    (diag.sample(1 << 20) ** 2).sum().backward()  # G = R with a million rows: segment partials and the ordered finish
    assert torch.isfinite(diag.mean_.grad).all() and torch.isfinite(diag.log_std_.grad).all()
    with torch.no_grad():
        empty = diag.log_prob(torch.empty(0, 5, device=dev))
    assert empty.shape == (0,)


@pytest.mark.parametrize("D", [6, 64])
def test_backward_is_deterministic(dev, D):
    R, n = 1 << 20, 1024
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(R, D, generator=g, device=dev)
    gy = torch.randn(R, D, generator=g, device=dev)
    w = torch.randn(R, generator=g, device=dev)
    for group, rows in ((1, R), (n, R // n), (R, 1)):
        params = torch.randn(rows, 2 * D, generator=g, device=dev) * 0.3
        a = ops.diagnormal_log_prob_backward(x, params, group, w)
        b = ops.diagnormal_log_prob_backward(x, params, group, w)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), group
        a = ops.diagnormal_sample_backward(x, params, group, gy)
        b = ops.diagnormal_sample_backward(x, params, group, gy)
        assert torch.equal(a, b), group
        if group > 1:  # the group sums against fp64
            want = gy.double().reshape(rows, group, D).sum(1)
            _check_grad(a[:, :D], want.cpu(), "sample grad_mean G=%d" % group, rtol=1e-4)


@pytest.mark.parametrize("rows", [1, 129, 641])
@pytest.mark.parametrize("D", [3, 64])
def test_guard_bands(dev, rows, D):
    x = torch.randn(rows, D, device=dev)
    w, gy = torch.randn(rows, device=dev), torch.randn(rows, D, device=dev)
    for group in (1, 7, 64, rows):
        P = -(-rows // group)
        params = torch.randn(P, 2 * D, device=dev) * 0.3
        with GuardedAllocations() as g:
            lp = ops.diagnormal_log_prob(x, params, group, w)
            gx, gp = ops.diagnormal_log_prob_backward(x, params, group, w)
            y = ops.diagnormal_sample(x, params, group)
            gps = ops.diagnormal_sample_backward(x, params, group, gy)
        g.check("diagnormal D=%d rows=%d group=%d" % (D, rows, group))
        rep = torch.arange(rows, device=dev) // group
        m, s = params[rep, :D], params[rep, D:]
        assert torch.allclose(lp, dno.normal_log_prob(x, m, s) + w, rtol=1e-5, atol=1e-4)
        assert torch.allclose(y, m + torch.exp(s) * x, rtol=1e-5, atol=1e-5)
        want = torch.zeros(P, D, device=dev).index_add_(0, rep, gy)
        assert torch.allclose(gps[:, :D], want, rtol=1e-4, atol=1e-4) and torch.isfinite(gp).all()
        assert torch.allclose(gx, -w[:, None] * (x - m) * torch.exp(-2 * s), rtol=1e-4, atol=1e-5)


def _flow(name, dev, seed=0):
    wl = workloads.get_workload(name)
    flow = workloads.build_flow(wl, seed=seed)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    flow.load_state_dict(state)
    return wl, flow.to(dev).eval(), state


FLOWS = ["cond_prq_diag_small", "maf_diag_small"]


def _context(wl, rows, seed):
    if wl["context_features"] is None:
        return None
    return torch.randn(rows, wl["context_features"], generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("name", FLOWS)
def test_flow_log_prob_and_sampling(dev, name):
    wl, flow, state = _flow(name, dev)
    specs, base = workloads.oracle_specs(wl), wl["base"]
    s64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    x = torch.randn(4099, 6, generator=torch.Generator().manual_seed(5))
    ctx = _context(wl, 4099, 6)
    _cabi.STATS.reset()
    with torch.no_grad():
        lp = flow.log_prob(x.to(dev), None if ctx is None else ctx.to(dev))
    assert _cabi.STATS.counts.get("fc_diagnormal_log_prob") == 1
    want32 = dno.flow_log_prob(state, specs, base, x, ctx)
    want64 = dno.flow_log_prob(s64, specs, base, x.double(), None if ctx is None else ctx.double())
    assert_parity(lp, want32, want64, 1e-5, 1.0, name + " log_prob")
    C, n = (7, 300) if ctx is not None else (None, 2048)
    c = None if ctx is None else _context(wl, C, 8).to(dev)
    with torch.no_grad():
        torch.manual_seed(7)
        got, got_lp = flow.sample_and_log_prob(n, c)
        torch.manual_seed(7)
        rows = n if c is None else C * n
        noise = torch.randn(rows, 6, device=dev)
        m, s = dno.base_params({k: v.to(dev) for k, v in state.items()}, base, 6, c, torch.float32)
        m64, s64b = dno.base_params({k: v.to(dev) for k, v in s64.items()}, base, 6, c, torch.float64)
        bs = dno.sample_from_noise(m, s, noise, n if c is not None else rows).reshape(rows, 6).cpu()
        bs64 = dno.sample_from_noise(m64, s64b, noise.double(), n if c is not None else rows).reshape(rows, 6).cpu()
        reps = None if c is None else torch.repeat_interleave(c, n, dim=0).cpu()
        want = dno.flow_sample_from_noise(state, specs, bs, reps)
        want64 = dno.flow_sample_from_noise(s64, specs, bs64, None if reps is None else reps.double())
        assert_parity(got.reshape(rows, 6), want, want64, 1e-5, 1.0, name + " samples", max_ratio=1e3)
        tame = got.reshape(rows, 6).abs().amax(1) < 20
        assert int(tame.sum()) >= 10
        lp_of = flow.log_prob(got.reshape(rows, 6)[tame], None if reps is None else reps.to(dev)[tame])
        assert torch.allclose(got_lp.reshape(rows)[tame], lp_of, rtol=1e-4, atol=1e-3)
        torch.manual_seed(7)
        assert torch.equal(flow.sample(n, c), got)


@pytest.mark.parametrize("name", FLOWS)
def test_capture_sampler_replays(dev, name):
    wl, flow, _ = _flow(name, dev)
    c = None if wl["context_features"] is None else _context(wl, 5, 9).to(dev)
    s = graphs.capture_sampler(flow, 64, c)
    a = (s(c) if c is not None else s()).clone()
    b = s(c) if c is not None else s()
    assert a.shape == ((5, 64, 6) if c is not None else (64, 6)) and torch.isfinite(a).all()
    assert not torch.equal(a, b) and s.records == 1  # fresh noise on every replay
    sl = graphs.capture_sampler(flow, 64, c, with_log_prob=True)
    out = sl(c) if c is not None else sl()
    assert torch.isfinite(out[1]).all()


@pytest.mark.parametrize("name", FLOWS)
def test_graphed_training_step_matches_eager(dev, name):
    wl = workloads.get_workload(name)
    flows_ = [workloads.build_flow(wl, seed=2) for _ in range(2)]
    state = workloads.trained_like_({k: v.clone() for k, v in flows_[0].state_dict().items()}, wl)
    for f in flows_:
        f.load_state_dict(state)
    flows_ = [f.to(dev).train() for f in flows_]
    opts = [torch.optim.Adam(f.parameters(), lr=1e-3, capturable=True) for f in flows_]
    g = torch.Generator().manual_seed(8)
    batches = [torch.randn(4099, 6, generator=g).to(dev) for _ in range(3)]
    ctxs = [None if wl["context_features"] is None else _context(wl, 4099, 20 + i).to(dev) for i in range(3)]

    def loss_of(f):
        return (lambda x: -f.log_prob(x).mean()) if ctxs[0] is None else (lambda x, c: -f.log_prob(x, c).mean())

    example = (batches[0],) if ctxs[0] is None else (batches[0], ctxs[0])
    stepper = graphs.GraphedTrainStep(flows_[1], opts[1], loss_of(flows_[1]), *example)
    for x, c in zip(batches, ctxs):
        opts[0].zero_grad(set_to_none=True)
        loss = loss_of(flows_[0])(*((x,) if c is None else (x, c)))
        loss.backward()
        opts[0].step()
        assert loss.item() == stepper.step(*((x,) if c is None else (x, c))).item()
    for k, v in flows_[0].state_dict().items():
        assert torch.equal(v, flows_[1].state_dict()[k]), k
    for k, v in flows_[0].state_dict().items():  # the base was trained
        if k.startswith("_distribution."):
            assert not torch.equal(v.cpu(), state[k]), k
