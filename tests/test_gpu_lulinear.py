"""LULinear on the B200: fc_lulinear (D < 64) and the tensor-core GEMM (D >= 64) against the fp64 oracle, the layer's
identities, gradients in both directions, determinism, flows with LU layers (graphs included), guard bands, and the
reference's state_dict where the reference tree is available."""
import pytest
import torch

from flowconductor_b200 import _cabi, graphs, ops, transforms, workloads
from oracle import locate, restated
from tests import lu_oracle
from tests.helpers import assert_parity
from tests.test_gpu_guard import GuardedAllocations

pytestmark = pytest.mark.gpu
KERNEL_D = [1, 2, 3, 7, 16, 33, 63]
TC_D = [64, 65, 128, 256]
SPEC = {"kind": "lu_linear", "prefix": ""}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def make_layer(D, init, seed=0):
    torch.manual_seed(seed)
    layer = transforms.LULinear(D, identity_init=(init == "identity"))
    if init == "trained":  # every entry non-zero, the bias too, at the non-identity init scale
        with torch.no_grad():
            for p in layer.parameters():
                p.uniform_(-D ** -0.5, D ** -0.5)
    return layer


def oracle(layer, x, inverse):
    """(fp32, fp64) oracle outputs on the device of x."""
    s32 = {k: v.detach().to(x.device) for k, v in layer.state_dict().items()}
    s64 = {k: v.double() for k, v in s32.items()}
    with torch.no_grad():
        return (lu_oracle.apply_layer(s32, SPEC, x, inverse=inverse),
                lu_oracle.apply_layer(s64, SPEC, x.double(), inverse=inverse))


def inputs(B, D, dev, strided, seed=1):
    g = torch.Generator().manual_seed(seed)
    if strided:  # a column slice of a wider tensor: row stride D + 5, base offset 3 floats (not 16-byte aligned)
        return torch.randn(B, D + 5, generator=g).to(dev)[:, 3:3 + D]
    return torch.randn(B, D, generator=g).to(dev)


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("init", ["identity", "random", "trained"])
@pytest.mark.parametrize("D", KERNEL_D + TC_D)
def test_parity(dev, D, init, inverse):
    layer = make_layer(D, init).to(dev)
    for B in (1, 129, 4099):
        for strided in (False, True):
            x = inputs(B, D, dev, strided)
            _cabi.STATS.reset()
            with torch.no_grad():
                y, lad = layer.inverse(x) if inverse else layer(x)
            assert _cabi.STATS.counts.get("fc_lulinear_apply", 0) == (1 if D < 64 else 0)
            (r32, l32), (r64, l64) = oracle(layer, x, inverse)
            what = "D={} {} inverse={} B={} strided={}".format(D, init, inverse, B, strided)
            assert_parity(y, r32, r64, 1e-5, 1.0, what)
            assert_parity(lad, l32, l64, 1e-5, 1.0, what + " logabsdet")


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("D", [16, 63, 128])
def test_parity_million_rows(dev, D, inverse):
    """1 M rows (thousands of tiles per CTA ring), strided input; fp32 / fp64 oracle on the GPU."""
    layer = make_layer(D, "trained").to(dev)
    x = inputs(1 << 20, D, dev, strided=True)
    with torch.no_grad():
        y, lad = layer.inverse(x) if inverse else layer(x)
    (r32, l32), (r64, l64) = oracle(layer, x, inverse)
    err = (y.double() - r64).abs().max().item()
    noise = (r32.double() - r64).abs().max().item()
    assert err <= 10 * noise + 1e-5, (err, noise)
    rows = torch.arange(0, 1 << 20, 61, device=dev)
    assert_parity(y[rows], r32[rows], r64[rows], 1e-5, 1.0, "1M rows D={} inverse={}".format(D, inverse))
    assert (lad == lad[0]).all() and abs(lad[0].item() - l64[0].item()) <= 1e-5 * max(1.0, abs(l64[0].item()))


@pytest.mark.parametrize("D", [2, 7, 33, 63, 128])
def test_identities(dev, D):
    layer = make_layer(D, "trained", seed=D).to(dev)
    x = inputs(4099, D, dev, strided=False)
    with torch.no_grad():
        y, lad = layer(x)
        xr, lad_inv = layer.inverse(y)
        W64 = layer.weight().double()
        wi, ld = layer.weight_inverse().double(), layer.logabsdet().double()
    sign, logdet = torch.linalg.slogdet(W64)
    assert sign.item() == 1.0
    assert (xr - x).abs().max().item() <= 1e-4 * max(1.0, x.abs().max().item())
    assert (lad.double() - logdet).abs().max().item() <= 1e-5 * max(1.0, abs(logdet.item()))
    assert (lad_inv.double() + logdet).abs().max().item() <= 1e-5 * max(1.0, abs(logdet.item()))
    s64 = {k: v.detach().double().cpu() for k, v in layer.state_dict().items()}
    eye = torch.eye(D, dtype=torch.float64)
    W_ref, _ = lu_oracle.apply_layer(s64, SPEC, eye)  # rows: W e_i + bias
    W_ref = (W_ref - s64["bias"]).t()
    assert torch.allclose(W64.cpu(), W_ref, atol=1e-6)
    assert torch.allclose(wi.cpu(), torch.linalg.inv(W_ref), atol=1e-5 * max(1.0, torch.linalg.inv(W_ref).abs().max().item()))
    assert abs(ld.item() - logdet.item()) <= 1e-5 * max(1.0, abs(logdet.item()))


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("D", [1, 3, 16, 33, 63, 64])
def test_gradients(dev, D, inverse):
    """Gradients of the input and of all four parameters against fp64 autograd through the restated oracle."""
    layer = make_layer(D, "trained", seed=3).to(dev)
    g = torch.Generator().manual_seed(4)
    x0 = torch.randn(4099, D, generator=g)
    wy = torch.randn(4099, D, generator=g)
    wl = torch.randn(4099, generator=g)
    x = x0.to(dev).requires_grad_(True)
    _cabi.STATS.reset()
    y, lad = layer.inverse(x) if inverse else layer(x)
    ((y * wy.to(dev)).sum() + (lad * wl.to(dev)).sum()).backward()
    if D < 64:
        assert _cabi.STATS.counts.get("fc_lulinear_backward", 0) >= 1
    s64 = {k: v.detach().double().cpu().requires_grad_(True) for k, v in layer.state_dict().items()}
    x64 = x0.double().requires_grad_(True)
    y64, lad64 = lu_oracle.apply_layer(s64, SPEC, x64, inverse=inverse)
    ((y64 * wy.double()).sum() + (lad64 * wl.double()).sum()).backward()
    named = dict(layer.named_parameters())
    for name, got, want in [("x", x.grad, x64.grad)] + [(k, named[k].grad, s64[k].grad) for k in s64]:
        if want.numel() == 0:
            continue
        err = (got.double().cpu() - want).abs().max().item()
        assert err <= 2e-4 * max(1.0, want.abs().max().item()), (name, err, want.abs().max().item())


def test_backward_is_deterministic(dev):
    x = torch.randn(1 << 18, 33, device=dev)
    gy = torch.randn(1 << 18, 33, device=dev)
    M = torch.randn(33, 33, device=dev)
    a = ops.lulinear_layer_backward(x, M, gy)
    b = ops.lulinear_layer_backward(x, M, gy)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert torch.allclose(a[1], gy.t() @ x, rtol=1e-4, atol=1e-2) and torch.allclose(a[2], gy.sum(0), atol=1e-2)


def test_kernel_requires_fp32(dev):
    M, c, ld = torch.eye(4, device=dev), torch.zeros(4, device=dev), torch.zeros((), device=dev)
    with pytest.raises(RuntimeError, match="float32"):
        ops.lulinear_layer(torch.randn(3, 4, device=dev, dtype=torch.float64), M, c, ld)
    with pytest.raises(RuntimeError, match="float32"):
        transforms.LULinear(4).to(dev)(torch.randn(3, 4, device=dev, dtype=torch.float16))


def _nsf_small(dev):
    wl = workloads.get_workload("nsf_lu_small")
    flow = workloads.build_flow(wl)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    flow.load_state_dict(state)
    return wl, flow.to(dev), state


def test_flow_log_prob_and_sampling(dev):
    wl, flow, state = _nsf_small(dev)
    specs = workloads.oracle_specs(wl)
    s64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    x = torch.randn(4099, 6, generator=torch.Generator().manual_seed(5))
    with torch.no_grad():
        lp = flow.log_prob(x.to(dev))
        z = torch.randn(4099, 6, generator=torch.Generator().manual_seed(6))
        samples, _ = flow._transform.inverse(z.to(dev))
        want32, want64 = lu_oracle.flow_log_prob(state, specs, x), lu_oracle.flow_log_prob(s64, specs, x.double())
        assert_parity(lp, want32, want64, 1e-5, 1.0, "nsf_lu_small log_prob")
        s32 = lu_oracle.flow_sample_from_noise(state, specs, z)
        s64_ = lu_oracle.flow_sample_from_noise(s64, specs, z.double())
        assert_parity(samples, s32, s64_, 1e-5, 1.0, "nsf_lu_small sample")
        # the same base draw through the oracle: samples and log N(z) - logabsdet of the inverse cascade
        torch.manual_seed(7)
        got, got_lp = flow.sample_and_log_prob(2048)
        torch.manual_seed(7)
        noise = torch.randn(2048, 6, device=dev).cpu()
        want = []
        for st, zz in ((state, noise), (s64, noise.double())):
            smp, lad = lu_oracle.composite(st, specs, zz, inverse=True)
            want.append((smp, restated.standard_normal_log_prob(zz) - lad))
        assert_parity(got, want[0][0], want[1][0], 1e-5, 1.0, "nsf_lu_small sample_and_log_prob samples")
        assert_parity(got_lp, want[0][1], want[1][1], 1e-5, 1.0, "nsf_lu_small sample_and_log_prob log_prob")
        torch.manual_seed(7)
        assert torch.equal(flow.sample(2048), got)


def test_inverse_transform(dev):
    layer = make_layer(9, "trained").to(dev)
    inv = transforms.InverseTransform(layer)
    x = torch.randn(300, 9, device=dev)
    with torch.no_grad():
        a, la = inv(x)
        b, lb = layer.inverse(x)
        c, lc = inv.inverse(x)
        d, ld = layer(x)
    assert torch.equal(a, b) and torch.equal(la, lb) and torch.equal(c, d) and torch.equal(lc, ld)


def test_graph_capture_follows_parameter_updates(dev):
    _, flow, _ = _nsf_small(dev)
    flow.eval()
    x = torch.randn(512, 6, device=dev)
    g = graphs.capture(flow.log_prob, x)
    with torch.no_grad():
        assert torch.equal(g(x), flow.log_prob(x))
        for name, p in flow.named_parameters():
            if "lower_entries" in name or "unconstrained_upper_diag" in name or name.endswith("1.bias"):
                p.add_(0.05)
        eager = flow.log_prob(x)
    assert torch.equal(g(x), eager) and g.records == 2


def test_graphed_training_step_matches_eager(dev):
    wl = workloads.get_workload("nsf_lu_small")
    flows_ = [workloads.build_flow(wl, seed=2) for _ in range(2)]
    state = workloads.trained_like_({k: v.clone() for k, v in flows_[0].state_dict().items()}, wl)
    for f in flows_:
        f.load_state_dict(state)
    flows_ = [f.to(dev) for f in flows_]
    opts = [torch.optim.Adam(f.parameters(), lr=1e-3, capturable=True) for f in flows_]
    g = torch.Generator().manual_seed(8)
    batches = [torch.randn(4099, 6, generator=g).to(dev) for _ in range(3)]
    stepper = graphs.GraphedTrainStep(flows_[1], opts[1], lambda x: -flows_[1].log_prob(x).mean(), batches[0])
    for x in batches:
        opts[0].zero_grad(set_to_none=True)
        loss = -flows_[0].log_prob(x).mean()
        loss.backward()
        opts[0].step()
        assert loss.item() == stepper.step(x).item()
    for pe, pg in zip(flows_[0].parameters(), flows_[1].parameters()):
        assert torch.equal(pe, pg)


@pytest.mark.parametrize("rows", [1, 129, 300, 641])
@pytest.mark.parametrize("D", [3, 16, 33, 63])
def test_guard_bands(dev, rows, D):
    layer = make_layer(D, "trained").to(dev)
    x = torch.randn(rows, D, device=dev)
    gy = torch.randn(rows, D, device=dev)
    M, c, ld = torch.randn(D, D, device=dev), torch.randn(D, device=dev), torch.randn((), device=dev)
    with GuardedAllocations() as g:
        with torch.no_grad():
            y, lad = layer(x)
            xi, _ = layer.inverse(x)
        yo, lo = ops.lulinear_layer(x, M, c, ld)
        gx, gM, gc = ops.lulinear_layer_backward(x, M, gy)
    g.check("lulinear D=%d rows=%d" % (D, rows))
    assert torch.allclose(yo, x @ M.t() + c, atol=1e-4) and torch.equal(lo, ld.expand(rows))
    assert torch.allclose(gx, gy @ M, atol=1e-4) and torch.allclose(gM, gy.t() @ x, atol=1e-3)
    assert torch.allclose(gc, gy.sum(0), atol=1e-4)
    assert torch.isfinite(y).all() and torch.isfinite(xi).all()


@pytest.mark.skipif(not locate.have_reference(), reason="reference tree not found")
@pytest.mark.parametrize("D", [5, 33, 80])
def test_reference_state_dict(dev, D):
    flowcon = locate.import_reference()
    from flowcon.transforms.lu import LULinear as RefLULinear

    torch.manual_seed(11)
    ref = RefLULinear(D, identity_init=False)
    with torch.no_grad():
        ref.bias.uniform_(-0.3, 0.3)
    ours = transforms.LULinear(D)
    ours.load_state_dict(ref.state_dict(), strict=True)
    ours = ours.to(dev)
    x = torch.randn(257, D)
    with torch.no_grad():
        for inverse in (False, True):
            want, want_lad = ref.inverse(x) if inverse else ref(x)
            got, got_lad = ours.inverse(x.to(dev)) if inverse else ours(x.to(dev))
            assert torch.allclose(got.cpu(), want, atol=1e-4, rtol=1e-4)
            assert torch.allclose(got_lad.cpu(), want_lad, atol=1e-4)
    assert flowcon is not None
