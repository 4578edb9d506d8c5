"""The element-wise squashing layers on the B200 (csrc/fc_pointwise.cu) against the fp64 oracle (tests/pointwise_oracle.py):
every layer in both directions at D = 1 ... 257 and up to 1 M rows, on normal, heavy-tailed and near-edge inputs, strided
and [B, 3, 4] layouts, the domain checks and CUDA-graph capture, gradients for the inputs and the temperature, bitwise
determinism, the bounded_maf_small flow (log_prob, sampling, captured sampler, graphed training step) and, where the
reference tree is present, class-by-class parity with flowcon.transforms.nonlinearities."""
import math

import pytest
import torch

from flowconductor_b200 import _cabi, graphs, transforms, workloads
from oracle import locate
from tests import pointwise_oracle as pwo
from tests.helpers import assert_parity

pytestmark = pytest.mark.gpu
DS = [1, 3, 6, 32, 64, 257]
BS = [1, 129, 4099, 1 << 20]
T_SIG, SLOPE = 1.3, 0.05


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def layer_and_oracle(name, dev):
    """(our layer, oracle(x, inverse) -> (y, lad) in x's dtype, inverse directions that check the domain)"""
    T = torch.tensor([T_SIG])
    table = {
        "sigmoid": (transforms.Sigmoid(temperature=T_SIG), lambda x, inv: pwo.sigmoid(x, T, 1e-6, inv)),
        "logit": (transforms.Logit(temperature=T_SIG), lambda x, inv: pwo.sigmoid(x, T, 1e-6, not inv)),
        "tanh": (transforms.Tanh(), lambda x, inv: pwo.tanh(x, inv)),
        "leaky_relu": (transforms.LeakyReLU(SLOPE), lambda x, inv: pwo.leaky_relu(x, SLOPE, inv)),
        "exp": (transforms.Exp(), lambda x, inv: pwo.exp(x, inv)),
        "cauchy": (transforms.CauchyCDF(), lambda x, inv: pwo.cauchy_cdf(x, inv)),
        "cauchy_inverse": (transforms.CauchyCDFInverse(), lambda x, inv: pwo.cauchy_cdf(x, not inv)),
    }
    layer, fn = table[name]
    return layer.to(dev), fn


# the direction of each layer whose input lives on a bounded set: (layer, inverse) -> domain kind
BOUNDED = {("sigmoid", True): "unit", ("logit", False): "unit", ("tanh", True): "sym", ("exp", True): "pos",
           ("cauchy", True): "unit", ("cauchy_inverse", False): "unit"}
LAYERS = ["sigmoid", "logit", "tanh", "leaky_relu", "exp", "cauchy", "cauchy_inverse"]
CASES = [(name, inv) for name in LAYERS for inv in (False, True)]


def make_inputs(name, inverse, B, D, kind, seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, D, generator=g)
    dom = BOUNDED.get((name, inverse))
    if kind == "heavy":
        z = z * 10
    if dom is None:
        if kind == "edge":  # zeros and tiny magnitudes of both signs
            z.view(-1)[::3] = 0.0
            z.view(-1)[1::7] = 1e-30
            z.view(-1)[2::11] = -1e-30
        return z
    if dom == "pos":
        x = torch.exp(z.clamp(-80, 80))
        if kind == "edge":
            x.view(-1)[::5] = 1e-38
        return x
    u = torch.sigmoid(z)
    if dom == "sym":
        u = (2 * u - 1).clamp(-1 + 6e-8, 1 - 6e-8)
        if kind == "edge":
            u.view(-1)[::5] = 1 - 6e-8
            u.view(-1)[1::5] = -(1 - 6e-8)
        return u
    if kind == "edge":  # the clamp's bounds and the interval's ends
        edge = torch.tensor([0.0, 1.0, 1e-6, 1 - 1e-6, 1e-7, 1 - 1e-7, 0.5])
        u.view(-1)[: min(u.numel(), 3 * edge.numel())] = edge.repeat(3)[: min(u.numel(), 3 * edge.numel())]
    return u


def check(name, inverse, x_dev, y, lad, fn, what):
    x = x_dev.cpu()
    with torch.no_grad():
        y32, l32 = fn(x, inverse)
        y64, l64 = fn(x.double(), inverse)
    if name == "tanh" and not inverse:
        l64 = pwo.tanh_stable_logdet(x.double())
        inf = ~torch.isfinite(l32)  # the reference's fp32 log(1 − y²) is −inf there: held against fp64 only
        if inf.any():
            got = lad.detach().cpu().double()[inf]
            assert ((got - l64[inf]).abs() <= 1e-5 * l64[inf].abs().clamp_min(1.0)).all(), what + " stable log-det"
        l32 = torch.where(inf, l64.float(), l32)
    assert_parity(y.reshape(x.shape), y32, y64, 1e-5, 1.0, what + " outputs")
    assert_parity(lad, l32, l64, 1e-5, 1.0, what + " logabsdet")


def _sizes():
    for D in DS:
        for B in BS:
            if B < (1 << 20) or D <= 6:
                yield D, B


@pytest.mark.parametrize("name,inverse", CASES)
@pytest.mark.parametrize("D,B", list(_sizes()))
def test_parity(dev, name, inverse, D, B):
    layer, fn = layer_and_oracle(name, dev)
    call = layer.inverse if inverse else layer.forward
    for i, kind in enumerate(("normal", "heavy", "edge")):
        x = make_inputs(name, inverse, B, D, kind, seed=D * 7 + B + i).to(dev)
        with torch.no_grad():
            y, lad = call(x)
        assert y.shape == x.shape and lad.shape == (B,) and lad.device == x.device and lad.dtype == torch.float32
        check(name, inverse, x, y, lad, fn, "{} inverse={} D={} B={} {}".format(name, inverse, D, B, kind))


@pytest.mark.parametrize("name,inverse", CASES)
def test_layouts(dev, name, inverse):
    layer, fn = layer_and_oracle(name, dev)
    call = layer.inverse if inverse else layer.forward
    wide = make_inputs(name, inverse, 4099, 37, "normal", seed=11).to(dev)
    x = wide[:, 2:34]  # a column slice: row stride 37, no copy
    with torch.no_grad():
        y, lad = call(x)
    check(name, inverse, x, y, lad, fn, name + " column slice")
    x3 = make_inputs(name, inverse, 513, 12, "heavy", seed=12).reshape(513, 3, 4).to(dev)
    with torch.no_grad():
        y3, lad3 = call(x3)
    assert y3.shape == (513, 3, 4)
    check(name, inverse, x3, y3, lad3, fn, name + " [B, 3, 4]")


def test_domain_checks(dev):
    cases = {"sigmoid": ([-1e-7, 1.0 + 1e-7], [0.0, 1.0]), "logit": ([-1e-7, 1.0 + 1e-7], [0.0, 1.0]),
             "tanh": ([-1.0, 1.0], [-0.999, 0.999]), "exp": ([0.0, -1.0], [1e-38, 5.0]),
             "cauchy": ([-1e-7, 1.0 + 1e-7], [0.0, 1.0]), "cauchy_inverse": ([-1e-7, 1.0 + 1e-7], [0.0, 1.0])}
    for name, (outside, inside) in cases.items():
        layer, _ = layer_and_oracle(name, dev)
        checking = layer.forward if (name, False) in BOUNDED else layer.inverse
        other = layer.inverse if (name, False) in BOUNDED else layer.forward
        base = torch.full((300, 5), 0.5, device=dev)
        for bad in outside:
            x = base.clone()
            x[123, 3] = bad
            with pytest.raises(transforms.InputOutsideDomain):
                checking(x)
            other(x)  # the unchecked direction never raises
            x = base.clone()
            x[7, 1] = inside[0]
            x[299, 4] = inside[1]
            checking(x)  # a fresh status word: clean on the next call
    for name in ("tanh", "leaky_relu"):  # no domain at all in the forward direction
        layer, _ = layer_and_oracle(name, dev)
        layer.forward(torch.full((8, 3), 1e30, device=dev))
    transforms.LeakyReLU().inverse(torch.full((8, 3), -1e30, device=dev))


def test_capture_of_a_checking_direction_raises(dev):
    for layer, call in ((transforms.Logit(), "forward"), (transforms.Sigmoid(), "inverse"),
                        (transforms.Exp(), "inverse"), (transforms.Tanh(), "inverse")):
        x = torch.full((64, 4), 0.5, device=dev)
        with pytest.raises(RuntimeError, match="CUDA graph"):
            graphs.capture(getattr(layer.to(dev), call), x)
    for layer, call in ((transforms.Sigmoid(learn_temperature=True), "forward"), (transforms.Logit(), "inverse"),
                        (transforms.Tanh(), "forward"), (transforms.Exp(), "forward"),
                        (transforms.CauchyCDF(), "forward"), (transforms.LeakyReLU(), "inverse")):
        layer = layer.to(dev)
        x = torch.randn(64, 4, device=dev)
        g = graphs.capture(getattr(layer, call), x)
        got = g(x)
        with torch.no_grad():
            want = getattr(layer, call)(x)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    sig = transforms.Sigmoid(learn_temperature=True).to(dev)  # the graph reads the temperature on the device
    x = torch.randn(64, 4, device=dev)
    g = graphs.capture(sig.forward, x)
    with torch.no_grad():
        sig.temperature.fill_(2.5)
        want = sig.forward(x)
    got = g(x)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def grads(layer_fn, oracle_fn, x, gy, gl, T, inverse, dtype, learn):
    """(grad_x, grad_T) of <gy, y> + <gl, lad>."""
    x = x.to(dtype).detach().requires_grad_(True)
    if T is not None:
        T = T.to(dtype).detach().requires_grad_(learn)
    y, lad = layer_fn(x) if layer_fn is not None else oracle_fn(x, T, inverse)
    loss = (gy.to(dtype) * y).sum() + (gl.to(dtype) * lad).sum()
    wrt = [x] + ([T] if (T is not None and learn) else [])
    out = torch.autograd.grad(loss, wrt)
    return out[0], (out[1] if len(out) > 1 else None)


ORACLE_T = {"sigmoid": lambda x, T, inv: pwo.sigmoid(x, T, 1e-6, inv),
            "logit": lambda x, T, inv: pwo.sigmoid(x, T, 1e-6, not inv)}


@pytest.mark.parametrize("name,inverse", CASES)
@pytest.mark.parametrize("D", [3, 64])
def test_gradients(dev, name, inverse, D):
    B = 4099
    learn = name in ("sigmoid", "logit")
    T = torch.tensor([T_SIG])
    if name == "sigmoid":
        layer = transforms.Sigmoid(temperature=T_SIG, learn_temperature=True).to(dev)
        t_param = layer.temperature
    elif name == "logit":
        layer = transforms.InverseTransform(transforms.Sigmoid(temperature=T_SIG, learn_temperature=True)).to(dev)
        t_param = layer._transform.temperature
    else:
        layer, fn = layer_and_oracle(name, dev)
        t_param = None
    if name in ORACLE_T:
        ofn = ORACLE_T[name]
    else:
        _, fn = layer_and_oracle(name, dev)
        ofn = (lambda f: lambda x, T, inv: f(x, inv))(fn)
    g = torch.Generator().manual_seed(D)
    x = make_inputs(name, inverse, B, D, "normal", seed=D)
    if (name, inverse) in BOUNDED:  # keep the population away from the clamp and the ends
        x = x.clamp(1e-3, 1 - 1e-3) if BOUNDED[(name, inverse)] == "unit" else x
    gy, gl = torch.randn(B, D, generator=g), torch.randn(B, generator=g)
    call = layer.inverse if inverse else layer.forward
    results = []
    for _ in range(2):
        xg = x.to(dev).requires_grad_(True)
        y, lad = call(xg)
        params = [xg] + ([t_param] if t_param is not None else [])
        results.append(torch.autograd.grad((gy.to(dev) * y).sum() + (gl.to(dev) * lad).sum(), params))
    for a, b in zip(*results):  # two backward calls are bitwise equal
        assert torch.equal(a, b)
    gx32, gt32 = grads(None, ofn, x, gy, gl, T, inverse, torch.float32, learn)
    gx64, gt64 = grads(None, ofn, x, gy, gl, T, inverse, torch.float64, learn)
    what = "{} inverse={} D={}".format(name, inverse, D)
    assert_parity(results[0][0], gx32, gx64, 1e-5, max(1.0, float(gx64.abs().mean())), what + " grad x")
    if learn:
        got = float(results[0][1])
        assert abs(got - float(gt64)) <= 1e-4 * max(1.0, abs(float(gt64))) + 2 * abs(float(gt32) - float(gt64)), (
            what, got, float(gt32), float(gt64))


def test_composite_cdf_transform(dev):
    torch.manual_seed(0)
    layer = transforms.CompositeCDFTransform(transforms.Sigmoid(temperature=0.7, learn_temperature=True),
                                             transforms.PiecewiseRationalQuadraticCDF([6], 8)).to(dev)
    state = {k: v.detach().cpu() for k, v in layer.state_dict().items()}
    s64 = {k: v.double() for k, v in state.items()}
    x = torch.randn(4099, 6, generator=torch.Generator().manual_seed(1)) * 3
    for inverse in (False, True):
        with torch.no_grad():
            y, lad = (layer.inverse if inverse else layer.forward)(x.to(dev))
            y32, l32 = pwo.composite_cdf(state, "", x, 8, inverse)
            y64, l64 = pwo.composite_cdf(s64, "", x.double(), 8, inverse)
        assert_parity(y, y32, y64, 1e-5, 1.0, "composite outputs inverse={}".format(inverse))
        assert_parity(lad, l32, l64, 1e-5, 1.0, "composite logabsdet inverse={}".format(inverse))
    xg = x.to(dev).requires_grad_(True)
    y, lad = layer(xg)
    (y.sum() + lad.sum()).backward()
    t = layer._transforms[0].temperature
    assert t.grad is not None and torch.isfinite(t.grad).all() and torch.isfinite(xg.grad).all()
    assert layer._transforms[1].unnormalized_widths.grad is not None


def _flow(name, dev, seed=0):
    wl = workloads.get_workload(name)
    flow = workloads.build_flow(wl, seed=seed)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    flow.load_state_dict(state)
    return wl, flow.to(dev), state


def test_bounded_flow_log_prob_and_sampling(dev):
    wl, flow, state = _flow("bounded_maf_small", dev)
    specs = workloads.oracle_specs(wl)
    s64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    x = workloads.sample_data(wl, 4099, seed=5)
    with torch.no_grad():
        lp = flow.log_prob(x.to(dev))
    assert_parity(lp, pwo.flow_log_prob(state, specs, x), pwo.flow_log_prob(s64, specs, x.double()), 1e-5, 1.0,
                  "bounded_maf_small log_prob")
    with torch.no_grad():
        torch.manual_seed(7)
        got, got_lp = flow.sample_and_log_prob(2048)
        torch.manual_seed(7)
        noise = torch.randn(2048, 6, device=dev).cpu()
    want, want_lp = pwo.flow_sample_and_log_prob(state, specs, noise)
    want64, want_lp64 = pwo.flow_sample_and_log_prob(s64, specs, noise.double())
    assert bool((got > 0).all()) and bool((got < 1).all())
    assert_parity(got, want, want64, 1e-5, 1.0, "bounded_maf_small samples", max_ratio=1e3)
    assert_parity(got_lp, want_lp, want_lp64, 1e-5, 1.0, "bounded_maf_small sample log_prob", max_ratio=1e3)


def test_bounded_flow_captured_sampler(dev):
    _, flow, _ = _flow("bounded_maf_small", dev)
    s = graphs.capture_sampler(flow, 512)
    a = s().clone()
    b = s()
    assert a.shape == (512, 6) and not torch.equal(a, b) and bool(((a > 0) & (a < 1)).all())
    z = torch.randn(512, 6, device=dev)  # the sampler's cascade on given noise, captured and eager
    g = graphs.capture(lambda n: flow._transform.inverse(n), z)
    got = g(z)
    with torch.no_grad():
        want = flow._transform.inverse(z)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_bounded_flow_graphed_training_by_sampling(dev):
    """A sampling-direction objective (reverse KL to a quadratic energy on the box): the logit's learned temperature
    trains, and a GraphedTrainStep replays the eager steps bitwise."""
    flows_ = [_flow("bounded_maf_small", dev, seed=2)[1].train() for _ in range(2)]
    opts = [torch.optim.Adam(f.parameters(), lr=1e-2, capturable=True) for f in flows_]
    t0 = float(flows_[0]._transform._transforms[0]._transform.temperature)

    def loss_of(f):
        def loss(z):
            x, lad = f._transform.inverse(z)
            return (20.0 * ((x - 0.3) ** 2).sum(1) - lad).mean()
        return loss

    g = torch.Generator().manual_seed(8)
    batches = [torch.randn(4099, 6, generator=g).to(dev) for _ in range(3)]
    stepper = graphs.GraphedTrainStep(flows_[1], opts[1], loss_of(flows_[1]), batches[0])
    for z in batches:
        opts[0].zero_grad(set_to_none=True)
        loss = loss_of(flows_[0])(z)
        loss.backward()
        opts[0].step()
        assert loss.item() == stepper.step(z).item()
    for k, v in flows_[0].state_dict().items():
        assert torch.equal(v, flows_[1].state_dict()[k]), k
    assert float(flows_[0]._transform._transforms[0]._transform.temperature) != t0


@pytest.mark.skipif(not locate.have_reference(), reason="the FlowConductor reference tree is not available")
def test_reference_classes(dev):
    nl = locate.import_reference().transforms.nonlinearities
    g = torch.Generator().manual_seed(0)
    x = torch.randn(257, 5, generator=g)
    u = torch.rand(257, 5, generator=g) * 0.98 + 0.01
    pairs = [(transforms.Sigmoid(1.3, learn_temperature=True), nl.Sigmoid(1.3, learn_temperature=True), x, u),
             (transforms.Logit(0.8), nl.Logit(0.8), u, x), (transforms.Tanh(), nl.Tanh(), x, 2 * u - 1),
             (transforms.Exp(), nl.Exp(), x, u), (transforms.CauchyCDF(), nl.CauchyCDF(), x, u),
             (transforms.CauchyCDFInverse(), nl.CauchyCDFInverse(), u, x)]
    for ours, ref, xf, xi in pairs:
        ours.load_state_dict(ref.state_dict(), strict=True)
        ours = ours.to(dev)
        for inverse, inp in ((False, xf), (True, xi)):
            with torch.no_grad():
                want = (ref.inverse if inverse else ref)(inp)
                got = (ours.inverse if inverse else ours)(inp.to(dev))
            assert torch.allclose(got[0].cpu(), want[0], rtol=1e-5, atol=1e-5), (type(ours).__name__, inverse)
            assert torch.allclose(got[1].cpu(), want[1], rtol=1e-5, atol=1e-4), (type(ours).__name__, inverse)
    ref = nl.LeakyReLU(0.1)  # the reference's mask is a CPU tensor: compare on the CPU
    with torch.no_grad():
        got = transforms.LeakyReLU(0.1).forward(x.to(dev))
    want = (torch.nn.functional.leaky_relu(x, 0.1), ref.log_negative_slope * (x < 0).float().sum(1))
    assert torch.allclose(got[0].cpu(), want[0]) and torch.allclose(got[1].cpu(), want[1], atol=1e-5)
    refc = nl.CompositeCDFTransform(nl.Sigmoid(learn_temperature=True), nl.PiecewiseRationalQuadraticCDF([5], 8))
    ours = transforms.CompositeCDFTransform(transforms.Sigmoid(learn_temperature=True),
                                            transforms.PiecewiseRationalQuadraticCDF([5], 8))
    ours.load_state_dict(refc.state_dict(), strict=True)
    ours = ours.to(dev)
    with torch.no_grad():
        want, got = refc(x), ours(x.to(dev))
    assert torch.allclose(got[0].cpu(), want[0], atol=1e-5) and torch.allclose(got[1].cpu(), want[1], atol=1e-4)
