"""BatchNorm on the B200 (csrc/fc_batchnorm.cu) against the fp64 oracle in both modes: forward, inverse, batch
statistics and running buffers, gradients, determinism, errors, the packaged flows (maf_bn_small / realnvp_bn_small:
log_prob, sampling, training steps, CUDA graphs), guard bands, and the reference's state_dicts where the reference tree
is available."""
import pytest
import torch

from flowconductor_b200 import _cabi, flows, graphs, ops, transforms, workloads
from oracle import locate
from tests import bn_oracle
from tests.helpers import assert_parity
from tests.test_gpu_guard import GuardedAllocations

pytestmark = pytest.mark.gpu
MAX_D = 4096
SPEC = {"kind": "batchnorm", "prefix": ""}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def make_layer(D, seed=0):
    torch.manual_seed(seed)
    layer = transforms.BatchNorm(D)
    with torch.no_grad():
        layer.unconstrained_weight.add_(0.4 * torch.randn(D))
        layer.bias.normal_(0.0, 0.5)
    return layer


def inputs(B, D, dev, dist, seed=1):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(B, D, generator=g, device=dev)
    if dist == "offset":  # |mean| >> std: the case a composed shift or Σx² − Bμ² gets wrong
        return 1000.0 + 0.01 * x
    if dist == "heavy":  # a Gaussian scale mixture: heavy tails, occasional |x| in the hundreds
        return x * torch.exp(1.5 * torch.randn(B, D, generator=g, device=dev))
    return x


def states(layer):
    s32 = {k: v.detach().clone() for k, v in layer.state_dict().items()}
    return s32, {k: v.double() for k, v in s32.items()}


@pytest.mark.parametrize("dist", ["normal", "offset", "heavy"])
@pytest.mark.parametrize("D", [1, 3, 6, 21, 64, 257, MAX_D])
def test_parity(dev, D, dist):
    """Three training steps (outputs, logabsdet, batch statistics, running buffers), then eval forward and inverse."""
    for B in (2, 129, 4099, 1 << 20):
        if B * D > (1 << 24):  # 1 M rows at D <= 6 (the CPU-side parity check is capped at 2^24 elements)
            continue
        # offset rows: every fp32 result carries the rounding of μ ~ 1000 (ulp 6e-5) divided by σ = 0.01, in ours and in
        # the reference alike, so the element-wise criteria give way to the population ones (quantiles and max no worse
        # than the reference's fp32 error)
        frac = 1.0 if dist == "offset" else 2e-2
        layer = make_layer(D).to(dev)
        s32, s64 = states(layer)
        for step in range(3):
            x = inputs(B, D, dev, dist, seed=step)
            if B == 4099 and step == 1:  # a column slice: row stride D + 5, base not 16-byte aligned
                x = inputs(B, D + 5, dev, dist, step)[:, 3:3 + D]
            what = "D={} {} B={} step {}".format(D, dist, B, step)
            _cabi.STATS.reset()
            y, lad = layer(x)
            assert _cabi.STATS.counts == {"fc_batchnorm_stats": 1, "fc_batchnorm_apply": 1}, _cabi.STATS.counts
            _, _, mean, var = ops.batchnorm_train(x, layer.unconstrained_weight, layer.bias, layer.eps)
            with torch.no_grad():
                r32 = bn_oracle.batch_norm(s32, "", x, training=True)
                r64 = bn_oracle.batch_norm(s64, "", x.double(), training=True)
                st32, st64 = bn_oracle.batch_stats(x), bn_oracle.batch_stats(x.double())
            assert_parity(y, r32[0], r64[0], 1e-5, 1.0, what, max_fail_frac=frac)
            assert_parity(lad, r32[1], r64[1], 1e-5, 1.0, what + " logabsdet")
            assert_parity(mean, st32[0], st64[0], 1e-5, 1.0, what + " mean")
            assert_parity(var, st32[1], st64[1], 1e-5, 1e-4, what + " var")
            bn_oracle.update_running(s32, "", x)
            bn_oracle.update_running(s64, "", x.double())
        for name, floor in (("running_mean", 1.0), ("running_var", 1e-4)):
            assert_parity(getattr(layer, name), s32[name], s64[name], 1e-5, floor, "D={} {} B={} {}".format(D, dist, B, name))
        layer.eval()
        s32, s64 = states(layer)
        x = inputs(B, D, dev, dist, seed=9)
        with torch.no_grad():
            for inverse in (False, True):
                _cabi.STATS.reset()
                y, lad = layer.inverse(x) if inverse else layer(x)
                assert _cabi.STATS.counts == {"fc_batchnorm_apply": 1}
                r32 = bn_oracle.batch_norm(s32, "", x, inverse=inverse)
                r64 = bn_oracle.batch_norm(s64, "", x.double(), inverse=inverse)
                what = "eval D={} {} B={} inverse={}".format(D, dist, B, inverse)
                assert_parity(y, r32[0], r64[0], 1e-5, 1.0, what, max_fail_frac=frac)
                assert_parity(lad, r32[1], r64[1], 1e-5, 1.0, what + " logabsdet")


def test_eval_before_training_uses_zero_running_variance(dev):
    layer = make_layer(5).to(dev).eval()
    x = torch.randn(300, 5, device=dev)
    with torch.no_grad():
        y, lad = layer(x)
    w = layer.weight.detach()
    assert torch.allclose(y, w * (x / torch.sqrt(torch.tensor(1e-5))) + layer.bias.detach(), rtol=1e-5)
    assert torch.allclose(lad, (torch.log(w) - 0.5 * torch.log(torch.tensor(1e-5))).sum().expand(300), rtol=1e-6)


@pytest.mark.parametrize("mode", ["train", "eval_forward", "eval_inverse"])
@pytest.mark.parametrize("D", [1, 6, 43, 64, 257])
def test_gradients(dev, D, mode):
    """Gradients of the input, unconstrained_weight and bias against fp64 autograd through the oracle, with both upstream
    gradients and with each alone."""
    layer = make_layer(D, seed=3).to(dev)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        layer.running_mean.copy_(torch.randn(D, generator=g))
        layer.running_var.copy_(torch.exp(torch.randn(D, generator=g)))
    if mode != "train":
        layer.eval()
    B = 4099
    x0 = torch.randn(B, D, generator=g) * 2 + 1
    wys = torch.randn(B, D, generator=g)
    wls = torch.randn(B, generator=g)
    for wy, wl in ((wys, wls), (wys, None), (None, wls)):
        layer.zero_grad(set_to_none=True)
        x = x0.to(dev).requires_grad_(True)
        y, lad = layer.inverse(x) if mode == "eval_inverse" else layer(x)
        loss = 0.0
        if wy is not None:
            loss = loss + (y * wy.to(dev)).sum()
        if wl is not None:
            loss = loss + (lad * wl.to(dev)).sum()
        _cabi.STATS.reset()
        loss.backward()
        assert _cabi.STATS.counts.get("fc_batchnorm_backward", 0) == 1
        s64 = {k: v.detach().double().cpu() for k, v in layer.state_dict().items()}
        s64["unconstrained_weight"].requires_grad_(True)
        s64["bias"].requires_grad_(True)
        x64 = x0.double().requires_grad_(True)
        y64, lad64 = bn_oracle.batch_norm(s64, "", x64, inverse=mode == "eval_inverse", training=mode == "train")
        loss64 = 0.0
        if wy is not None:
            loss64 = loss64 + (y64 * wy.double()).sum()
        if wl is not None:
            loss64 = loss64 + (lad64 * wl.double()).sum()
        loss64.backward()
        for name, got, want in (("x", x.grad, x64.grad), ("uw", layer.unconstrained_weight.grad,
                                                          s64["unconstrained_weight"].grad),
                                ("bias", layer.bias.grad, s64["bias"].grad)):
            if want is None:
                want = torch.zeros_like(got, dtype=torch.float64).cpu()
            got = torch.zeros_like(want) if got is None else got.double().cpu()
            err = (got - want).abs().max().item()
            assert err <= 2e-4 * max(1.0, want.abs().max().item()), (mode, D, name, wy is None, wl is None, err)


def test_determinism(dev):
    x = inputs(1 << 20, 43, dev, "normal")
    uw, bias = torch.randn(43, device=dev), torch.randn(43, device=dev)
    a = ops.batchnorm_train(x, uw, bias, 1e-5)
    b = ops.batchnorm_train(x, uw, bias, 1e-5)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    gy, gl = torch.randn_like(x), torch.randn(x.shape[0], device=dev)
    for mode in (_cabi.BATCHNORM_TRAIN, _cabi.BATCHNORM_EVAL_FORWARD, _cabi.BATCHNORM_EVAL_INVERSE):
        r1 = ops.batchnorm_backward(x, a[2], a[3], uw, bias, 1e-5, gy, gl, mode)
        r2 = ops.batchnorm_backward(x, a[2], a[3], uw, bias, 1e-5, gy, gl, mode)
        for u, v in zip(r1, r2):
            assert torch.equal(u, v), mode


def test_errors_and_single_row(dev):
    layer = make_layer(4).to(dev)
    with pytest.raises(transforms.InverseNotAvailable):
        layer.inverse(torch.randn(8, 4, device=dev))
    with pytest.raises(ValueError):
        layer(torch.randn(8, 4, 2, device=dev))
    with pytest.raises(RuntimeError, match="float32"):
        layer(torch.randn(8, 4, device=dev, dtype=torch.float64))
    x = torch.randn(1, 4, device=dev, requires_grad=True)
    y, lad = layer(x)  # unbiased variance of one row: NaN statistics, as the reference
    (y.sum() + lad.sum()).backward()
    torch.cuda.synchronize()
    assert torch.isnan(y).all() and torch.isnan(layer.running_var).all()
    with torch.no_grad():
        empty_y, empty_lad = layer.eval()(torch.empty(0, 4, device=dev))
    assert empty_y.shape == (0, 4) and empty_lad.shape == (0,)


def _flow(name, dev, seed=0):
    wl = workloads.get_workload(name)
    flow = workloads.build_flow(wl, seed=seed)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    flow.load_state_dict(state)
    return wl, flow.to(dev), state


FLOWS = ["maf_bn_small", "realnvp_bn_small"]


@pytest.mark.parametrize("name", FLOWS)
def test_flow_log_prob_and_sampling(dev, name):
    wl, flow, state = _flow(name, dev)
    specs = workloads.oracle_specs(wl)
    s64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    x = torch.randn(4099, 6, generator=torch.Generator().manual_seed(5))
    for training in (False, True):  # eval first: the training-mode call moves the running buffers
        flow.train(training)
        with torch.no_grad():
            lp = flow.log_prob(x.to(dev))
        want32 = bn_oracle.flow_log_prob(dict(state), specs, x, training=training)
        want64 = bn_oracle.flow_log_prob(dict(s64), specs, x.double(), training=training)
        assert_parity(lp, want32, want64, 1e-5, 1.0, "{} log_prob training={}".format(name, training))
    # the training-mode call moved the running buffers exactly as the reference's update does
    st = dict(state)
    bn_oracle.flow_log_prob(st, specs, x, training=True, update=True)
    for k, v in flow.state_dict().items():
        if "running" in k:
            assert torch.allclose(v.cpu(), st[k], rtol=1e-5, atol=1e-6), k
            state[k] = v.cpu().clone()
    flow.eval()
    s64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    with torch.no_grad():
        torch.manual_seed(7)
        got, got_lp = flow.sample_and_log_prob(2048)
        torch.manual_seed(7)
        noise = torch.randn(2048, 6, device=dev).cpu()
        want = bn_oracle.flow_sample_from_noise(state, specs, noise)
        want64 = bn_oracle.flow_sample_from_noise(s64, specs, noise.double())
        assert_parity(got, want, want64, 1e-5, 1.0, name + " sample_and_log_prob samples")
        # the trained-like inverse cascade throws most samples far out (|x| up to 1e14), where log_prob is
        # ill-conditioned; the samples themselves were held to the oracle above
        tame = got.abs().amax(1) < 100
        assert int(tame.sum()) >= 10
        lp_of_sample = flow.log_prob(got[tame])
        assert torch.allclose(got_lp[tame], lp_of_sample, rtol=1e-4, atol=1e-3)
        torch.manual_seed(7)
        assert torch.equal(flow.sample(2048), got)


@pytest.mark.parametrize("name", FLOWS)
def test_flow_training_step_gradients(dev, name):
    wl, flow, state = _flow(name, dev)
    specs = workloads.oracle_specs(wl)
    x = torch.randn(4099, 6, generator=torch.Generator().manual_seed(6))
    flow.train()
    (-flow.log_prob(x.to(dev)).mean()).backward()
    s64 = {k: (v.double().requires_grad_(True) if v.is_floating_point() else v) for k, v in state.items()}
    (-bn_oracle.flow_log_prob(s64, specs, x.double(), training=True).mean()).backward()
    for k, p in flow.named_parameters():
        want = s64[k].grad
        assert want is not None, k
        err = (p.grad.double().cpu() - want).abs().max().item()
        assert err <= 1e-3 * max(1.0, want.abs().max().item()), (k, err, want.abs().max().item())


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
    stepper = graphs.GraphedTrainStep(flows_[1], opts[1], lambda x: -flows_[1].log_prob(x).mean(), batches[0])
    for k, v in flows_[1].state_dict().items():  # the warm-up is undone, running statistics included
        assert torch.equal(v, flows_[0].state_dict()[k]), k
    for x in batches:
        opts[0].zero_grad(set_to_none=True)
        loss = -flows_[0].log_prob(x).mean()
        loss.backward()
        opts[0].step()
        assert loss.item() == stepper.step(x).item()
    for k, v in flows_[0].state_dict().items():
        assert torch.equal(v, flows_[1].state_dict()[k]), k


@pytest.mark.parametrize("name", FLOWS)
def test_graph_capture_follows_running_stats_and_parameters(dev, name):
    _, flow, _ = _flow(name, dev)
    flow.eval()
    x = torch.randn(512, 6, device=dev)
    g = graphs.capture(flow.log_prob, x)
    with torch.no_grad():
        assert torch.equal(g(x), flow.log_prob(x))
        for k, b in flow.named_buffers():
            if "running" in k:
                b.mul_(1.3).add_(0.05)
        eager = flow.log_prob(x)
        assert torch.equal(g(x), eager) and g.records == 1  # the kernels read the buffers: no new recording
        for k, p in flow.named_parameters():
            if "unconstrained_weight" in k or k.endswith("2.bias") or k.endswith("3.bias"):
                p.add_(0.05)
        eager = flow.log_prob(x)
    assert torch.equal(g(x), eager)


@pytest.mark.parametrize("rows", [1, 129, 300, 641])
@pytest.mark.parametrize("D", [3, 43, 64])
def test_guard_bands(dev, rows, D):
    layer = make_layer(D).to(dev)
    x = torch.randn(rows, D, device=dev)
    gy, gl = torch.randn(rows, D, device=dev), torch.randn(rows, device=dev)
    with GuardedAllocations() as g:
        y, lad, mean, var = ops.batchnorm_train(x, layer.unconstrained_weight.detach(), layer.bias.detach(), 1e-5)
        outs = [ops.batchnorm_backward(x, mean, var, layer.unconstrained_weight.detach(), layer.bias.detach(), 1e-5, gy,
                                       gl, mode) for mode in range(3)]
        ye, le = ops.batchnorm_eval(x, mean, var, layer.unconstrained_weight.detach(), layer.bias.detach(), 1e-5, False)
        yi, li = ops.batchnorm_eval(ye, mean, var, layer.unconstrained_weight.detach(), layer.bias.detach(), 1e-5, True)
    g.check("batchnorm D=%d rows=%d" % (D, rows))
    if rows > 1:
        assert torch.allclose(mean, x.mean(0), atol=1e-5) and torch.allclose(var, x.var(0), rtol=1e-4, atol=1e-6)
        assert torch.allclose(ye, y) and torch.allclose(yi, x, atol=1e-4) and torch.allclose(li, -le)
        for gx, guw, gb in outs:
            assert torch.isfinite(gx).all() and torch.isfinite(guw).all()
        assert torch.allclose(outs[0][2], gy.sum(0), atol=1e-4) and torch.allclose(outs[1][2], gy.sum(0), atol=1e-4)


@pytest.mark.skipif(not locate.have_reference(), reason="reference tree not found")
def test_reference_state_dicts(dev):
    flowcon = locate.import_reference()
    from flowcon.flows.autoregressive import MaskedAutoregressiveFlow as RefMAF
    from flowcon.flows.realnvp import SimpleRealNVP as RefRealNVP
    from flowcon.transforms.normalization import BatchNorm as RefBatchNorm

    torch.manual_seed(11)
    ref = RefBatchNorm(7)
    ours = transforms.BatchNorm(7)
    x = torch.randn(257, 7) * 3 + 2
    with torch.no_grad():
        ref.unconstrained_weight.add_(0.3 * torch.randn(7))
        ref.bias.normal_()
        ref(x)
    ours.load_state_dict(ref.state_dict(), strict=True)
    ours = ours.to(dev)
    for training in (True, False):
        ref.train(training)
        ours.train(training)
        with torch.no_grad():
            want, want_lad = ref(x)
            got, got_lad = ours(x.to(dev))
        assert torch.allclose(got.cpu(), want, atol=1e-4, rtol=1e-4)
        assert torch.allclose(got_lad.cpu(), want_lad, atol=1e-4)
        if not training:
            with torch.no_grad():
                want, want_lad = ref.inverse(x)
                got, got_lad = ours.inverse(x.to(dev))
            assert torch.allclose(got.cpu(), want, atol=1e-4, rtol=1e-4)
    for cls, ref_cls in ((flows.MaskedAutoregressiveFlow, RefMAF), (flows.SimpleRealNVP, RefRealNVP)):
        torch.manual_seed(12)
        ref_flow = ref_cls(6, 16, 2, 2, batch_norm_between_layers=True)
        with torch.no_grad():
            ref_flow.log_prob(torch.randn(300, 6))  # non-trivial running statistics
        ref_flow.eval()
        ours = cls(6, 16, 2, 2, batch_norm_between_layers=True)
        ours.load_state_dict(ref_flow.state_dict(), strict=True)
        ours = ours.to(dev).eval()
        x = torch.randn(257, 6)
        with torch.no_grad():
            assert torch.allclose(ours.log_prob(x.to(dev)).cpu(), ref_flow.log_prob(x), atol=1e-4, rtol=1e-4)
    assert flowcon is not None
