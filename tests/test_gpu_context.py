"""GPU tests of conditional coupling / masked autoregressive layers on the fused conditioner kernel (a ResidualNet or
residual MADE with `context_features`, inference): every case against the oracle (oracle/restated.py apply_layer with
the context) in fp32 and fp64, under the criteria the suite applies to the context-free twin of the case."""
import math

import pytest
import torch

from flowconductor_b200 import _cabi, conditioner as fcond, graphs, linear as fl, transforms, workloads
from flowconductor_b200.nn import tensorcore
from flowconductor_b200.nn.nets.resnet import ResidualNet
from flowconductor_b200.transforms import splines
from oracle import restated
from tests.helpers import assert_parity
from tests.test_gpu_guard import GuardedAllocations

pytestmark = pytest.mark.gpu

OUT_TOL = 1e-5
AR_INV_TOL = 1e-3  # autoregressive D-pass inverses (test_gpu_parity.test_flow_matches_reference)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _trained_like(layer, net_name, P, wh_slots, seed, gain=8.0):
    """workloads.trained_like_ for one layer (final weight x 8, seeded final bias with std 16 on spline width / height
    slots), and context layers / second block layers drawn at 1 / sqrt(fan-in) so that the context terms matter."""
    g = torch.Generator().manual_seed(seed)
    net = getattr(layer, net_name)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if "context_layer" in name or "linear_layers.1" in name:
                scale = 1.0 / math.sqrt(p.shape[-1]) if p.dim() == 2 else 0.3
                p.copy_(torch.randn(p.shape, generator=g) * scale)
        fin = net.final_layer
        std = torch.ones(fin.bias.numel())
        if wh_slots:
            std = std.view(-1, P)
            std[:, :wh_slots] = 16.0
            std = std.reshape(-1)
        fin.weight.mul_(gain)
        fin.bias.add_(torch.randn(fin.bias.numel(), generator=g) * std)
    return layer


def _prq_coupling(D, H, K, C, blocks, tails="linear", seed=0):
    torch.manual_seed(seed)
    layer = transforms.PiecewiseRationalQuadraticCouplingTransform(
        mask=workloads.make_mask(D, "alternating_even"),
        transform_net_create_fn=lambda i, o: ResidualNet(i, o, hidden_features=H, context_features=C, num_blocks=blocks),
        num_bins=K, tails=tails, tail_bound=3.0)
    P = 3 * K - 1 if tails == "linear" else 3 * K + 1
    spec = {"kind": "prq_coupling", "num_bins": K, "tails": tails, "tail_bound": 3.0, "hidden_features": H,
            "num_blocks": blocks, "prefix": ""}
    return _trained_like(layer, "transform_net", P, 2 * K, seed + 1), spec


def _check_layer(layer, spec, x, ctx, inverse, tol=OUT_TOL, rows=None, yfloor=1.0):
    """Layer on the GPU against the oracle in fp32 / fp64 (on `rows` only when given)."""
    dev = x.device
    with torch.no_grad():
        y, lad = (layer.inverse if inverse else layer)(x, context=ctx)
    torch.cuda.synchronize()
    assert fcond.kernel_error() == 0
    sel = slice(None) if rows is None else rows
    xs, cs = x[sel].cpu(), ctx[sel].cpu()
    state = {k: v.cpu() for k, v in layer.state_dict().items()}
    state64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    with torch.no_grad():
        y32, l32 = restated.apply_layer(state, spec, xs, cs, inverse)
        y64, l64 = restated.apply_layer(state64, spec, xs.double(), cs.double(), inverse)
    what = "{} inverse={} B={}".format(spec["kind"], inverse, x.shape[0])
    assert_parity(y[sel], y32, y64, tol, yfloor, what + " outputs")
    assert_parity(lad[sel], l32, l64, tol, 1.0, what + " logabsdet")
    assert y.device == dev


def _counts(fn):
    _cabi.STATS.reset()
    with torch.no_grad():
        fn()
    torch.cuda.synchronize()
    return dict(_cabi.STATS.counts)


@pytest.mark.parametrize("C", [16, 5, 96])
@pytest.mark.parametrize("inverse", [False, True])
def test_prq_coupling_with_context(dev, C, inverse):
    """cfg 2 shapes (D = 64, H = 256, K = 8 linear tails) with a context: C = 16, an odd C = 5 (padded input columns) and
    C = 96 (context terms from the tensor-core GEMM).  Parity at 4096 rows (the rule of test_cfg2_layers_match_oracle);
    batches of 1 / 129 / 300 / 641 rows (ragged row tiles and tile pairs) return exactly the rows of the large batch."""
    layer, spec = _prq_coupling(64, 256, 8, C, 2, seed=C)
    layer = layer.to(dev).eval()
    g = torch.Generator().manual_seed(C)
    x = (torch.randn(4096, 64, generator=g) * 1.5).to(dev)
    ctx = torch.randn(4096, C, generator=g).to(dev)
    _check_layer(layer, spec, x, ctx, inverse)
    fn = layer.inverse if inverse else layer
    with torch.no_grad():
        y, lad = fn(x, context=ctx)
        for B in (1, 129, 300, 641):
            yb, ladb = fn(x[:B].clone(), context=ctx[:B].clone())
            assert torch.equal(yb, y[:B]) and torch.equal(ladb, lad[:B]), B


@pytest.mark.parametrize("C", [16, 96])
@pytest.mark.parametrize("inverse", [False, True])
def test_prq_coupling_with_context_full_size(dev, C, inverse):
    """2^20 rows in one launch; the oracle checks rows at both ends of the same launch."""
    layer, spec = _prq_coupling(64, 256, 8, C, 2, seed=7 + C)
    layer = layer.to(dev).eval()
    B = 1 << 20
    g = torch.Generator(device=dev).manual_seed(11)
    x = torch.randn(B, 64, generator=g, device=dev) * 1.5
    ctx = torch.randn(B, C, generator=g, device=dev)
    rows = torch.cat([torch.arange(1024), torch.arange(B - 1024, B)]).to(dev)
    _check_layer(layer, spec, x, ctx, inverse, rows=rows)


@pytest.mark.parametrize("H,blocks", [(64, 2), (256, 1), (128, 4)])
def test_prq_coupling_with_context_widths_and_blocks(dev, H, blocks):
    """A narrow net (64 units zero-padded to the kernel's 128: the padding units' terms are zero), 1 and 4 blocks."""
    layer, spec = _prq_coupling(32, H, 8, 12, blocks, seed=H + blocks)
    layer = layer.to(dev).eval()
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(700, 32, generator=g) * 1.5).to(dev)
    ctx = torch.randn(700, 12, generator=g).to(dev)
    for inverse in (False, True):
        _check_layer(layer, spec, x, ctx, inverse)


def test_prq_coupling_no_tails_with_context(dev):
    """K = 10 without tails (3 K + 1 parameters, the unit box): parity inside, InputOutsideDomain through the status word."""
    layer, spec = _prq_coupling(16, 128, 10, 8, 2, tails=None, seed=5)
    layer = layer.to(dev).eval()
    g = torch.Generator().manual_seed(4)
    x = torch.rand(500, 16, generator=g).to(dev) * 0.98 + 0.01
    ctx = torch.randn(500, 8, generator=g).to(dev)
    with torch.no_grad():
        assert tensorcore.usable(layer.transform_net, x, ctx)
    counts = _counts(lambda: layer(x, context=ctx))
    assert counts.get("fc_conditioner_rqs_apply") == 1, counts
    _check_layer(layer, spec, x, ctx, False)
    bad = x.clone()
    bad[17, 0] = 1.5  # a transformed feature outside [0, 1]
    with pytest.raises(splines.InputOutsideDomain), torch.no_grad():
        layer(bad, context=ctx)


@pytest.mark.parametrize("inverse", [False, True])
def test_affine_coupling_with_context(dev, inverse):
    torch.manual_seed(2)
    layer = transforms.AffineCouplingTransform(
        workloads.make_mask(24, "mid_split"),
        lambda i, o: ResidualNet(i, o, hidden_features=128, context_features=10, num_blocks=2))
    layer = _trained_like(layer, "transform_net", 2, 0, 3).to(dev).eval()
    spec = {"kind": "affine_coupling", "scale_activation": "sigmoid2", "hidden_features": 128, "num_blocks": 2,
            "prefix": ""}
    g = torch.Generator().manual_seed(6)
    x = torch.randn(641, 24, generator=g).to(dev)
    ctx = torch.randn(641, 10, generator=g).to(dev)
    counts = _counts(lambda: layer(x, context=ctx))
    assert counts.get("fc_conditioner_affine_apply") == 1 and counts.get("fc_context_terms") == 1, counts
    _check_layer(layer, spec, x, ctx, inverse)


def test_quadratic_coupling_with_context(dev):
    """The store variant (conditioner outputs written out, element-wise spline kernel afterwards)."""
    torch.manual_seed(4)
    layer = transforms.PiecewiseQuadraticCouplingTransform(
        workloads.make_mask(16, "alternating_odd"),
        lambda i, o: ResidualNet(i, o, hidden_features=128, context_features=6, num_blocks=2),
        num_bins=8, tails="linear", tail_bound=3.0)
    layer = _trained_like(layer, "transform_net", 15, 0, 5).to(dev).eval()
    spec = {"kind": "pquad_coupling", "num_bins": 8, "tails": "linear", "tail_bound": 3.0, "hidden_features": 128,
            "num_blocks": 2, "prefix": ""}
    g = torch.Generator().manual_seed(8)
    x = torch.randn(300, 16, generator=g).to(dev)
    ctx = torch.randn(300, 6, generator=g).to(dev)
    counts = _counts(lambda: layer(x, context=ctx))
    assert counts.get("fc_conditioner_store_apply") == 1 and "fc_linear_apply" not in counts, counts
    for inverse in (False, True):
        _check_layer(layer, spec, x, ctx, inverse)


def _maf(kind, D, H, C, seed, **kw):
    torch.manual_seed(seed)
    if kind == "maf_prq":
        layer = transforms.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(
            features=D, hidden_features=H, context_features=C, num_bins=kw["K"], tails="linear", tail_bound=3.0,
            num_blocks=2)
        P, wh = 3 * kw["K"] - 1, 0
        spec = {"kind": kind, "num_bins": kw["K"], "tails": "linear", "tail_bound": 3.0, "hidden_features": H}
    elif kind == "maf_affine":
        layer = transforms.MaskedAffineAutoregressiveTransform(features=D, hidden_features=H, context_features=C,
                                                               num_blocks=2)
        P, wh = 2, 0
        spec = {"kind": kind, "hidden_features": H}
    else:
        layer = transforms.MaskedSumOfSigmoidsTransform(features=D, hidden_features=H, n_sigmoids=10, context_features=C,
                                                        num_blocks=2)
        P, wh = 31, 0
        spec = {"kind": kind, "n_sigmoids": 10, "hidden_features": H}
    spec.update(num_blocks=2, prefix="")
    # (an affine MAF with the x 8 final-layer gain has scales near 1e-3: its inverse amplifies the reference's own fp32
    # noise by ~1e9 over 16 features, no criterion can be met there)
    return _trained_like(layer, "autoregressive_net", P, wh, seed + 1, gain=1.0 if kind == "maf_affine" else 8.0), spec


@pytest.mark.parametrize("kind,entry", [("maf_prq", "fc_conditioner_rqs_apply"),
                                        ("maf_affine", "fc_conditioner_affine_apply"),
                                        ("maf_sos", "fc_conditioner_sos_apply")])
def test_masked_autoregressive_forward_with_context(dev, kind, entry):
    """cfg 3 shapes (D = 16, K = 16, H = 256) with an 8-wide context."""
    layer, spec = _maf(kind, 16, 256, 8, seed=21, K=16)
    layer = layer.to(dev).eval()
    g = torch.Generator().manual_seed(9)
    x = torch.randn(641, 16, generator=g).to(dev)
    ctx = torch.randn(641, 8, generator=g).to(dev)
    counts = _counts(lambda: layer(x, context=ctx))
    # one fused launch plus one term producer, no per-layer GEMM
    assert counts.get(entry) == 1 and counts.get("fc_context_terms") == 1 and "fc_linear_apply" not in counts, counts
    yfloor = 1.0
    _check_layer(layer, spec, x, ctx, False, yfloor=yfloor)


@pytest.mark.parametrize("kind,entry", [("maf_prq", "fc_conditioner_rqs_apply"),
                                        ("maf_affine", "fc_conditioner_affine_apply")])
def test_masked_autoregressive_inverse_with_context(dev, kind, entry):
    """The D-pass inverse at 4096 rows: the context terms once, then one fused launch per pass."""
    D = 16
    layer, spec = _maf(kind, D, 256, 8, seed=31, K=16)
    layer = layer.to(dev).eval()
    g = torch.Generator().manual_seed(10)
    z = torch.randn(4096, D, generator=g).to(dev)
    ctx = torch.randn(4096, 8, generator=g).to(dev)
    counts = _counts(lambda: layer.inverse(z, context=ctx))
    assert counts.get(entry) == D and counts.get("fc_context_terms") == 1 and "fc_linear_apply" not in counts, counts
    _check_layer(layer, spec, z, ctx, True, tol=AR_INV_TOL)


def test_launches_of_a_conditional_coupling_layer(dev):
    """One term producer + one fused conditioner launch, no per-layer GEMM, for both term producers."""
    for C, producer in ((16, "fc_context_terms"), (96, "fc_linear_apply")):
        layer, _ = _prq_coupling(64, 256, 8, C, 2, seed=1)
        layer = layer.to(dev).eval()
        x = torch.randn(1000, 64, device=dev)
        ctx = torch.randn(1000, C, device=dev)
        for fn in (lambda: layer(x, context=ctx), lambda: layer.inverse(x, context=ctx)):
            _counts(fn)  # packs the weights
            counts = _counts(fn)
            assert counts.get("fc_conditioner_rqs_apply") == 1 and counts.get(producer) == 1, counts
            assert sum(counts.values()) == 2, counts


def _conditional_cfg2(C, rows=None):
    wl = workloads.get_workload("cfg2")
    wl["context_features"] = C
    flow = workloads.build_flow(wl)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    g = torch.Generator().manual_seed(C)
    for k in state:  # the context layers away from their default initialisation, so that the gates matter
        if "context_layer" in k:
            state[k] = torch.randn(state[k].shape, generator=g) * (1.0 / math.sqrt(C) if state[k].dim() == 2 else 0.3)
    flow.load_state_dict(state)
    return wl, flow, state


def test_conditional_coupling_stack_log_prob(dev):
    """8 conditional PRQ coupling layers (cfg 2 shapes, C = 16): log_prob against the oracle on rows of one full-size
    launch, with the rule of test_full_size_cfg2_log_prob."""
    wl, flow, state = _conditional_cfg2(16)
    flow = flow.to(dev).eval()
    B = wl["batch"]
    g = torch.Generator(device=dev).manual_seed(1234)
    x = torch.randn(B, 64, generator=g, device=dev)
    ctx = torch.randn(B, 16, generator=g, device=dev)
    with torch.no_grad():
        lp = flow.log_prob(x, context=ctx)
    assert torch.isfinite(lp).all()
    specs = workloads.oracle_specs(wl)
    rows = torch.cat([torch.arange(512), torch.arange(B - 512, B)])
    cpu_state = {k: v.cpu() for k, v in flow.state_dict().items()}
    with torch.no_grad():
        o32 = restated.flow_log_prob(cpu_state, specs, x[rows].cpu(), ctx[rows].cpu())
        o64 = restated.flow_log_prob({k: (v.double() if v.is_floating_point() else v) for k, v in cpu_state.items()},
                                     specs, x[rows].cpu().double(), ctx[rows].cpu().double())
    assert_parity(lp[rows.to(dev)], o32, o64, OUT_TOL, 1.0, "conditional cfg2 log_prob rows", max_ratio=30.0)


def test_cuda_graph_replay_with_context(dev):
    """graphs.capture of a conditional log_prob and of the sampling cascade replays bit for bit what the eager calls return;
    capture_sampler(flow, n, context) draws finite samples of the same distribution as eager sampling."""
    wl = workloads.get_workload("cfg2_tc_small")
    wl["context_features"] = 12
    flow = workloads.build_flow(wl, seed=3).to(dev).eval()
    B = 384
    g = torch.Generator().manual_seed(5)
    xs = [torch.randn(B, 64, generator=g).to(dev) for _ in range(3)]
    cs = [torch.randn(B, 12, generator=g).to(dev) for _ in range(3)]
    with torch.no_grad():
        assert tensorcore.usable(flow._transform._transforms[0].transform_net, xs[0], cs[0])
        glp = graphs.capture(lambda x, c: flow.log_prob(x, context=c), xs[0], cs[0])
        ginv = graphs.capture(lambda z, c: flow._transform.inverse(z, context=c), xs[0], cs[0])
        for i in (1, 2, 0):
            lp = glp(xs[i], cs[i], clone=True)
            assert torch.equal(lp, flow.log_prob(xs[i], context=cs[i]))
            inv, lad = ginv(xs[i], cs[i], clone=True)
            e_inv, e_lad = flow._transform.inverse(xs[i], context=cs[i])
            assert torch.equal(inv, e_inv) and torch.equal(lad, e_lad)
        ctx = torch.randn(4, 12, generator=g).to(dev)
        sampler = graphs.capture_sampler(flow, 256, ctx)
        a, b = sampler(ctx, clone=True), sampler(ctx, clone=True)
        assert a.shape == (4, 256, 64) and torch.isfinite(a).all() and not torch.equal(a, b)
        # graph samples are distributed like eager samples: their log_prob under the flow is comparable
        reps = ctx.repeat_interleave(256, 0)
        lp_g = flow.log_prob(a.reshape(-1, 64), context=reps).mean().item()
        lp_e = flow.log_prob(flow.sample(256, ctx).reshape(-1, 64), context=reps).mean().item()
        assert abs(lp_g - lp_e) < 3.0


@pytest.mark.parametrize("rows", [1, 129, 300, 641])
def test_guard_bands_around_conditional_layers(dev, rows):
    """Every buffer allocated while a conditional layer runs (outputs, the T128 term buffer) sits inside sentinel bands
    that must stay untouched."""
    layers = [_prq_coupling(64, 256, 8, 16, 2, seed=2)[0], _prq_coupling(64, 256, 8, 96, 2, seed=2)[0],
              _maf("maf_affine", 16, 256, 8, seed=3)[0]]
    for layer in layers:
        layer = layer.to(dev).eval()
        D = 16 if isinstance(layer, transforms.MaskedAffineAutoregressiveTransform) else 64
        net = getattr(layer, "transform_net", None) or layer.autoregressive_net
        C = fcond.pack_context(net).features
        x = torch.randn(rows, D, device=dev)
        ctx = torch.randn(rows, C, device=dev)
        with torch.no_grad():
            layer(x, context=ctx)  # packs outside the guarded window
            with GuardedAllocations() as g:
                y, _ = layer(x, context=ctx)
                xi, _ = layer.inverse(y, context=ctx)
                terms = tensorcore.context_terms(net, ctx)
        g.check("%s rows=%d C=%d" % (type(layer).__name__, rows, C))
        assert isinstance(terms, fl.T128) and torch.isfinite(xi).all()


def test_conditioner_abi_rejects_bad_term_modes(dev):
    layer, _ = _prq_coupling(64, 128, 8, 8, 1, seed=1)
    net = layer.to(dev).transform_net
    plan = tensorcore.context_plan_for(net)
    d_t = 32
    ccols = layer._ccols
    packed = fcond.pack_rqs(net, 8, d_t, col_map=torch.cat((ccols, torch.arange(64, 72, device=dev,
                                                                                  dtype=torch.int32))),
                            k_in=72, context=plan)
    B = 256
    x = torch.randn(B, 64, device=dev)
    a = torch.cat((x, torch.randn(B, 8, device=dev)), 1)
    y, lad = torch.empty_like(x), torch.empty(B, device=dev)
    cfg = _cabi.RqsConfig(8, _cabi.TAILS_LINEAR, 0, 0, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3, 1.0 / math.sqrt(128))
    terms = fcond.context_terms(plan, a[:, 64:])
    L = _cabi.lib()

    def call():
        return L.fc_conditioner_rqs_apply(ctypes_ref(packed.struct), a.data_ptr(), a.stride(0), B, x.data_ptr(), 64,
                                          y.data_ptr(), 64, lad.data_ptr(), 0, d_t, _cabi.cols(layer._tcols),
                                          _cabi.cols(ccols), ctypes_ref(cfg), None, _cabi.stream_ptr(dev))

    fcond._bind_terms(packed, terms, B)
    assert call() == _cabi.FC_OK
    gate = packed.struct.layers[2]
    gate.term_mode = _cabi.COND_TERM_ADD  # ADD belongs to a block's first layer
    assert call() == -1
    gate.term_mode = 7
    assert call() == -1
    gate.term_mode = _cabi.COND_TERM_GATE
    packed.struct.layers[0].term_mode = _cabi.COND_TERM_GATE  # on the initial layer
    assert call() == -1
    packed.struct.layers[0].term_mode = _cabi.COND_TERM_NONE
    saved = gate.terms
    gate.terms = saved + 4  # misaligned
    assert call() == -2
    gate.terms = saved
    gate.term_width = 120  # narrower than the layer
    assert call() == -2
    gate.term_width = terms.width
    gate.terms = None
    assert call() == -1
    gate.terms = saved
    assert call() == _cabi.FC_OK
    torch.cuda.synchronize()
    # the context-term producer's own argument checks
    assert L.fc_context_terms(ctx_ptr(a), 72, B, 0, plan.weight.data_ptr(), plan.bias.data_ptr(), plan.width,
                              terms.buf.data_ptr(), _cabi.stream_ptr(dev)) == -1
    assert L.fc_context_terms(ctx_ptr(a), 72, B, 8, plan.weight.data_ptr(), plan.bias.data_ptr(), 120,
                              terms.buf.data_ptr(), _cabi.stream_ptr(dev)) == -1
    assert L.fc_context_terms(ctx_ptr(a), 72, B, 8, plan.weight.data_ptr(), plan.bias.data_ptr(), plan.width,
                              terms.buf.data_ptr() + 4, _cabi.stream_ptr(dev)) == -2


def ctypes_ref(s):
    import ctypes

    return ctypes.byref(s)


def ctx_ptr(a):
    return a.data_ptr() + 64 * 4
