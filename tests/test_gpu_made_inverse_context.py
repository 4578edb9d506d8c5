"""GPU tests of the incremental autoregressive inverse of a conditional MADE (`context_features`; csrc/fc_made_inverse.cuh
with the context prefill, C ABI fc_made_inverse_*): one context-term launch plus one fc_made_inverse_* launch per layer,
against the oracle (oracle/restated.py apply_layer with the context) in fp32 / fp64 and against this package's own D-pass
path."""
import ctypes
import math

import pytest
import torch

from flowconductor_b200 import _cabi, graphs, made_inverse, transforms, workloads
from flowconductor_b200.nn import tensorcore
from flowconductor_b200.transforms.base import InputOutsideDomain
from oracle import restated
from tests.helpers import assert_parity
from tests.test_gpu_guard import GuardedAllocations

pytestmark = pytest.mark.gpu

AR_INV_TOL = 1e-3  # autoregressive inverses (test_gpu_parity.test_flow_matches_reference)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _layer(kind, D=16, H=48, C=8, blocks=2, seed=0, K=8, tails="linear", gain=1.0):
    """A conditional masked autoregressive layer of family `kind` and its oracle spec; the context layers and second block
    layers drawn at 1 / sqrt(fan-in) so that the context terms matter."""
    torch.manual_seed(seed)
    common = dict(features=D, hidden_features=H, context_features=C, num_blocks=blocks)
    spec = {"kind": kind, "hidden_features": H, "num_blocks": blocks, "prefix": ""}
    if kind == "maf_affine":
        layer = transforms.MaskedAffineAutoregressiveTransform(**common)
    elif kind == "maf_prq":
        layer = transforms.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(num_bins=K, tails=tails, tail_bound=3.0,
                                                                                   **common)
        spec.update(num_bins=K, tails=tails, tail_bound=3.0)
    elif kind == "maf_sos":
        layer = transforms.MaskedSumOfSigmoidsTransform(n_sigmoids=10, **common)
        spec.update(n_sigmoids=10)
    elif kind == "maf_plin":
        layer = transforms.MaskedPiecewiseLinearAutoregressiveTransform(K, **common)
        spec.update(num_bins=K)
    elif kind == "maf_pquad":
        layer = transforms.MaskedPiecewiseQuadraticAutoregressiveTransform(num_bins=K, tails="linear", tail_bound=3.0,
                                                                           **common)
        spec.update(num_bins=K, tails="linear", tail_bound=3.0)
    else:
        layer = transforms.MaskedPiecewiseCubicAutoregressiveTransform(K, **common)
        spec.update(num_bins=K)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in layer.autoregressive_net.named_parameters():
            if "context_layer" in name or "linear_layers.1" in name:
                scale = 1.0 / math.sqrt(p.shape[-1]) if p.dim() == 2 else 0.3
                p.copy_(torch.randn(p.shape, generator=g) * scale)
        layer.autoregressive_net.final_layer.weight.mul_(gain)
    return layer, spec


UNIT_BOX = ("maf_plin", "maf_pcubic")  # the constrained unit box, no tails


def _inputs(kind, B, D, C, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, D, generator=g) * 0.98 + 0.01 if kind in UNIT_BOX else torch.randn(B, D, generator=g)
    return x.to(dev), torch.randn(B, C, generator=g).to(dev)


def _counts(fn):
    _cabi.STATS.reset()
    with torch.no_grad():
        out = fn()
    torch.cuda.synchronize()
    return out, dict(_cabi.STATS.counts)


def _d_pass(layer, z, ctx):
    made_inverse.ENABLED = False
    try:
        with torch.no_grad():
            return layer.inverse(z, context=ctx)
    finally:
        made_inverse.ENABLED = True


def _oracle(layer, spec, z, ctx, rows=None):
    sel = slice(None) if rows is None else rows
    zs, cs = z[sel].cpu(), ctx[sel].cpu()
    state = {k: v.cpu() for k, v in layer.state_dict().items()}
    state64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    with torch.no_grad():
        x32, l32 = restated.apply_layer(state, spec, zs, cs, True)
        x64, l64 = restated.apply_layer(state64, spec, zs.double(), cs.double(), True)
    return x32, l32, x64, l64


def _check(layer, spec, z, ctx, x, lad, what, rows=None):
    sel = slice(None) if rows is None else rows
    x32, l32, x64, l64 = _oracle(layer, spec, z, ctx, rows)
    assert_parity(x[sel], x32, x64, AR_INV_TOL, 1.0, what + " outputs")
    assert_parity(lad[sel], l32, l64, AR_INV_TOL, 1.0, what + " logabsdet")


FAMILIES = [("maf_affine", "fc_made_inverse_affine"), ("maf_prq", "fc_made_inverse_rqs"),
            ("maf_sos", "fc_made_inverse_sos"), ("maf_plin", "fc_made_inverse_linspline"),
            ("maf_pquad", "fc_made_inverse_quadspline"), ("maf_pcubic", "fc_made_inverse_cubicspline")]


@pytest.mark.parametrize("kind,entry", FAMILIES)
def test_narrow_conditional_layer_per_family(dev, kind, entry):
    """D = 16, H = 48 (below the fused kernel's widths), C = 8, 2 blocks: one term launch + one incremental launch,
    the oracle's three-way rule, and the D-pass path."""
    layer, spec = _layer(kind, seed=3)
    layer = layer.to(dev).eval()
    x, ctx = _inputs(kind, 1000, 16, 8, dev, seed=4)
    with torch.no_grad():
        z, _ = layer(x, context=ctx)
        assert not tensorcore.usable(layer.autoregressive_net, z, ctx, z) and made_inverse.usable(layer.autoregressive_net,
                                                                                                   z, ctx)
        layer.inverse(z, context=ctx)  # compiles the program
    (xi, ladi), counts = _counts(lambda: layer.inverse(z, context=ctx))
    assert counts == {"fc_context_terms": 1, entry: 1}, counts
    _check(layer, spec, z, ctx, xi, ladi, kind)
    xd, ladd = _d_pass(layer, z, ctx)
    scale = max(1.0, float(xd.abs().max()))
    assert float((xi - xd).abs().max()) < 1e-3 * scale and float((ladi - ladd).abs().max()) < 1e-3 * max(
        1.0, float(ladd.abs().max()))
    assert float((xi - x).abs().max()) < 1e-3 * max(1.0, float(x.abs().max()))


@pytest.mark.parametrize("C,producer", [(8, "fc_context_terms"), (96, "fc_linear_apply")])
def test_both_term_producers(dev, C, producer):
    layer, spec = _layer("maf_prq", C=C, seed=5)
    layer = layer.to(dev).eval()
    x, ctx = _inputs("maf_prq", 777, 16, C, dev, seed=6)
    with torch.no_grad():
        z, _ = layer(x, context=ctx)
        layer.inverse(z, context=ctx)
    (xi, ladi), counts = _counts(lambda: layer.inverse(z, context=ctx))
    assert counts == {producer: 1, "fc_made_inverse_rqs": 1}, counts
    _check(layer, spec, z, ctx, xi, ladi, "C=%d" % C)


def test_ragged_batches_and_domain(dev):
    """A tails=None RQ layer: in-domain inputs at ragged batches raise nothing and return the rows of the 4096-row batch bit
    for bit; an input outside the box raises.  The ragged calls run with every buffer they allocate — the T128 terms
    included — filled with a sentinel (98765.4321), so a row tile that read the unwritten T128 rows past the batch would
    put that value into its hidden units: out of the spline's box, it would set the status word and raise."""
    layer, spec = _layer("maf_prq", tails=None, seed=7)
    layer = layer.to(dev).eval()
    g = torch.Generator().manual_seed(8)
    x = (torch.rand(4096, 16, generator=g) * 1.8 - 0.9).to(dev)
    ctx = torch.randn(4096, 8, generator=g).to(dev)
    with torch.no_grad():
        z, _ = layer(x, context=ctx)
        assert float(z.abs().max()) < 1.2
        x_all, lad_all = layer.inverse(z, context=ctx)
        for B in (1, 31, 32, 33, 641):
            zb, cb = z[:B].clone(), ctx[:B].clone()
            with GuardedAllocations() as guard:
                xb, ladb = layer.inverse(zb, context=cb)
            guard.check("ragged inverse B=%d" % B)
            assert torch.equal(xb, x_all[:B]) and torch.equal(ladb, lad_all[:B]), B
    _check(layer, spec, z, ctx, x_all, lad_all, "tails=None", rows=torch.arange(0, 4096, 7))
    bad = z[:33].clone()
    bad[32, 5] = 1.5
    with pytest.raises(InputOutsideDomain):
        with torch.no_grad():
            layer.inverse(bad, context=ctx[:33].clone())


def test_cfg3_shapes_keep_the_fused_path_and_the_kernel_matches(dev):
    """H = 256, K = 16, C = 8: layer.inverse stays on the D fused launches; the incremental kernel called directly on
    32 768 rows passes the three-way rule on 512 rows at both ends."""
    D = 16
    layer, spec = _layer("maf_prq", H=256, K=16, seed=9, gain=8.0)
    layer = layer.to(dev).eval()
    net = layer.autoregressive_net
    g = torch.Generator().manual_seed(10)
    z = torch.randn(32768, D, generator=g).to(dev)
    ctx = torch.randn(32768, 8, generator=g).to(dev)
    _, counts = _counts(lambda: layer.inverse(z[:4096], context=ctx[:4096]))
    assert counts.get("fc_conditioner_rqs_apply") == D and "fc_made_inverse_rqs" not in counts, counts
    P = layer._spline.params_per_feature()
    prog = made_inverse.program_for(net, P)
    assert prog is not None and len(prog.term_arrays) == 3
    cfg, _ = layer._spline.config(True, None)
    with torch.no_grad():
        x, lad = made_inverse.apply_rqs(prog, z, cfg, None, context=ctx)
    rows = torch.cat((torch.arange(512), torch.arange(32768 - 512, 32768)))
    _check(layer, spec, z, ctx, x, lad, "cfg3 shapes", rows=rows.to(dev))


def _cfg3_small_conditional(dev):
    wl = workloads.get_workload("cfg3_small")
    wl["context_features"] = 8
    return workloads.build_flow(wl, seed=3).to(dev).eval()


def test_conditional_flow_sampling(dev):
    """cfg3_small (H = 32) with an 8-wide context: every MAF layer of the sampling cascade is one incremental launch;
    sample shapes, sample_and_log_prob against log_prob, graph replay of the inverse, graph-captured sampling."""
    flow = _cfg3_small_conditional(dev)
    n_maf = sum(1 for t in flow._transform._transforms if hasattr(t, "autoregressive_net"))
    g = torch.Generator().manual_seed(11)
    zs = [torch.randn(300, 16, generator=g).to(dev) for _ in range(3)]
    cs = [torch.randn(300, 8, generator=g).to(dev) for _ in range(3)]
    with torch.no_grad():
        flow._transform.inverse(zs[0], context=cs[0])
    _, counts = _counts(lambda: flow._transform.inverse(zs[0], context=cs[0]))
    assert counts.get("fc_made_inverse_rqs") == n_maf == 2, counts
    ctx = torch.randn(5, 8, generator=g).to(dev)
    with torch.no_grad():
        s = flow.sample(64, ctx)
        assert s.shape == (5, 64, 16) and torch.isfinite(s).all()
        samples, lp = flow.sample_and_log_prob(64, context=ctx)
        lp2 = flow.log_prob(samples.reshape(-1, 16), context=ctx.repeat_interleave(64, 0)).reshape(5, 64)
        assert float((lp - lp2).abs().max()) < 1e-3 * max(1.0, float(lp2.abs().max()))
        ginv = graphs.capture(lambda z, c: flow._transform.inverse(z, context=c), zs[0], cs[0])
        for i in (1, 2, 0):
            inv, lad = ginv(zs[i], cs[i], clone=True)
            e_inv, e_lad = flow._transform.inverse(zs[i], context=cs[i])
            assert torch.equal(inv, e_inv) and torch.equal(lad, e_lad)
        sampler = graphs.capture_sampler(flow, 128, ctx)
        a, b = sampler(ctx, clone=True), sampler(ctx, clone=True)
        assert a.shape == (5, 128, 16) and torch.isfinite(a).all() and not torch.equal(a, b)


def test_context_weights_change_rebuilds_program_and_plan(dev):
    layer, spec = _layer("maf_affine", seed=12)
    layer = layer.to(dev).eval()
    net = layer.autoregressive_net
    x, ctx = _inputs("maf_affine", 300, 16, 8, dev, seed=13)
    with torch.no_grad():
        z, _ = layer(x, context=ctx)
        x0, _ = layer.inverse(z, context=ctx)
        prog0 = made_inverse.program_for(net, 2)
        net.blocks[1].context_layer.weight.add_(torch.randn_like(net.blocks[1].context_layer.weight) * 0.5)
        x1, lad1 = layer.inverse(z, context=ctx)
        prog1 = made_inverse.program_for(net, 2)
        xd, _ = _d_pass(layer, z, ctx)
    assert prog1 is not prog0 and not torch.equal(prog1.context.weight, prog0.context.weight)
    assert float((x1 - x0).abs().max()) > 1e-3 and float((x1 - xd).abs().max()) < 1e-3 * max(1.0, float(xd.abs().max()))
    _check(layer, spec, z, ctx, x1, lad1, "after the weight change")


@pytest.mark.parametrize("rows", [1, 129, 300, 641])
def test_guard_bands(dev, rows):
    """Every buffer allocated during a conditional incremental inverse (outputs, the T128 terms) sits inside sentinel
    bands that must stay untouched, for both term producers."""
    for C in (8, 96):
        layer, _ = _layer("maf_prq", C=C, seed=14)
        layer = layer.to(dev).eval()
        z = torch.randn(rows, 16, device=dev) * 0.5
        ctx = torch.randn(rows, C, device=dev)
        with torch.no_grad():
            layer.inverse(z, context=ctx)  # compiles outside the guarded window
            with GuardedAllocations() as g:
                x, lad = layer.inverse(z, context=ctx)
        g.check("conditional incremental inverse rows=%d C=%d" % (rows, C))
        assert torch.isfinite(x).all() and torch.isfinite(lad).all()


def test_abi_rejects_bad_context_arguments(dev):
    layer, _ = _layer("maf_affine", H=50, blocks=3, seed=15)
    layer = layer.to(dev).eval()
    net = layer.autoregressive_net
    prog = made_inverse.program_for(net, 2)
    B = 100
    z = torch.randn(B, 16, device=dev)
    ctx = torch.randn(B, 8, device=dev)
    terms = made_inverse._bind_terms(prog, ctx, B)
    st = prog.struct
    x, lad = torch.empty_like(z), torch.empty(B, device=dev)
    L = _cabi.lib()

    def call():
        return L.fc_made_inverse_affine(ctypes.byref(st), z.data_ptr(), 16, x.data_ptr(), 16, lad.data_ptr(), 0, B,
                                        _cabi.SCALE_SOFTPLUS_EPS, _cabi.stream_ptr(dev))

    assert call() == _cabi.FC_OK
    torch.cuda.synchronize()
    ta = st.term_arrays
    cases = [("n_term_arrays", st, "n_term_arrays", -1), ("n_term_arrays", st, "n_term_arrays", 9),
             ("terms", st, "terms", None), ("terms", st, "terms", terms.buf.data_ptr() + 4),
             ("term_width", st, "term_width", st.term_width - 8), ("term_width", st, "term_width", 0),
             ("column", ta[1], "column", ta[1].column + 2), ("column", ta[3], "column", st.term_width - 48),
             ("array", ta[0], "array", 0), ("array", ta[2], "array", prog.n_arrays + 1), ("array", ta[2], "array", 1),
             ("b_off", ta[3], "b_off", prog.bias.numel() - 49), ("b_off", ta[0], "b_off", -4)]
    for what, obj, field, bad in cases:
        saved = getattr(obj, field)
        setattr(obj, field, bad)
        assert call() == -1, (what, bad)
        setattr(obj, field, saved)
    assert call() == _cabi.FC_OK
    torch.cuda.synchronize()
    assert torch.isfinite(x).all()
