"""GPU parity tests: the CUDA path (through torch.ops.flowcon_b200 -> C ABI) against
  (1) golden vectors from the unmodified reference (fp32 + fp64),
  (2) the oracle restatement on fresh seeded inputs,
  (3) size-independent properties at BASELINE.json's full sizes (forward o inverse = id, logabsdet
      antisymmetry, identity-init known answer, outside-tail identity).

Tolerances (north_star): outputs and logabsdet within 1e-5 relative in fp32, gradients within 1e-4, judged
with the three-way rule of tests/helpers.assert_parity (the reference's own fp32 noise floor is ~1e-5).
"""
import math

import pytest
import torch

from flowconductor_b200 import _cabi, ops, transforms, workloads
from flowconductor_b200.transforms import splines
from oracle import restated
from tests.helpers import assert_parity, golden_state, load_golden

pytestmark = pytest.mark.gpu

OUT_TOL = 1e-5
GRAD_TOL = 1e-4


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def fn_gold():
    return load_golden("functions")


def _spline_call(gold, name, dev, requires_grad=False):
    k, lin, tb, inv, ident = gold[name + "/meta"].tolist()
    k = int(k)
    x = gold[name + "/x"].to(dev).requires_grad_(requires_grad)
    p = gold[name + "/params"].to(dev).requires_grad_(requires_grad)
    uw, uh, ud = p[..., :k], p[..., k:2 * k], p[..., 2 * k:]
    kw = dict(inverse=bool(inv), enable_identity_init=bool(ident))
    if lin:
        y, lad = transforms.unconstrained_rational_quadratic_spline(x, uw, uh, ud, tails="linear", tail_bound=tb,
                                                                    **kw)
    else:
        y, lad = transforms.rational_quadratic_spline(x, uw, uh, ud, **kw)
    return x, p, y, lad, tb


RQ_CASES = ["rq_fwd_lin_k8", "rq_inv_lin_k8", "rq_fwd_lin_k16_id", "rq_inv_lin_k16_id", "rq_fwd_none_k5",
            "rq_inv_none_k5", "rq_fwd_lin_k10_b1", "rq_fwd_lin_k8_zero_id"]


@pytest.mark.parametrize("name", RQ_CASES)
def test_spline_functions_match_reference(fn_gold, dev, name):
    _, _, y, lad, tb = _spline_call(fn_gold, name, dev)
    assert_parity(y, fn_gold[name + "/y32"], fn_gold[name + "/y64"], OUT_TOL, max(tb, 1.0), name + " outputs")
    assert_parity(lad, fn_gold[name + "/lad32"], fn_gold[name + "/lad64"], OUT_TOL, 1.0, name + " logabsdet")


@pytest.mark.parametrize("name", ["rq_fwd_lin_k8", "rq_inv_lin_k8", "rq_fwd_lin_k16_id", "rq_fwd_none_k5"])
def test_spline_gradients_match_reference(fn_gold, dev, name):
    x, p, y, lad, _ = _spline_call(fn_gold, name, dev, requires_grad=True)
    gy, gl = fn_gold[name + "/gy"].to(dev), fn_gold[name + "/gl"].to(dev)
    gx, gp = torch.autograd.grad((y * gy).sum() + (lad * gl).sum(), [x, p])
    s = max(1.0, fn_gold[name + "/gx64"].abs().median().item())
    assert_parity(gx, fn_gold[name + "/gx32"], fn_gold[name + "/gx64"], GRAD_TOL, s, name + " grad x")
    s = max(1e-2, fn_gold[name + "/gp64"].abs().mean().item())
    assert_parity(gp, fn_gold[name + "/gp32"], fn_gold[name + "/gp64"], GRAD_TOL, s, name + " grad params")


def test_bin_parity_through_outputs(fn_gold, dev):
    """Bins identical except within 1e-6 (normalised units) of a knot: a wrong bin away from a knot would
    move the output by O(bin width); near a knot the spline is C1 so outputs still agree."""
    name = "rq_fwd_lin_k8"
    _, _, y, _, _ = _spline_call(fn_gold, name, dev)
    err = (y.cpu().double() - fn_gold[name + "/y64"]).abs()
    assert err.max() < 1e-4


def test_identity_init_known_answers(dev):
    # tests/transforms/splines/rational_quadratic_test.py:33-62 (constrained, K+1 zero derivatives)
    k, shape = 10, (2, 3, 4)
    z = torch.zeros(*shape, k, device=dev)
    zd = torch.zeros(*shape, k + 1, device=dev)
    x = torch.rand(*shape, device=dev)
    for inverse in (False, True):
        y, lad = transforms.rational_quadratic_spline(x, z, z, zd, inverse=inverse, enable_identity_init=True)
        assert (y - x).abs().max() <= 1e-6
        assert lad.abs().max() <= 1e-6
    # :116-146 all inputs in the tails -> identity, zero logabsdet
    xt = torch.sign(torch.randn(*shape, device=dev)) * (1.0 + torch.rand(*shape, device=dev))
    y, lad = transforms.unconstrained_rational_quadratic_spline(xt, z, z, zd[..., :k - 1], tail_bound=1.0,
                                                                enable_identity_init=True)
    assert torch.equal(y, xt) and torch.equal(lad, torch.zeros_like(lad))


def test_domain_errors(dev):
    # tests/transforms/nonlinearities_test.py:60-76
    p = torch.zeros(1, 16, device=dev)
    for bad in (-1.0, -0.1, 1.1, 2.0):
        with pytest.raises(transforms.InputOutsideDomain):
            transforms.rational_quadratic_spline(torch.tensor([bad], device=dev), p[:, :5], p[:, 5:10], p[:, 10:])
    with pytest.raises(ValueError):
        transforms.rational_quadratic_spline(torch.zeros(1, device=dev), p[:, :5], p[:, 5:10], p[:, 10:],
                                             min_bin_width=0.3)
    with pytest.raises(RuntimeError):
        transforms.unconstrained_rational_quadratic_spline(torch.zeros(1, device=dev), p[:, :5], p[:, 5:10],
                                                           p[:, 10:14], tails="cubic")


@pytest.mark.parametrize("k,tb,ident", [(8, 3.0, False), (16, 3.0, True), (7, 2.0, False), (33, 5.0, True)])
def test_spline_matches_oracle_on_fresh_inputs(dev, k, tb, ident):
    """Fresh seeded inputs vs the oracle (fp32 and fp64), incl. an odd K and a K on the runtime-K path."""
    g = torch.Generator().manual_seed(100 + k)
    x = torch.randn(513, 11, generator=g) * tb * 0.6
    p = torch.randn(513, 11, 3 * k - 1, generator=g) * 2
    for inverse in (False, True):
        args = lambda t: (t[..., :k], t[..., k:2 * k], t[..., 2 * k:])  # noqa: E731
        kw = dict(inverse=inverse, tails="linear", tail_bound=tb, enable_identity_init=ident)
        r32y, r32l = restated.unconstrained_rational_quadratic_spline(x, *args(p), **kw)
        r64y, r64l = restated.unconstrained_rational_quadratic_spline(x.double(), *args(p.double()), **kw)
        y, lad = transforms.unconstrained_rational_quadratic_spline(x.to(dev), *args(p.to(dev)), **kw)
        assert_parity(y, r32y, r64y, OUT_TOL, tb, "oracle outputs K=%d inv=%s" % (k, inverse))
        assert_parity(lad, r32l, r64l, OUT_TOL, 1.0, "oracle logabsdet K=%d inv=%s" % (k, inverse))


def test_empty_and_ragged_batches(dev):
    k = 8
    for n in (0, 1, 7, 255, 257):
        x = torch.randn(n, 5, device=dev)
        p = torch.randn(n, 5 * 23, device=dev)
        y, lad, _ = ops.rqs_layer(x, p, None, None, k, _cabi.TAILS_LINEAR, False, False, -3.0, 3.0, -3.0, 3.0, 1e-3,
                                  1e-3, 1e-3, 1.0)
        assert y.shape == (n, 5) and lad.shape == (n,)
        if n:
            ry, rl = restated.rq_elementwise(x.cpu(), p.cpu(), k, "linear", 3.0, False, None, False)
            assert (y.cpu() - ry).abs().max() < 1e-4 and (lad.cpu() - rl).abs().max() < 1e-3


def test_pipelined_and_staged_kernels_agree(dev, monkeypatch):
    """The TMA-pipelined fast path and the staged kernel run the same element arithmetic: bit-identical."""
    g = torch.Generator().manual_seed(9)
    for B, D, k, coupling in ((4099, 64, 8, True), (1000, 16, 16, False), (333, 8, 5, True)):
        d_t = D // 2 if coupling else D
        x = (torch.randn(B, D, generator=g) * 1.5).to(dev)
        p = (torch.randn(B, d_t * (3 * k - 1), generator=g) * 2).to(dev)
        tc = torch.arange(0, D, 2, dtype=torch.int32, device=dev) if coupling else None
        cc = torch.arange(1, D, 2, dtype=torch.int32, device=dev) if coupling else None
        for inverse in (False, True):
            args = (x, p, tc, cc, k, _cabi.TAILS_LINEAR, inverse, False, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3, 0.25)
            monkeypatch.setenv("FC_PIPE", "0")
            y0, l0, _ = ops.rqs_layer(*args)
            monkeypatch.delenv("FC_PIPE")
            y1, l1, _ = ops.rqs_layer(*args)
            assert torch.equal(y0, y1) and torch.equal(l0, l1), (B, D, k, inverse)


def test_strided_inputs_and_column_lists(dev):
    """Coupling-style call: full-width rows, int32 column lists, non-contiguous row stride."""
    g = torch.Generator().manual_seed(5)
    B, D, k = 300, 10, 8
    big = torch.randn(B, D + 6, generator=g).to(dev)
    x = big[:, 3:3 + D]  # row stride D+6, last dim dense
    tc = torch.tensor([0, 3, 4, 8], dtype=torch.int32, device=dev)
    cc = torch.tensor([1, 2, 5, 6, 7, 9], dtype=torch.int32, device=dev)
    p = (torch.randn(B, 4 * 23, generator=g) * 2).to(dev)
    y, lad, _ = ops.rqs_layer(x, p, tc, cc, k, _cabi.TAILS_LINEAR, False, False, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3,
                              1e-3, 0.25)
    xc = x.cpu()
    ry, rl = restated.rq_elementwise(xc[:, tc.cpu().long()], p.cpu(), k, "linear", 3.0, False, 4.0, False)
    assert torch.equal(y[:, cc.long()].cpu(), xc[:, cc.cpu().long()])
    assert (y[:, tc.long()].cpu() - ry).abs().max() < 1e-4
    assert (lad.cpu() - rl).abs().max() < 1e-3


# ------------------------------------------------------------------------------------------------
# affine / sum of sigmoids function level
# ------------------------------------------------------------------------------------------------
def test_affine_kernels(fn_gold, dev):
    x = fn_gold["affine/x"].to(dev)
    p = fn_gold["affine/params"].to(dev)
    for act, name in ((_cabi.SCALE_SIGMOID2, "blocked_sigmoid2"), (_cabi.SCALE_SOFTPLUS_CLAMP3,
                                                                    "blocked_softplus_clamp3")):
        y, lad = ops.affine_layer(x, p, None, None, _cabi.AFFINE_BLOCKED, act, False)
        assert_parity(y, fn_gold["affine/%s_fwd_y32" % name], fn_gold["affine/%s_fwd_y64" % name], OUT_TOL, 1.0, name)
        assert_parity(lad, fn_gold["affine/%s_fwd_lad32" % name], fn_gold["affine/%s_fwd_lad64" % name], OUT_TOL, 1.0,
                      name + " lad")
        yi, ladi = ops.affine_layer(x, p, None, None, _cabi.AFFINE_BLOCKED, act, True)
        assert_parity(yi, fn_gold["affine/%s_inv_y32" % name], fn_gold["affine/%s_inv_y64" % name], OUT_TOL, 1.0,
                      name + " inverse")
        assert torch.equal(ladi, -lad)
    y, lad = ops.affine_layer(x, p, None, None, _cabi.AFFINE_INTERLEAVED, _cabi.SCALE_SOFTPLUS_EPS, False)
    assert_parity(y, fn_gold["affine/interleaved_fwd_y32"], fn_gold["affine/interleaved_fwd_y64"], OUT_TOL, 1.0, "maf")
    assert_parity(lad, fn_gold["affine/interleaved_fwd_lad32"], fn_gold["affine/interleaved_fwd_lad64"], OUT_TOL, 1.0,
                  "maf lad")


@pytest.mark.parametrize("name", ["sos_n10", "sos_n3_wide"])
def test_sum_of_sigmoids_kernels(fn_gold, dev, name):
    ns = int(fn_gold[name + "/meta"][0])
    x = fn_gold[name + "/x"].to(dev).requires_grad_(True)
    raw = fn_gold[name + "/params"].to(dev).requires_grad_(True)
    n, d = x.shape
    y, lad = ops.sos_layer(x, raw.reshape(n, -1), ns, 0.0, False, 50, 120.0)
    floor = max(1.0, fn_gold[name + "/y64"].abs().median().item())
    assert_parity(y, fn_gold[name + "/y32"], fn_gold[name + "/y64"], OUT_TOL, floor, name + " y")
    assert_parity(lad, fn_gold[name + "/lad32"], fn_gold[name + "/lad64"], OUT_TOL, 1.0, name + " lad")
    gy, gl = fn_gold[name + "/gy"].to(dev), fn_gold[name + "/gl"].to(dev)
    gx, gp = torch.autograd.grad((y * gy).sum() + (lad * gl).sum(), [x, raw])
    s = max(1e-2, fn_gold[name + "/gx64"].abs().mean().item())
    assert_parity(gx, fn_gold[name + "/gx32"], fn_gold[name + "/gx64"], GRAD_TOL, s, name + " gx")
    s = max(1e-2, fn_gold[name + "/gp64"].abs().mean().item())
    assert_parity(gp, fn_gold[name + "/gp32"], fn_gold[name + "/gp64"], GRAD_TOL, s, name + " gp")
    # numerical inverse: reference tests accept eps 1e-5 .. 1e-3 (adaptive_sigmoid_test.py:40-41,64-79)
    with torch.no_grad():
        xi, ladi = ops.sos_layer(fn_gold[name + "/y32"].to(dev), raw.reshape(n, -1), ns, 0.0, True, 50, 120.0)
    ref = fn_gold[name + "/inv_x64"]
    scale = ref.abs().clamp_min(1.0)
    assert ((xi.cpu().double() - ref).abs() / scale).max() < 1e-3
    assert (ladi.cpu().double() - fn_gold[name + "/inv_lad64"]).abs().max() < 5e-3


def test_sum_of_sigmoids_large_inputs(dev):
    # adaptive_sigmoid_test.py:64-79: inverse at |x| ~ 200 still consistent
    t = transforms.SumOfSigmoids(features=3, n_sigmoids=5).to(dev)
    x = torch.tensor([[200.0, -200.0, 150.0], [-180.0, 0.5, 199.0]], device=dev)
    with torch.no_grad():
        y, lad = t(x)
        xi, ladi = t.inverse(y)
    assert ((xi - x).abs() / x.abs().clamp_min(1)).max() < 1e-4
    assert (lad + ladi).abs().max() < 1e-3


# ------------------------------------------------------------------------------------------------
# model level: the drop-in classes with the reference's weights
# ------------------------------------------------------------------------------------------------
MODELS = ["cfg1", "cfg2_small", "cfg3_small", "cfg4_small", "affine_coupling_small", "cond_prq_small",
          "maf_sos_small", "prq_coupling_notails_small", "prq_coupling_uncond_small", "plin_coupling_small",
          "maf_plin_small", "pquad_coupling_small", "maf_pquad_small", "pcubic_coupling_small", "maf_pcubic_small", "actnorm_maf_small"]


def _load(name, dev):
    gold = load_golden(name)
    wl = workloads.get_workload(name)
    flow = workloads.build_flow(wl)
    flow.load_state_dict(golden_state(gold), strict=True)
    if "actnorm" in name:
        flow.eval()  # as the fixture was generated: a training-mode ActNorm re-initialises itself from its first batch
    return gold, wl, flow.to(dev)


@pytest.mark.parametrize("name", MODELS)
def test_flow_matches_reference(dev, name):
    gold, wl, flow = _load(name, dev)
    x = gold["x"].to(dev)
    ctx = gold["context"].to(dev) if "context" in gold else None
    with torch.no_grad():
        z, lad = flow._transform(x, context=ctx)
        lp = flow.log_prob(x, context=ctx)
        xi, ladi = flow._transform.inverse(gold["noise"].to(dev), context=ctx)
    yfloor = max(1.0, gold["fwd_y64"].abs().median().item())
    assert_parity(z, gold["fwd_y32"], gold["fwd_y64"], OUT_TOL, yfloor, name + " forward outputs")
    assert_parity(lad, gold["fwd_lad32"], gold["fwd_lad64"], OUT_TOL, 1.0, name + " forward logabsdet")
    assert_parity(lp, gold["log_prob32"], gold["log_prob64"], OUT_TOL, 1.0, name + " log_prob")
    # tolerance-level parity only for (a) the numerical sum-of-sigmoids inverse and (b) autoregressive inverses,
    # which re-run the conditioner D times on partially inverted outputs (SURVEY.md §7): reference test eps 1e-3
    numerical = "sos" in name or name in ("cfg4_small", "cfg3_small")
    tol = 1e-3 if numerical else OUT_TOL
    yfloor = max(1.0, gold["inv_y64"].abs().median().item())
    assert_parity(xi, gold["inv_y32"], gold["inv_y64"], tol, yfloor, name + " inverse outputs")
    assert_parity(ladi, gold["inv_lad32"], gold["inv_lad64"], 10 * tol if numerical else tol, 1.0,
                  name + " inverse logabsdet")


@pytest.mark.parametrize("name", ["cfg1", "cfg2_small", "cfg3_small", "cfg4_small", "affine_coupling_small",
                                  "cond_prq_small", "actnorm_maf_small"])
def test_flow_parameter_gradients_match_reference(dev, name):
    """loss = -log_prob(x).mean(); backward through our kernels vs the reference's autograd."""
    gold, wl, flow = _load(name, dev)
    x = gold["x"].to(dev)
    ctx = gold["context"].to(dev) if "context" in gold else None
    loss = -flow.log_prob(x, context=ctx).mean()
    loss.backward()
    assert_parity(loss, gold["loss32"], gold["loss64"], OUT_TOL, 1.0, name + " loss")
    for pn, p in flow.named_parameters():
        r32, r64 = gold["grad32/" + pn], gold["grad64/" + pn]
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        if "gradrows/" + pn in gold:  # a large gradient is stored at a fixed sample of its rows
            g = g[gold["gradrows/" + pn].to(g.device)]
        scale = max(1e-6, r64.abs().max().item())
        assert_parity(g / scale, r32 / scale, r64 / scale, GRAD_TOL, 1.0, name + " grad " + pn)


def test_actnorm_data_dependent_initialisation(dev):
    """normalization.py:177-178,204-218: in training mode the first batch sets log_scale / shift so that the outputs have
    zero mean and unit variance; later calls leave them alone.  Large ragged batch: the vector path and the tail."""
    layer = transforms.ActNorm(12).to(dev)
    x = torch.randn(4097, 12, device=dev) * 3.0 + 1.5
    layer.train()
    y, lad = layer(x)
    assert bool(layer.initialized)
    assert y.mean(0).abs().max() < 1e-4 and (y.std(0) - 1).abs().max() < 1e-4
    ref_lad = layer.log_scale.sum()
    assert (lad - ref_lad).abs().max() < 1e-5
    ls = layer.log_scale.detach().clone()
    layer(x * 2)
    assert torch.equal(layer.log_scale.detach(), ls)
    xi, ladi = layer.inverse(y)
    assert (xi - x).abs().max() < 1e-4 and (lad + ladi).abs().max() < 1e-5
    # gradients against torch autograd of the reference's formula, odd width (scalar path)
    layer = transforms.ActNorm(7).to(dev).eval()
    with torch.no_grad():
        layer.log_scale.normal_(0, 0.3)
        layer.shift.normal_(0, 0.5)
    x = torch.randn(333, 7, device=dev, requires_grad=True)
    w = torch.randn(333, 7, device=dev)
    wl = torch.randn(333, device=dev)
    for inverse in (False, True):
        for p in (layer.log_scale, layer.shift, x):
            p.grad = None
        y, lad = layer.inverse(x) if inverse else layer(x)
        ((y * w).sum() + (lad * wl).sum()).backward()
        got = [x.grad.clone(), layer.log_scale.grad.clone(), layer.shift.grad.clone()]
        xr = x.detach().double().requires_grad_(True)
        lsr = layer.log_scale.detach().double().requires_grad_(True)
        shr = layer.shift.detach().double().requires_grad_(True)
        if inverse:
            yr, ladr = (xr - shr) / torch.exp(lsr), -lsr.sum() * torch.ones(333, device=dev, dtype=torch.float64)
        else:
            yr, ladr = torch.exp(lsr) * xr + shr, lsr.sum() * torch.ones(333, device=dev, dtype=torch.float64)
        ((yr * w.double()).sum() + (ladr * wl.double()).sum()).backward()
        for g, r in zip(got, (xr.grad, lsr.grad, shr.grad)):
            assert ((g.double() - r).abs() / r.abs().clamp_min(1.0)).max() < 1e-4


def test_sample_and_log_prob_consistency(dev):
    # tests/flows/base_test.py:54-69: sample_and_log_prob == log_prob(sample).  Freshly initialised flow (smooth):
    # with the synthetic "trained-like" weights even the reference's own fp32 inverse->forward chain drifts.
    wl = workloads.get_workload("cfg2_small")
    flow = workloads.build_flow(wl).to(dev)
    with torch.no_grad():
        samples, lp = flow.sample_and_log_prob(64)
        lp2 = flow.log_prob(samples)
        assert flow.sample(10).shape == (10, 64)
    assert samples.shape == (64, 64) and lp.shape == (64,)
    assert ((lp - lp2).abs() / lp2.abs().clamp_min(1)).max() < 1e-4


def test_patch_reference_functions(dev):
    """The function-level seam with the reference's own calling convention (strided views of one
    [B, D, 3K-1] tensor, coupling.py:550-552)."""
    g = torch.Generator().manual_seed(3)
    B, D, K = 64, 6, 8
    x = (torch.randn(B, D, generator=g) * 2).to(dev)
    tp = torch.randn(B, D, 3 * K - 1, generator=g).to(dev)
    y, lad = splines.unconstrained_rational_quadratic_spline(x, tp[..., :K], tp[..., K:2 * K], tp[..., 2 * K:],
                                                             tails="linear", tail_bound=3.0)
    ry, rl = restated.unconstrained_rational_quadratic_spline(x.cpu(), tp.cpu()[..., :K], tp.cpu()[..., K:2 * K],
                                                              tp.cpu()[..., 2 * K:], tails="linear", tail_bound=3.0)
    assert (y.cpu() - ry).abs().max() < 1e-4 and (lad.cpu() - rl).abs().max() < 1e-3


# ------------------------------------------------------------------------------------------------
# full-size properties (BASELINE.json sizes; the oracle is too slow here, so size-independent checks)
# ------------------------------------------------------------------------------------------------
def test_full_size_cfg2_log_prob(dev):
    """cfg 2 at its full batch (1M rows): finite, log_prob == N(z) + logabsdet, and an oracle spot check on rows
    of the SAME full-size launch.  (No 8-layer round trip here: with the synthetic trained-like weights the
    reference algorithm itself cannot invert the stack in fp32 — oracle median |x_rt - x| is 0.3.)"""
    wl = workloads.get_workload("cfg2")
    flow = workloads.build_flow(wl)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    flow.load_state_dict(state)
    flow = flow.to(dev)
    B = wl["batch"]
    x = torch.randn(B, 64, generator=torch.Generator(device=dev).manual_seed(1234), device=dev)
    with torch.no_grad():
        z, lad = flow._transform(x)
        lp = flow.log_prob(x)
    assert torch.isfinite(lp).all() and torch.isfinite(z).all()
    ref_lp = -0.5 * (z.double() ** 2).sum(1) - 0.5 * 64 * math.log(2 * math.pi) + lad.double()
    assert (lp.double() - ref_lp).abs().max() < 1e-3
    specs = workloads.oracle_specs(wl)
    rows = torch.cat([torch.arange(512), torch.arange(B - 512, B)])
    cpu_state = {k: v.cpu() for k, v in flow.state_dict().items()}
    with torch.no_grad():
        o32 = restated.flow_log_prob(cpu_state, specs, x[rows].cpu())
        o64 = restated.flow_log_prob({k: (v.double() if v.is_floating_point() else v) for k, v in cpu_state.items()},
                                     specs, x[rows].cpu().double())
    # eight ill-conditioned layers in sequence: the per-row error is heavy-tailed (profiles/r01_tc_error_by_layer.txt)
    # and the max over 1024 rows is a noisy statistic, so the whole-stack check bounds it at 30x the reference's
    # own max; every layer is checked on its own at the usual 10x in test_cfg2_layers_match_oracle.
    assert_parity(lp[rows], o32, o64, OUT_TOL, 1.0, "cfg2 full-size log_prob rows", max_ratio=30.0)


@pytest.mark.parametrize("tc", [True, False])
def test_cfg2_layers_match_oracle(dev, tc, monkeypatch):
    """Every layer of the full-size cfg 2 model on its own: the layer's input is the fp32 oracle's output of the
    previous layer, so the comparison sees one conditioner + spline evaluation, not the chaotic amplification of
    the whole stack.  tc=True is the tensor-core inference path (3xTF32 GEMMs, spline in the epilogue), tc=False
    the unfused path (torch conditioner + element-wise kernel)."""
    from flowconductor_b200.nn import tensorcore

    monkeypatch.setattr(tensorcore, "ENABLED", tc)
    wl = workloads.get_workload("cfg2")
    flow = workloads.build_flow(wl)
    state = workloads.trained_like_({k: v.clone() for k, v in flow.state_dict().items()}, wl)
    flow.load_state_dict(state)
    specs = workloads.oracle_specs(wl)
    state64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    flow = flow.to(dev)
    h = torch.randn(4096, 64, generator=torch.Generator().manual_seed(99))
    with torch.no_grad():
        for li, (layer, spec) in enumerate(zip(flow._transform._transforms, specs)):
            y64, l64 = restated.apply_layer(state64, spec, h.double())
            y32, l32 = restated.apply_layer(state, spec, h)
            y, lad = layer(h.to(dev))
            assert_parity(y, y32, y64, OUT_TOL, 1.0, "cfg2 layer {} outputs (tc={})".format(li, tc))
            assert_parity(lad, l32, l64, OUT_TOL, 1.0, "cfg2 layer {} logabsdet (tc={})".format(li, tc))
            h = y32


@pytest.mark.parametrize("d,k", [(64, 8), (256, 8)])
def test_full_size_layer_round_trip(dev, d, k):
    """One coupling layer at the full batch: inverse(forward(x)) == x, forward(inverse(y)) == y, logabsdet
    antisymmetric, identity columns bit-exact, points outside the tails untouched.  Size-independent properties
    (the oracle is too slow at 1M x 32..128 x 23)."""
    B = 1 << 20 if d == 64 else 1 << 18
    d_t = d // 2
    g = torch.Generator(device=dev).manual_seed(7)
    x = torch.randn(B, d, generator=g, device=dev) * 1.5
    p = torch.randn(B, d_t * (3 * k - 1), generator=g, device=dev)
    tc = torch.arange(0, d, 2, dtype=torch.int32, device=dev)
    cc = torch.arange(1, d, 2, dtype=torch.int32, device=dev)
    hyper = (k, _cabi.TAILS_LINEAR)
    tail = (False, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3, 1.0)
    y, lad, _ = ops.rqs_layer(x, p, tc, cc, *hyper, False, *tail)
    xr, ladr, _ = ops.rqs_layer(y, p, tc, cc, *hyper, True, *tail)
    y2, _, _ = ops.rqs_layer(xr, p, tc, cc, *hyper, False, *tail)
    assert torch.equal(y[:, 1::2], x[:, 1::2]) and torch.equal(xr[:, 1::2], x[:, 1::2])
    outside = x[:, 0::2].abs() > 3.0
    assert outside.any() and torch.equal(y[:, 0::2][outside], x[:, 0::2][outside])
    err = (xr - x).abs()[:, 0::2].flatten()
    q = torch.quantile(err[: 1 << 22].double(), torch.tensor([0.5, 0.999], dtype=torch.float64, device=dev))
    assert q[0] < 1e-6 and q[1] < 2e-4 and err.max() < 0.2   # 1/slope amplification in the flattest bins
    assert (y2 - y).abs().max() < 1e-4
    asym = (lad + ladr).abs()
    assert asym.median() < 1e-4 and torch.quantile(asym[: 1 << 20], 0.999) < 5e-3
    assert torch.isfinite(lad).all()


# ------------------------------------------------------------------------------------------------
# tensor-core GEMM entry points (fc_linear_*), called through the C ABI by flowconductor_b200.linear
# ------------------------------------------------------------------------------------------------
def _gemm_err(got, want64):
    return (got.double() - want64).abs().max().item() / want64.abs().max().item()


@pytest.mark.parametrize("M,K,N,relu_in,relu_out,res,a_t,o_t", [
    (1, 32, 4, False, False, False, False, False),        # a single row, narrowest output
    (128, 32, 256, False, False, False, False, False),
    (1000, 256, 256, True, True, True, False, False),     # ragged last tile, ReLU both sides, skip connection
    (4099, 256, 512, True, False, True, False, False),    # two N tiles of the 256-wide kernel
    (5000, 8, 64, False, True, False, False, False),      # K shorter than one ring slot
    (300, 752, 32, False, False, False, False, False),    # input-gradient shape: long reduction, narrow output
    (777, 256, 132, True, True, True, False, False),      # row-major staged store: last 32-column box clipped to 4
    (130, 96, 100, False, False, True, False, False),     # two row tiles, one partial column tile, skip connection
    (70001, 256, 256, True, False, True, False, False),   # row-major staged store, ~4 work units per CTA pair, ragged
    (1000, 256, 256, False, False, False, True, False),   # T128 in, rows out
    (1000, 64, 256, False, False, False, False, True),    # rows in, T128 out: staged kernel
    (1000, 256, 256, True, True, True, True, True),       # staged kernel with skip connection, CTA pairs, ragged
    (257, 256, 384, True, False, True, True, True),       # three 128-wide tiles, odd number of row tiles
    (70000, 32, 64, True, False, True, True, True),       # T128 but not a multiple of 128 wide: direct stores
])
def test_linear_store_kernels(dev, M, K, N, relu_in, relu_out, res, a_t, o_t):
    """fc_linear_apply against an fp64 matmul; the yardstick is the fp32 cuBLAS result of the same product."""
    from flowconductor_b200 import linear as fl

    g = torch.Generator(device=dev).manual_seed(M * 7 + K)
    a = torch.randn(M, K, generator=g, device=dev)
    w = torch.randn(N, K, generator=g, device=dev) / math.sqrt(K)
    b = torch.randn(N, generator=g, device=dev)
    r = torch.randn(M, N, generator=g, device=dev) if res else None
    pk = fl.pack(w, b)
    out = fl.linear(fl.T128.from_rows(a) if a_t else a, pk, relu_in=relu_in, relu_out=relu_out,
                    residual=(fl.T128.from_rows(r) if (o_t and res) else r), out_t128=o_t)
    if o_t:
        out = out.to_rows()
    a64 = a.double().relu() if relu_in else a.double()
    want = a64 @ w.double().t() + b.double() + (r.double() if res else 0.0)
    ref32 = torch.nn.functional.linear(a.relu() if relu_in else a, w, b) + (r if res else 0.0)
    if relu_out:
        want, ref32 = want.relu(), ref32.relu()
    assert out.shape == (M, N) and torch.isfinite(out).all()
    assert _gemm_err(out, want) <= 2.0 * _gemm_err(ref32, want) + 2e-7


@pytest.mark.parametrize("N,K,B,slices", [(256, 256, 8192, None), (752, 256, 20000, 7), (64, 100, 4096, 1),
                                          (256, 256, 131072, None)])  # 148 ranges: two work units per CTA pair
def test_linear_splitk_t_weight_gradient_shape(dev, N, K, B, slices):
    """fc_linear_splitk_t_apply: grad_W = grad_y^T @ x as a split-K product over the batch, against fp64."""
    from flowconductor_b200 import linear as fl

    g = torch.Generator(device=dev).manual_seed(N + B)
    gy = torch.randn(B, N, generator=g, device=dev)
    x = torch.randn(B, K, generator=g, device=dev)
    # grad_y untransposed (operand via TMEM), bias gradient accumulated on the way
    got3, colsum = fl.linear_splitk_t(gy, fl.pack_transposed(x), k_slices=slices, column_sums=True)
    assert torch.equal(got3, fl.linear_splitk_t(gy, fl.pack_transposed(x), k_slices=slices))
    want_cs = gy.double().sum(0)
    assert colsum.shape == (N,)
    assert (colsum.double() - want_cs).abs().max() <= 4.0 * (gy.sum(0).double() - want_cs).abs().max() + \
        2e-6 * want_cs.abs().max()
    want = gy.double().t() @ x.double()
    ref32 = gy.t() @ x
    assert got3.shape == (N, K)
    assert _gemm_err(got3, want) <= 2.0 * _gemm_err(ref32, want) + 2e-7


def test_linear_pack_folds_mask_and_column_scatter(dev):
    from flowconductor_b200 import linear as fl

    g = torch.Generator(device=dev).manual_seed(2)
    x = torch.randn(777, 64, generator=g, device=dev)
    ident = torch.arange(1, 64, 2, device=dev)
    w = torch.randn(256, 32, generator=g, device=dev)
    mask = (torch.rand(256, 32, generator=g, device=dev) > 0.5).float()
    b = torch.randn(256, generator=g, device=dev)
    pk = fl.pack(w, b, mask=mask, col_map=ident.to(torch.int32), k_in=64)
    out = fl.linear(x, pk)
    want = x[:, ident].double() @ (w * mask).double().t() + b.double()
    assert _gemm_err(out, want) < 1e-6


@pytest.mark.parametrize("M,D,K,H,inverse,coupling,h_t", [
    (1000, 64, 8, 256, False, True, True), (3001, 64, 8, 256, True, True, False), (500, 16, 16, 256, False, False, True),
    (129, 20, 8, 64, False, True, False), (1, 6, 8, 64, True, False, False),
])
def test_linear_rqs_fused_kernel(dev, M, D, K, H, inverse, coupling, h_t):
    """fc_linear_rqs_apply (final layer + spline) against fp64 GEMM -> fp32 parameters -> element-wise kernel; the
    yardstick is the same with the fp32 cuBLAS GEMM (the spline amplifies parameter noise, 1/slope in the inverse)."""
    from flowconductor_b200 import linear as fl

    g = torch.Generator(device=dev).manual_seed(M + D)
    P = 3 * K - 1
    tcols = torch.arange(0, D, 2, device=dev, dtype=torch.int32) if coupling else None
    ccols = torch.arange(1, D, 2, device=dev, dtype=torch.int32) if coupling else None
    d_t = D // 2 if coupling else D
    x = torch.randn(M, D, generator=g, device=dev) * 1.5
    hid = torch.randn(M, H, generator=g, device=dev)
    w = torch.randn(d_t * P, H, generator=g, device=dev) * (4.0 / math.sqrt(H))
    b = torch.randn(d_t * P, generator=g, device=dev)
    pk = fl.pack(w, b, row_map=fl.grouped_row_map(d_t, P, fl.RQS_PPAD[K], dev), n_tile=fl.N_TILE_RQS)
    cfg = _cabi.RqsConfig(K, _cabi.TAILS_LINEAR, 0, int(inverse), -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3,
                          1.0 / math.sqrt(H))
    y, lad = torch.empty_like(x), torch.empty(M, device=dev)
    fl.linear_rqs(fl.T128.from_rows(hid) if h_t else hid, pk, x, y, lad, False, d_t, tcols, ccols, cfg, None)
    args = (K, _cabi.TAILS_LINEAR, inverse, False, -3.0, 3.0, -3.0, 3.0, 1e-3, 1e-3, 1e-3, 1.0 / math.sqrt(H))
    p64 = (hid.double() @ w.double().t() + b.double()).float()
    y2, lad2, _ = ops.rqs_layer(x, p64, tcols, ccols, *args)
    y3, lad3, _ = ops.rqs_layer(x, torch.nn.functional.linear(hid, w, b), tcols, ccols, *args)
    if coupling:
        assert torch.equal(y[:, 1::2], x[:, 1::2])
    q = torch.tensor([0.5, 0.99, 1.0], device=dev)
    for ours, ref, yard, slack in ((y, y2, y3, 3e-6), (lad, lad2, lad3, 3e-5)):
        eo = torch.quantile((ours - ref).abs().flatten().float(), q)
        ey = torch.quantile((yard - ref).abs().flatten().float(), q)
        assert bool((eo <= 4 * ey + slack * max(1.0, ref.abs().max().item())).all()), (eo, ey)


@pytest.mark.parametrize("layout,act,inverse,D,H", [
    (_cabi.AFFINE_BLOCKED, _cabi.SCALE_SIGMOID2, False, 64, 256), (_cabi.AFFINE_BLOCKED, _cabi.SCALE_SOFTPLUS_CLAMP3, True, 10, 64),
    (_cabi.AFFINE_INTERLEAVED, _cabi.SCALE_SOFTPLUS_EPS, False, 100, 64), (_cabi.AFFINE_INTERLEAVED, _cabi.SCALE_SOFTPLUS_EPS, True, 2, 64),
])
def test_linear_affine_fused_kernel(dev, layout, act, inverse, D, H):
    from flowconductor_b200 import linear as fl

    g = torch.Generator(device=dev).manual_seed(D)
    M = 1500
    blocked = layout == _cabi.AFFINE_BLOCKED
    tcols = torch.arange(0, D, 2, device=dev, dtype=torch.int32) if blocked else None
    ccols = torch.arange(1, D, 2, device=dev, dtype=torch.int32) if blocked else None
    d_t = D // 2 if blocked else D
    x = torch.randn(M, D, generator=g, device=dev)
    hid = torch.randn(M, H, generator=g, device=dev)
    w = torch.randn(2 * d_t, H, generator=g, device=dev) / math.sqrt(H)
    b = torch.randn(2 * d_t, generator=g, device=dev) * 0.5
    pk = fl.pack(w, b, row_map=fl.affine_row_map(d_t, layout, dev), n_tile=fl.N_TILE_AFFINE)
    y, lad = torch.empty_like(x), torch.empty(M, device=dev)
    fl.linear_affine(fl.T128.from_rows(hid), pk, x, y, lad, False, d_t, tcols, ccols, act, inverse)
    p64 = (hid.double() @ w.double().t() + b.double()).float()
    y2, lad2 = ops.affine_layer(x, p64, tcols, ccols, layout, act, inverse)
    assert (y - y2).abs().max() < 2e-5 * max(1.0, y2.abs().max().item())
    assert (lad - lad2).abs().max() < 2e-4


def test_linear_argument_errors(dev):
    """The C ABI returns FC_ERR_* (raised by _cabi.check) instead of launching on bad arguments."""
    from flowconductor_b200 import linear as fl

    w = torch.randn(64, 64, device=dev)
    pk = fl.pack(w, None)
    a = torch.randn(10, 64, device=dev)
    with pytest.raises(ValueError):
        fl.linear(torch.randn(10, 32, device=dev), pk)        # wrong reduction length
    with pytest.raises(RuntimeError):
        fl.linear(torch.randn(10, 65, device=dev)[:, :64], pk)  # row pitch not a multiple of 16 bytes (TMA operand)
    with pytest.raises(RuntimeError):
        fl.linear(a.cpu(), pk)                                  # no CPU path
    out = fl.linear(a[:0], pk)                                  # empty batch: no launch, empty result
    assert out.shape == (0, 64)
    with pytest.raises(ValueError):
        fl.T128(10, 20, dev)


def test_tensorcore_path_variants_agree(dev, monkeypatch):
    """The tensor-core inference path with its optimisations switched off one at a time: in-place intermediates
    change nothing bit for bit; the T128 activation layout switches the hidden layers to the staged kernel, which adds
    the skip connection after the GEMM partials instead of before (different fp32 rounding order), so that variant
    agrees to rounding noise.  None of them touches the caller's input."""
    from flowconductor_b200.nn import tensorcore

    wl = workloads.get_workload("cfg2")
    flow = workloads.build_flow(wl)  # fresh initialisation: a smooth map, so rounding-order noise is not amplified
    flow = flow.to(dev)
    x = torch.randn(3000, 64, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    x0 = x.clone()
    outs = []
    with torch.no_grad():
        for inplace, t128 in ((True, True), (False, True), (True, False)):
            monkeypatch.setattr(tensorcore, "INPLACE", inplace)
            monkeypatch.setattr(tensorcore, "T128_ENABLED", t128)
            z, lad = flow._transform(x)
            outs.append((z.clone(), lad.clone()))
            assert torch.equal(x, x0)
    assert torch.equal(outs[1][0], outs[0][0]) and torch.equal(outs[1][1], outs[0][1])
    assert (outs[2][0] - outs[0][0]).abs().max() < 1e-5
    assert (outs[2][1] - outs[0][1]).abs().max() < 1e-4 * max(1.0, outs[0][1].abs().max().item())


def test_stacked_autoregressive_layers_tensorcore_vs_unfused(dev, monkeypatch):
    """Two autoregressive layers back to back (no permutation between them), forward and inverse: the tensor-core
    path (fused final layer, in-place intermediates) against the unfused path.  The inverse re-reads its input D
    times, so it must never be overwritten in place."""
    from flowconductor_b200 import transforms as T
    from flowconductor_b200.nn import tensorcore

    torch.manual_seed(11)
    flows = {
        "affine": T.CompositeTransform([T.MaskedAffineAutoregressiveTransform(6, 64) for _ in range(3)]),
        "prq": T.CompositeTransform([T.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(
            6, 64, num_bins=8, tails="linear", tail_bound=3.0) for _ in range(3)]),
    }
    x = torch.randn(777, 6, generator=torch.Generator().manual_seed(3)).to(dev)
    for name, tr in flows.items():
        tr = tr.to(dev)
        for p in tr.parameters():
            p.data.add_(0.3 * torch.randn_like(p))
        res = {}
        with torch.no_grad():
            for tc in (True, False):
                monkeypatch.setattr(tensorcore, "ENABLED", tc)
                x_in = x.clone()
                y, lad = tr(x_in)
                xi, ladi = tr.inverse(y.clone())
                assert torch.equal(x_in, x)
                res[tc] = (y, lad, xi, ladi)
        # forward: tolerance-level agreement of two fp32 evaluation orders; inverse (D conditioner passes on partially
        # inverted outputs, 1/slope amplification): the round trip of the tensor-core path must be as good as the
        # unfused path's
        # (6 features: the conditioner inputs are padded to 8 columns for the kernels; three strongly perturbed layers in
        # a row amplify single fp32 roundings near knots, hence a quantile + a loose bound on the maximum)
        for a, b in zip(res[True][:2], res[False][:2]):
            err = ((a - b).abs() / max(1.0, b.abs().max().item())).flatten()
            assert torch.quantile(err, 0.999) < 5e-4 and err.max() < 5e-3, (name, float(err.max()))
        rt_tc = (res[True][2] - x).abs().flatten().double()
        rt_un = (res[False][2] - x).abs().flatten().double()
        assert rt_tc.median() <= 2 * rt_un.median() + 1e-6 and rt_tc.max() <= 4 * rt_un.max() + 1e-5, name


def test_host_log_prob_streams_chunks(dev):
    """distributed.host_log_prob (pinned host batch, double-buffered chunks) == flow.log_prob on the whole batch."""
    from flowconductor_b200 import distributed as fdist

    wl = workloads.get_workload("cfg2_tc_small")
    flow = workloads.build_flow(wl).to(dev)
    x = torch.randn(1000, 64, generator=torch.Generator().manual_seed(4)).pin_memory()
    with torch.no_grad():
        want = flow.log_prob(x.to(dev))
    got = fdist.host_log_prob(flow, x, chunk_rows=300)   # 4 chunks, the last one ragged
    torch.cuda.synchronize()
    assert got.shape == (1000,) and (got - want.cpu()).abs().max() < 1e-4 * max(1.0, want.abs().max().item())
    wl4 = workloads.get_workload("cfg4_small")
    flow4 = workloads.build_flow(wl4).to(dev)
    x4, c4 = torch.randn(257, 8).pin_memory(), torch.randn(257, 8).pin_memory()
    with torch.no_grad():
        want4 = flow4.log_prob(x4.to(dev), context=c4.to(dev))
    got4 = fdist.host_log_prob(flow4, x4, chunk_rows=100, context_host=c4)
    torch.cuda.synchronize()
    assert (got4 - want4.cpu()).abs().max() < 1e-4 * max(1.0, want4.abs().max().item())


def test_full_size_cfg3_training_step_is_finite(dev):
    wl = workloads.get_workload("cfg3")
    flow = workloads.build_flow(wl).to(dev)
    opt = torch.optim.Adam(flow.parameters(), lr=1e-3, weight_decay=1e-5)
    x = torch.randn(32768, 16, device=dev)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        loss = -flow.log_prob(x).mean()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(math.isfinite(v) for v in losses) and losses[-1] < losses[0]


@pytest.mark.parametrize("name", ["cfg1", "cfg2_tc_small", "cfg3_small", "cfg4_small", "plin_coupling_small",
                                  "pquad_coupling_small", "prq_coupling_uncond_small"])
def test_cuda_graph_replay_matches_eager(dev, name):
    """graphs.capture (SURVEY §8(f) n2/n4): a replayed graph of log_prob and of the inverse cascade returns exactly
    what the eager call returns, for new inputs copied into the static buffers, and leaves the inputs untouched."""
    from flowconductor_b200 import graphs

    wl = workloads.get_workload(name)
    flow = workloads.build_flow(wl, seed=3).to(dev).eval()
    B, D, C = 384, wl["features"], wl.get("context_features")
    g = torch.Generator().manual_seed(5)
    xs = [torch.randn(B, D, generator=g).to(dev) for _ in range(3)]
    cs = [torch.randn(B, C, generator=g).to(dev) for _ in range(3)] if C else None
    with torch.no_grad():
        if C:
            glp = graphs.capture(lambda x, c: flow.log_prob(x, context=c), xs[0], cs[0])
            ginv = graphs.capture(lambda z, c: flow._transform.inverse(z, context=flow._embedding_net(c)), xs[0], cs[0])
        else:
            glp = graphs.capture(flow.log_prob, xs[0])
            ginv = graphs.capture(flow._transform.inverse, xs[0])
        for i in (1, 2, 0):
            args = (xs[i], cs[i]) if C else (xs[i],)
            keep = xs[i].clone()
            lp = glp(*args, clone=True)
            eager = flow.log_prob(xs[i], context=cs[i]) if C else flow.log_prob(xs[i])
            assert torch.equal(lp, eager), name
            inv, lad = ginv(*args, clone=True)
            e_inv, e_lad = flow._transform.inverse(xs[i], context=cs[i] if C else None)
            assert torch.equal(inv, e_inv) and torch.equal(lad, e_lad), name
            assert torch.equal(xs[i], keep)
    assert glp.replays == 3 and ginv.replays == 3
    with pytest.raises(ValueError):
        glp(*([xs[0][:10]] + ([cs[0][:10]] if C else [])))


def test_cuda_graph_sampler_draws_fresh_noise(dev):
    from flowconductor_b200 import graphs

    flow = workloads.build_flow(workloads.get_workload("cfg3_small"), seed=1).to(dev).eval()
    sampler = graphs.capture_sampler(flow, 256)
    a = sampler(clone=True)
    b = sampler(clone=True)
    assert a.shape == (256, 16) and torch.isfinite(a).all() and torch.isfinite(b).all()
    assert not torch.equal(a, b)  # philox offset advances between replays
    with torch.no_grad():  # samples are distributed like eager samples: log_prob of both is comparable
        lp_g = flow.log_prob(a).mean().item()
        lp_e = flow.log_prob(flow.sample(256)).mean().item()
    assert abs(lp_g - lp_e) < 3.0


@pytest.mark.parametrize("rows,width,masked", [(1000, 64, False), (4100, 256, False), (8192, 128, True)])
def test_fused_residual_block_gradients(dev, rows, width, masked, monkeypatch):
    """tc_autograd.residual_block (ReLU fused into the GEMM operands, ReLU backward gating the input-gradient epilogue,
    bias gradients from the weight-gradient kernel) against the same block in fp64 torch; the yardstick is the error of
    the unfused fp32 torch block."""
    from flowconductor_b200.nn import nets, tc_autograd
    from flowconductor_b200.transforms import made as made_module

    torch.manual_seed(rows + width)
    if masked:
        deg = torch.arange(width) % 7 + 1
        block = made_module.MaskedResidualBlock(deg, autoregressive_features=8, zero_initialization=False)
    else:
        block = nets.resnet.ResidualBlock(width, None, zero_initialization=False)
    block = block.to(dev)
    x = torch.randn(rows, width, device=dev)
    gy = torch.randn(rows, width, device=dev)

    def run(module, inp, g):
        inp = inp.clone().requires_grad_(True)
        out = module(inp)
        grads = torch.autograd.grad((out * g).sum(), [inp] + list(module.parameters()))
        return [out.detach()] + [t.detach() for t in grads]

    launches_before = dict(_cabi.STATS.counts)
    fused = run(block, x, gy)
    assert _cabi.STATS.counts.get("fc_linear_apply", 0) - launches_before.get("fc_linear_apply", 0) == 4
    monkeypatch.setattr(tc_autograd, "ENABLED", False)  # plain torch fp32
    ref32 = run(block, x, gy)
    ref64 = run(block.double(), x.double(), gy.double())
    for got, r32, r64 in zip(fused, ref32, ref64):
        scale = r64.abs().max().item()
        assert (got.double() - r64).abs().max().item() <= 3.0 * (r32.double() - r64).abs().max().item() + 2e-6 * scale


def test_short_reduction_layer_keeps_tensor_core_weight_gradient(dev, monkeypatch):
    """A 16 -> 256 layer (first layer of the cfg-3 MADE): forward / input gradient on cuBLAS fp32 (K < MIN_K), weight and
    bias gradients from fc_linear_splitk_t_apply."""
    from flowconductor_b200.nn import tc_autograd

    g = torch.Generator(device=dev).manual_seed(9)
    x = torch.randn(8192, 16, generator=g, device=dev)
    w = (torch.randn(256, 16, generator=g, device=dev) / 4).requires_grad_(True)
    b = torch.randn(256, generator=g, device=dev).requires_grad_(True)
    mask = (torch.rand(256, 16, generator=g, device=dev) > 0.3).float()
    gy = torch.randn(8192, 256, generator=g, device=dev)
    before = _cabi.STATS.counts.get("fc_linear_splitk_t_apply", 0)
    y = tc_autograd.linear(x, w, b, mask)
    gw, gb = torch.autograd.grad((y * gy).sum(), [w, b])
    assert _cabi.STATS.counts.get("fc_linear_splitk_t_apply", 0) == before + 1
    want_w = (gy.double().t() @ x.double()) * mask.double()
    want_b = gy.double().sum(0)
    ref_w = (gy.t() @ x) * mask
    assert torch.equal(y, torch.nn.functional.linear(x, w * mask, b))
    assert _gemm_err(gw, want_w) <= 2.0 * _gemm_err(ref_w, want_w) + 2e-7
    assert (gb.double() - want_b).abs().max() <= 2e-6 * want_b.abs().max()


@pytest.mark.parametrize("rows,cols", [(4099, 100), (128, 32), (1000, 256), (5, 3)])
def test_pack_transposed_ragged_shapes(dev, rows, cols):
    """fc_linear_pack_transposed on ragged shapes (vector and scalar store paths)."""
    from flowconductor_b200 import linear as fl

    g = torch.Generator(device=dev).manual_seed(rows)
    x = torch.randn(rows, cols, generator=g, device=dev)
    for relu in (False, True):
        pk = fl.pack_transposed(x, relu=relu)
        planes = pk.w  # [2, n_pad, k_pad]: tf32 hi / lo planes of x^T, zero padded
        src = x.relu() if relu else x
        hi = planes[0, :cols, :rows]
        assert (hi.contiguous().view(torch.int32) & 0x1FFF).abs().max() == 0  # tf32: low 13 mantissa bits clear
        assert (hi - src.t()).abs().max() <= 2.0 ** -11 * src.abs().max()
        lo = planes[1, :cols, :rows]
        assert (hi.double() + lo.double() - src.t().double()).abs().max() <= 2.0 ** -21 * src.abs().max()
        assert planes[:, cols:, :].abs().sum() == 0 and planes[:, :, rows:].abs().sum() == 0  # zero padding


def test_cuda_graph_training_step_matches_eager(dev):
    """graphs.GraphedTrainStep: three replayed steps (zero_grad, -log_prob.mean, backward, Adam) leave exactly the
    parameters three eager steps leave; constructing the graph does not train."""
    from flowconductor_b200 import graphs

    wl = workloads.get_workload("cfg3_small")
    flows_ = [workloads.build_flow(wl, seed=2).to(dev) for _ in range(2)]
    flows_[1].load_state_dict(flows_[0].state_dict())
    opts = [torch.optim.Adam(f.parameters(), lr=1e-3, weight_decay=1e-5, capturable=True) for f in flows_]
    g = torch.Generator().manual_seed(8)
    batches = [torch.randn(256, wl["features"], generator=g).to(dev) for _ in range(3)]
    before = [p.detach().clone() for p in flows_[1].parameters()]
    stepper = graphs.GraphedTrainStep(flows_[1], opts[1], lambda x: -flows_[1].log_prob(x).mean(), batches[0])
    for p, b in zip(flows_[1].parameters(), before):
        assert torch.equal(p, b)
    losses = []
    for x in batches:
        opts[0].zero_grad(set_to_none=True)
        loss = -flows_[0].log_prob(x).mean()
        loss.backward()
        opts[0].step()
        losses.append((loss.item(), stepper.step(x).item()))
    for le, lg in losses:
        assert le == lg
    for pe, pg in zip(flows_[0].parameters(), flows_[1].parameters()):
        assert torch.equal(pe, pg)
    with pytest.raises(ValueError):
        graphs.GraphedTrainStep(flows_[0], torch.optim.Adam(flows_[0].parameters()), lambda x: x.sum(), batches[0])


@pytest.mark.parametrize("name", ["lin_fwd_k8", "lin_inv_k8", "lin_fwd_tails_k10", "lin_inv_tails_k10", "lin_fwd_k5"])
def test_linear_spline_kernels(dev, name):
    """fc_linspline_apply / fc_linspline_backward (through transforms.linear_spline / unconstrained_linear_spline,
    the reference's functional API) against golden vectors of the reference's splines/linear.py."""
    gold = load_golden("functions_linear")
    k, has_tails, tb, inverse = gold[name + "/meta"].tolist()
    x = gold[name + "/x"].to(dev).requires_grad_(True)
    u = gold[name + "/params"].to(dev).requires_grad_(True)
    if has_tails:
        y, lad = transforms.unconstrained_linear_spline(x, u, inverse=bool(inverse), tail_bound=tb, tails="linear")
    else:
        y, lad = transforms.linear_spline(x, u, inverse=bool(inverse))
    assert_parity(y, gold[name + "/y32"], gold[name + "/y64"], OUT_TOL, 1.0, name + " y")
    assert_parity(lad, gold[name + "/lad32"], gold[name + "/lad64"], OUT_TOL, 1.0, name + " lad")
    gx, gu = torch.autograd.grad((y * gold[name + "/gy"].to(dev)).sum() + (lad * gold[name + "/gl"].to(dev)).sum(), [x, u])
    s = max(1e-2, gold[name + "/gx64"].abs().mean().item())
    assert_parity(gx, gold[name + "/gx32"], gold[name + "/gx64"], GRAD_TOL, s, name + " gx")
    s = max(1e-2, gold[name + "/gp64"].abs().mean().item())
    assert_parity(gu, gold[name + "/gp32"], gold[name + "/gp64"], GRAD_TOL, s, name + " gp")


def test_linear_spline_domain_error_and_wide_layer(dev):
    """linear.py:45-46 raises InputOutsideDomain without tails; a 64-feature layer exercises the TMA-ring kernel and
    round-trips."""
    with pytest.raises(transforms.InputOutsideDomain):
        transforms.linear_spline(torch.tensor([0.5, 1.5], device=dev), torch.zeros(2, 8, device=dev))
    g = torch.Generator(device=dev).manual_seed(4)
    layer = transforms.PiecewiseLinearCDF([64], num_bins=8, tails="linear", tail_bound=3.0).to(dev)
    x = torch.randn(20000, 64, generator=g, device=dev) * 2
    with torch.no_grad():
        y, lad = layer(x)
        xi, ladi = layer.inverse(y)
        ref_y, ref_lad = restated.linear_cdf({"unnormalized_pdf": layer.unnormalized_pdf.detach().cpu().double()}, "",
                                             x.cpu().double(), 8, "linear", 3.0, False)
    assert (y.cpu().double() - ref_y).abs().max() < 2e-5 and (lad.cpu().double() - ref_lad).abs().max() < 2e-4
    assert (xi - x).abs().max() < 2e-4 and (lad + ladi).abs().max() < 2e-3


def test_cfg3_gradients_tensorcore_path_vs_cublas_path(dev, monkeypatch):
    """cfg 3 (full architecture, trained-like weights) at 8192 rows: loss and every parameter gradient of the
    tensor-core training path (staged row-major GEMMs, fused residual blocks, untransposed-grad_y weight gradients with
    in-kernel bias gradients) and of the same model with every dense layer on cuBLAS fp32 (tc_autograd.ENABLED = False),
    both against the fp64 CPU oracle's autograd."""
    from flowconductor_b200.nn import tc_autograd

    wl = workloads.get_workload("cfg3")
    flow = workloads.build_flow(wl, seed=4)
    # (the SURVEY 8d "trained-like" perturbation makes this 5-layer model's gradient ill-conditioned in fp32 — the
    # cuBLAS path itself is then 90 % away from fp64 — so the weights are a mild random perturbation of the init)
    g = torch.Generator().manual_seed(2)
    state = {k: (v + 0.03 * torch.randn(v.shape, generator=g) if v.is_floating_point() and "mask" not in k else v.clone())
             for k, v in flow.state_dict().items()}
    flow.load_state_dict(state)
    x = torch.randn(8192, wl["features"], generator=torch.Generator().manual_seed(6))
    # fp64 oracle
    specs = workloads.oracle_specs(wl)
    names = [n for n, _ in flow.named_parameters()]
    st64 = {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}
    for n in names:
        st64[n] = st64[n].clone().requires_grad_(True)
    loss64 = -restated.flow_log_prob(st64, specs, x.double(), None).mean()
    ref = dict(zip(names, torch.autograd.grad(loss64, [st64[n] for n in names], allow_unused=True)))
    flow = flow.to(dev)
    xd = x.to(dev)
    errs = {}
    for enabled in (True, False):
        monkeypatch.setattr(tc_autograd, "ENABLED", enabled)
        before = _cabi.STATS.counts.get("fc_linear_splitk_t_apply", 0)
        flow.zero_grad(set_to_none=True)
        loss = -flow.log_prob(xd).mean()
        loss.backward()
        assert (_cabi.STATS.counts.get("fc_linear_splitk_t_apply", 0) > before) == enabled
        assert abs(loss.item() - loss64.item()) <= 2e-5 * abs(loss64.item())
        worst = 0.0
        for n, p in flow.named_parameters():
            r = ref[n] if ref[n] is not None else torch.zeros_like(p, dtype=torch.float64, device="cpu")
            worst = max(worst, ((p.grad.cpu().double() - r).abs().max() / (r.abs().max() + 1e-12)).item())
        errs[enabled] = worst
    # the tensor-core path is as close to fp64 as the cuBLAS fp32 path (factor 3 + an absolute floor)
    assert errs[True] <= 3.0 * errs[False] + 1e-4, errs


@pytest.mark.parametrize("name", ["quad_fwd_k8", "quad_inv_k8", "quad_fwd_tails_k10", "quad_inv_tails_k10", "quad_fwd_k5"])
def test_quadratic_spline_kernels(dev, name):
    """fc_quadspline_apply / fc_quadspline_backward (through transforms.quadratic_spline /
    unconstrained_quadratic_spline) against golden vectors of the reference's splines/quadratic.py."""
    gold = load_golden("functions_quadratic")
    k, has_tails, tb, inverse = gold[name + "/meta"].tolist()
    x = gold[name + "/x"].to(dev).requires_grad_(True)
    uw = gold[name + "/uw"].to(dev).requires_grad_(True)
    uh = gold[name + "/uh"].to(dev).requires_grad_(True)
    if has_tails:
        y, lad = transforms.unconstrained_quadratic_spline(x, uw, uh, inverse=bool(inverse), tail_bound=tb)
    else:
        y, lad = transforms.quadratic_spline(x, uw, uh, inverse=bool(inverse))
    assert_parity(y, gold[name + "/y32"], gold[name + "/y64"], OUT_TOL, 1.0, name + " y")
    assert_parity(lad, gold[name + "/lad32"], gold[name + "/lad64"], OUT_TOL, 1.0, name + " lad")
    gx, gw, gh = torch.autograd.grad((y * gold[name + "/gy"].to(dev)).sum() + (lad * gold[name + "/gl"].to(dev)).sum(),
                                     [x, uw, uh])
    for got, key in ((gx, "gx"), (gw, "gw"), (gh, "gh")):
        s = max(1e-2, gold[name + "/" + key + "64"].abs().mean().item())
        assert_parity(got, gold[name + "/" + key + "32"], gold[name + "/" + key + "64"], GRAD_TOL, s, name + " " + key)


def test_quadratic_spline_wide_layer_round_trip(dev):
    """A 64-feature PiecewiseQuadraticCDF (TMA-ring kernel): forward against the fp64 oracle, inverse round trip."""
    g = torch.Generator(device=dev).manual_seed(5)
    layer = transforms.PiecewiseQuadraticCDF([64], num_bins=8, tails="linear", tail_bound=3.0).to(dev)
    x = torch.randn(20000, 64, generator=g, device=dev) * 2
    with torch.no_grad():
        y, lad = layer(x)
        xi, ladi = layer.inverse(y)
        st = {"unnormalized_widths": layer.unnormalized_widths.detach().cpu().double(),
              "unnormalized_heights": layer.unnormalized_heights.detach().cpu().double()}
        ref_y, ref_lad = restated.quadratic_cdf(st, "", x.cpu().double(), 8, "linear", 3.0, False)
    assert (y.cpu().double() - ref_y).abs().max() < 2e-5 and (lad.cpu().double() - ref_lad).abs().max() < 5e-4
    assert (xi - x).abs().max() < 5e-4 and (lad + ladi).abs().max() < 5e-3


def test_linear_kernels_stay_inside_their_buffers(dev):
    """Guard bands around every output of fc_linear_apply (row-major and T128, ragged and odd tile counts): nothing outside
    the buffer may change.  (Round 2: a T128 output with an odd number of 128-row tiles was written one tile past its end;
    the T128 container now holds an even number of tiles.)"""
    from flowconductor_b200 import linear as fl

    sent, guard = 12345.0, 1 << 16
    torch.manual_seed(0)
    for M in (1, 32, 129, 300, 641):
        for K, N in ((256, 256), (256, 384), (64, 64)):
            W = torch.randn(N, K, device=dev) * 0.1
            b = torch.randn(N, device=dev)
            packed = fl.pack(W, b)
            a_rows = torch.randn(M, K, device=dev)
            ref = a_rows @ W.t() + b
            for a_t, o_t in ((False, False), (False, True), (True, True), (True, False)):
                a = fl.T128.from_rows(a_rows) if a_t else a_rows
                if o_t:
                    out = fl.T128(M, N, dev)
                    n = out.buf.numel()
                    big = torch.full((n + 2 * guard,), sent, device=dev)
                    out.buf = big[guard:guard + n]
                else:
                    n = M * N
                    big = torch.full((n + 2 * guard,), sent, device=dev)
                    out = big[guard:guard + n].view(M, N)
                got = fl.linear(a, packed, out=out, out_t128=o_t, n_out=N)
                torch.cuda.synchronize()
                tag = "M=%d K=%d N=%d a_t128=%s out_t128=%s" % (M, K, N, a_t, o_t)
                assert bool((big[:guard] == sent).all()) and bool((big[guard + n:] == sent).all()), "out-of-bounds write: " + tag
                g = got.to_rows() if o_t else got
                assert (g - ref).abs().max() < 1e-3, tag
