"""Host logic of the incremental autoregressive inverse of a conditional MADE (`context_features`): the program
`made_inverse.compile_made` emits for it, interpreted on the CPU as csrc/fc_made_inverse.cuh does — the context arrays
prefilled with bias + act(term) from the T128 term matrix, every other unit NaN until a task writes it — must reproduce
the reference's D-pass inverse with the context (oracle/restated.py `_autoregressive`)."""
import pytest
import torch

from flowconductor_b200 import _cabi, made_inverse
from flowconductor_b200 import conditioner as fcond
from flowconductor_b200.transforms import made as made_module
from oracle import restated

INIT_BIAS = made_inverse.INIT_BIAS


def _t128(rows_mat):
    """fp64 T128 buffer of a row-major [B, T] matrix (the layout of linear.T128, kept in double)."""
    B, T = rows_mat.shape
    tiles = (B + 127) // 128
    tiles += tiles & 1
    padded = torch.zeros((tiles * 128, T), dtype=torch.float64)
    padded[:B] = rows_mat
    return padded.view(tiles, 128, T // 4, 4).permute(0, 2, 1, 3).reshape(-1)


def _terms(prog, ctx):
    """The context terms of `ctx` in fp64, as the T128 buffer the kernel reads."""
    plan = prog.context
    return _t128(ctx.double() @ plan.weight.double().t() + plan.bias.double())


def emulate_context_program(prog, z, terms, invert_feature):
    """The kernel's interpretation of `prog` in fp64 (as tests/helpers.py emulate_made_program), with the prefill of the
    context arrays: unit j of array `array` starts at bias[b_off + j] + act(terms[r, column + j]), read at the T128 index
    (r / 128) * 128 T + (c / 4) * 512 + (r % 128) * 4 + c % 4.  Unwritten state is NaN."""
    z = z.double()
    B, T = z.shape[0], prog.context.width
    X = z.t().clone()
    H = torch.full((prog.n_arrays, prog.hidden, B), float("nan"), dtype=torch.float64)
    PT = torch.full((prog.params_per_feature, B), float("nan"), dtype=torch.float64)
    lad = torch.zeros((B,), dtype=torch.float64)
    w = prog.weights.detach().double().cpu()
    bias = prog.bias.detach().double().cpu()
    r = torch.arange(B)[None, :]
    for array, column, b_off, relu in prog.term_arrays:
        c = column + torch.arange(prog.hidden)[:, None]
        g = terms[(r // 128) * 128 * T + (c // 4) * 512 + (r % 128) * 4 + c % 4]
        H[array - 1] = bias[b_off:b_off + prog.hidden][:, None] + (g.clamp_min(0) if relu else g)
    for _, hdr, tasks in prog.tasks():
        rows, width, woff, feat = hdr["rows"], hdr["width"], hdr["w_off4"], hdr["feature"]
        mat = w[woff * 4 + 128: woff * 4 + 128 + rows * width].reshape(rows, width)
        results = []
        for t in tasks:
            nj, kn, k0, j0, c0 = t["nj"], t["kn"], t["k0"], t["j0"], t["c0"]
            dst = H[t["out_array"] - 1] if t["out_array"] > 0 else PT
            v = bias[t["b_off"]:t["b_off"] + nj][:, None].expand(nj, B).clone() if t["flags"] & INIT_BIAS \
                else dst[j0:j0 + nj].clone()
            if kn > 0:
                a = (X if t["in_array"] == 0 else H[t["in_array"] - 1])[k0:k0 + kn]
                if t["flags"] & made_inverse.RELU_IN:
                    a = a.clamp_min(0)
                v = v + mat[:kn, c0:c0 + nj].t() @ a
            if t["res_array"]:
                v = v + H[t["res_array"] - 1][j0:j0 + nj]
            results.append((dst, j0, nj, v))
        for dst, j0, nj, v in results:
            dst[j0:j0 + nj] = v
        if feat >= 0:
            assert not torch.isnan(PT).any()
            xf, lf = invert_feature(X[feat].clone(), PT.t().clone())
            X[feat] = xf
            lad = lad + lf
            PT.fill_(float("nan"))
    return X.t().contiguous(), lad


def _net(D, H, blocks, C, P=2, seed=0):
    torch.manual_seed(seed)
    net = made_module.MADE(features=D, hidden_features=H, context_features=C, num_blocks=blocks, output_multiplier=P)
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * 0.1)
    return net


def _affine_inverse(zf, params):
    y, lad = restated.affine_elementwise(zf[:, None], params, "interleaved", "softplus_eps", True)
    return y[:, 0], lad


@pytest.mark.parametrize("D,H,blocks,C", [(1, 32, 1, 3), (2, 256, 2, 8), (5, 6, 3, 1), (16, 50, 2, 8), (16, 4, 1, 3),
                                          (21, 32, 5, 70), (5, 50, 4, 70), (21, 6, 2, 8), (16, 256, 1, 1)])
def test_context_program_reproduces_d_pass_inverse(D, H, blocks, C):
    net = _net(D, H, blocks, C, seed=D * 100 + H + C)
    prog = made_inverse.compile_made(net, 2)
    assert prog is not None and prog.context is not None
    g = torch.Generator().manual_seed(blocks)
    B = 37
    z = torch.randn(B, D, generator=g, dtype=torch.float64) * 1.3
    ctx = torch.randn(B, C, generator=g, dtype=torch.float64)
    x, lad = emulate_context_program(prog, z, _terms(prog, ctx), _affine_inverse)
    state = {"autoregressive_net." + k: v.double() for k, v in net.state_dict().items()}
    spec = {"kind": "maf_affine", "prefix": "", "num_blocks": blocks, "hidden_features": H}
    x_ref, lad_ref = restated.apply_layer(state, spec, z, ctx, inverse=True)
    # (relative to the outputs' scale: the 16-feature nets push some rows to |x| ~ 1e7)
    assert (x - x_ref).abs().max() < 1e-9 * max(1.0, float(x_ref.abs().max()))
    assert (lad - lad_ref).abs().max() < 1e-9 * max(1.0, float(lad_ref.abs().max()))


def test_context_program_rq_spline():
    """A rational-quadratic layer (cfg 3's family: P = 3 K + 1 without tails) with a context, on 140 rows (two T128 tiles)."""
    D, H, blocks, C, K = 5, 32, 2, 8, 4
    P = 3 * K + 1
    net = _net(D, H, blocks, C, P=P, seed=5)
    prog = made_inverse.compile_made(net, P)
    g = torch.Generator().manual_seed(1)
    z = torch.rand(140, D, generator=g, dtype=torch.float64) * 2 - 1
    ctx = torch.randn(140, C, generator=g, dtype=torch.float64)
    spec = {"kind": "maf_prq", "prefix": "", "num_blocks": blocks, "hidden_features": H, "num_bins": K, "tails": None}

    def invert(zf, params):
        y, lad = restated.rq_elementwise(zf[:, None], params, K, None, 1.0, True, None, True, constrained_bound=1.2)
        return y[:, 0], lad

    x, lad = emulate_context_program(prog, z, _terms(prog, ctx), invert)
    state = {"autoregressive_net." + k: v.double() for k, v in net.state_dict().items()}
    x_ref, lad_ref = restated.apply_layer(state, spec, z, ctx, inverse=True)
    assert (x - x_ref).abs().max() < 1e-9 and (lad - lad_ref).abs().max() < 1e-9


@pytest.mark.parametrize("D,H,blocks", [(16, 48, 2), (5, 6, 3), (2, 256, 1)])
def test_context_program_is_the_plain_program_without_init_bias(D, H, blocks):
    """The conditional program is the context-free program of the same weights, except that the tasks writing a context
    array (1 and 2 b + 2) accumulate onto the prefill instead of initialising from the bias."""
    net = _net(D, H, blocks, 8)
    plain = made_module.MADE(features=D, hidden_features=H, num_blocks=blocks, output_multiplier=2)
    plain.load_state_dict({k: v for k, v in net.state_dict().items() if "context_layer" not in k})
    prog, ref = made_inverse.compile_made(net, 2), made_inverse.compile_made(plain, 2)
    assert ref.context is None and ref.term_arrays == []
    ctx_arrays = {1} | {2 * b + 2 for b in range(blocks)}
    assert [a for a, _, _, _ in prog.term_arrays] == sorted(ctx_arrays)
    # (the weight streams differ in the flag words of the phase records they carry)
    assert prog.weights.shape == ref.weights.shape and torch.equal(prog.bias, ref.bias)
    n_ctx_tasks = 0
    for (_, _, tasks), (_, _, ref_tasks) in zip(prog.tasks(), ref.tasks()):
        for t, rt in zip(tasks, ref_tasks):
            if t["out_array"] in ctx_arrays:
                n_ctx_tasks += 1
                assert not t["flags"] & INIT_BIAS
                rt = dict(rt, flags=rt["flags"] & ~INIT_BIAS)
            assert t == rt
    assert n_ctx_tasks > 0
    assert (prog.phases_np.shape == ref.phases_np.shape)


def test_term_plan_layout():
    """Columns i * ceil4(H) + j hold the i-th context layer's row of sorted unit j (degree order, the program's `perm`);
    padding columns are zero; the width is a multiple of 16; each array's bias offset is its layer's."""
    D, H, blocks, C = 7, 50, 3, 5
    net = _net(D, H, blocks, C)
    prog = made_inverse.compile_made(net, 2)
    plan = prog.context
    stride = 52
    assert plan.width == 208 and plan.width % 16 == 0 and plan.features == C
    perm = torch.argsort(net.initial_layer.degrees, stable=True)
    assert bool((net.initial_layer.degrees[perm][1:] >= net.initial_layer.degrees[perm][:-1]).all())
    layers = [net.context_layer] + [b.context_layer for b in net.blocks]
    for i, (lin, (array, column, b_off, relu)) in enumerate(zip(layers, prog.term_arrays)):
        assert column == i * stride and relu == int(i == 0)
        assert array == (1 if i == 0 else 2 * i)
        assert torch.equal(plan.weight[column:column + H], lin.weight.detach()[perm])
        assert torch.equal(plan.bias[column:column + H], lin.bias.detach()[perm])
        assert not plan.weight[column + H:column + stride].any() and not plan.bias[column + H:column + stride].any()
        src = net.initial_layer if i == 0 else net.blocks[i - 1].linear_layers[0]
        assert torch.equal(prog.bias[b_off:b_off + H], src.bias.detach()[perm])
    assert not plan.weight[len(layers) * stride:].any()
    assert plan.layers == [(a, _cabi.COND_TERM_ADD_RELU if r else _cabi.COND_TERM_ADD, c) for a, c, _, r in prog.term_arrays]


def test_too_many_context_layers_do_not_compile():
    net = _net(4, 16, _cabi.MADE_MAX_TERM_ARRAYS, 3)  # 1 + 8 context layers
    assert made_inverse.supported_made(net) and made_inverse.compile_made(net, 2) is None
    net = _net(4, 16, _cabi.MADE_MAX_TERM_ARRAYS - 1, 3)
    assert len(made_inverse.compile_made(net, 2).term_arrays) == _cabi.MADE_MAX_TERM_ARRAYS


def _old_pack_context(net):
    """The fused path's stacking as it was written before `stack_context` was factored out of it."""
    blocks = list(net.blocks)
    if hasattr(net, "context_layer"):
        src = [(0, _cabi.COND_TERM_ADD_RELU, net.context_layer)]
        src += [(1 + 2 * i, _cabi.COND_TERM_ADD, b.context_layer) for i, b in enumerate(blocks)]
    else:
        src = [(2 + 2 * i, _cabi.COND_TERM_GATE, b.context_layer) for i, b in enumerate(blocks)]
    hp = fcond.padded_hidden(net.initial_layer.weight.shape[0])
    C = src[0][2].weight.shape[1]
    weight = torch.zeros((hp * len(src), C))
    bias = torch.zeros((hp * len(src),))
    layers = []
    for i, (layer, mode, lin) in enumerate(src):
        n = lin.weight.shape[0]
        weight[i * hp:i * hp + n] = lin.weight.detach()
        bias[i * hp:i * hp + n] = lin.bias.detach()
        layers.append((layer, mode, i * hp))
    return weight, bias, layers, weight.shape[0]


@pytest.mark.parametrize("kind,hidden,blocks,C", [("made", 256, 2, 8), ("made", 64, 3, 5), ("resnet", 100, 2, 16),
                                                  ("resnet", 128, 4, 40)])
def test_fused_context_plan_unchanged(kind, hidden, blocks, C):
    from flowconductor_b200.nn.nets.resnet import ResidualNet

    torch.manual_seed(hidden + C)
    net = (_net(12, hidden, blocks, C, P=3) if kind == "made"
           else ResidualNet(10, 23, hidden, context_features=C, num_blocks=blocks))
    plan = fcond.pack_context(net)
    weight, bias, layers, width = _old_pack_context(net)
    assert torch.equal(plan.weight, weight) and torch.equal(plan.bias, bias)
    assert plan.layers == layers and plan.width == width and plan.features == C


def test_routing_keeps_unsupported_calls_on_the_d_pass_path():
    """Context layers on some blocks only, batch norm: not compiled.  A net with context layers called without context,
    a plain net called with one, CPU tensors: not routed to the kernel."""
    net = _net(6, 16, 2, 3)
    assert made_inverse.supported_made(net)
    del net.blocks[1].context_layer
    assert not made_inverse.supported_made(net)
    assert not made_inverse.supported_made(made_module.MADE(6, 16, context_features=3, use_batch_norm=True))
    net, plain = _net(6, 16, 2, 3), made_module.MADE(6, 16)
    z, ctx = torch.zeros(4, 6), torch.zeros(4, 3)
    with torch.no_grad():
        assert not made_inverse.usable(net, z, None)
        assert not made_inverse.usable(plain, z, ctx)
        assert not made_inverse.usable(net, z, ctx)  # CPU
