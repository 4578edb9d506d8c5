"""CPU checks of the conditional-conditioner plan (no GPU needed).

The fused conditioner kernel (csrc/fc_conditioner.cu) evaluates a ResidualNet / residual MADE with a context by reading
precomputed context terms g = Wc ctx + bc: one [B, T] matrix in the T128 layout whose columns are the stacked
`context_layer`s of the net (conditioner.pack_context), consumed by the hidden layers in the modes FC_COND_TERM_ADD /
ADD_RELU / GATE.  Here that plan is interpreted in fp64 exactly as the kernel consumes it (T128 indexing from each
layer's first column, padding units of a narrow net, the mode arithmetic) and compared with the mirror modules and with
the oracle's restatement of the reference (oracle/restated.py residual_net / made_net).

The oracle's context branches are not pinned by a golden fixture (the reference package was not available to
generate one); the agreement of these two independent restatements with the kernel's plan is the evidence here.
"""
import ctypes
import os
import subprocess
import tempfile

import pytest
import torch

from flowconductor_b200 import _cabi, conditioner as fcond, linear as fl
from flowconductor_b200.nn import tensorcore
from flowconductor_b200.nn.nets.resnet import ResidualNet
from flowconductor_b200.transforms.made import MADE
from oracle import restated
from tests.helpers import ROOT


def _randomise(net, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in net.parameters():  # away from the near-identity initialisation of the blocks
            scale = 1.0 / p.shape[-1] ** 0.5 if p.dim() == 2 else 0.3
            p.copy_(torch.randn(p.shape, generator=g) * scale)
    return net


def test_path_selection_with_context():
    ctx = torch.zeros(3, 4)
    assert tensorcore.supported_net(ResidualNet(32, 100, 64, context_features=4), ctx)
    assert tensorcore.supported_net(MADE(8, 128, context_features=4, output_multiplier=3), ctx)
    # a context net without its context, a plain net with one: both unsupported
    assert not tensorcore.supported_net(ResidualNet(32, 100, 64, context_features=4), None)
    assert not tensorcore.supported_net(ResidualNet(32, 100, 64), ctx)
    assert not tensorcore.supported_net(MADE(8, 128, context_features=4), None)
    assert not tensorcore.supported_net(MADE(8, 128), ctx)
    # shapes the fused kernel does not cover keep the torch modules
    assert not tensorcore.supported_net(ResidualNet(32, 100, 64, context_features=4, use_batch_norm=True), ctx)
    assert not tensorcore.supported_net(MADE(8, 128, context_features=4, use_residual_blocks=False), ctx)
    assert not tensorcore.supported_net(ResidualNet(32, 100, 32, context_features=4), ctx)  # below MIN_K
    # CPU tensors never take a kernel path
    assert not tensorcore.usable(ResidualNet(32, 100, 64, context_features=4), torch.zeros(3, 32), ctx)


def test_context_fusability_limits():
    # usable() asks the fused conditioner's shape rules with the context columns included (D + C <= 256)
    assert tensorcore.context_k_in(ResidualNet(32, 100, 64, context_features=4), 32, torch.zeros(1, 4)) == 36
    assert tensorcore.context_k_in(MADE(8, 128, context_features=4), 8, torch.zeros(1, 4)) == 8
    assert fcond.supported_store_shape(256, 252, 2, 100)
    assert not fcond.supported_store_shape(256, 260, 2, 100)


def _t128_column_block(terms, col, width_used):
    """[B, width_used] block of a T128 matrix from column `col` on, read as the kernel reads it: pointer
    base + 128 * col, element (r, c) at (r / 128) * 128 * T + ((c / 4) * 128 + r % 128) * 4 + c % 4."""
    buf = terms.buf
    T = terms.width
    r = torch.arange(terms.rows)[:, None]
    c = torch.arange(width_used)[None, :]
    off = 128 * col + (r // 128) * 128 * T + ((c // 4) * 128 + r % 128) * 4 + c % 4
    return buf[off]


def _padded(layer, rows, cols, masked):
    w = layer.weight.detach().double()
    if masked:
        w = w * layer.mask.double()
    W = torch.zeros((rows, cols), dtype=torch.float64)
    W[:w.shape[0], :w.shape[1]] = w
    b = torch.zeros((rows,), dtype=torch.float64)
    b[:w.shape[0]] = layer.bias.detach().double()
    return W, b


def _interpret(net, a, plan, terms, masked):
    """The kernel's layer program in fp64: hidden layers at the padded width, context terms consumed per mode."""
    hp = fcond.padded_hidden(net.initial_layer.weight.shape[0])
    modes = {layer: (mode, col) for layer, mode, col in plan.layers}

    def term(layer):
        mode, col = modes[layer]
        return mode, _t128_column_block(terms, col, hp).double()

    W, b = _padded(net.initial_layer, hp, a.shape[1], masked)
    acc = a.double() @ W.t() + b
    if 0 in modes:
        mode, g = term(0)
        assert mode == _cabi.COND_TERM_ADD_RELU
        acc = acc + g.clamp_min(0)
    h = acc
    for i, blk in enumerate(net.blocks):
        W0, b0 = _padded(blk.linear_layers[0], hp, hp, masked)
        W1, b1 = _padded(blk.linear_layers[1], hp, hp, masked)
        t = h.clamp_min(0) @ W0.t() + b0
        if 1 + 2 * i in modes:
            mode, g = term(1 + 2 * i)
            assert mode == _cabi.COND_TERM_ADD
            t = t + g
        u = t.clamp_min(0) @ W1.t() + b1
        if 2 + 2 * i in modes:
            mode, g = term(2 + 2 * i)
            assert mode == _cabi.COND_TERM_GATE
            h = u * torch.sigmoid(g) + h
        else:
            h = h + u
    Wf, bf = _padded(net.final_layer, net.final_layer.weight.shape[0], hp, masked)
    return h @ Wf.t() + bf


@pytest.mark.parametrize("hidden,blocks,C,B", [(64, 1, 5, 130), (256, 2, 16, 300), (128, 4, 48, 257)])
def test_residual_net_context_plan(hidden, blocks, C, B):
    D_in, out = 10, 23
    net = _randomise(ResidualNet(D_in, out, hidden, context_features=C, num_blocks=blocks), seed=hidden + C)
    g = torch.Generator().manual_seed(B)
    x = torch.randn(B, D_in, generator=g)
    ctx = torch.randn(B, C, generator=g)
    plan = fcond.pack_context(net)
    hp = fcond.padded_hidden(hidden)
    assert plan.width == blocks * hp and plan.width % 16 == 0
    assert [(l, m) for l, m, _ in plan.layers] == [(2 + 2 * i, _cabi.COND_TERM_GATE) for i in range(blocks)]
    assert [c for _, _, c in plan.layers] == [i * hp for i in range(blocks)]
    # the padding rows of the stacked weight are zero
    for i in range(blocks):
        assert not plan.weight[i * hp + hidden:(i + 1) * hp].any() and not plan.bias[i * hp + hidden:(i + 1) * hp].any()
    terms = fl.T128.from_rows((ctx.double() @ plan.weight.double().t() + plan.bias.double()).float())
    # (terms rounded to fp32, as the kernel receives them: compare against the modules fed the same rounding)
    ours = _interpret(net, torch.cat((x, ctx), 1), plan, terms, masked=False)
    net64 = net.double()
    state = {k: v.double() for k, v in net.state_dict().items()}
    with torch.no_grad():
        ref_mod = net64(x.double(), ctx.double())
        ref_or = restated.residual_net(state, "", x.double(), ctx.double(), num_blocks=blocks)
    assert torch.allclose(ref_mod, ref_or, rtol=0, atol=1e-12)
    tol = 1e-5 * max(1.0, float(ref_or.abs().max()))  # fp32 rounding of the terms
    assert float((ours - ref_or).abs().max()) <= tol
    # with fp64 terms the interpretation is the reference to 1e-12
    t64 = fl.T128(B, plan.width, "cpu")
    t64.buf = _t128_fp64(ctx.double() @ plan.weight.double().t() + plan.bias.double(), plan.width)
    ours64 = _interpret(net, torch.cat((x, ctx), 1), plan, t64, masked=False)
    assert float((ours64 - ref_or).abs().max()) <= 1e-12 * max(1.0, float(ref_or.abs().max()))


def _t128_fp64(rows_mat, width):
    """T128 buffer (fp64) of a row-major matrix: the layout of linear.T128.from_rows, kept in double."""
    rows = rows_mat.shape[0]
    tiles = (rows + 127) // 128
    tiles += tiles & 1
    padded = torch.zeros((tiles * 128, width), dtype=torch.float64)
    padded[:rows] = rows_mat
    return padded.view(tiles, 128, width // 4, 4).permute(0, 2, 1, 3).reshape(-1)


@pytest.mark.parametrize("hidden,blocks,C,B", [(256, 2, 8, 200), (64, 1, 3, 129), (128, 3, 40, 300)])
def test_made_context_plan(hidden, blocks, C, B):
    D, mult = 12, 7
    net = _randomise(MADE(D, hidden, context_features=C, num_blocks=blocks, output_multiplier=mult), seed=hidden + C)
    g = torch.Generator().manual_seed(B)
    x = torch.randn(B, D, generator=g)
    ctx = torch.randn(B, C, generator=g)
    plan = fcond.pack_context(net)
    hp = fcond.padded_hidden(hidden)
    assert plan.width == (1 + blocks) * hp
    assert [(l, m) for l, m, _ in plan.layers] == (
        [(0, _cabi.COND_TERM_ADD_RELU)] + [(1 + 2 * i, _cabi.COND_TERM_ADD) for i in range(blocks)])
    terms = fl.T128(B, plan.width, "cpu")
    terms.buf = _t128_fp64(ctx.double() @ plan.weight.double().t() + plan.bias.double(), plan.width)
    ours = _interpret(net, x, plan, terms, masked=True)
    state = {k: (v.double() if v.is_floating_point() else v) for k, v in net.state_dict().items()}
    with torch.no_grad():
        ref_mod = net.double()(x.double(), ctx.double())
        ref_or = restated.made_net(state, "", x.double(), ctx.double(), num_blocks=blocks)
    scale = max(1.0, float(ref_or.abs().max()))
    assert float((ref_mod - ref_or).abs().max()) <= 1e-12 * scale
    assert float((ours - ref_or).abs().max()) <= 1e-12 * scale


def test_plain_nets_have_no_context_plan():
    assert fcond.pack_context(ResidualNet(8, 10, 64)) is None
    assert fcond.pack_context(MADE(8, 64)) is None


def test_gate_sigmoid_host_arithmetic():
    """fc_sigmoid of fc_math.cuh (the context gate) against torch.sigmoid in fp64.  The host build evaluates the same
    formula with libm's exp2f and an IEEE reciprocal; on the device ex2.approx / rcp.approx + Newton add ~2 ulp."""
    src = os.path.join(ROOT, "flowconductor_b200", "csrc", "fc_math.cuh")
    with tempfile.TemporaryDirectory() as tmp:
        shim = os.path.join(tmp, "gate.cpp")
        lib = os.path.join(tmp, "libgate.so")
        with open(shim, "w") as f:
            f.write('#include "%s"\nextern "C" void gate(const float* z, float* s, long n) {\n'
                    '  for (long i = 0; i < n; ++i) s[i] = fc::fc_sigmoid(z[i]);\n}\n' % src)
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", shim, "-o", lib])
        L = ctypes.CDLL(lib)
        z = torch.cat((torch.linspace(-40.0, 40.0, 200001), torch.randn(100000) * 3)).float()
        s = torch.empty_like(z)
        L.gate(ctypes.c_void_p(z.data_ptr()), ctypes.c_void_p(s.data_ptr()), ctypes.c_long(z.numel()))
    ref = torch.sigmoid(z.double())
    err = (s.double() - ref).abs()
    assert float(err.max()) < 1.5e-7
    # relative: the rounding of the argument |z| log2(e) costs |z| 8.6e-8 of e^-|z| (fc_math.cuh, fc_sigmoid_parts)
    assert bool((err / ref <= z.double().abs() * 1e-7 + 3e-7).all())
