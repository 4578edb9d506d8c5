"""Host side of the fused conditioner kernel (csrc/fc_conditioner.cu, C ABI `fc_conditioner_*`).

`PackedConditioner` is the packed form of a whole ResidualNet (flowcon/nn/nets/resnet.py:59-100) or residual MADE
(flowcon/transforms/made.py:205-283): every layer's weights as fp16 (hi, lo) planes in the shared-memory image of the
kernel's weight ring, in one buffer, plus the per-layer bias / inverse-scale vectors and the layer table
(`struct fc_conditioner`).  `rqs_apply` launches conditioner + rational-quadratic spline as ONE kernel on torch's current
stream.  No fallback: CPU tensors or a missing library raise.

Conditional nets (`context_features`): every `context_layer` of the net is stacked into one [T, C] matrix
(`ContextPlan`, T = hidden width padded to the kernel's x the number of context layers), `context_terms` evaluates
Wc ctx + bc for the whole batch in one launch as a T128 matrix, and the `*_apply` calls hand it to the kernel, whose
hidden layers consume their columns (FC_COND_TERM_* of include/flowcon_b200.h).  The terms do not depend on the
conditioner's inputs: a D-pass autoregressive inverse computes them once.
"""
import ctypes

import torch

from . import _cabi

HIDDEN_WIDTHS = (128, 256)  # what the kernel runs; narrower nets are zero-padded to 128 at pack time (exact: the padding
                            # units are relu(0) = 0 and multiply zero weights)
MAX_K_IN = 256
RQS_PPAD = {8: 24, 16: 48}  # linear tails (kept for callers of the first fused shapes)
RQS_BINS = (8, 10, 16)      # bin counts with a register-resident instantiation of the fused kernel
SOS_PPAD = 48               # 3 n + 1 = 31 parameters per feature for n = 10, two features per 96-column tile
SOS_SIGMOIDS = (10,)
AFFINE_PPAD = 24            # a 24-column slot holds the (raw scale, shift) pairs of AFFINE_GROUP consecutive features
AFFINE_GROUP = 12
MAX_BLOCKS = (_cabi.COND_MAX_LAYERS - 2) // 2


def _ceil_to(v, m):
    return (v + m - 1) // m * m


class PackedConditioner:
    """Packed weights of a whole conditioner.  Keeps the device buffers alive; `struct` is what the C ABI takes."""

    def __init__(self, weights, vectors, struct, hidden, k_in, n_final_tiles, num_bins, context=None):
        self.weights, self.vectors, self.struct = weights, vectors, struct
        # hidden: the width the kernel runs (128 / 256); num_bins: bins of the spline, or None for other bijections
        self.hidden, self.k_in, self.n_final_tiles, self.num_bins = hidden, k_in, n_final_tiles, num_bins
        self.context = context  # ContextPlan of a conditional net, else None


MIN_K_TC = 64  # context widths from here on take the tensor-core GEMM for their terms (nn/tc_autograd.py MIN_K)


class ContextPlan:
    """The context layers of a conditional net stacked into one affine map ctx -> [B, width] (T128).  `layers`: the
    (conditioner layer index, FC_COND_TERM_* mode, first column) of every layer that consumes terms; the columns of
    padding units (a net narrower than the kernel's width) have zero weights and bias."""

    def __init__(self, weight, bias, layers, width, linear):
        self.weight, self.bias, self.layers, self.width = weight, bias, layers, width
        self.features = weight.shape[1]
        self.linear = linear  # linear.PackedLinear for the tensor-core GEMM (C >= MIN_K_TC), else None


def pack_context(net):
    """ContextPlan of a conditional ResidualNet (a gate per block, resnet.py:45-52) or residual MADE (initial layer
    made.py:274-279, the first layer of every block made.py:170-181); None for a net without context layers."""
    blocks = list(net.blocks)
    if hasattr(net, "context_layer"):  # MADE
        src = [(0, _cabi.COND_TERM_ADD_RELU, net.context_layer)]
        src += [(1 + 2 * i, _cabi.COND_TERM_ADD, b.context_layer) for i, b in enumerate(blocks)]
    elif getattr(net, "context_features", None) is not None:  # ResidualNet
        src = [(2 + 2 * i, _cabi.COND_TERM_GATE, b.context_layer) for i, b in enumerate(blocks)]
    else:
        return None
    return stack_context(src, padded_hidden(net.initial_layer.weight.shape[0]))


def stack_context(src, stride, order=None):
    """ContextPlan of the context layers `src` [(consumer, FC_COND_TERM_* mode, nn.Linear)]: layer i's outputs at
    columns i * stride + j, taken in the order `order` (an index into the outputs) when given; the width is padded to a
    multiple of 16 and the padding columns have zero weights and bias.  The incremental MADE inverse (made_inverse.py)
    stacks its context layers here too, in the degree order of its hidden units."""
    from . import linear as fl

    ref = src[0][2].weight
    C = ref.shape[1]
    width = _ceil_to(stride * len(src), 16)
    weight = torch.zeros((width, C), dtype=torch.float32, device=ref.device)
    bias = torch.zeros((width,), dtype=torch.float32, device=ref.device)
    layers = []
    for i, (layer, mode, lin) in enumerate(src):
        w = lin.weight.detach()
        b = lin.bias.detach() if lin.bias is not None else None
        if order is not None:
            w = w[order]
            b = b[order] if b is not None else None
        n = w.shape[0]
        weight[i * stride:i * stride + n] = w
        if b is not None:
            bias[i * stride:i * stride + n] = b
        layers.append((layer, mode, i * stride))
    linear = None
    if C >= MIN_K_TC and ref.is_cuda:  # (a plan of CPU modules only serves host-side tests of the stacking)
        c4 = _ceil_to(C, 4)
        cm = None if c4 == C else torch.arange(C, dtype=torch.int32, device=ref.device)
        linear = fl.pack(weight, bias, col_map=cm, k_in=c4)
    return ContextPlan(weight, bias, layers, width, linear)


def context_terms(packed, ctx):
    """Wc ctx + bc of every context layer, [B, width] as a linear.T128: ONE launch (fc_context_terms below the tensor-core
    GEMM's minimum reduction, else fc_linear_apply).  `packed`: a PackedConditioner of a conditional net or its ContextPlan."""
    from . import linear as fl

    plan = packed.context if isinstance(packed, PackedConditioner) else packed
    if plan is None:
        raise ValueError("the conditioner has no context layers")
    _cabi.require_cuda_f32(ctx, "context")
    if ctx.dim() != 2 or ctx.shape[1] != plan.features:
        raise ValueError("context has shape {}, the net expects {} features".format(tuple(ctx.shape), plan.features))
    if plan.linear is not None:
        a = ctx
        k = plan.linear.k_in
        if not (k == ctx.shape[1] and ctx.stride(1) == 1 and ctx.stride(0) % 4 == 0 and ctx.data_ptr() % 16 == 0):
            a = ctx.new_zeros((ctx.shape[0], k))  # 16-byte row pitch for the GEMM's TMA loads
            a[:, :ctx.shape[1]] = ctx
        return fl.linear(a, plan.linear, out_t128=True)
    L = _cabi.lib()
    ctx, cp, ldc = _cabi.rows(ctx)
    out = fl.T128(ctx.shape[0], plan.width, ctx.device)
    with torch.cuda.device(ctx.device), _cabi.launch("fc_context_terms", ctx.device):
        rc = L.fc_context_terms(cp, ldc, ctx.shape[0], plan.features, plan.weight.data_ptr(), plan.bias.data_ptr(),
                                plan.width, out.buf.data_ptr(), _cabi.stream_ptr(ctx.device))
    _cabi.check(rc, "fc_context_terms")
    return out


def _bind_terms(packed, terms, B):
    """Point the layer table at this call's context terms (a conditional net needs them, any other net takes none)."""
    if packed.context is None:
        if terms is not None:
            raise ValueError("context terms given for a conditioner without context layers")
        return
    if terms is None:
        raise ValueError("a conditioner with context layers needs its context terms (conditioner.context_terms)")
    if terms.rows != B or terms.width != packed.context.width:
        raise ValueError("context terms are [{}, {}], expected [{}, {}]".format(terms.rows, terms.width, B,
                                                                                  packed.context.width))
    base = terms.buf.data_ptr()
    for layer, _, col in packed.context.layers:
        e = packed.struct.layers[layer]
        e.terms = base + 4 * terms.TILE * col  # T128: a column group is the slow index inside a 128-row tile
        e.term_width = terms.width


def _pack_layer(L, dev, blob, offset, layer, mask, n_pad, k_pad, bn, row_map=None, col_map=None):
    w = _cabi.require_cuda_f32(layer.weight.detach(), "weight")
    if w.stride(1) != 1:
        w = w.contiguous()
    N, K = w.shape
    b = layer.bias
    if b is not None:
        b = _cabi.require_cuda_f32(b.detach(), "bias").contiguous()
    if mask is not None:
        mask = _cabi.require_cuda_f32(mask.detach(), "mask")
        if mask.stride(1) != 1:
            mask = mask.contiguous()
    vec = (torch.empty((n_pad,), dtype=torch.float32, device=dev), torch.empty((2,), dtype=torch.float32, device=dev))
    for m in (row_map, col_map):
        if m is not None:
            assert m.dtype == torch.int32 and m.is_cuda and m.is_contiguous()
    with _cabi.launch("fc_conditioner_pack_layer", dev):
        rc = L.fc_conditioner_pack_layer(w.data_ptr(), w.stride(0), mask.data_ptr() if mask is not None else None,
                                         mask.stride(0) if mask is not None else 0,
                                         b.data_ptr() if b is not None else None, N, K,
                                         row_map.data_ptr() if row_map is not None else None,
                                         col_map.data_ptr() if col_map is not None else None, n_pad, k_pad, bn,
                                         blob.data_ptr() + offset, vec[0].data_ptr(), vec[1].data_ptr(),
                                         _cabi.stream_ptr(dev))
    _cabi.check(rc, "fc_conditioner_pack_layer")
    return vec


def padded_hidden(hidden):
    """Width the kernel runs for a net of this hidden width, or None."""
    if hidden <= 0 or hidden % 4:
        return None
    return 128 if hidden <= 128 else (256 if hidden <= 256 else None)


def rqs_ppad(num_bins, tails):
    """Accumulator columns per feature of the final layer's tiles for a spline with these bins / tails, or None."""
    P = 3 * num_bins - 1 if tails == "linear" else 3 * num_bins + 1
    if num_bins not in RQS_BINS or P > 48:
        return None
    return 24 if P <= 24 else 48


VEC_BYTES = 20480  # kVecBytes of the kernel: the bias of every output column of every layer is staged in shared memory


def _vectors_fit(hidden, num_blocks, ppad, d_t, group=1):
    """The kernel keeps every layer's bias in shared memory: (1 + 2 blocks) hidden-wide layers + the final layer's tiles."""
    if d_t is None:
        return True
    feats = 96 // ppad * group
    total_cols = (1 + 2 * num_blocks) * padded_hidden(hidden) + (d_t + feats - 1) // feats * 96
    return total_cols * 4 + 4 * _cabi.COND_MAX_LAYERS <= VEC_BYTES


def supported_shape(hidden, k_in, num_blocks, num_bins, tails="linear", d_t=None):
    ppad = rqs_ppad(num_bins, tails)
    return (padded_hidden(hidden) is not None and 0 < k_in <= MAX_K_IN and k_in % 4 == 0
            and 1 <= num_blocks <= MAX_BLOCKS and ppad is not None and _vectors_fit(hidden, num_blocks, ppad, d_t))


def supported_sos_shape(hidden, k_in, num_blocks, n_sigmoids, d_t=None):
    return (padded_hidden(hidden) is not None and 0 < k_in <= MAX_K_IN and k_in % 4 == 0
            and 1 <= num_blocks <= MAX_BLOCKS and n_sigmoids in SOS_SIGMOIDS
            and _vectors_fit(hidden, num_blocks, SOS_PPAD, d_t))


def supported_affine_shape(hidden, k_in, num_blocks, d_t=None):
    return (padded_hidden(hidden) is not None and 0 < k_in <= MAX_K_IN and k_in % 4 == 0
            and 1 <= num_blocks <= MAX_BLOCKS and _vectors_fit(hidden, num_blocks, AFFINE_PPAD, d_t, AFFINE_GROUP))


STORE_PPAD = 48


def supported_store_shape(hidden, k_in, num_blocks, n_out):
    """`fc_conditioner_store_apply`: any final width (padded to whole 96-column tiles)."""
    return (n_out > 0 and padded_hidden(hidden) is not None and 0 < k_in <= MAX_K_IN and k_in % 4 == 0
            and 1 <= num_blocks <= MAX_BLOCKS and _vectors_fit(hidden, num_blocks, STORE_PPAD, (n_out + 47) // 48))


def pack(net, P, ppad, d_t, col_map=None, k_in=None, num_bins=None, final_row_map=None, group=1, context=None):
    """Pack `net` (initial_layer, blocks[*].linear_layers[0..1], final_layer; optional `.mask` per layer, made.py:72)
    for the `fc_conditioner_*_apply` kernels: P parameters per feature in `ppad` accumulator columns (final_row_map /
    group: explicit placement of the final layer's rows, `group` features per `ppad`-column slot).  col_map / k_in:
    scatter of the first layer's input columns (a coupling layer's conditioner reads the full-width inputs:
    coupling.py:82-86 folded into the weights; a conditional ResidualNet's initial layer reads [inputs | context]).
    context: the net's ContextPlan (conditional nets)."""
    L = _cabi.lib()
    init, fin = net.initial_layer, net.final_layer
    dev = init.weight.device
    hidden_real = init.weight.shape[0]
    hidden = padded_hidden(hidden_real)
    k_in = init.weight.shape[1] if k_in is None else k_in
    nb = len(net.blocks)
    if hidden is None or not (0 < k_in <= MAX_K_IN and k_in % 4 == 0 and 1 <= nb <= MAX_BLOCKS) or 96 % ppad or P > ppad:
        raise ValueError("conditioner shape not supported by the fused kernel")
    if final_row_map is None and fin.weight.shape[0] != d_t * P:
        raise ValueError("final layer has {} outputs, expected {} x {}".format(fin.weight.shape[0], d_t, P))
    feats = 96 // ppad * group
    n_final_tiles = (d_t + feats - 1) // feats
    # k-values the layers after the first multiply: the 128-wide kernel skips a padding chunk (nets of <= 64 units)
    hk = _ceil_to(hidden_real, 64) if hidden == 128 else hidden
    layers = [(init, _cabi.COND_INITIAL, 128, _ceil_to(k_in, 64), hidden)]
    for blk in net.blocks:
        layers.append((blk.linear_layers[0], _cabi.COND_BLOCK_FIRST, 128, hk, hidden))
        layers.append((blk.linear_layers[1], _cabi.COND_BLOCK_SECOND, 128, hk, hidden))
    layers.append((fin, _cabi.COND_FINAL, 96, hk, n_final_tiles * 96))
    sizes = [int(L.fc_conditioner_layer_bytes(n_pad, k_pad, bn)) for (_, _, bn, k_pad, n_pad) in layers]
    assert all(s > 0 for s in sizes)
    blob = torch.empty((sum(sizes),), dtype=torch.uint8, device=dev)
    assert blob.data_ptr() % 16 == 0
    st = _cabi.Conditioner()
    st.weights = blob.data_ptr()
    st.n_layers, st.hidden, st.k_in, st.hidden_k = len(layers), hidden, k_in, (_ceil_to(hidden_real, 4) if hidden == 128 else 0)
    vectors = []
    offset = 0
    with torch.cuda.device(dev):
        for i, ((layer, kind, bn, k_pad, n_pad), size) in enumerate(zip(layers, sizes)):
            row_map = None
            if kind == _cabi.COND_FINAL and final_row_map is not None:
                row_map = final_row_map.to(device=dev, dtype=torch.int32)
            elif kind == _cabi.COND_FINAL:
                j = torch.arange(d_t, device=dev).repeat_interleave(P)
                ii = torch.arange(P, device=dev).repeat(d_t)
                row_map = (j * ppad + ii).to(torch.int32)
            vec = _pack_layer(L, dev, blob, offset, layer, getattr(layer, "mask", None), n_pad, k_pad, bn, row_map=row_map,
                              col_map=col_map if kind == _cabi.COND_INITIAL else None)
            vectors.append(vec)
            e = st.layers[i]
            e.kind, e.n_tiles = kind, n_pad // bn
            # the next layer multiplies relu(result) unless it is the final layer (resnet.py:99 / made.py:282: the final
            # layer reads the residual stream itself) or this is the final layer
            nxt = layers[i + 1][1] if i + 1 < len(layers) else None
            e.relu_next = int(nxt in (_cabi.COND_BLOCK_FIRST, _cabi.COND_BLOCK_SECOND))
            e.w_offset = offset
            e.bias, e.winv = vec[0].data_ptr(), vec[1].data_ptr()
            offset += size
    if context is not None:
        for layer, mode, _ in context.layers:
            st.layers[layer].term_mode = mode
    return PackedConditioner(blob, vectors, st, hidden, k_in, n_final_tiles, num_bins, context)


def pack_rqs(net, num_bins, d_t, col_map=None, k_in=None, tails="linear", context=None):
    """`pack` for `fc_conditioner_rqs_apply` (3 K - 1 parameters per feature with linear tails, 3 K + 1 without)."""
    ppad = rqs_ppad(num_bins, tails)
    if ppad is None:
        raise ValueError("conditioner shape not supported by the fused kernel")
    P = 3 * num_bins - 1 if tails == "linear" else 3 * num_bins + 1
    return pack(net, P, ppad, d_t, col_map=col_map, k_in=k_in, num_bins=num_bins, context=context)


def pack_sos(net, n_sigmoids, d_t, col_map=None, k_in=None, context=None):
    """`pack` for `fc_conditioner_sos_apply` (3 n + 1 parameters per feature)."""
    if n_sigmoids not in SOS_SIGMOIDS:
        raise ValueError("conditioner shape not supported by the fused kernel")
    return pack(net, 3 * n_sigmoids + 1, SOS_PPAD, d_t, col_map=col_map, k_in=k_in, context=context)


def pack_affine(net, d_t, layout, col_map=None, k_in=None, context=None):
    """`pack` for `fc_conditioner_affine_apply`: feature j's (raw scale, shift) in final-layer rows (2 j, 2 j + 1)."""
    from . import linear as fl

    rm = fl.affine_row_map(d_t, layout, net.final_layer.weight.device)
    return pack(net, 2, AFFINE_PPAD, d_t, col_map=col_map, k_in=k_in, final_row_map=rm, group=AFFINE_GROUP,
                context=context)


def rqs_apply(packed, a, x, y, logabsdet, accumulate, d_t, tcols, ccols, cfg, status=None, terms=None):
    """Whole conditioner + rational-quadratic spline in one kernel (fc_conditioner_rqs_apply).  a: [B, k_in] matrix the
    initial layer multiplies; writes y[:, tcols] (and y[:, ccols] = x[:, ccols] unless y is x) and logabsdet.
    terms: `context_terms` of this call's context (conditional nets only)."""
    _cabi.require_cuda_f32(a, "conditioner inputs")
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    a, ap, lda = _cabi.rows(a)
    if a.shape[1] != packed.k_in:
        raise ValueError("conditioner inputs have {} columns, the packed net expects {}".format(a.shape[1], packed.k_in))
    assert x.stride(1) == 1 and y.stride(1) == 1 and logabsdet.is_contiguous()
    B = a.shape[0]
    _bind_terms(packed, terms, B)
    with torch.cuda.device(x.device), _cabi.launch("fc_conditioner_rqs_apply", x.device):
        rc = L.fc_conditioner_rqs_apply(ctypes.byref(packed.struct), ap, lda, B, x.data_ptr(), x.stride(0), y.data_ptr(),
                                        y.stride(0), logabsdet.data_ptr(), int(accumulate), d_t, _cabi.cols(tcols),
                                        _cabi.cols(ccols), ctypes.byref(cfg),
                                        status.data_ptr() if status is not None else None, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_conditioner_rqs_apply")
    return y, logabsdet


def sos_apply(packed, a, x, y, logabsdet, accumulate, d_t, n_sigmoids, offset, terms=None):
    """Whole conditioner + sum-of-sigmoids transform (forward) in one kernel (fc_conditioner_sos_apply).  a: [B, k_in]
    matrix the initial layer multiplies (the context of a conditional layer, the inputs of a MADE); terms as `rqs_apply`."""
    _cabi.require_cuda_f32(a, "conditioner inputs")
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    a, ap, lda = _cabi.rows(a)
    if a.shape[1] != packed.k_in:
        raise ValueError("conditioner inputs have {} columns, the packed net expects {}".format(a.shape[1], packed.k_in))
    if a.shape[0] != x.shape[0]:
        raise ValueError("conditioner inputs and inputs differ in rows")
    assert x.stride(1) == 1 and y.stride(1) == 1 and logabsdet.is_contiguous()
    _bind_terms(packed, terms, a.shape[0])
    with torch.cuda.device(x.device), _cabi.launch("fc_conditioner_sos_apply", x.device):
        rc = L.fc_conditioner_sos_apply(ctypes.byref(packed.struct), ap, lda, a.shape[0], x.data_ptr(), x.stride(0),
                                        y.data_ptr(), y.stride(0), logabsdet.data_ptr(), int(accumulate), d_t,
                                        _cabi.cols(None), _cabi.cols(None), int(n_sigmoids), float(offset),
                                        _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_conditioner_sos_apply")
    return y, logabsdet


def affine_apply(packed, a, x, y, logabsdet, accumulate, d_t, tcols, ccols, activation, inverse, terms=None):
    """Whole conditioner + affine transform in one kernel (fc_conditioner_affine_apply); arguments as `rqs_apply`."""
    _cabi.require_cuda_f32(a, "conditioner inputs")
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    a, ap, lda = _cabi.rows(a)
    if a.shape[1] != packed.k_in:
        raise ValueError("conditioner inputs have {} columns, the packed net expects {}".format(a.shape[1], packed.k_in))
    if a.shape[0] != x.shape[0]:
        raise ValueError("conditioner inputs and inputs differ in rows")
    assert x.stride(1) == 1 and y.stride(1) == 1 and logabsdet.is_contiguous()
    _bind_terms(packed, terms, a.shape[0])
    with torch.cuda.device(x.device), _cabi.launch("fc_conditioner_affine_apply", x.device):
        rc = L.fc_conditioner_affine_apply(ctypes.byref(packed.struct), ap, lda, a.shape[0], x.data_ptr(), x.stride(0),
                                           y.data_ptr(), y.stride(0), logabsdet.data_ptr(), int(accumulate), d_t,
                                           _cabi.cols(tcols), _cabi.cols(ccols), int(activation), int(bool(inverse)),
                                           _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_conditioner_affine_apply")
    return y, logabsdet


def pack_store(net, col_map=None, k_in=None, context=None):
    """`pack` for `fc_conditioner_store_apply` (the conditioner's outputs, no bijection): final-layer rows in their own order."""
    n_out = net.final_layer.weight.shape[0]
    rm = torch.arange(n_out, dtype=torch.int32, device=net.final_layer.weight.device)
    packed = pack(net, STORE_PPAD, STORE_PPAD, (n_out + 47) // 48, col_map=col_map, k_in=k_in, final_row_map=rm,
                  context=context)
    packed.n_out = n_out
    return packed


def store_apply(packed, a, out, terms=None):
    """The whole conditioner in one kernel, outputs to `out` [B, out_features] (fc_conditioner_store_apply); terms as
    `rqs_apply`."""
    _cabi.require_cuda_f32(a, "conditioner inputs")
    L = _cabi.lib()
    a, ap, lda = _cabi.rows(a)
    if a.shape[1] != packed.k_in:
        raise ValueError("conditioner inputs have {} columns, the packed net expects {}".format(a.shape[1], packed.k_in))
    assert out.shape == (a.shape[0], packed.n_out) and out.stride(1) == 1 and out.is_cuda and out.dtype == torch.float32
    _bind_terms(packed, terms, a.shape[0])
    with torch.cuda.device(a.device), _cabi.launch("fc_conditioner_store_apply", a.device):
        rc = L.fc_conditioner_store_apply(ctypes.byref(packed.struct), ap, lda, a.shape[0], out.data_ptr(), out.stride(0),
                                          packed.n_out, _cabi.stream_ptr(a.device))
    _cabi.check(rc, "fc_conditioner_store_apply")
    return out


def kernel_error():
    """Non-zero if a barrier wait inside the last fused kernels timed out (synchronises; debugging aid)."""
    out = ctypes.c_int32(0)
    _cabi.check(_cabi.lib().fc_conditioner_error(ctypes.byref(out)), "fc_conditioner_error")
    return out.value


PROFILE_FIELDS = {0: "mma total", 1: "mma wait operand", 2: "mma wait accumulator", 3: "mma wait weights", 4: "mma slots",
                  8: "row total", 9: "row initial operand", 10: "row final hand-off", 11: "row hidden wait",
                  12: "row hidden drain", 13: "row hidden skip/relu", 14: "row hidden convert", 15: "row final wait",
                  16: "row final drain", 17: "row spline", 18: "bij total", 19: "bij wait", 20: "bij work"}


def kernel_profile():
    """Cycle counters of the last fused launch (library built with FC_LINEAR_PROFILE_BUILD=1; zeros otherwise)."""
    buf = (ctypes.c_uint64 * 32)()
    _cabi.check(_cabi.lib().fc_conditioner_profile(buf), "fc_conditioner_profile")
    return {name: int(buf[i]) for i, name in PROFILE_FIELDS.items()}
