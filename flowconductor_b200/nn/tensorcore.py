"""Inference path of the conditioner networks on the tensor cores (csrc/fc_linear.cu).

`ResidualNet` (flowcon/nn/nets/resnet.py:59-100) and `MADE` (flowcon/transforms/made.py:205-283) are chains of
Linear / MaskedLinear layers with pre-activation residual blocks.  When no gradient is needed, every layer runs as
one `fc_linear_apply` launch (3xTF32 tcgen05 GEMM, ReLU / bias / skip connection fused) and the final layer
runs as `fc_linear_rqs_apply` (spline in the GEMM epilogue) where the bijection is a linear-tails
rational-quadratic spline with 8 or 16 bins; otherwise the final layer's parameters are materialised by
`fc_linear_apply` and handed to the stand-alone element-wise kernel.

Conditional nets (a ResidualNet with `context_features`, a MADE with a `context_layer`) run only on the fused
conditioner kernel: their context layers become one launch of precomputed terms (`context_terms`) that the kernel's
hidden layers consume; a conditional net of a shape the fused kernel does not cover stays on the torch modules.

The packed weights are cached on the module and rebuilt when any parameter changes (data pointer or
in-place version counter).  Training (autograd) keeps using the torch.nn modules and the custom ops of
`flowconductor_b200.ops`: this path has no backward.
"""
import math
import os
import threading

import torch
from torch import nn
from torch.nn import functional as F

from .. import _cabi, conditioner as fcond, linear as fl
from . import tc_autograd

ENABLED = True  # set False to force the unfused (torch.nn + element-wise kernel) path everywhere


# ---------------------------------------------------------------------------------------------------------
# In-place layers inside a CompositeTransform: a coupling layer rewrites only its transformed columns, so when its
# input is an intermediate that nothing but the running cascade references, it can work in place and the identity
# columns need not be copied (coupling.py:96-98 copies them into a fresh tensor).  Two facts are required, and
# both are established per layer call:  the CASCADE says "this input is my private intermediate" (begin_layer),
# and the PREVIOUS layer call says "I allocated that tensor myself" (mark_fresh).  User-visible tensors never
# satisfy both.
# ---------------------------------------------------------------------------------------------------------
class _Ownership(threading.local):
    consent = None      # the tensor the cascade allows the next layer to overwrite (consumed by the first kernel layer)
    fresh = None        # the tensor allocated by the layer call that is running / has just returned
    prev_fresh = None   # ... by the layer call before it


_own = _Ownership()


def begin_layer(private_input):
    """Called by CompositeTransform._cascade before each layer; `private_input` is the previous layer's output
    (None for the first layer, whose input belongs to the caller)."""
    _own.consent = private_input
    _own.prev_fresh, _own.fresh = _own.fresh, None


def end_cascade():
    _own.consent = _own.fresh = _own.prev_fresh = None


def mark_fresh(t):
    _own.fresh = t


def may_overwrite(t):
    """True exactly once per cascade step, and only for the very tensor object the cascade handed to its direct child:
    a view of it, a tensor that merely shares its storage, or a second kernel layer called by a wrapper transform on the
    same input never qualify (identity, not data_ptr, is compared; the consent is consumed on first use)."""
    ok = (INPLACE and not torch.is_grad_enabled() and _own.consent is not None
          and t is _own.consent and t is _own.prev_fresh)
    return ok


def consume_consent():
    _own.consent = None


INPLACE = True


def _is_relu(act):
    return act is F.relu or act is torch.relu or isinstance(act, nn.ReLU)


def wants_grad(net, *tensors):
    if not torch.is_grad_enabled():
        return False
    if any(t is not None and t.requires_grad for t in tensors):
        return True
    return any(p.requires_grad for p in net.parameters())


def supported_net(net, context):
    """True if `net` is a ResidualNet / MADE configuration the kernels cover, called with a context exactly when it has
    context layers."""
    from ..transforms import made as made_module
    from .nets.resnet import ResidualNet

    if not ENABLED:
        return False
    if isinstance(net, ResidualNet):
        if (net.context_features is not None) != (context is not None):
            return False
        blocks = net.blocks
    elif isinstance(net, made_module.MADE):
        if (not net.use_residual_blocks or hasattr(net, "context_layer") != (context is not None)
                or not _is_relu(net.activation)):
            return False
        blocks = net.blocks
    else:
        return False
    for blk in blocks:
        if getattr(blk, "use_batch_norm", False) or not _is_relu(blk.activation):
            return False
        if blk.dropout.p > 0 and blk.training:
            return False
    hidden_width = net.initial_layer.weight.shape[0]
    # narrow nets stay on the torch path: below a reduction length of 64 the 3xTF32 error floor is above the fp32
    # FMA chain's rounding noise (nn/tc_autograd.py MIN_K) and there is no time to gain
    return hidden_width % 4 == 0 and hidden_width >= tc_autograd.MIN_K


def usable(net, a, context, *other_inputs):
    """Should this conditioner call take the tensor-core path?  `a` is the matrix the first layer multiplies."""
    if not supported_net(net, context) or wants_grad(net, a, context, *other_inputs):
        return False
    # (the TMA operand constraints — 16-byte aligned base and row pitch — are met by `aligned_inputs` below)
    if not (a.is_cuda and a.dtype == torch.float32 and a.dim() == 2 and a.shape[0] > 0):
        return False
    if context is None:
        return True
    # only the fused conditioner takes a context (the per-layer kernels do not): its store variant, which every layer
    # can fall back to, must cover the net
    return (context.is_cuda and context.dtype == torch.float32 and context.dim() == 2 and context.shape[0] == a.shape[0]
            and FUSED_CONDITIONER and fcond.supported_store_shape(
                net.initial_layer.weight.shape[0], _pad4(context_k_in(net, a.shape[1], context)), len(net.blocks),
                net.final_layer.weight.shape[0]))


def context_k_in(net, k_in, context):
    """Input width of the initial layer: a conditional ResidualNet multiplies [inputs | context] (resnet.py:93-95), a
    MADE only the inputs (its context enters through the terms)."""
    from .nets.resnet import ResidualNet

    return k_in + context.shape[1] if context is not None and isinstance(net, ResidualNet) else k_in


def _with_context(net, a, col_map, k_in, context):
    """(a, col_map, k_in) for the initial layer of `net` called with `context`: for a ResidualNet one zero-padded
    [B, k_in + C] copy of [inputs | context] (16-byte row pitch) whose context columns the packed weights read through
    col_map; unchanged otherwise."""
    from .nets.resnet import ResidualNet

    if context is None or not isinstance(net, ResidualNet):
        return a, col_map, k_in
    k = a.shape[1] if k_in is None else k_in
    C = context.shape[1]
    width = (k + C + 3) // 4 * 4
    cat = a.new_empty((a.shape[0], width))
    cat[:, :a.shape[1]] = a
    cat[:, k:k + C] = context
    if width > k + C:
        cat[:, k + C:] = 0
    n_in = net.initial_layer.weight.shape[1] - C  # the input columns of the initial layer come first (resnet.py:93-95)
    # cached on the net (the col_map of a coupling layer is a buffer of the layer that owns the net)
    key = (None,) if col_map is None else (id(col_map), col_map.data_ptr(), col_map._version)
    key += (n_in, k, C, str(a.device))
    cached = getattr(net, "_fc_ctx_cols", None)
    if cached is None or cached[0] != key:
        base = col_map if col_map is not None else torch.arange(n_in, dtype=torch.int32, device=a.device)
        cm = torch.cat((base.to(torch.int32), torch.arange(k, k + C, dtype=torch.int32, device=a.device)))
        cached = (key, cm)
        object.__setattr__(net, "_fc_ctx_cols", cached)
    return cat, cached[1], width


def context_plan_for(net):
    """ContextPlan (stacked context layers) of a conditional net, cached on the module like the packed weights."""
    key = _param_key(net)
    plan = getattr(net, "_fc_ctx_plan", None)
    if plan is not None and plan[0] == key:
        return plan[1]
    packed = fcond.pack_context(net)
    object.__setattr__(net, "_fc_ctx_plan", (key, packed))
    _generation[0] += 1
    return packed


def context_terms(net, context):
    """The context terms of one call (conditioner.context_terms): computed once, shared by every pass of a D-pass
    autoregressive inverse."""
    return fcond.context_terms(context_plan_for(net), context)


def _terms(net, context, terms):
    if context is None:
        return None
    return terms if terms is not None else context_terms(net, context)


def aligned_inputs(a, col_map, k_in):
    """(a, col_map, k_in) with a 16-byte aligned base and row pitch for the TMA loads of the first layer.  A feature count that
    is not a multiple of 4 (the tabular data sets of the reference's experiments: 6, 21, 43, 63 columns) gets a zero-padded
    copy of the inputs — B x D floats, noise next to the conditioner — and the first layer's packed weights the matching
    zero columns (col_map scatters the real ones)."""
    k = a.shape[1] if k_in is None else k_in
    if a.stride(1) == 1 and a.stride(0) % 4 == 0 and a.data_ptr() % 16 == 0 and k % 4 == 0:
        return a, col_map, k_in
    k4 = (a.shape[1] + 3) // 4 * 4
    padded = a.new_zeros((a.shape[0], k4))
    padded[:, :a.shape[1]] = a
    if col_map is None:
        col_map = _identity_cols(a.shape[1], a.device)
    return padded, col_map, k4


_identity_cache = {}


def _identity_cols(n, device):
    key = (n, str(device))
    if key not in _identity_cache:
        _identity_cache[key] = torch.arange(n, dtype=torch.int32, device=device)
    return _identity_cache[key]


def _param_key(net):
    return tuple((p.data_ptr(), p._version) for p in net.parameters())


_generation = [0]  # bumped whenever a packed-weight plan is built or dropped


def cache_generation():
    return _generation[0]


def module_param_key(module):
    """(pointer, in-place version) of every parameter under `module`: changes on optimizer steps / load_state_dict."""
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


def invalidate(module):
    """Drop the packed-weight plans cached on `module` and its sub-modules.  The cache key is (data pointer, in-place
    version counter) of every parameter; a write through `.data` (EMA swaps such as `p.data.copy_(...)`, collectives on
    `p.data`) changes neither, so code that updates weights that way must call this afterwards.  Optimizer steps,
    `load_state_dict` and `distributed.broadcast_parameters` are covered without it."""
    for m in module.modules():
        if getattr(m, "_fc_plan", None) is not None:
            object.__setattr__(m, "_fc_plan", None)
        if getattr(m, "_fc_cond_plan", None) is not None:
            object.__setattr__(m, "_fc_cond_plan", None)
        if getattr(m, "_fc_made_plan", None) is not None:
            object.__setattr__(m, "_fc_made_plan", None)
        if getattr(m, "_fc_ctx_plan", None) is not None:
            object.__setattr__(m, "_fc_ctx_plan", None)
    _generation[0] += 1


class _Plan:
    __slots__ = ("key", "initial", "blocks", "final", "final_kind", "col_map")


def _pack_layer(layer, **kw):
    mask = getattr(layer, "mask", None)
    return fl.pack(layer.weight, layer.bias, mask=mask, **kw)


def plan_for(net, col_map, k_in, final_kind, final_group=None):
    """Packed layers of `net`, cached on the module.  col_map / k_in: scatter of the first layer's input columns
    (coupling layers read the full-width inputs).  final_kind: ("store",) or ("rqs", K)."""
    key = (_param_key(net), final_kind, k_in)
    plan = getattr(net, "_fc_plan", None)
    if plan is not None and plan.key == key:
        return plan
    plan = _Plan()
    plan.key = key
    # a short first reduction (e.g. an 8-wide context) runs as a torch fp32 GEMM, see MIN_K
    plan.initial = _pack_layer(net.initial_layer, col_map=col_map, k_in=k_in) if k_in >= tc_autograd.MIN_K else None
    plan.col_map = col_map
    plan.blocks = [(_pack_layer(b.linear_layers[0]), _pack_layer(b.linear_layers[1])) for b in net.blocks]
    plan.final_kind = final_kind
    fin = net.final_layer
    if final_kind[0] == "affine":
        d_t = fin.weight.shape[0] // 2
        rm = fl.affine_row_map(d_t, final_kind[1], fin.weight.device)
        plan.final = _pack_layer(fin, row_map=rm, n_tile=fl.N_TILE_AFFINE)
    elif final_kind[0] == "rqs":
        K = final_kind[1]
        P = 3 * K - 1
        d_t = fin.weight.shape[0] // P
        rm = fl.grouped_row_map(d_t, P, fl.RQS_PPAD[K], fin.weight.device)
        plan.final = _pack_layer(fin, row_map=rm, n_tile=fl.N_TILE_RQS)
    else:
        plan.final = _pack_layer(fin)
    object.__setattr__(net, "_fc_plan", plan)
    _generation[0] += 1
    return plan


T128_ENABLED = True  # keep the activations between the conditioner's layers in the T128 layout (coalesced epilogues)


def hidden(net, plan, a):
    """Everything up to (not including) the final layer: ResidualNet.hidden / MADE.hidden.  Returns a
    linear.T128 when every hidden width allows it, else a row-major tensor."""
    t128 = T128_ENABLED and net.initial_layer.weight.shape[0] % 16 == 0 and all(
        l0.n_out % 16 == 0 and l1.n_out % 16 == 0 for l0, l1 in plan.blocks)
    if plan.initial is not None:
        h = fl.linear(a, plan.initial, out_t128=t128)
    else:
        lin = net.initial_layer
        cols = a if plan.col_map is None else a[:, plan.col_map.long()]
        h = F.linear(cols, lin.weight if getattr(lin, "mask", None) is None else lin.weight * lin.mask, lin.bias)
        if t128:
            h = fl.T128.from_rows(h)
    for l0, l1 in plan.blocks:
        # relu(W0 relu(h) + b0): only ever consumed through ReLU
        t = fl.linear(h, l0, relu_in=True, relu_out=True, out_t128=t128)
        h = fl.linear(t, l1, residual=h, out_t128=t128)  # h + W1 t + b1
    return h


def params(net, a, col_map=None, k_in=None, context=None, terms=None):
    """Full conditioner output [B, out_features] (final layer materialised).  context: the call's context (conditional
    nets; `terms`: its context_terms when the caller already has them)."""
    a, col_map, k_in = _with_context(net, a, col_map, k_in, context)
    a, col_map, k_in = aligned_inputs(a, col_map, k_in)
    k = k_in if k_in is not None else a.shape[1]
    if context is not None or store_fusable(net, k):  # the whole conditioner as one launch
        key = (_param_key(net), "store", k)
        plan = getattr(net, "_fc_cond_plan", None)
        if plan is None or plan[0] != key:
            ctx = context_plan_for(net) if context is not None else None
            plan = (key, fcond.pack_store(net, col_map=col_map, k_in=k, context=ctx))
            object.__setattr__(net, "_fc_cond_plan", plan)
            _generation[0] += 1
        out = torch.empty((a.shape[0], net.final_layer.weight.shape[0]), dtype=a.dtype, device=a.device)
        return fcond.store_apply(plan[1], a, out, terms=_terms(net, context, terms))
    plan = plan_for(net, col_map, k_in if k_in is not None else a.shape[1], ("store",))
    n = plan.final.n_out
    n4 = (n + 3) // 4 * 4  # the store epilogue writes 16-byte vectors: round up into the zero-weight padding
    out = fl.linear(hidden(net, plan, a), plan.final, n_out=n4)
    return out if n4 == n else out[:, :n]


def _output_buffer(inputs, allow_inplace=True):
    """(x, y) for a fused final layer: in place when the running cascade owns `inputs`, else a fresh tensor.
    allow_inplace=False for callers that need `inputs` again (the D passes of an autoregressive inverse)."""
    x = inputs if inputs.stride(1) == 1 else inputs.contiguous()
    y = x if (allow_inplace and may_overwrite(inputs) and x is inputs) else torch.empty_like(x)
    consume_consent()  # whatever this call decided, no later kernel layer of the same cascade step may write in place
    mark_fresh(y)
    return x, y


def affine_layer(net, a, inputs, tcols, ccols, layout, activation, inverse, col_map=None, k_in=None,
                 allow_inplace=True, context=None, terms=None):
    """Conditioner + affine transform for one layer (final layer fused: fc_linear_affine_apply).  A conditional net
    (context given) must pass `affine_fusable` with its context_k_in."""
    d_t = tcols.numel() if tcols is not None else inputs.shape[1]
    a, col_map, k_in = _with_context(net, a, col_map, k_in, context)
    a, col_map, k_in = aligned_inputs(a, col_map, k_in)
    k_in = k_in if k_in is not None else a.shape[1]
    if affine_fusable(net, k_in, d_t):
        packed = affine_cond_plan_for(net, col_map, k_in, d_t, layout, context is not None)
        x, y = _output_buffer(inputs, allow_inplace)
        lad = torch.empty((x.shape[0],), dtype=x.dtype, device=x.device)
        fcond.affine_apply(packed, a, x, y, lad, False, d_t, tcols, ccols, activation, inverse,
                           terms=_terms(net, context, terms))
        return y, lad
    assert context is None, "conditional nets run on the fused conditioner only"
    plan = plan_for(net, col_map, k_in, ("affine", layout))
    h = hidden(net, plan, a)
    x, y = _output_buffer(inputs, allow_inplace)
    lad = torch.empty((x.shape[0],), dtype=x.dtype, device=x.device)
    fl.linear_affine(h, plan.final, x, y, lad, False, d_t, tcols, ccols, activation, inverse)
    return y, lad


def rqs_fusable(spline, final_out_features, d_t, net=None, k_in=None, context=None):
    """Can the bijection run inside a tensor-core kernel?  Either in the final layer's epilogue (fc_linear_rqs_apply: linear
    tails, 8 or 16 bins) or — `net` / `k_in` given — inside the fused conditioner (more bin counts, also without tails).
    With a context only the fused conditioner qualifies."""
    if not ENABLED or final_out_features != d_t * spline.params_per_feature():
        return False
    if context is not None:
        return net is not None and conditioner_fusable(net, context_k_in(net, k_in, context), spline, d_t)
    if spline.tails == "linear" and spline.num_bins in fl.RQS_PPAD:
        return True
    return net is not None and conditioner_fusable(net, k_in, spline, d_t)


FUSED_AFFINE = os.environ.get("FC_FUSED_AFFINE", "1") != "0"  # A/B switch of the fused affine conditioner
FUSED_CONDITIONER = True  # whole conditioner + spline as ONE persistent kernel (csrc/fc_conditioner.cu) where it applies


def cond_plan_for(net, col_map, k_in, num_bins, d_t, tails="linear", context=False):
    """PackedConditioner of `net`, cached on the module like the per-layer plans (same key rules).  context: pack the
    net's context layers as well (a conditional net called with its context)."""
    key = (_param_key(net), num_bins, tails, k_in, d_t, context)
    plan = getattr(net, "_fc_cond_plan", None)
    if plan is not None and plan[0] == key:
        return plan[1]
    packed = fcond.pack_rqs(net, num_bins, d_t, col_map=col_map, k_in=k_in, tails=tails,
                            context=context_plan_for(net) if context else None)
    object.__setattr__(net, "_fc_cond_plan", (key, packed))
    _generation[0] += 1
    return packed


def affine_cond_plan_for(net, col_map, k_in, d_t, layout, context=False):
    """PackedConditioner of `net` for the fused affine kernel, cached like the spline plans."""
    key = (_param_key(net), "affine", layout, k_in, d_t, context)
    plan = getattr(net, "_fc_cond_plan", None)
    if plan is not None and plan[0] == key:
        return plan[1]
    packed = fcond.pack_affine(net, d_t, layout, col_map=col_map, k_in=k_in,
                               context=context_plan_for(net) if context else None)
    object.__setattr__(net, "_fc_cond_plan", (key, packed))
    _generation[0] += 1
    return packed


FUSED_STORE = os.environ.get("FC_FUSED_STORE", "1") != "0"  # A/B switch: fc_conditioner_store_apply behind `params`
FUSED_SOS = os.environ.get("FC_FUSED_SOS", "1") != "0"      # A/B: sum of sigmoids inside the conditioner kernel, or store + layer kernel


def store_fusable(net, k_in):
    return FUSED_CONDITIONER and FUSED_STORE and fcond.supported_store_shape(
        net.initial_layer.weight.shape[0], _pad4(k_in), len(net.blocks), net.final_layer.weight.shape[0])


def _pad4(k_in):
    """Input width the kernels see: `aligned_inputs` pads to a multiple of 4 columns."""
    return None if k_in is None else (k_in + 3) // 4 * 4


def affine_fusable(net, k_in, d_t=None):
    return FUSED_CONDITIONER and FUSED_AFFINE and k_in is not None and fcond.supported_affine_shape(
        net.initial_layer.weight.shape[0], _pad4(k_in), len(net.blocks), d_t)


def sos_cond_plan_for(net, k_in, n_sigmoids, d_t, col_map=None, context=False):
    """PackedConditioner of `net` for the fused sum-of-sigmoids kernel, cached like the spline plans."""
    key = (_param_key(net), "sos", n_sigmoids, k_in, d_t, context)
    plan = getattr(net, "_fc_cond_plan", None)
    if plan is not None and plan[0] == key:
        return plan[1]
    packed = fcond.pack_sos(net, n_sigmoids, d_t, col_map=col_map, k_in=k_in,
                            context=context_plan_for(net) if context else None)
    object.__setattr__(net, "_fc_cond_plan", (key, packed))
    _generation[0] += 1
    return packed


def sos_fusable(net, k_in, n_sigmoids, d_t=None):
    return FUSED_CONDITIONER and FUSED_SOS and fcond.supported_sos_shape(net.initial_layer.weight.shape[0], _pad4(k_in), len(net.blocks),
                                                           n_sigmoids, d_t)


def sos_layer(net, a, inputs, n_sigmoids, offset, context=None, terms=None):
    """Conditioner + sum-of-sigmoids transform (forward) as one kernel; returns (outputs, logabsdet).  `a` feeds the
    conditioner (context / MADE inputs), `inputs` the bijection; `context`: the context of a conditional net."""
    a, col_map, k_in = _with_context(net, a, None, None, context)
    a, col_map, k_in = aligned_inputs(a, col_map, k_in)
    packed = sos_cond_plan_for(net, a.shape[1], int(n_sigmoids), inputs.shape[1], col_map, context is not None)
    x = inputs if inputs.stride(1) == 1 else inputs.contiguous()
    y = torch.empty_like(x)
    consume_consent()
    mark_fresh(y)
    lad = torch.empty((x.shape[0],), dtype=x.dtype, device=x.device)
    fcond.sos_apply(packed, a, x, y, lad, False, inputs.shape[1], n_sigmoids, offset, terms=_terms(net, context, terms))
    return y, lad


def conditioner_fusable(net, k_in, spline, d_t=None):
    """`spline`: RationalQuadraticSettings (or a bin count, meaning linear tails); d_t: transformed features (the final
    layer's bias vector must fit in the kernel's shared memory)."""
    num_bins, tails = (spline, "linear") if isinstance(spline, int) else (int(spline.num_bins), spline.tails)
    return FUSED_CONDITIONER and k_in is not None and fcond.supported_shape(
        net.initial_layer.weight.shape[0], _pad4(k_in), len(net.blocks), num_bins, tails, d_t)


def rqs_layer(net, a, inputs, spline, tcols, ccols, inverse, hidden_for_scaling, col_map=None, k_in=None,
              allow_inplace=True, context=None, terms=None):
    """Conditioner + spline for one layer; returns (outputs, logabsdet).  A conditional net (context given) must pass
    `rqs_fusable` with the context."""
    d_t = tcols.numel() if tcols is not None else inputs.shape[1]
    a, col_map, k_in = _with_context(net, a, col_map, k_in, context)
    a, col_map, k_in = aligned_inputs(a, col_map, k_in)
    k_in = k_in if k_in is not None else a.shape[1]
    cfg, tails = spline.config(inverse, hidden_for_scaling)
    if conditioner_fusable(net, k_in, spline, d_t):
        from ..transforms import splines as fsplines

        packed = cond_plan_for(net, col_map, k_in, int(spline.num_bins), d_t, spline.tails, context is not None)
        x, y = _output_buffer(inputs, allow_inplace)
        lad = torch.empty((x.shape[0],), dtype=x.dtype, device=x.device)
        # without tails the reference raises InputOutsideDomain after a host-side check (rational_quadratic.py:81-82): the
        # kernel reports through the status word instead
        status = torch.zeros((1,), dtype=torch.int32, device=x.device) if (tails == _cabi.TAILS_NONE or fsplines.STRICT) \
            else None
        fcond.rqs_apply(packed, a, x, y, lad, False, d_t, tcols, ccols, cfg, status, terms=_terms(net, context, terms))
        if status is not None:
            fsplines.check_status(status, tails)
        return y, lad
    assert context is None, "conditional nets run on the fused conditioner only"
    plan = plan_for(net, col_map, k_in, ("rqs", spline.num_bins))
    h = hidden(net, plan, a)
    x, y = _output_buffer(inputs, allow_inplace)
    lad = torch.empty((x.shape[0],), dtype=x.dtype, device=x.device)
    fl.linear_rqs(h, plan.final, x, y, lad, False, d_t, tcols, ccols, cfg, None)
    return y, lad
