"""Host side of the incremental autoregressive inverse (csrc/fc_made_inverse.cu, C ABI `fc_made_inverse_*`).

`AutoregressiveTransform.inverse` of the reference (flowcon/transforms/autoregressive/autoregressive.py:44-53) runs the whole
MADE D times.  `compile_made` turns a residual MADE (flowcon/transforms/made.py:205-283) into the straight-line program the
kernel interprets: the hidden units are ordered by degree, so that every masked weight row (made.py:28-51,72) reads a PREFIX
of the layer below; pass f then computes only the units that become valid with feature f - 1 and the P parameters of
feature f, after which the kernel inverts that feature.  The schedule is derived from the MASKS, not from the degree
formula: any mask pattern with the prefix property compiles, anything else returns None (the D-pass inverse runs).

A conditional MADE (`context_features`) compiles to the same program.  Its context layers (initial layer made.py:138-140,
first layer of every block made.py:100-102) do not depend on x: they are stacked into one `conditioner.ContextPlan`, rows
in the program's degree order, and each call evaluates them for the whole batch in one launch
(`conditioner.context_terms`).  The kernel starts the hidden arrays that consume them from bias + act(term), so the tasks
that write those arrays accumulate instead of initialising from the bias.

No fallback inside: `apply_*` needs CUDA fp32 tensors and the library.
"""
import ctypes

import numpy as np
import torch

from . import _cabi, conditioner

MAX_NJ = 24      # FC_MADE_MAX_NJ
TASKS = 8        # FC_MADE_TASKS
ROWS = 32        # rows per CTA of the kernel
SMEM_LIMIT = 232448  # opt-in shared memory per CTA on sm_100
SLOT_FLOATS = 2048   # ring slot of the kernel
RELU_IN, INIT_BIAS = 1, 2
# tasks per narrow (dependent-chain) phase.  Measured on cfg 3 at 32 768 rows: 8 tasks 7.45 ms, 2 tasks 7.51 ms, 1 task (as
# few as the 24-output limit allows) 7.92 ms — the chain is latency-bound, so the outputs are spread over all warps.
CHAIN_PARTS = int(__import__("os").environ.get("FC_MADE_CHAIN_PARTS", str(TASKS)))
PHASE_INTS = 4 + 12 * TASKS
RECORD_FLOATS = 128  # FC_MADE_RECORD_FLOATS: the phase record (padded) in front of the phase's matrix
TASK_FIELDS = ("in_array", "out_array", "k0", "kn", "j0", "nj", "c0", "flags", "res_array", "b_off", "reserved0", "reserved1")


class MadeProgram:
    """Compiled program + its device buffers (`phases`, `weights`, `bias` keep the memory alive)."""

    def __init__(self, phases_np, weights, bias, features, params_per_feature, n_arrays, hidden, device, context=None,
                 term_arrays=()):
        self.phases_np = phases_np  # [n_phases, 100] int32 (host copy: tests, debugging)
        self.phases = torch.from_numpy(phases_np.copy()).to(device)
        self.weights, self.bias = weights, bias
        self.features, self.params_per_feature, self.n_arrays, self.hidden = features, params_per_feature, n_arrays, hidden
        # conditional MADE: the stacked context layers, and per consuming hidden array (array, column, b_off, relu)
        self.context, self.term_arrays = context, list(term_arrays)
        self.struct = None
        if weights.is_cuda:
            st = _cabi.MadeProgramStruct()
            st.phases, st.weights, st.bias = self.phases.data_ptr(), weights.data_ptr(), bias.data_ptr()
            st.n_phases, st.features, st.params_per_feature = phases_np.shape[0], features, params_per_feature
            st.n_arrays, st.hidden, st.n_bias = n_arrays, hidden, bias.numel()
            if context is not None:
                st.term_width, st.n_term_arrays = context.width, len(self.term_arrays)
                for i, t in enumerate(self.term_arrays):
                    st.term_arrays[i].array, st.term_arrays[i].column, st.term_arrays[i].b_off, st.term_arrays[i].relu = t
            self.struct = st

    @property
    def n_phases(self):
        return self.phases_np.shape[0]

    def tasks(self):
        """[(phase index, header dict, [task dicts])] of the host copy (tests)."""
        out = []
        for i, row in enumerate(self.phases_np.tolist()):
            hdr = dict(zip(("rows", "width", "w_off4", "feature"), row[:4]))
            ts = [dict(zip(TASK_FIELDS, row[4 + 12 * t: 16 + 12 * t])) for t in range(TASKS)]
            out.append((i, hdr, [t for t in ts if t["nj"] > 0]))
        return out


def smem_bytes(features, params_per_feature, n_arrays, hidden, n_bias=None):
    """Mirror of fc_made_inverse_smem_bytes (kept in sync by tests/test_host_api.py): the row tile's state, every bias, and
    the smallest weight ring (2 slots)."""
    if n_bias is None:
        n_bias = n_arrays * hidden + features * params_per_feature
    ring = 2 * SLOT_FLOATS * 4
    return ring + 4 * (features * ROWS + n_arrays * hidden * ROWS + params_per_feature * ROWS + (n_bias + 3) // 4 * 4) \
        + 8 * 2 * 8 + 128


def _prefix_counts(mask):
    """mask [N, K] of 0/1 -> per-row count of leading ones, or None if some row is not of the form 1..1 0..0."""
    cnt = mask.sum(dim=1).round().long()
    k = torch.arange(mask.shape[1], device=mask.device)
    if not bool(((k[None, :] < cnt[:, None]).to(mask.dtype) == mask).all()):
        return None
    return cnt


def supported_made(net):
    """Structure the compiler handles: residual blocks, ReLU, no batch norm / active dropout; context layers on the initial
    layer and every block, or none."""
    from .nn import tensorcore

    if not getattr(net, "use_residual_blocks", False):
        return False
    if not tensorcore._is_relu(net.activation):
        return False
    ctx = hasattr(net, "context_layer")
    for blk in net.blocks:
        if getattr(blk, "use_batch_norm", False) or not tensorcore._is_relu(blk.activation) or hasattr(blk, "context_layer") != ctx:
            return False
        if blk.dropout.p > 0 and blk.training:
            return False
    return True


def _split_even(n, parts):
    """n outputs -> consecutive slices whose widths are multiples of 4 (the last one may be ragged) and at most MAX_NJ: `parts`
    of them when that is enough, more otherwise (the caller spreads more than TASKS slices over several phases)."""
    n4 = (n + 3) // 4
    parts = max(1, min(parts, n4), (n + MAX_NJ - 1) // MAX_NJ)
    while True:
        base, extra = divmod(n4, parts)
        if 4 * (base + (1 if extra else 0)) <= MAX_NJ:
            break
        parts += 1
    out, j = [], 0
    for i in range(parts):
        w = 4 * (base + (1 if i < extra else 0))
        out.append((j, min(w, n - j)))
        j += w
    return [(a, b) for a, b in out if b > 0]


def compile_made(net, params_per_feature):
    """-> MadeProgram, or None when the network does not have the structure the kernel needs."""
    init, fin = net.initial_layer, net.final_layer
    dev = init.weight.device
    H, D = init.weight.shape
    P = params_per_feature
    if fin.weight.shape[0] != D * P:
        return None
    nb = len(net.blocks)
    n_arrays = 1 + 2 * nb
    if smem_bytes(D, P, n_arrays, H) > SMEM_LIMIT:
        return None
    conditional = hasattr(net, "context_layer")
    if conditional and 1 + nb > _cabi.MADE_MAX_TERM_ARRAYS:
        return None
    # hidden arrays that start from bias + act(context term): the initial layer's (ReLU) and each block's first layer's
    ctx_arrays = {1} | {2 * b + 2 for b in range(nb)} if conditional else set()
    with torch.no_grad():
        deg = init.degrees.detach().cpu()
        for blk in net.blocks:
            for lin in blk.linear_layers:
                if not torch.equal(lin.degrees.detach().cpu(), deg):
                    return None
        perm = torch.argsort(deg, stable=True).to(dev)
        # layers: (module, input array, output array (0 = parameter tile), relu on the input, skip-connection array)
        layers = [(init, 0, 1, 0, 0)]
        for b, blk in enumerate(net.blocks):
            h_in = 1 if b == 0 else 2 * b + 1
            layers.append((blk.linear_layers[0], h_in, 2 * b + 2, 1, 0))
            layers.append((blk.linear_layers[1], 2 * b + 2, 2 * b + 3, 1, h_in))
        layers.append((fin, n_arrays, 0, 0, 0))
        sorted_w, counts, bias_parts, bias_base = [], [], [], []
        off = 0
        for lin, in_a, out_a, _, _ in layers:
            w = (lin.weight * lin.mask).detach().float()
            m = lin.mask.detach().float()
            b = lin.bias.detach().float() if lin.bias is not None else torch.zeros(w.shape[0], device=dev)
            if in_a != 0:
                w, m = w[:, perm], m[:, perm]
            if out_a != 0:
                w, m, b = w[perm], m[perm], b[perm]
            cnt = _prefix_counts(m)
            if cnt is None:
                return None
            sorted_w.append(w.contiguous())
            counts.append(cnt.cpu().numpy())
            bias_parts.append(b)
            bias_base.append(off)
            off += b.numel()
        fl = len(layers) - 1
        phases, blocks = [], []
        w_floats = [0]

        def add_phase(tasks, feature):
            """tasks: [(layer index, j_lo, nj, k0, kn, init_bias, final, j_base)] -> one phase record + its weight matrix."""
            assert 0 < len(tasks) <= TASKS
            rows = max(t[4] for t in tasks)
            width = sum(4 * ((t[2] + 3) // 4) for t in tasks)
            assert width <= SLOT_FLOATS - RECORD_FLOATS and w_floats[0] % 4 == 0
            rec = [rows, width, w_floats[0] // 4, feature]
            mat = torch.zeros((max(rows, 1), width), dtype=torch.float32, device=dev) if rows > 0 else None
            c0 = 0
            for li, j_lo, nj, k0, kn, init_bias, final, j_base in tasks:
                _, in_a, out_a, relu_in, res_a = layers[li]
                flags = (RELU_IN if relu_in else 0) | (INIT_BIAS if init_bias and out_a not in ctx_arrays else 0)
                rec += [in_a, out_a, k0, kn, j_lo - j_base, nj, c0, flags, res_a if final else 0, bias_base[li] + j_lo, 0, 0]
                if kn > 0:
                    mat[:kn, c0:c0 + nj] = sorted_w[li][j_lo:j_lo + nj, k0:k0 + kn].t()
                c0 += 4 * ((nj + 3) // 4)
            rec += [0] * (PHASE_INTS - len(rec))
            phases.append(rec)
            # the record itself travels through the kernel's weight ring, in front of the matrix
            rec_words = torch.tensor(rec + [0] * (RECORD_FLOATS - PHASE_INTS), dtype=torch.int32, device=dev)
            blocks.append(rec_words.view(torch.float32))
            w_floats[0] += RECORD_FLOATS
            if rows > 0:
                blocks.append(mat.reshape(-1))
                w_floats[0] += rows * width

        def chunks(li, j_lo, j_hi, k0, kn, init_bias, final, j_base):
            return [(li, j, min(MAX_NJ, j_hi - j), k0, kn, init_bias, final, j_base) for j in range(j_lo, j_hi, MAX_NJ)]

        def balance(tasks):
            """Fewer tasks than warps: halve the most expensive ones (k-values x instructions per k-value) so that every
            warp has work and the slowest task of the phase is as short as possible."""
            tasks = list(tasks)

            def cost(t):
                return (t[4] + 4) * (1 + 3 * ((t[2] + 3) // 4))

            while len(tasks) < TASKS:
                cand = [i for i in range(len(tasks)) if tasks[i][2] > 4]
                if not cand:
                    break
                i = max(cand, key=lambda t: cost(tasks[t]))
                li, j, nj, k0, kn, ib, fn, jb = tasks[i]
                half = 4 * (((nj + 3) // 4 + 1) // 2)
                tasks[i:i + 1] = [(li, j, half, k0, kn, ib, fn, jb), (li, j + half, nj - half, k0, kn, ib, fn, jb)]
            return tasks

        def emit(tasks, feature=-1):
            for i in range(0, len(tasks), TASKS):
                last = i + TASKS >= len(tasks)
                add_phase(tasks[i:i + TASKS], feature if last else -1)

        ready = 0  # units [0, ready) of EVERY hidden array are final
        for f in range(D):
            c = counts[fl][f * P:(f + 1) * P]
            hi = int(c.max())
            lo = ready
            if hi < lo:
                return None  # features must need non-decreasing prefixes (degrees 1..D in order)
            new = hi > lo
            if new:
                # the initial layer of the new units reads features < f only (else the net is not autoregressive in order)
                kx = int(counts[0][lo:hi].max())
                if kx > f:
                    return None
                for li in range(1, fl):
                    need = int(counts[li][lo:hi].max())
                    if need > hi:
                        return None
            # ---- wide phase: everything that depends on earlier passes only
            wide = []
            if new:
                wide += chunks(0, lo, hi, 0, int(counts[0][lo:hi].max()), True, True, 0)
                if lo > 0:
                    for li in range(1, fl):
                        wide += chunks(li, lo, hi, 0, lo, True, False, 0)
            if lo > 0 or not new:
                # the feature's parameters from the units that were final before this pass (bias only when there are none)
                wide += chunks(fl, f * P, (f + 1) * P, 0, min(lo, hi), True, False, f * P)
            if not new:
                # nothing new to compute: the wide phase completes the parameters
                emit(balance(wide), f)
                continue
            if wide:
                emit(balance(wide))
            # ---- the dependent chain: one narrow phase per layer over the new units of the layer below
            for li in range(1, fl):
                need = int(counts[li][lo:hi].max())
                tasks = [(li, lo + j, nj, lo, max(need - lo, 0), lo == 0, True, 0)
                         for j, nj in _split_even(hi - lo, CHAIN_PARTS)]
                emit(tasks)
            tasks = [(fl, f * P + j, nj, lo, hi - lo, lo == 0, False, f * P) for j, nj in _split_even(P, CHAIN_PARTS)]
            emit(tasks, f)
            ready = hi
        phases_np = np.asarray(phases, dtype=np.int32).reshape(-1, PHASE_INTS)
        weights = torch.cat(blocks) if blocks else torch.zeros((4,), dtype=torch.float32, device=dev)
        bias = torch.cat(bias_parts).contiguous()
        context, term_arrays = None, []
        if conditional:
            # columns i * ceil4(H) + j: sorted unit j of the i-th consuming array (the kernel reads whole float4 groups)
            src = [(1, _cabi.COND_TERM_ADD_RELU, net.context_layer)]
            src += [(2 * b + 2, _cabi.COND_TERM_ADD, blk.context_layer) for b, blk in enumerate(net.blocks)]
            context = conditioner.stack_context(src, (H + 3) // 4 * 4, order=perm)
            b_off = {1: bias_base[0]}
            b_off.update({2 * b + 2: bias_base[1 + 2 * b] for b in range(nb)})
            term_arrays = [(arr, col, b_off[arr], int(mode == _cabi.COND_TERM_ADD_RELU)) for arr, mode, col in context.layers]
    return MadeProgram(phases_np, weights.contiguous(), bias, D, P, n_arrays, H, dev, context, term_arrays)


def _io(prog, z):
    _cabi.require_cuda_f32(z, "inputs")
    if z.dim() != 2 or z.shape[1] != prog.features:
        raise ValueError("expected inputs of shape [B, {}]".format(prog.features))
    z, zp, ldz = _cabi.rows(z)
    x = torch.empty((z.shape[0], prog.features), dtype=torch.float32, device=z.device)
    lad = torch.empty((z.shape[0],), dtype=torch.float32, device=z.device)
    return z, zp, ldz, x, lad


def _bind_terms(prog, context, B):
    """The context terms of this call (one launch, conditioner.context_terms), bound into the program struct; None for a
    MADE without context layers.  The binding is valid for one launch only: the caller keeps the result alive until the
    launch is enqueued and then clears `prog.struct.terms` (the buffer goes back to the caching allocator)."""
    if prog.context is None:
        if context is not None:
            raise ValueError("a context was given for a MADE without context layers")
        prog.struct.terms = None
        return None
    if context is None:
        raise ValueError("a MADE with context layers needs its context")
    if context.dim() != 2 or context.shape[0] != B:
        raise ValueError("context has shape {}, expected [{}, {}]".format(tuple(context.shape), B, prog.context.features))
    terms = conditioner.context_terms(prog.context, context)
    if terms.width != prog.context.width:  # the kernel addresses the T128 tiles with the plan's width
        raise ValueError("context terms are {} wide, the program expects {}".format(terms.width, prog.context.width))
    prog.struct.terms = terms.buf.data_ptr()
    return terms


def _apply(entry, prog, z, context, *tail):
    """Shared launch plumbing of the fc_made_inverse_* entry points: (x, logabsdet)."""
    L = _cabi.lib()
    z, zp, ldz, x, lad = _io(prog, z)
    terms = _bind_terms(prog, context, z.shape[0])  # noqa: F841 (alive until the launch is enqueued)
    try:
        with torch.cuda.device(z.device), _cabi.launch(entry, z.device):
            rc = getattr(L, entry)(ctypes.byref(prog.struct), zp, ldz, x.data_ptr(), x.stride(0), lad.data_ptr(), 0,
                                   z.shape[0], *tail, _cabi.stream_ptr(z.device))
    finally:
        prog.struct.terms = None  # a later direct use of the struct must bind its own terms
    _cabi.check(rc, entry)
    return x, lad


def _sptr(status):
    return status.data_ptr() if status is not None else None


def apply_rqs(prog, z, cfg, status=None, context=None):
    """Inverse of a MAF layer with rational-quadratic splines: (x, logabsdet) = layer.inverse(z, context).  `context`:
    the [B, C] context of a conditional MADE (required exactly when the program has context layers); likewise below."""
    return _apply("fc_made_inverse_rqs", prog, z, context, ctypes.byref(cfg), _sptr(status))


def apply_affine(prog, z, activation, context=None):
    """Inverse of a MaskedAffineAutoregressiveTransform layer."""
    return _apply("fc_made_inverse_affine", prog, z, context, int(activation))


def apply_sos(prog, z, n_sigmoids, offset, iterations, lim, context=None):
    """Inverse of a MaskedSumOfSigmoidsTransform layer (numerical inverse per feature, as fc_sos_apply)."""
    return _apply("fc_made_inverse_sos", prog, z, context, int(n_sigmoids), float(offset), int(iterations), float(lim))


def apply_linspline(prog, z, num_bins, tails, lo, hi, status=None, context=None):
    return _apply("fc_made_inverse_linspline", prog, z, context, int(num_bins), int(tails), float(lo), float(hi), float(lo),
                  float(hi), _sptr(status))


def apply_quadspline(prog, z, cfg, status=None, context=None):
    return _apply("fc_made_inverse_quadspline", prog, z, context, ctypes.byref(cfg), _sptr(status))


def apply_cubicspline(prog, z, cfg, status=None, context=None):
    return _apply("fc_made_inverse_cubicspline", prog, z, context, ctypes.byref(cfg), _sptr(status))


PROFILE_FIELDS = ("phase record", "wait weights", "multiply", "store units", "phase barrier", "invert feature", "total",
                  "phases")


def kernel_profile():
    """Cycle counters of the last launch (library built with FC_LINEAR_PROFILE_BUILD=1; zeros otherwise): warps 0 and 5 of
    CTA 0, wide phases (rows > 40) and narrow phases separately."""
    buf = (ctypes.c_uint64 * 32)()
    _cabi.check(_cabi.lib().fc_made_inverse_profile(buf), "fc_made_inverse_profile")
    out = {}
    for w, base in (("warp0", 0), ("warp5", 16)):
        for kind, off in (("wide", 0), ("narrow", 8)):
            out[w + " " + kind] = {n: int(buf[base + off + i]) for i, n in enumerate(PROFILE_FIELDS)}
    return out


ENABLED = True  # False: every autoregressive inverse takes the D-pass path


def program_for(net, params_per_feature):
    """Compiled program of `net` (with the stacked context layers of a conditional MADE), cached on the module with the
    same key rules as the packed tensor-core weights (nn/tensorcore.py: data pointer + in-place version of every parameter,
    the context layers' included).  None if the net does not compile."""
    from .nn import tensorcore

    key = (tensorcore._param_key(net), params_per_feature, bool(net.training))
    cached = getattr(net, "_fc_made_plan", None)
    if cached is not None and cached[0] == key:
        return cached[1]
    prog = compile_made(net, params_per_feature) if supported_made(net) else None
    object.__setattr__(net, "_fc_made_plan", (key, prog))
    tensorcore._generation[0] += 1
    return prog


def usable(net, inputs, context):
    """Should this inverse call take the incremental kernel?  A call with a context does when the net has context layers
    and the fused conditioner does not cover the call (there the D-pass inverse runs one fused launch per pass:
    AutoregressiveTransform.inverse)."""
    from .nn import tensorcore
    from .transforms import made as made_module

    if not ENABLED or not isinstance(net, made_module.MADE) or hasattr(net, "context_layer") != (context is not None):
        return False
    if tensorcore.wants_grad(net, inputs, context):
        return False
    if not (inputs.is_cuda and inputs.dtype == torch.float32 and inputs.dim() == 2 and inputs.shape[0] > 0):
        return False
    if context is None:
        return True
    return (context.is_cuda and context.dtype == torch.float32 and context.dim() == 2
            and context.shape[0] == inputs.shape[0] and not tensorcore.usable(net, inputs, context, inputs))
