"""Host side of the tensor-core conditioner path (csrc/fc_linear.cu, C ABI `fc_linear_*`).

`PackedLinear` is the packed ("3xTF32" hi/lo planes, padded) form of one nn.Linear / MaskedLinear
(flowcon/nn/nets/resnet.py:26-28,69-91, flowcon/transforms/made.py:15-72); `linear` and `linear_rqs` launch the
kernels on torch's current stream.  No fallback: CPU tensors or a missing library raise.
"""
import ctypes

import torch

from . import _cabi

N_TILE_STORE = 256  # fc_linear_apply
N_TILE_RQS = 192    # fc_linear_rqs_apply
N_TILE_AFFINE = 64  # fc_linear_affine_apply
RQS_PPAD = {8: 24, 16: 48}  # accumulator columns per feature for the supported bin counts (P = 3K-1 -> P_pad)


def _ceil_to(v, m):
    return (v + m - 1) // m * m


class PackedLinear:
    """Packed weights of one dense layer.  `n_out` = logical output width (before padding)."""

    def __init__(self, w, b, n_out, k_in):
        self.w = w          # [2, n_pad, k_pad] fp32 (tf32 hi plane, tf32 lo plane)
        self.b = b          # [n_pad]
        self.n_out = n_out
        self.k_in = k_in    # width of the activation matrix the layer multiplies (after any column scatter)
        self.struct = _cabi.LinearWeights(w.data_ptr(), b.data_ptr(), w.shape[1], w.shape[2])

    @property
    def n_pad(self):
        return self.w.shape[1]

    @property
    def k_pad(self):
        return self.w.shape[2]


def pack(weight, bias, mask=None, row_map=None, col_map=None, k_in=None, n_pad=None, n_tile=N_TILE_STORE):
    """fc_linear_pack.  weight [N, K] (+ optional {0,1} mask [N, K], made.py:72), bias [N] or None.
    row_map int32[N]: packed row of each weight row; col_map int32[K]: activation column each weight column
    multiplies (k_in = width of that activation matrix)."""
    _cabi.require_cuda_f32(weight, "weight")
    L = _cabi.lib()
    weight = weight.detach()
    N, K = weight.shape
    if weight.stride(1) != 1:
        weight = weight.contiguous()
    k_in = K if k_in is None else k_in
    k_pad = _ceil_to(k_in, 32)
    rows = N if row_map is None else int(row_map.max().item()) + 1
    n_pad = _ceil_to(max(rows, n_pad or 0), n_tile)
    dev = weight.device
    w = torch.empty((2, n_pad, k_pad), dtype=torch.float32, device=dev)
    b = torch.empty((n_pad,), dtype=torch.float32, device=dev)
    if bias is not None:
        bias = _cabi.require_cuda_f32(bias.detach(), "bias").contiguous()
    if mask is not None:
        mask = _cabi.require_cuda_f32(mask.detach(), "mask")
        if mask.stride(1) != 1:
            mask = mask.contiguous()
    for m in (row_map, col_map):
        if m is not None:
            assert m.dtype == torch.int32 and m.is_cuda and m.is_contiguous()
    with torch.cuda.device(dev), _cabi.launch("fc_linear_pack", dev):
        rc = L.fc_linear_pack(weight.data_ptr(), weight.stride(0), mask.data_ptr() if mask is not None else None,
                              mask.stride(0) if mask is not None else 0,
                              bias.data_ptr() if bias is not None else None, N, K,
                              row_map.data_ptr() if row_map is not None else None,
                              col_map.data_ptr() if col_map is not None else None, n_pad, k_pad, w.data_ptr(),
                              b.data_ptr(), _cabi.stream_ptr(dev))
    _cabi.check(rc, "fc_linear_pack")
    return PackedLinear(w, b, rows, k_in)


def grouped_row_map(n_groups, group, group_pad, device):
    """row j*group + i  ->  j*group_pad + i  (per-feature parameter groups padded to the epilogue's stride)."""
    j = torch.arange(n_groups, device=device).repeat_interleave(group)
    i = torch.arange(group, device=device).repeat(n_groups)
    return (j * group_pad + i).to(torch.int32)


class T128:
    """An activation matrix [rows, width] in the T128 layout of include/flowcon_b200.h (128-row tiles, 16-byte
    column groups slowest inside a tile).  Only the conditioner's own layers read it."""
    TILE = 128

    def __init__(self, rows, width, device):
        if width % 16 != 0:
            raise ValueError("T128 needs a width that is a multiple of 16")
        self.rows, self.width = rows, width
        # The staged kernels work on CTA PAIRS (cta_group::2): one unit = 256 rows = two tiles, and the pair stores (and
        # loads) both tiles of its last unit even when the second one lies beyond `rows`.  The buffer therefore always holds
        # an EVEN number of tiles; with ceil(rows / 128) tiles an odd tile count made the kernel write one tile past the
        # end (found by scripts/fuzz_made_inverse.py: a neighbouring mask buffer was overwritten).
        tiles = (rows + self.TILE - 1) // self.TILE
        tiles += tiles & 1
        self.buf = torch.empty((tiles * self.TILE * width,), dtype=torch.float32, device=device)

    @staticmethod
    def from_rows(t):
        """Row-major [rows, width] tensor -> T128 (test helper; the kernels produce T128 directly)."""
        rows, width = t.shape
        out = T128(rows, width, t.device)
        tiles = out.buf.numel() // (T128.TILE * width)
        padded = torch.zeros((tiles * T128.TILE, width), dtype=torch.float32, device=t.device)
        padded[:rows] = t
        out.buf.copy_(padded.view(tiles, T128.TILE, width // 4, 4).permute(0, 2, 1, 3).reshape(-1))
        return out

    def to_rows(self):
        tiles = self.buf.numel() // (self.TILE * self.width)
        return (self.buf.view(tiles, self.width // 4, self.TILE, 4).permute(0, 2, 1, 3)
                .reshape(tiles * self.TILE, self.width)[:self.rows].contiguous())


def linear(a, packed, relu_in=False, relu_out=False, residual=None, out=None, out_t128=False, n_out=None,
           residual_gates=False):
    """out = act_out(act_in(a) @ W.T + b (+ residual)).  a: [M, K] fp32 row-major (row stride a multiple of 4
    floats) or a T128; the result (and the residual) is a T128 when out_t128 is set, else row-major.
    residual_gates=True: the residual is not added, it gates the result, out = where(residual > 0, a @ W.T + b, 0) — the
    ReLU backward of an input-gradient product."""
    L = _cabi.lib()
    layouts = _cabi.LINEAR_RESIDUAL_GATES if residual_gates else 0
    if isinstance(a, T128):
        layouts |= _cabi.LINEAR_A_T128
        M, k_in, ap, lda, dev = a.rows, a.width, a.buf.data_ptr(), a.width, a.buf.device
    else:
        _cabi.require_cuda_f32(a, "activations")
        a, ap, lda = _cabi.rows(a)
        M, k_in, dev = a.shape[0], a.shape[1], a.device
    if k_in != packed.k_in:
        raise ValueError("activations have {} columns, the packed layer expects {}".format(k_in, packed.k_in))
    n_out = packed.n_out if n_out is None else n_out  # may include zero-weight padding columns (<= n_pad)
    rp, ldr = None, 0
    if out_t128:
        layouts |= _cabi.LINEAR_OUT_T128
        if out is None:
            out = T128(M, n_out, dev)
        op, ldo = out.buf.data_ptr(), out.width
        if residual is not None:
            assert isinstance(residual, T128) and residual.width == n_out and residual.rows == M
            rp, ldr = residual.buf.data_ptr(), residual.width
    else:
        if out is None:
            out = torch.empty((M, n_out), dtype=torch.float32, device=dev)
        op, ldo = out.data_ptr(), out.stride(0)
        if residual is not None:
            residual, rp, ldr = _cabi.rows(_cabi.require_cuda_f32(residual, "residual"))
    with torch.cuda.device(dev), _cabi.launch("fc_linear_apply", dev):
        rc = L.fc_linear_apply(ap, lda, M, k_in, ctypes.byref(packed.struct), int(relu_in), op, ldo, n_out,
                               int(relu_out), rp, ldr, layouts, _cabi.stream_ptr(dev))
    _cabi.check(rc, "fc_linear_apply")
    return out


def linear_rqs(hidden, packed, x, y, logabsdet, accumulate, d_t, tcols, ccols, cfg, status, relu_in=False):
    """Final conditioner layer + rational-quadratic spline in one kernel (fc_linear_rqs_apply).
    Writes y[:, tcols] (and y[:, ccols] = x[:, ccols] unless y is x) and logabsdet in place."""
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    layouts = 0
    if isinstance(hidden, T128):
        layouts |= _cabi.LINEAR_A_T128
        B, H, hp, ldh = hidden.rows, hidden.width, hidden.buf.data_ptr(), hidden.width
    else:
        _cabi.require_cuda_f32(hidden, "hidden activations")
        hidden, hp, ldh = _cabi.rows(hidden)
        B, H = hidden.shape
    assert x.stride(1) == 1 and y.stride(1) == 1 and logabsdet.is_contiguous()
    with torch.cuda.device(x.device), _cabi.launch("fc_linear_rqs_apply", x.device):
        rc = L.fc_linear_rqs_apply(hp, ldh, B, H, ctypes.byref(packed.struct), int(relu_in),
                                   x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), logabsdet.data_ptr(),
                                   int(accumulate), d_t, _cabi.cols(tcols), _cabi.cols(ccols), ctypes.byref(cfg),
                                   status.data_ptr() if status is not None else None, layouts,
                                   _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_linear_rqs_apply")
    return y, logabsdet


def affine_row_map(d_t, layout, device):
    """Packed row of each final-layer output so that feature j's (raw scale, shift) sit in rows (2j, 2j+1)."""
    j = torch.arange(d_t, device=device)
    if layout == _cabi.AFFINE_BLOCKED:      # [shift_0..shift_{D-1} | raw_0..raw_{D-1}]  (coupling.py:234-238)
        return torch.cat((2 * j + 1, 2 * j)).to(torch.int32)
    return torch.arange(2 * d_t, device=device, dtype=torch.int32)  # already (raw, shift) pairs (autoregressive.py:124-129)


def linear_affine(hidden, packed, x, y, logabsdet, accumulate, d_t, tcols, ccols, activation, inverse, relu_in=False):
    """Final conditioner layer + affine transform in one kernel (fc_linear_affine_apply)."""
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    layouts = 0
    if isinstance(hidden, T128):
        layouts |= _cabi.LINEAR_A_T128
        B, H, hp, ldh = hidden.rows, hidden.width, hidden.buf.data_ptr(), hidden.width
    else:
        _cabi.require_cuda_f32(hidden, "hidden activations")
        hidden, hp, ldh = _cabi.rows(hidden)
        B, H = hidden.shape
    assert x.stride(1) == 1 and y.stride(1) == 1 and logabsdet.is_contiguous()
    with torch.cuda.device(x.device), _cabi.launch("fc_linear_affine_apply", x.device):
        rc = L.fc_linear_affine_apply(hp, ldh, B, H, ctypes.byref(packed.struct), int(relu_in), x.data_ptr(),
                                      x.stride(0), y.data_ptr(), y.stride(0), logabsdet.data_ptr(), int(accumulate),
                                      d_t, _cabi.cols(tcols), _cabi.cols(ccols), int(activation), int(bool(inverse)),
                                      layouts, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_linear_affine_apply")
    return y, logabsdet


def linear_splitk_t(a_t, packed, k_slices=None, column_sums=False):
    """a_t.T @ W.T for a_t given TRANSPOSED ([K, M] row-major, e.g. grad_y [B, N]) — fc_linear_splitk_t_apply: the
    weight-gradient product without a transposed copy of grad_y.  Returns [M, n_out]; `packed` must carry a zero bias.
    column_sums=True also returns a_t.sum(0) (the bias gradient), accumulated while a_t passes through the kernel."""
    _cabi.require_cuda_f32(a_t, "activations")
    L = _cabi.lib()
    a_t, ap, ld = _cabi.rows(a_t)
    K, M = a_t.shape
    if K != packed.k_in:
        raise ValueError("activations have {} rows, the packed layer expects {}".format(K, packed.k_in))
    n4 = (packed.n_out + 3) // 4 * 4
    if k_slices is None:
        # two waves of (row-tile pair, range) units over the SM pairs, at least 512 reduction steps each (measured at
        # 32768 rows, 256 x 256: 16 ranges 0.108 ms, 32: 0.067, 64: 0.046, 128: 0.051)
        pairs = (M + 255) // 256
        clusters = torch.cuda.get_device_properties(a_t.device).multi_processor_count // 2
        k_slices = max(1, min(K // 512, (2 * clusters) // pairs))
    slice_rows = _ceil_to(M, 256)
    partials = torch.empty((k_slices, slice_rows, n4), dtype=torch.float32, device=a_t.device)
    csum = torch.empty((k_slices, slice_rows), dtype=torch.float32, device=a_t.device) if column_sums else None
    with torch.cuda.device(a_t.device), _cabi.launch("fc_linear_splitk_t_apply", a_t.device):
        rc = L.fc_linear_splitk_t_apply(ap, ld, M, K, ctypes.byref(packed.struct), k_slices, partials.data_ptr(),
                                        slice_rows, n4, n4, csum.data_ptr() if column_sums else None,
                                        _cabi.stream_ptr(a_t.device))
    _cabi.check(rc, "fc_linear_splitk_t_apply")
    out = partials[0] if k_slices == 1 else partials.sum(0)
    out = out[:M] if n4 == packed.n_out else out[:M, :packed.n_out]
    if column_sums:
        return out, (csum[0] if k_slices == 1 else csum.sum(0))[:M]
    return out


def pack_transposed(x, n_tile=N_TILE_STORE, relu=False):
    """Packed hi / lo planes of x^T (zero bias) for linear_splitk_t: x [B, K] -> PackedLinear with n_out = K, k_in = B.
    relu=True packs max(x, 0)."""
    _cabi.require_cuda_f32(x, "activations")
    L = _cabi.lib()
    x, xp, ld = _cabi.rows(x)
    B, K = x.shape
    n_pad, k_pad = _ceil_to(K, n_tile), _ceil_to(B, 32)
    w = torch.empty((2, n_pad, k_pad), dtype=torch.float32, device=x.device)
    b = torch.empty((n_pad,), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_linear_pack_transposed", x.device):
        rc = L.fc_linear_pack_transposed(xp, ld, B, K, n_pad, k_pad, int(relu), w.data_ptr(), b.data_ptr(),
                                         _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_linear_pack_transposed")
    return PackedLinear(w, b, K, B)
