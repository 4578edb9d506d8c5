"""Training path of the conditioner's dense layers on the tensor cores.

`linear(x, weight, bias, mask)` is F.linear(x, weight * mask, bias) (flowcon/nn/nets/resnet.py:26-28,
flowcon/transforms/made.py:71-72) as an autograd function whose forward and input-gradient GEMMs run on the
3xTF32 tcgen05 kernel (`fc_linear_apply`, fp32-faithful):

    forward   y  = x  @ (W*mask)^T + b          tensor cores
    backward  gx = gy @ (W*mask)                tensor cores (the packed operand is the transposed weight)
              gW = (gy^T @ x) * mask            tensor cores, split-K: the reduction runs over the batch, so it is cut
              gb = gy.sum(0)                    into ranges that run as independent work units (fc_linear_splitk_t_apply)

The weights change every optimizer step, so they are re-packed on every call (two tiny kernels per layer).
Anything the kernel does not cover (CPU tensors, other dtypes, misaligned operands) takes F.linear.
"""
import torch
from torch.nn import functional as F

from .. import linear as fl

ENABLED = True
# Shortest reduction the tensor-core GEMM is used for.  Every 3xTF32 product carries ~2^-22 relative error (dropped
# lo*lo term, truncation inside the MMA); an fp32 FMA chain rounds at 2^-24 per step, so its error grows with the
# chain length.  Measured (scripts/check_linear.py, Gaussian operands): at K = 32 the tensor-core result is 1.3x
# noisier than cuBLAS fp32, at K = 64 equal, at K = 256 15% better.  Below 64 there is no time to gain either.
MIN_K = 64


def _eligible(x, weight):
    return (ENABLED and x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32 and x.dim() == 2
            and x.shape[0] > 0 and x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0
            and weight.shape[1] >= MIN_K        # forward reduction length
            and weight.shape[0] >= MIN_K)       # input-gradient reduction length


def _gemm(a, packed, n, relu_in=False):
    """a @ packed^T, first n columns.  The store epilogue writes 16-byte vectors: n is rounded up into the packed
    layer's zero-weight padding and sliced off again."""
    n4 = (n + 3) // 4 * 4
    out = fl.linear(a, packed, n_out=n4, relu_in=relu_in)
    return out if n4 == n else out[:, :n]


class _TCLinear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, mask):
        y = _gemm(x, fl.pack(weight, bias, mask=mask), weight.shape[0])
        ctx.save_for_backward(x, weight, mask)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, mask = ctx.saved_tensors
        gy = gy.contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            wm = weight if mask is None else weight * mask
            gx = _gemm(gy, fl.pack(wm.t().contiguous(), None), weight.shape[1])
            if gx.stride(0) != weight.shape[1]:
                gx = gx.contiguous()
        if ctx.needs_input_grad[1]:
            gw, gb = _wgrad(gy, x, weight, mask, ctx.has_bias and ctx.needs_input_grad[2])
        if gb is None and ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gy.sum(0)
        return gx, gw, gb, None


def _wgrad(gy, x, weight, mask, want_bias, relu_x=False):
    """(grad_W, grad_b or None) of y = relu?(x) @ (W*mask)^T + b for upstream gy."""
    gb = None
    # (the reduction runs over the batch, so a narrow layer input does not shorten it: no MIN_K condition here)
    if (x.shape[0] >= 4096 and x.shape[0] % 4 == 0 and gy.shape[1] % 4 == 0
            and x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0):
        xt = fl.pack_transposed(x, relu=relu_x)
        if want_bias:
            gw, gb = fl.linear_splitk_t(gy, xt, column_sums=True)
        else:
            gw = fl.linear_splitk_t(gy, xt)
        if gw.stride(0) != weight.shape[1]:
            gw = gw.contiguous()
    else:
        gw = gy.t().mm(x.relu() if relu_x else x)
        if want_bias:
            gb = gy.sum(0)
    if mask is not None:
        gw = gw * mask
    return gw, gb


FUSED_BLOCKS = True  # residual blocks as one autograd node with the activations fused into the GEMMs


class _TCResidualBlock(torch.autograd.Function):
    """out = x + L1(relu(L0(relu(x))))  (ResidualBlock.forward, flowcon/nn/nets/resnet.py:40-52, and
    MaskedResidualBlock.forward, flowcon/transforms/made.py:170-181, without batch norm / dropout / context).

    Forward: two GEMMs; ReLU is applied to the operand while it is split for the tensor cores, the skip connection is
    added by the second GEMM's epilogue.  Backward: the ReLU derivative gates the input-gradient GEMMs in their
    epilogue (FC_LINEAR_RESIDUAL_GATES, the saved pre-activation is the gate), the weight-gradient products read
    max(x, 0) while packing and return the bias gradients.  7 launches of 5 kernels instead of 14 launches."""

    @staticmethod
    def forward(ctx, x, w0, b0, m0, w1, b1, m1):
        t1 = _gemm(x, fl.pack(w0, b0, mask=m0), w0.shape[0], relu_in=True)
        out = fl.linear(t1, fl.pack(w1, b1, mask=m1), relu_in=True, residual=x)
        ctx.save_for_backward(x, t1, w0, m0, w1, m1)
        ctx.bias = (b0 is not None, b1 is not None)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, t1, w0, m0, w1, m1 = ctx.saved_tensors
        g_out = g_out.contiguous()
        need = ctx.needs_input_grad
        gw0 = gb0 = gw1 = gb1 = gx = None
        if need[4] or (ctx.bias[1] and need[5]):
            gw1, gb1 = _wgrad(g_out, t1, w1, m1, ctx.bias[1] and need[5], relu_x=True)
        w1m = w1 if m1 is None else w1 * m1
        g_t1 = fl.linear(g_out, fl.pack(w1m.t().contiguous(), None), residual=t1, residual_gates=True)
        if need[1] or (ctx.bias[0] and need[2]):
            gw0, gb0 = _wgrad(g_t1, x, w0, m0, ctx.bias[0] and need[2], relu_x=True)
        if need[0]:
            w0m = w0 if m0 is None else w0 * m0
            gx = fl.linear(g_t1, fl.pack(w0m.t().contiguous(), None), residual=x, residual_gates=True)
            gx = gx.add_(g_out)
        return gx, gw0, gb0, None, gw1, gb1, None


def is_relu(activation):
    return activation is F.relu or activation is torch.relu or isinstance(activation, torch.nn.ReLU)


def residual_block_eligible(x, lin0, lin1):
    w0, w1 = lin0.weight, lin1.weight
    return (FUSED_BLOCKS and _eligible(x, w0) and _eligible(x, w1) and w0.shape[0] == w0.shape[1] == w1.shape[0]
            == w1.shape[1] and w0.shape[0] % 4 == 0 and x.stride(0) == x.shape[1] and torch.is_grad_enabled())


def residual_block(x, lin0, lin1):
    """x + lin1(relu(lin0(relu(x)))) for two nn.Linear / MaskedLinear modules of equal width."""
    return _TCResidualBlock.apply(x, lin0.weight, lin0.bias, getattr(lin0, "mask", None), lin1.weight, lin1.bias,
                                  getattr(lin1, "mask", None))


class _TCWgradLinear(torch.autograd.Function):
    """A layer whose forward reduction is too short for the 3xTF32 product (K < MIN_K, e.g. the first layer of a MADE
    over 16 features): forward and input gradient stay cuBLAS fp32, the weight gradient — a reduction over the whole
    batch — still runs on the tensor cores (and returns the bias gradient)."""

    @staticmethod
    def forward(ctx, x, weight, bias, mask):
        ctx.save_for_backward(x, weight, mask)
        ctx.has_bias = bias is not None
        return F.linear(x, weight if mask is None else weight * mask, bias)

    @staticmethod
    def backward(ctx, gy):
        x, weight, mask = ctx.saved_tensors
        gy = gy.contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = gy.mm(weight if mask is None else weight * mask)
        want_bias = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1]:
            gw, gb = _wgrad(gy, x, weight, mask, want_bias)
        if gb is None and want_bias:
            gb = gy.sum(0)
        return gx, gw, gb, None


def linear(x, weight, bias=None, mask=None):
    if not _eligible(x, weight) or gy_misaligned(weight):
        if (ENABLED and x.is_cuda and x.dtype == torch.float32 and x.dim() == 2
                and weight.dtype == torch.float32 and x.shape[0] >= 4096 and x.shape[0] % 4 == 0
                and weight.shape[0] % 4 == 0 and weight.shape[0] >= MIN_K and weight.requires_grad
                and torch.is_grad_enabled()):
            return _TCWgradLinear.apply(x, weight, bias, mask)
        return F.linear(x, weight if mask is None else weight * mask, bias)
    return _TCLinear.apply(x, weight, bias, mask)


def gy_misaligned(weight):
    # the input-gradient GEMM reads gy [M, N] through TMA: N * 4 bytes must be a multiple of 16
    return weight.shape[0] % 4 != 0


def module_linear(module, x):
    """`module(x)` for an nn.Linear / MaskedLinear, through `linear`."""
    return linear(x, module.weight, module.bias, getattr(module, "mask", None))
