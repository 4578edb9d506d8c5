"""torch custom ops (`torch.ops.flowcon_b200.*`) over the C-ABI kernels, with autograd.

Each op is one kernel launch on torch's current CUDA stream.  Layer ops take the FULL-width input
[B, D] plus int32 column lists, so the coupling split / scatter of the reference
(flowcon/transforms/coupling.py:82-83,96-98) happens inside the kernel; autoregressive / conditional
layers pass no column lists.  Backward ops recompute the forward intermediates from (x, params)
(SURVEY.md Appendix B) — nothing else is saved.
"""
import ctypes
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _cabi


def _cfg(num_bins, tails, inverse, identity_init, left, right, bottom, top, min_w, min_h, min_d, wh_scale):
    return _cabi.RqsConfig(int(num_bins), int(tails), int(identity_init), int(inverse), left, right, bottom, top,
                           min_w, min_h, min_d, wh_scale)


# ------------------------------------------------------------------------------------------------
# RQ-spline layer
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::rqs_layer", mutates_args=())
def rqs_layer(x: Tensor, params: Tensor, tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int,
              tails: int, inverse: bool, identity_init: bool, left: float, right: float, bottom: float, top: float,
              min_bin_width: float, min_bin_height: float, min_derivative: float,
              wh_scale: float) -> Tuple[Tensor, Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params, broadcast_ok=True)
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    y = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    status = torch.zeros((1,), dtype=torch.int32, device=x.device)
    cfg = _cfg(num_bins, tails, inverse, identity_init, left, right, bottom, top, min_bin_width, min_bin_height,
               min_derivative, wh_scale)
    p_per = 3 * num_bins - 1 if tails == _cabi.TAILS_LINEAR else 3 * num_bins + 1
    if params.shape[1] != d_t * p_per:
        raise ValueError("transform params have {} columns, expected {} x {}".format(params.shape[1], d_t, p_per))
    with torch.cuda.device(x.device), _cabi.launch("fc_rqs_apply", x.device):
        rc = L.fc_rqs_apply(xp, xs, pp, ps, y.data_ptr(), y.shape[1], lad.data_ptr(), 0, B, d_t, _cabi.cols(tcols),
                            _cabi.cols(ccols), ctypes.byref(cfg), status.data_ptr(), _cabi.stream_ptr(x.device))
    if rc == -1 and (min_bin_width * num_bins > 1.0 or min_bin_height * num_bins > 1.0):
        # flowcon/transforms/splines/rational_quadratic.py:86-89
        raise ValueError("Minimal bin width/height too large for the number of bins")
    _cabi.check(rc, "fc_rqs_apply")
    return y, lad, status


def rqs_bins(x, params, tcols, num_bins, tails, inverse, identity_init, left, right, bottom, top, min_bin_width,
             min_bin_height, min_derivative, wh_scale):
    """Parity aid (fc_rqs_bins): (bins int32 [B, D_t], knot distance [B, D_t]) as the kernels' own arithmetic sees them;
    bin -1 = outside the linear tails.  Same argument meaning as `rqs_layer`."""
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    bins = torch.empty((B, d_t), dtype=torch.int32, device=x.device)
    dist = torch.empty((B, d_t), dtype=torch.float32, device=x.device)
    cfg = _cfg(num_bins, tails, inverse, identity_init, left, right, bottom, top, min_bin_width, min_bin_height,
               min_derivative, wh_scale)
    with torch.cuda.device(x.device), _cabi.launch("fc_rqs_bins", x.device):
        rc = L.fc_rqs_bins(xp, xs, pp, ps, B, d_t, _cabi.cols(tcols), ctypes.byref(cfg), bins.data_ptr(), dist.data_ptr(),
                           _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_rqs_bins")
    return bins, dist


@rqs_layer.register_fake
def _(x, params, tcols, ccols, num_bins, tails, inverse, identity_init, left, right, bottom, top, min_bin_width,
      min_bin_height, min_derivative, wh_scale):
    return torch.empty_like(x), x.new_empty((x.shape[0],)), x.new_empty((1,), dtype=torch.int32)


@torch.library.custom_op("flowcon_b200::rqs_layer_backward", mutates_args=())
def rqs_layer_backward(x: Tensor, params: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                       tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int, tails: int, inverse: bool,
                       identity_init: bool, left: float, right: float, bottom: float, top: float,
                       min_bin_width: float, min_bin_height: float, min_derivative: float,
                       wh_scale: float) -> Tuple[Tensor, Tensor]:
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    gx = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    gp = torch.empty((B, params.shape[1]), dtype=x.dtype, device=x.device)
    if tcols is not None and (tcols.numel() + (ccols.numel() if ccols is not None else 0)) < x.shape[1]:
        gx.zero_()
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    cfg = _cfg(num_bins, tails, inverse, identity_init, left, right, bottom, top, min_bin_width, min_bin_height,
               min_derivative, wh_scale)
    with torch.cuda.device(x.device), _cabi.launch("fc_rqs_backward", x.device):
        rc = L.fc_rqs_backward(xp, xs, pp, ps, gyp, gys, glp, gx.data_ptr(), gx.shape[1], gp.data_ptr(), gp.shape[1],
                               B, d_t, _cabi.cols(tcols), _cabi.cols(ccols), ctypes.byref(cfg),
                               _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_rqs_backward")
    return gx, gp


@rqs_layer_backward.register_fake
def _(x, params, grad_y, grad_lad, tcols, ccols, *args):
    return torch.empty_like(x), torch.empty_like(params)


def _rqs_setup(ctx, inputs, output):
    x, params, tcols, ccols = inputs[:4]
    ctx.save_for_backward(x, params, tcols, ccols)
    ctx.hyper = inputs[4:]


def _rqs_backward(ctx, gy, gl, gstatus):
    x, params, tcols, ccols = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gp = rqs_layer_backward(x, params, gy, gl, tcols, ccols, *ctx.hyper)
    return (gx, gp) + (None,) * (2 + len(ctx.hyper))


rqs_layer.register_autograd(_rqs_backward, setup_context=_rqs_setup)


# ------------------------------------------------------------------------------------------------
# piecewise-linear spline layer
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::linspline_layer", mutates_args=())
def linspline_layer(x: Tensor, params: Tensor, tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int,
                    tails: int, inverse: bool, left: float, right: float, bottom: float,
                    top: float) -> Tuple[Tensor, Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params, broadcast_ok=True)
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    if params.shape[1] != d_t * num_bins:
        raise ValueError("transform params have {} columns, expected {} x {}".format(params.shape[1], d_t, num_bins))
    y = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    status = torch.zeros((1,), dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_linspline_apply", x.device):
        rc = L.fc_linspline_apply(xp, xs, pp, ps, y.data_ptr(), y.shape[1], lad.data_ptr(), 0, B, d_t,
                                  _cabi.cols(tcols), _cabi.cols(ccols), int(num_bins), int(tails), left, right, bottom,
                                  top, int(inverse), status.data_ptr(), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_linspline_apply")
    return y, lad, status


@linspline_layer.register_fake
def _(x, params, tcols, ccols, num_bins, tails, inverse, left, right, bottom, top):
    return torch.empty_like(x), x.new_empty((x.shape[0],)), x.new_empty((1,), dtype=torch.int32)


@torch.library.custom_op("flowcon_b200::linspline_layer_backward", mutates_args=())
def linspline_layer_backward(x: Tensor, params: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                             tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int, tails: int, inverse: bool,
                             left: float, right: float, bottom: float, top: float) -> Tuple[Tensor, Tensor]:
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    gx = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    gp = torch.empty((B, params.shape[1]), dtype=x.dtype, device=x.device)
    if tcols is not None and (tcols.numel() + (ccols.numel() if ccols is not None else 0)) < x.shape[1]:
        gx.zero_()
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch("fc_linspline_backward", x.device):
        rc = L.fc_linspline_backward(xp, xs, pp, ps, gyp, gys, glp, gx.data_ptr(), gx.shape[1], gp.data_ptr(),
                                     gp.shape[1], B, d_t, _cabi.cols(tcols), _cabi.cols(ccols), int(num_bins),
                                     int(tails), left, right, bottom, top, int(inverse), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_linspline_backward")
    return gx, gp


@linspline_layer_backward.register_fake
def _(x, params, grad_y, grad_lad, tcols, ccols, *args):
    return torch.empty_like(x), torch.empty_like(params)


def _linspline_setup(ctx, inputs, output):
    x, params, tcols, ccols = inputs[:4]
    ctx.save_for_backward(x, params, tcols, ccols)
    ctx.hyper = inputs[4:]


def _linspline_backward(ctx, gy, gl, gstatus):
    x, params, tcols, ccols = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gp = linspline_layer_backward(x, params, gy, gl, tcols, ccols, *ctx.hyper)
    return (gx, gp) + (None,) * (2 + len(ctx.hyper))


linspline_layer.register_autograd(_linspline_backward, setup_context=_linspline_setup)


# ------------------------------------------------------------------------------------------------
# piecewise-quadratic spline layer
# ------------------------------------------------------------------------------------------------
def _quad_cfg(num_bins, tails, inverse, left, right, bottom, top, min_w, min_h, wh_scale):
    return _cabi.QuadSplineConfig(int(num_bins), int(tails), int(inverse), left, right, bottom, top, min_w, min_h,
                                  wh_scale)


@torch.library.custom_op("flowcon_b200::quadspline_layer", mutates_args=())
def quadspline_layer(x: Tensor, params: Tensor, tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int,
                     tails: int, inverse: bool, left: float, right: float, bottom: float, top: float,
                     min_bin_width: float, min_bin_height: float, wh_scale: float) -> Tuple[Tensor, Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params, broadcast_ok=True)
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    p_per = 2 * num_bins - 1 if tails == _cabi.TAILS_LINEAR else 2 * num_bins + 1
    if params.shape[1] != d_t * p_per:
        raise ValueError("transform params have {} columns, expected {} x {}".format(params.shape[1], d_t, p_per))
    if min_bin_width * num_bins > 1.0:  # quadratic.py:77-80
        raise ValueError("Minimal bin width too large for the number of bins")
    if min_bin_height * num_bins > 1.0:
        raise ValueError("Minimal bin height too large for the number of bins")
    y = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    status = torch.zeros((1,), dtype=torch.int32, device=x.device)
    cfg = _quad_cfg(num_bins, tails, inverse, left, right, bottom, top, min_bin_width, min_bin_height, wh_scale)
    with torch.cuda.device(x.device), _cabi.launch("fc_quadspline_apply", x.device):
        rc = L.fc_quadspline_apply(xp, xs, pp, ps, y.data_ptr(), y.shape[1], lad.data_ptr(), 0, B, d_t,
                                   _cabi.cols(tcols), _cabi.cols(ccols), ctypes.byref(cfg), status.data_ptr(),
                                   _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_quadspline_apply")
    return y, lad, status


@quadspline_layer.register_fake
def _(x, params, tcols, ccols, num_bins, tails, inverse, left, right, bottom, top, min_bin_width, min_bin_height,
      wh_scale):
    return torch.empty_like(x), x.new_empty((x.shape[0],)), x.new_empty((1,), dtype=torch.int32)


@torch.library.custom_op("flowcon_b200::quadspline_layer_backward", mutates_args=())
def quadspline_layer_backward(x: Tensor, params: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                              tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int, tails: int,
                              inverse: bool, left: float, right: float, bottom: float, top: float,
                              min_bin_width: float, min_bin_height: float, wh_scale: float) -> Tuple[Tensor, Tensor]:
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    gx = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    gp = torch.empty((B, params.shape[1]), dtype=x.dtype, device=x.device)
    if tcols is not None and (tcols.numel() + (ccols.numel() if ccols is not None else 0)) < x.shape[1]:
        gx.zero_()
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    cfg = _quad_cfg(num_bins, tails, inverse, left, right, bottom, top, min_bin_width, min_bin_height, wh_scale)
    with torch.cuda.device(x.device), _cabi.launch("fc_quadspline_backward", x.device):
        rc = L.fc_quadspline_backward(xp, xs, pp, ps, gyp, gys, glp, gx.data_ptr(), gx.shape[1], gp.data_ptr(),
                                      gp.shape[1], B, d_t, _cabi.cols(tcols), _cabi.cols(ccols), ctypes.byref(cfg),
                                      _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_quadspline_backward")
    return gx, gp


@quadspline_layer_backward.register_fake
def _(x, params, grad_y, grad_lad, tcols, ccols, *args):
    return torch.empty_like(x), torch.empty_like(params)


def _quadspline_setup(ctx, inputs, output):
    x, params, tcols, ccols = inputs[:4]
    ctx.save_for_backward(x, params, tcols, ccols)
    ctx.hyper = inputs[4:]


def _quadspline_backward(ctx, gy, gl, gstatus):
    x, params, tcols, ccols = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gp = quadspline_layer_backward(x, params, gy, gl, tcols, ccols, *ctx.hyper)
    return (gx, gp) + (None,) * (2 + len(ctx.hyper))


quadspline_layer.register_autograd(_quadspline_backward, setup_context=_quadspline_setup)


# ------------------------------------------------------------------------------------------------
# cubic spline layer (same configuration struct as the quadratic layer)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::cubicspline_layer", mutates_args=())
def cubicspline_layer(x: Tensor, params: Tensor, tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int,
                     tails: int, inverse: bool, left: float, right: float, bottom: float, top: float,
                     min_bin_width: float, min_bin_height: float, wh_scale: float) -> Tuple[Tensor, Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params, broadcast_ok=True)
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    p_per = 2 * num_bins + 2
    if params.shape[1] != d_t * p_per:
        raise ValueError("transform params have {} columns, expected {} x {}".format(params.shape[1], d_t, p_per))
    if min_bin_width * num_bins > 1.0:  # cubic.py:89-92
        raise ValueError("Minimal bin width too large for the number of bins")
    if min_bin_height * num_bins > 1.0:
        raise ValueError("Minimal bin height too large for the number of bins")
    y = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    status = torch.zeros((1,), dtype=torch.int32, device=x.device)
    cfg = _quad_cfg(num_bins, tails, inverse, left, right, bottom, top, min_bin_width, min_bin_height, wh_scale)
    with torch.cuda.device(x.device), _cabi.launch("fc_cubicspline_apply", x.device):
        rc = L.fc_cubicspline_apply(xp, xs, pp, ps, y.data_ptr(), y.shape[1], lad.data_ptr(), 0, B, d_t,
                                   _cabi.cols(tcols), _cabi.cols(ccols), ctypes.byref(cfg), status.data_ptr(),
                                   _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_cubicspline_apply")
    return y, lad, status


@cubicspline_layer.register_fake
def _(x, params, tcols, ccols, num_bins, tails, inverse, left, right, bottom, top, min_bin_width, min_bin_height,
      wh_scale):
    return torch.empty_like(x), x.new_empty((x.shape[0],)), x.new_empty((1,), dtype=torch.int32)


@torch.library.custom_op("flowcon_b200::cubicspline_layer_backward", mutates_args=())
def cubicspline_layer_backward(x: Tensor, params: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                              tcols: Optional[Tensor], ccols: Optional[Tensor], num_bins: int, tails: int,
                              inverse: bool, left: float, right: float, bottom: float, top: float,
                              min_bin_width: float, min_bin_height: float, wh_scale: float) -> Tuple[Tensor, Tensor]:
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    gx = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    gp = torch.empty((B, params.shape[1]), dtype=x.dtype, device=x.device)
    if tcols is not None and (tcols.numel() + (ccols.numel() if ccols is not None else 0)) < x.shape[1]:
        gx.zero_()
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    cfg = _quad_cfg(num_bins, tails, inverse, left, right, bottom, top, min_bin_width, min_bin_height, wh_scale)
    with torch.cuda.device(x.device), _cabi.launch("fc_cubicspline_backward", x.device):
        rc = L.fc_cubicspline_backward(xp, xs, pp, ps, gyp, gys, glp, gx.data_ptr(), gx.shape[1], gp.data_ptr(),
                                      gp.shape[1], B, d_t, _cabi.cols(tcols), _cabi.cols(ccols), ctypes.byref(cfg),
                                      _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_cubicspline_backward")
    return gx, gp


@cubicspline_layer_backward.register_fake
def _(x, params, grad_y, grad_lad, tcols, ccols, *args):
    return torch.empty_like(x), torch.empty_like(params)


def _cubicspline_setup(ctx, inputs, output):
    x, params, tcols, ccols = inputs[:4]
    ctx.save_for_backward(x, params, tcols, ccols)
    ctx.hyper = inputs[4:]


def _cubicspline_backward(ctx, gy, gl, gstatus):
    x, params, tcols, ccols = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gp = cubicspline_layer_backward(x, params, gy, gl, tcols, ccols, *ctx.hyper)
    return (gx, gp) + (None,) * (2 + len(ctx.hyper))


cubicspline_layer.register_autograd(_cubicspline_backward, setup_context=_cubicspline_setup)


# ------------------------------------------------------------------------------------------------
# affine layer
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::affine_layer", mutates_args=())
def affine_layer(x: Tensor, params: Tensor, tcols: Optional[Tensor], ccols: Optional[Tensor], layout: int,
                 activation: int, inverse: bool) -> Tuple[Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params, broadcast_ok=True)
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    if params.shape[1] != 2 * d_t:
        raise ValueError("affine params have {} columns, expected {}".format(params.shape[1], 2 * d_t))
    y = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_affine_apply", x.device):
        rc = L.fc_affine_apply(xp, xs, pp, ps, y.data_ptr(), y.shape[1], lad.data_ptr(), 0, B, d_t,
                               _cabi.cols(tcols), _cabi.cols(ccols), layout, activation, int(inverse),
                               _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_affine_apply")
    return y, lad


@affine_layer.register_fake
def _(x, params, tcols, ccols, layout, activation, inverse):
    return torch.empty_like(x), x.new_empty((x.shape[0],))


@torch.library.custom_op("flowcon_b200::affine_layer_backward", mutates_args=())
def affine_layer_backward(x: Tensor, params: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                          tcols: Optional[Tensor], ccols: Optional[Tensor], layout: int, activation: int,
                          inverse: bool) -> Tuple[Tensor, Tensor]:
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B = x.shape[0]
    d_t = tcols.numel() if tcols is not None else x.shape[1]
    gx = torch.empty((B, x.shape[1]), dtype=x.dtype, device=x.device)
    gp = torch.empty((B, params.shape[1]), dtype=x.dtype, device=x.device)
    if tcols is not None and (tcols.numel() + (ccols.numel() if ccols is not None else 0)) < x.shape[1]:
        gx.zero_()
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch("fc_affine_backward", x.device):
        rc = L.fc_affine_backward(xp, xs, pp, ps, gyp, gys, glp, gx.data_ptr(), gx.shape[1], gp.data_ptr(),
                                  gp.shape[1], B, d_t, _cabi.cols(tcols), _cabi.cols(ccols), layout, activation,
                                  int(inverse), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_affine_backward")
    return gx, gp


@affine_layer_backward.register_fake
def _(x, params, grad_y, grad_lad, tcols, ccols, layout, activation, inverse):
    return torch.empty_like(x), torch.empty_like(params)


def _affine_setup(ctx, inputs, output):
    x, params, tcols, ccols = inputs[:4]
    ctx.save_for_backward(x, params, tcols, ccols)
    ctx.hyper = inputs[4:]


def _affine_backward(ctx, gy, gl):
    x, params, tcols, ccols = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gp = affine_layer_backward(x, params, gy, gl, tcols, ccols, *ctx.hyper)
    return (gx, gp) + (None,) * (2 + len(ctx.hyper))


affine_layer.register_autograd(_affine_backward, setup_context=_affine_setup)


# ------------------------------------------------------------------------------------------------
# activation normalisation (per-feature affine, parameters shared by the batch)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::actnorm_layer", mutates_args=())
def actnorm_layer(x: Tensor, log_scale: Tensor, shift: Tensor, inverse: bool) -> Tuple[Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(log_scale, "log_scale")
    _cabi.require_cuda_f32(shift, "shift")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    B, D = x.shape
    if log_scale.numel() != D or shift.numel() != D:
        raise ValueError("log_scale / shift must have {} entries".format(D))
    log_scale, shift = log_scale.contiguous(), shift.contiguous()
    y = torch.empty((B, D), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_actnorm_apply", x.device):
        rc = L.fc_actnorm_apply(xp, xs, log_scale.data_ptr(), shift.data_ptr(), y.data_ptr(), D, lad.data_ptr(), 0, B, D,
                                int(inverse), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_actnorm_apply")
    return y, lad


@actnorm_layer.register_fake
def _(x, log_scale, shift, inverse):
    return torch.empty_like(x), x.new_empty((x.shape[0],))


@torch.library.custom_op("flowcon_b200::actnorm_layer_backward", mutates_args=())
def actnorm_layer_backward(x: Tensor, log_scale: Tensor, shift: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                           inverse: bool) -> Tuple[Tensor, Tensor, Tensor]:
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B, D = x.shape
    log_scale, shift = log_scale.contiguous(), shift.contiguous()
    gx = torch.empty((B, D), dtype=x.dtype, device=x.device)
    gls = torch.empty((D,), dtype=x.dtype, device=x.device)
    gsh = torch.empty((D,), dtype=x.dtype, device=x.device)
    ws = torch.empty((max(int(L.fc_actnorm_workspace_floats(B, D)), 1),), dtype=x.dtype, device=x.device)
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch("fc_actnorm_backward", x.device):
        rc = L.fc_actnorm_backward(xp, xs, log_scale.data_ptr(), shift.data_ptr(), gyp, gys, glp, gx.data_ptr(), D,
                                   gls.data_ptr(), gsh.data_ptr(), ws.data_ptr(), B, D, int(inverse),
                                   _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_actnorm_backward")
    return gx, gls, gsh


@actnorm_layer_backward.register_fake
def _(x, log_scale, shift, grad_y, grad_lad, inverse):
    return torch.empty_like(x), torch.empty_like(log_scale), torch.empty_like(shift)


def _actnorm_setup(ctx, inputs, output):
    x, log_scale, shift, inverse = inputs
    ctx.save_for_backward(x, log_scale, shift)
    ctx.inverse = inverse


def _actnorm_backward(ctx, gy, gl):
    x, log_scale, shift = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gls, gsh = actnorm_layer_backward(x, log_scale, shift, gy, gl, ctx.inverse)
    return gx, gls.reshape(log_scale.shape), gsh.reshape(shift.shape), None


actnorm_layer.register_autograd(_actnorm_backward, setup_context=_actnorm_setup)


# ------------------------------------------------------------------------------------------------
# dense D x D row map of LULinear (D < 64): y = x M^T + c, logabsdet = logdet on every row
# ------------------------------------------------------------------------------------------------
def _lu_operands(M, c, D):
    if M.shape != (D, D) or c.numel() != D:
        raise ValueError("M must be [{0}, {0}] and c must have {0} entries".format(D))
    return M.contiguous(), c.contiguous()


@torch.library.custom_op("flowcon_b200::lulinear_layer", mutates_args=())
def lulinear_layer(x: Tensor, M: Tensor, c: Tensor, logdet: Tensor) -> Tuple[Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(M, "M")
    _cabi.require_cuda_f32(c, "c")
    _cabi.require_cuda_f32(logdet, "logdet")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    B, D = x.shape
    M, c = _lu_operands(M, c, D)
    logdet = logdet.reshape(()).contiguous()
    y = torch.empty((B, D), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_lulinear_apply", x.device):
        rc = L.fc_lulinear_apply(xp, xs, M.data_ptr(), c.data_ptr(), logdet.data_ptr(), y.data_ptr(), D, lad.data_ptr(),
                                 0, B, D, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_lulinear_apply")
    return y, lad


@lulinear_layer.register_fake
def _(x, M, c, logdet):
    return x.new_empty(x.shape), x.new_empty((x.shape[0],))


@torch.library.custom_op("flowcon_b200::lulinear_layer_backward", mutates_args=())
def lulinear_layer_backward(x: Tensor, M: Tensor, grad_y: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """(grad_x, grad_M, grad_c) of y = x M^T + c; grad_logdet = sum(grad_logabsdet) is left to the caller."""
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B, D = x.shape
    M = M.contiguous()
    gx = torch.empty((B, D), dtype=x.dtype, device=x.device)
    gM = torch.empty((D, D), dtype=x.dtype, device=x.device)
    gc = torch.empty((D,), dtype=x.dtype, device=x.device)
    ws = torch.empty((max(int(L.fc_lulinear_workspace_floats(B, D)), 1),), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_lulinear_backward", x.device):
        rc = L.fc_lulinear_backward(xp, xs, M.data_ptr(), gyp, gys, gx.data_ptr(), D, gM.data_ptr(), gc.data_ptr(),
                                    ws.data_ptr(), B, D, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_lulinear_backward")
    return gx, gM, gc


@lulinear_layer_backward.register_fake
def _(x, M, grad_y):
    D = x.shape[1]
    return x.new_empty(x.shape), x.new_empty((D, D)), x.new_empty((D,))


def _lulinear_setup(ctx, inputs, output):
    x, M, c, logdet = inputs
    ctx.save_for_backward(x, M)
    ctx.c_shape, ctx.logdet_shape = c.shape, logdet.shape


def _lulinear_backward(ctx, gy, gl):
    x, M = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, gM, gc = lulinear_layer_backward(x, M, gy)
    gld = gl.sum() if gl is not None else x.new_zeros(())
    return gx, gM, gc.reshape(ctx.c_shape), gld.reshape(ctx.logdet_shape)


lulinear_layer.register_autograd(_lulinear_backward, setup_context=_lulinear_setup)


# ------------------------------------------------------------------------------------------------
# batch normalisation (BatchNorm): per-feature statistics of the batch (training) or running buffers (eval)
# ------------------------------------------------------------------------------------------------
def _bn_vectors(D, **named):
    for name, t in named.items():
        _cabi.require_cuda_f32(t, name)
        if t.numel() != D:
            raise ValueError("{} must have {} entries".format(name, D))
    return [t.contiguous() for t in named.values()]


def _bn_apply(x, mean, var, uw, bias, eps, inverse):
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    B, D = x.shape
    y = torch.empty((B, D), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_batchnorm_apply", x.device):
        rc = L.fc_batchnorm_apply(xp, xs, mean.data_ptr(), var.data_ptr(), uw.data_ptr(), bias.data_ptr(), eps,
                                  y.data_ptr(), D, lad.data_ptr(), B, D, int(inverse), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_batchnorm_apply")
    return y, lad


def _bn_workspace(L, B, D, device):
    n = int(L.fc_batchnorm_workspace_floats(B, D))
    if n < 0:
        _cabi.check(n, "fc_batchnorm_workspace_floats")
    return torch.empty((max(n, 1),), dtype=torch.float32, device=device)


@torch.library.custom_op("flowcon_b200::batchnorm_train", mutates_args=())
def batchnorm_train(x: Tensor, unconstrained_weight: Tensor, bias: Tensor,
                    eps: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Training-mode BatchNorm: (y, logabsdet, batch mean, unbiased batch variance).  Three launches: the statistics
    (per-CTA Welford, then a fixed-order merge) and the forward pass.  The statistics outputs carry no gradient."""
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    B, D = x.shape
    uw, bias = _bn_vectors(D, unconstrained_weight=unconstrained_weight, bias=bias)
    mean = torch.empty((D,), dtype=x.dtype, device=x.device)
    var = torch.empty((D,), dtype=x.dtype, device=x.device)
    ws = _bn_workspace(L, B, D, x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_batchnorm_stats", x.device):
        rc = L.fc_batchnorm_stats(xp, xs, mean.data_ptr(), var.data_ptr(), ws.data_ptr(), B, D,
                                  _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_batchnorm_stats")
    y, lad = _bn_apply(x, mean, var, uw, bias, eps, False)
    return y, lad, mean, var


@batchnorm_train.register_fake
def _(x, unconstrained_weight, bias, eps):
    D = x.shape[1]
    return torch.empty_like(x), x.new_empty((x.shape[0],)), x.new_empty((D,)), x.new_empty((D,))


@torch.library.custom_op("flowcon_b200::batchnorm_eval", mutates_args=())
def batchnorm_eval(x: Tensor, running_mean: Tensor, running_var: Tensor, unconstrained_weight: Tensor, bias: Tensor,
                   eps: float, inverse: bool) -> Tuple[Tensor, Tensor]:
    """Eval-mode BatchNorm in either direction, from the running buffers: (y, logabsdet).  One launch."""
    _cabi.require_cuda_f32(x, "inputs")
    D = x.shape[1]
    rm, rv, uw, bias = _bn_vectors(D, running_mean=running_mean, running_var=running_var,
                                   unconstrained_weight=unconstrained_weight, bias=bias)
    return _bn_apply(x, rm, rv, uw, bias, eps, inverse)


@batchnorm_eval.register_fake
def _(x, running_mean, running_var, unconstrained_weight, bias, eps, inverse):
    return torch.empty_like(x), x.new_empty((x.shape[0],))


@torch.library.custom_op("flowcon_b200::batchnorm_backward", mutates_args=())
def batchnorm_backward(x: Tensor, mean: Tensor, var: Tensor, unconstrained_weight: Tensor, bias: Tensor, eps: float,
                       grad_y: Tensor, grad_lad: Optional[Tensor], mode: int) -> Tuple[Tensor, Tensor, Tensor]:
    """(grad_x, grad_unconstrained_weight, grad_bias); mode _cabi.BATCHNORM_TRAIN differentiates through the batch
    statistics (mean, var), the eval modes treat them as constants."""
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B, D = x.shape
    mean, var, uw, bias = (t.contiguous() for t in (mean, var, unconstrained_weight, bias))
    gx = torch.empty((B, D), dtype=x.dtype, device=x.device)
    guw = torch.empty((D,), dtype=x.dtype, device=x.device)
    gb = torch.empty((D,), dtype=x.dtype, device=x.device)
    ws = _bn_workspace(L, B, D, x.device)
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch("fc_batchnorm_backward", x.device):
        rc = L.fc_batchnorm_backward(xp, xs, mean.data_ptr(), var.data_ptr(), uw.data_ptr(), bias.data_ptr(), eps, gyp,
                                     gys, glp, gx.data_ptr(), D, guw.data_ptr(), gb.data_ptr(), ws.data_ptr(), B, D,
                                     int(mode), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_batchnorm_backward")
    return gx, guw, gb


@batchnorm_backward.register_fake
def _(x, mean, var, unconstrained_weight, bias, eps, grad_y, grad_lad, mode):
    D = x.shape[1]
    return torch.empty_like(x), x.new_empty((D,)), x.new_empty((D,))


def _bn_train_setup(ctx, inputs, output):
    x, uw, bias, eps = inputs
    _, _, mean, var = output
    ctx.save_for_backward(x, mean, var, uw, bias)
    ctx.eps = eps
    ctx.mark_non_differentiable(mean, var)


def _bn_train_backward(ctx, gy, gl, _gmean, _gvar):
    x, mean, var, uw, bias = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    gx, guw, gb = batchnorm_backward(x, mean, var, uw, bias, ctx.eps, gy, gl, _cabi.BATCHNORM_TRAIN)
    return gx, guw.reshape(uw.shape), gb.reshape(bias.shape), None


batchnorm_train.register_autograd(_bn_train_backward, setup_context=_bn_train_setup)


def _bn_eval_setup(ctx, inputs, output):
    x, rm, rv, uw, bias, eps, inverse = inputs
    ctx.save_for_backward(x, rm, rv, uw, bias)
    ctx.eps, ctx.inverse = eps, inverse


def _bn_eval_backward(ctx, gy, gl):
    x, rm, rv, uw, bias = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    mode = _cabi.BATCHNORM_EVAL_INVERSE if ctx.inverse else _cabi.BATCHNORM_EVAL_FORWARD
    gx, guw, gb = batchnorm_backward(x, rm, rv, uw, bias, ctx.eps, gy, gl, mode)
    return gx, None, None, guw.reshape(uw.shape), gb.reshape(bias.shape), None, None


batchnorm_eval.register_autograd(_bn_eval_backward, setup_context=_bn_eval_setup)


# ------------------------------------------------------------------------------------------------
# sum-of-sigmoids layer
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::sos_layer", mutates_args=())
def sos_layer(x: Tensor, params: Tensor, n_sigmoids: int, offset: float, inverse: bool, bisection_iterations: int,
              lim: float) -> Tuple[Tensor, Tensor]:
    _cabi.require_cuda_f32(x, "inputs")
    _cabi.require_cuda_f32(params, "transform params")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params, broadcast_ok=True)
    B, D = x.shape
    if params.shape[1] != D * (3 * n_sigmoids + 1):
        raise ValueError("sum-of-sigmoids params have {} columns, expected {}".format(
            params.shape[1], D * (3 * n_sigmoids + 1)))
    y = torch.empty((B, D), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_sos_apply", x.device):
        rc = L.fc_sos_apply(xp, xs, pp, ps, y.data_ptr(), D, lad.data_ptr(), 0, B, D, n_sigmoids, offset,
                            int(inverse), bisection_iterations, lim, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_sos_apply")
    return y, lad


@sos_layer.register_fake
def _(x, params, n_sigmoids, offset, inverse, bisection_iterations, lim):
    return torch.empty_like(x), x.new_empty((x.shape[0],))


def _sos_adjoint(entry, x, params, grad_y, grad_lad, n_sigmoids):
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    params, pp, ps = _cabi.rows(params)
    grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs"))
    B, D = x.shape
    gx = torch.empty((B, D), dtype=x.dtype, device=x.device)
    gp = torch.empty((B, params.shape[1]), dtype=x.dtype, device=x.device)
    glp = None
    if grad_lad is not None:
        grad_lad = grad_lad.contiguous()
        glp = grad_lad.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch(entry, x.device):
        rc = getattr(L, entry)(xp, xs, pp, ps, gyp, gys, glp, gx.data_ptr(), D, gp.data_ptr(), gp.shape[1], B, D,
                               n_sigmoids, _cabi.stream_ptr(x.device))
    _cabi.check(rc, entry)
    return gx, gp


@torch.library.custom_op("flowcon_b200::sos_layer_backward", mutates_args=())
def sos_layer_backward(x: Tensor, params: Tensor, grad_y: Tensor, grad_lad: Optional[Tensor],
                       n_sigmoids: int) -> Tuple[Tensor, Tensor]:
    return _sos_adjoint("fc_sos_backward", x, params, grad_y, grad_lad, n_sigmoids)


@sos_layer_backward.register_fake
def _(x, params, grad_y, grad_lad, n_sigmoids):
    return torch.empty_like(x), torch.empty_like(params)


@torch.library.custom_op("flowcon_b200::sos_layer_inverse_backward", mutates_args=())
def sos_layer_inverse_backward(x_out: Tensor, params: Tensor, grad_out: Tensor, grad_lad: Optional[Tensor],
                               n_sigmoids: int) -> Tuple[Tensor, Tensor]:
    """Adjoint of `sos_layer(..., inverse=True)`: x_out is the inverse's output.  Returns the gradients of the inverse's
    input z and of the raw parameters (the offset, iteration count and bracket do not enter)."""
    return _sos_adjoint("fc_sos_inverse_backward", x_out, params, grad_out, grad_lad, n_sigmoids)


@sos_layer_inverse_backward.register_fake
def _(x_out, params, grad_out, grad_lad, n_sigmoids):
    return torch.empty_like(x_out), torch.empty_like(params)


def _sos_setup(ctx, inputs, output):
    x, params, n_sigmoids, offset, inverse = inputs[:5]
    # the inverse's adjoint is evaluated at its own output: saving it spares a second numerical solve
    ctx.save_for_backward(output[0] if inverse else x, params)
    ctx.n_sigmoids = n_sigmoids
    ctx.inverse = inverse


def _sos_backward(ctx, gy, gl):
    x, params = ctx.saved_tensors
    if gy is None:
        gy = torch.zeros_like(x)
    adjoint = sos_layer_inverse_backward if ctx.inverse else sos_layer_backward
    gx, gp = adjoint(x, params, gy, gl, ctx.n_sigmoids)
    return gx, gp, None, None, None, None, None


sos_layer.register_autograd(_sos_backward, setup_context=_sos_setup)


# ------------------------------------------------------------------------------------------------
# standard-normal tail
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowcon_b200::stdnormal_log_prob", mutates_args=())
def stdnormal_log_prob(z: Tensor, logabsdet: Optional[Tensor]) -> Tensor:
    _cabi.require_cuda_f32(z, "noise")
    L = _cabi.lib()
    z, zp, zs = _cabi.rows(z)
    B, D = z.shape
    out = torch.empty((B,), dtype=z.dtype, device=z.device)
    ladp = None
    if logabsdet is not None:
        logabsdet = _cabi.require_cuda_f32(logabsdet, "logabsdet").contiguous()
        ladp = logabsdet.data_ptr()
    with torch.cuda.device(z.device), _cabi.launch("fc_stdnormal_log_prob", z.device):
        rc = L.fc_stdnormal_log_prob(zp, zs, ladp, out.data_ptr(), B, D, _cabi.stream_ptr(z.device))
    _cabi.check(rc, "fc_stdnormal_log_prob")
    return out


@stdnormal_log_prob.register_fake
def _(z, logabsdet):
    return z.new_empty((z.shape[0],))


def _sn_setup(ctx, inputs, output):
    z, lad = inputs
    ctx.save_for_backward(z)
    ctx.has_lad = lad is not None


def _sn_backward(ctx, g):
    (z,) = ctx.saved_tensors
    return -z * g[:, None], (g if ctx.has_lad else None)


stdnormal_log_prob.register_autograd(_sn_backward, setup_context=_sn_setup)


# ------------------------------------------------------------------------------------------------
# diagonal Gaussian base densities (DiagonalNormal, ConditionalDiagonalNormal): params [C, 2D] = [means | log stds],
# data row r uses parameter row r // group
# ------------------------------------------------------------------------------------------------
def _dn_operands(rows, params, D, group):
    _cabi.require_cuda_f32(params, "base density params")
    if params.dim() != 2 or params.shape[1] != 2 * D:
        raise ValueError("base density params must be [C, {}], got {}".format(2 * D, tuple(params.shape)))
    want = max(1, -(-rows // group)) if group >= 1 else -1  # an empty batch still has its one shared row
    if params.shape[0] != want:
        raise ValueError("{} rows in groups of {} need {} parameter rows, got {}".format(
            rows, group, want, params.shape[0]))
    return _cabi.rows(params)


def _dn_workspace(L, R, D, group, device):
    n = int(L.fc_diagnormal_workspace_floats(R, D, group))
    if n < 0:
        _cabi.check(n, "fc_diagnormal_workspace_floats")
    return torch.empty((max(n, 1),), dtype=torch.float32, device=device)


@torch.library.custom_op("flowcon_b200::diagnormal_log_prob", mutates_args=())
def diagnormal_log_prob(x: Tensor, params: Tensor, group: int, logabsdet: Optional[Tensor]) -> Tensor:
    """log N(x; m, diag e^{2s}) per row (+ logabsdet) in one pass; row r reads parameter row r // group."""
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    R, D = x.shape
    params, pp, ps = _dn_operands(R, params, D, group)
    out = torch.empty((R,), dtype=x.dtype, device=x.device)
    ladp = None
    if logabsdet is not None:
        logabsdet = _cabi.require_cuda_f32(logabsdet, "logabsdet").contiguous()
        ladp = logabsdet.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch("fc_diagnormal_log_prob", x.device):
        rc = L.fc_diagnormal_log_prob(xp, xs, pp, ps, ladp, out.data_ptr(), R, D, group, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_diagnormal_log_prob")
    return out


@diagnormal_log_prob.register_fake
def _(x, params, group, logabsdet):
    return x.new_empty((x.shape[0],))


@torch.library.custom_op("flowcon_b200::diagnormal_log_prob_backward", mutates_args=())
def diagnormal_log_prob_backward(x: Tensor, params: Tensor, group: int, grad_out: Tensor) -> Tuple[Tensor, Tensor]:
    """(grad_x [R, D], grad_params [C, 2D]); the parameter gradients are group sums taken in a fixed order."""
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    R, D = x.shape
    params, pp, ps = _dn_operands(R, params, D, group)
    grad_out = _cabi.require_cuda_f32(grad_out, "grad outputs").contiguous()
    gx = torch.empty((R, D), dtype=x.dtype, device=x.device)
    gp = (torch.empty if R > 0 else torch.zeros)((params.shape[0], 2 * D), dtype=x.dtype, device=x.device)
    ws = _dn_workspace(L, R, D, group, x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_diagnormal_log_prob_backward", x.device):
        rc = L.fc_diagnormal_log_prob_backward(xp, xs, pp, ps, grad_out.data_ptr(), gx.data_ptr(), D, gp.data_ptr(),
                                               ws.data_ptr(), R, D, group, _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_diagnormal_log_prob_backward")
    return gx, gp


@diagnormal_log_prob_backward.register_fake
def _(x, params, group, grad_out):
    return torch.empty_like(x), params.new_empty((params.shape[0], 2 * x.shape[1]))


def _dn_lp_setup(ctx, inputs, output):
    x, params, group, lad = inputs
    ctx.save_for_backward(x, params)
    ctx.group = group
    ctx.has_lad = lad is not None


def _dn_lp_backward(ctx, g):
    x, params = ctx.saved_tensors
    gx, gp = diagnormal_log_prob_backward(x, params, ctx.group, g)
    return gx, gp, None, (g if ctx.has_lad else None)


diagnormal_log_prob.register_autograd(_dn_lp_backward, setup_context=_dn_lp_setup)


@torch.library.custom_op("flowcon_b200::diagnormal_sample", mutates_args=())
def diagnormal_sample(noise: Tensor, params: Tensor, group: int) -> Tensor:
    """m + e^{s} · noise per row; row r reads parameter row r // group (no repeated copies of the parameters)."""
    _cabi.require_cuda_f32(noise, "noise")
    L = _cabi.lib()
    noise, np_, ns = _cabi.rows(noise)
    R, D = noise.shape
    params, pp, ps = _dn_operands(R, params, D, group)
    y = torch.empty((R, D), dtype=noise.dtype, device=noise.device)
    with torch.cuda.device(noise.device), _cabi.launch("fc_diagnormal_sample", noise.device):
        rc = L.fc_diagnormal_sample(np_, ns, pp, ps, y.data_ptr(), D, R, D, group, _cabi.stream_ptr(noise.device))
    _cabi.check(rc, "fc_diagnormal_sample")
    return y


@diagnormal_sample.register_fake
def _(noise, params, group):
    return torch.empty_like(noise)


@torch.library.custom_op("flowcon_b200::diagnormal_sample_backward", mutates_args=())
def diagnormal_sample_backward(noise: Tensor, params: Tensor, group: int, grad_samples: Tensor) -> Tensor:
    """grad_params [C, 2D]: group sums of grad_samples and of grad_samples · e^{s} · noise, in a fixed order."""
    L = _cabi.lib()
    noise, np_, ns = _cabi.rows(noise)
    R, D = noise.shape
    params, pp, ps = _dn_operands(R, params, D, group)
    grad_samples, gsp, gss = _cabi.rows(_cabi.require_cuda_f32(grad_samples, "grad outputs"))
    gp = (torch.empty if R > 0 else torch.zeros)((params.shape[0], 2 * D), dtype=noise.dtype, device=noise.device)
    ws = _dn_workspace(L, R, D, group, noise.device)
    with torch.cuda.device(noise.device), _cabi.launch("fc_diagnormal_sample_backward", noise.device):
        rc = L.fc_diagnormal_sample_backward(np_, ns, pp, ps, gsp, gss, gp.data_ptr(), ws.data_ptr(), R, D, group,
                                             _cabi.stream_ptr(noise.device))
    _cabi.check(rc, "fc_diagnormal_sample_backward")
    return gp


@diagnormal_sample_backward.register_fake
def _(noise, params, group, grad_samples):
    return params.new_empty((params.shape[0], 2 * noise.shape[1]))


def _dn_sample_setup(ctx, inputs, output):
    noise, params, group = inputs
    ctx.save_for_backward(noise, params)
    ctx.group = group


def _dn_sample_backward(ctx, gy):
    noise, params = ctx.saved_tensors
    return None, diagnormal_sample_backward(noise, params, ctx.group, gy), None


diagnormal_sample.register_autograd(_dn_sample_backward, setup_context=_dn_sample_setup)


# ------------------------------------------------------------------------------------------------
# element-wise squashing layers (Sigmoid / Logit, Tanh, LeakyReLU, Exp, CauchyCDF): x [B, N] -> (y [B, N], logabsdet [B])
# ------------------------------------------------------------------------------------------------
def _pw_cfg(op, inverse, slope, eps, temperature):
    tp = None
    if op == _cabi.POINTWISE_SIGMOID:
        _cabi.require_cuda_f32(temperature, "temperature")
        if temperature.numel() != 1:
            raise ValueError("temperature must have one element")
        tp = temperature.data_ptr()
    return _cabi.PointwiseConfig(int(op), int(inverse), float(slope), float(eps), tp)


@torch.library.custom_op("flowcon_b200::pointwise_layer", mutates_args=())
def pointwise_layer(x: Tensor, temperature: Optional[Tensor], op: int, inverse: bool, slope: float,
                    eps: float) -> Tuple[Tensor, Tensor, Tensor]:
    """(y, logabsdet, status): one pass over x [B, N] (any row stride >= N); status carries
    FC_STATUS_INPUT_OUTSIDE_DOMAIN for the directions with a domain.  temperature: device [1] (Sigmoid only)."""
    _cabi.require_cuda_f32(x, "inputs")
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    B, N = x.shape
    if temperature is not None:
        temperature = temperature.contiguous()
    cfg = _pw_cfg(op, inverse, slope, eps, temperature)
    y = torch.empty((B, N), dtype=x.dtype, device=x.device)
    lad = torch.empty((B,), dtype=x.dtype, device=x.device)
    status = torch.zeros((1,), dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device), _cabi.launch("fc_pointwise_apply", x.device):
        rc = L.fc_pointwise_apply(xp, xs, y.data_ptr(), N, lad.data_ptr(), 0, B, N, ctypes.byref(cfg),
                                  status.data_ptr(), _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_pointwise_apply")
    return y, lad, status


@pointwise_layer.register_fake
def _(x, temperature, op, inverse, slope, eps):
    return torch.empty_like(x), x.new_empty((x.shape[0],)), x.new_empty((1,), dtype=torch.int32)


@torch.library.custom_op("flowcon_b200::pointwise_layer_backward", mutates_args=())
def pointwise_layer_backward(x: Tensor, temperature: Optional[Tensor], grad_y: Optional[Tensor],
                             grad_lad: Optional[Tensor], op: int, inverse: bool, slope: float, eps: float,
                             want_temperature: bool) -> Tuple[Tensor, Tensor]:
    """(grad_x [B, N], grad_temperature [1]) at the layer's input x; grad_temperature is a fixed-order sum over every
    element when want_temperature, else zero."""
    L = _cabi.lib()
    x, xp, xs = _cabi.rows(x)
    B, N = x.shape
    if temperature is not None:
        temperature = temperature.contiguous()
    cfg = _pw_cfg(op, inverse, slope, eps, temperature)
    gyp, gys = None, N
    if grad_y is not None:
        grad_y, gyp, gys = _cabi.rows(_cabi.require_cuda_f32(grad_y, "grad outputs").reshape(B, N))
    glp = None
    if grad_lad is not None:
        grad_lad = _cabi.require_cuda_f32(grad_lad, "grad logabsdet").contiguous()
        glp = grad_lad.data_ptr()
    gx = torch.empty((B, N), dtype=x.dtype, device=x.device)
    gt = torch.zeros((1,), dtype=x.dtype, device=x.device)
    gtp, ws = None, None
    if want_temperature:
        n = int(L.fc_pointwise_workspace_floats(B, N))
        _cabi.check(min(n, 0), "fc_pointwise_workspace_floats")
        ws = torch.empty((n,), dtype=torch.float32, device=x.device)
        gtp = gt.data_ptr()
    with torch.cuda.device(x.device), _cabi.launch("fc_pointwise_backward", x.device):
        rc = L.fc_pointwise_backward(xp, xs, gyp, gys, glp, gx.data_ptr(), N, gtp,
                                     None if ws is None else ws.data_ptr(), B, N, ctypes.byref(cfg),
                                     _cabi.stream_ptr(x.device))
    _cabi.check(rc, "fc_pointwise_backward")
    return gx, gt


@pointwise_layer_backward.register_fake
def _(x, temperature, grad_y, grad_lad, op, inverse, slope, eps, want_temperature):
    return torch.empty_like(x), x.new_empty((1,))


def _pw_setup(ctx, inputs, output):
    x, temperature, op, inverse, slope, eps = inputs
    ctx.save_for_backward(x, temperature)
    ctx.hyper = (op, inverse, slope, eps)
    ctx.mark_non_differentiable(output[2])


def _pw_backward(ctx, gy, gl, _gstatus):
    x, temperature = ctx.saved_tensors
    want_t = temperature is not None and ctx.needs_input_grad[1]
    gx, gt = pointwise_layer_backward(x, temperature, gy, gl, *ctx.hyper, want_t)
    return gx, (gt.reshape(temperature.shape) if want_t else None), None, None, None, None


pointwise_layer.register_autograd(_pw_backward, setup_context=_pw_setup)
