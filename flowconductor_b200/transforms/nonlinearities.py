"""Element-wise layers of flowcon/transforms/nonlinearities.py on the hot path.

The squashing layers (`Sigmoid` / `Logit`, `Tanh`, `LeakyReLU`, `Exp`, `CauchyCDF` / `CauchyCDFInverse`, and
`CompositeCDFTransform` around a CDF layer) run on csrc/fc_pointwise.cu: one pass computes the map and the summed
log-det, with the domain check of the reference's inverses as a device status word.

The unconditional element-wise CDF layers: `PiecewiseRationalQuadraticCDF`
(flowcon/transforms/nonlinearities.py:406-487) — a rational-quadratic spline whose parameters are learnable tensors
shared across the batch (`_share_across_batch` :246-247) instead of a conditioner output.  Same constructor, same
parameter names and shapes (`unnormalized_widths` [*shape, K], `unnormalized_heights` [*shape, K],
`unnormalized_derivatives` [*shape, K-1 | K+1]), so reference state_dicts load.  It is what
`PiecewiseRationalQuadraticCouplingTransform(apply_unconditional_transform=True)` puts on the identity features
(coupling.py:524-535).

The evaluation is the same kernel as every other RQ layer (`fc_rqs_apply` / `fc_rqs_backward` through
`splines.RationalQuadraticSettings`): no 1/sqrt(H) scaling, identity-init off, [0, 1] box when tails is None."""
import math

import numpy as np
import torch
from torch import nn

from .. import _cabi, ops
from . import splines
from .base import CompositeTransform, InputOutsideDomain, InverseTransform, Transform

__all__ = ["CauchyCDF", "CauchyCDFInverse", "CompositeCDFTransform", "Exp", "LeakyReLU", "Logit", "PiecewiseCubicCDF",
           "PiecewiseLinearCDF", "PiecewiseQuadraticCDF", "PiecewiseRationalQuadraticCDF", "Sigmoid", "Tanh"]


# ------------------------------------------------------------------------------------------------
# element-wise squashing layers (nonlinearities.py: Tanh, Sigmoid, Logit, LeakyReLU, Exp, CauchyCDF, CauchyCDFInverse,
# CompositeCDFTransform): one pass of fc_pointwise_apply per call, map and summed log-det together
# ------------------------------------------------------------------------------------------------
def _pointwise(inputs, op, inverse, check, temperature=None, slope=0.0, eps=0.0):
    """inputs [B, ...] viewed as [B, N] (copied only when no such view exists; a 2-D column slice keeps its row
    stride).  check: this direction raises InputOutsideDomain like the reference, which reads the kernel's status word
    on the host — a synchronisation a CUDA graph cannot record."""
    _cabi.require_cuda_f32(inputs, "inputs")
    if inputs.dim() < 2:
        raise ValueError("expected inputs of shape [batch, ...], got {}".format(tuple(inputs.shape)))
    if check and torch.cuda.is_current_stream_capturing():
        raise RuntimeError("this direction of the layer checks its inputs' domain on the host (the reference raises "
                           "InputOutsideDomain): that synchronisation cannot be recorded into a CUDA graph")
    flat = inputs.reshape(inputs.shape[0], math.prod(inputs.shape[1:]))
    y, lad, status = ops.pointwise_layer(flat, temperature, op, bool(inverse), float(slope), float(eps))
    if check and int(status.item()) & _cabi.STATUS_INPUT_OUTSIDE_DOMAIN:
        raise InputOutsideDomain()
    return y.reshape(inputs.shape), lad


class Tanh(Transform):
    """nonlinearities.py Tanh: y = tanh x.  The forward log-det is 2 (log 2 − |x| − softplus(−2|x|)) = log(1 − tanh² x),
    finite where the reference's fp32 rounds tanh x to ±1."""

    def forward(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_TANH, False, False)

    def inverse(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_TANH, True, True)


class Sigmoid(Transform):
    """nonlinearities.py Sigmoid: y = σ(T x); the inverse clamps its input to [eps, 1 − eps].  `temperature` is a [1]
    buffer, or a parameter with learn_temperature; the kernels read it on the device."""

    def __init__(self, temperature=1, eps=1e-6, learn_temperature=False):
        super().__init__()
        self.eps = eps
        if learn_temperature:
            self.temperature = nn.Parameter(torch.Tensor([temperature]))
        else:
            self.register_buffer("temperature", torch.Tensor([temperature]))

    def forward(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_SIGMOID, False, False, self.temperature, eps=self.eps)

    def inverse(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_SIGMOID, True, True, self.temperature, eps=self.eps)


class Logit(InverseTransform):
    """nonlinearities.py Logit: the inverse of Sigmoid (its temperature is `_transform.temperature`)."""

    def __init__(self, temperature=1, eps=1e-6):
        super().__init__(Sigmoid(temperature=temperature, eps=eps))


class LeakyReLU(Transform):
    """nonlinearities.py LeakyReLU; the log-det lives on the inputs' device, fp32."""

    def __init__(self, negative_slope=1e-2):
        if negative_slope <= 0:
            raise ValueError("Slope must be positive.")
        super().__init__()
        self.negative_slope = negative_slope
        self.log_negative_slope = torch.log(torch.as_tensor(self.negative_slope))

    def forward(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_LEAKY_RELU, False, False, slope=self.negative_slope)

    def inverse(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_LEAKY_RELU, True, False, slope=self.negative_slope)


class Exp(Transform):
    """nonlinearities.py Exp: y = eˣ, log-det x; the inverse raises for inputs <= 0."""

    def forward(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_EXP, False, False)

    def inverse(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_EXP, True, True)


class CauchyCDF(Transform):
    """nonlinearities.py CauchyCDF: y = atan(x) / π + ½ (location, scale and features are accepted and unused, as in the
    reference); the inverse raises for inputs outside [0, 1]."""

    def __init__(self, location=None, scale=None, features=None):
        super().__init__()

    def forward(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_CAUCHY_CDF, False, False)

    def inverse(self, inputs, context=None):
        return _pointwise(inputs, _cabi.POINTWISE_CAUCHY_CDF, True, True)


class CauchyCDFInverse(InverseTransform):
    """nonlinearities.py CauchyCDFInverse."""

    def __init__(self, location=None, scale=None, features=None):
        super().__init__(transform=CauchyCDF(location=location, scale=scale, features=features))


class CompositeCDFTransform(CompositeTransform):
    """nonlinearities.py CompositeCDFTransform: squash, apply the CDF on the unit box, unsquash."""

    def __init__(self, squashing_transform, cdf_transform):
        super().__init__([squashing_transform, cdf_transform, InverseTransform(squashing_transform)])


class PiecewiseRationalQuadraticCDF(Transform):
    def __init__(self, shape, num_bins=10, tails=None, tail_bound=1.0, identity_init=False,
                 min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH, min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT,
                 min_derivative=splines.DEFAULT_MIN_DERIVATIVE):
        super().__init__()
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.min_derivative = min_derivative
        self.tail_bound = tail_bound
        self.tails = tails
        if isinstance(shape, int):
            shape = (shape,)
        shape = tuple(shape)
        if len(shape) != 1:
            raise NotImplementedError("image-shaped CDF layers are outside the B200 hot path")
        num_derivatives = (num_bins - 1) if tails == "linear" else (num_bins + 1)
        if identity_init:  # nonlinearities.py:430-440
            constant = float(np.log(np.exp(1 - min_derivative) - 1))
            self.unnormalized_widths = nn.Parameter(torch.zeros(*shape, num_bins))
            self.unnormalized_heights = nn.Parameter(torch.zeros(*shape, num_bins))
            self.unnormalized_derivatives = nn.Parameter(constant * torch.ones(*shape, num_derivatives))
        else:  # :441-450 (same draw order as the reference: widths, heights, derivatives)
            self.unnormalized_widths = nn.Parameter(torch.rand(*shape, num_bins))
            self.unnormalized_heights = nn.Parameter(torch.rand(*shape, num_bins))
            self.unnormalized_derivatives = nn.Parameter(torch.rand(*shape, num_derivatives))
        # the reference never enables the identity-init boundary rule for this layer (it calls the spline functions
        # with their default enable_identity_init=False, :465-477)
        self._spline = splines.RationalQuadraticSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height,
                                                         min_derivative, identity_init=False,
                                                         constrained_box=(0.0, 1.0))

    def _shared_params(self, batch_size):
        """[D, P] per-feature blocks [w ; h ; d] -> one row, shared by every sample (expanded view)."""
        p = torch.cat((self.unnormalized_widths, self.unnormalized_heights, self.unnormalized_derivatives), dim=-1)
        return p.reshape(1, -1).expand(batch_size, -1)

    def apply_on_columns(self, inputs, tcols, ccols, inverse):
        """The layer applied to columns `tcols` of a wider tensor (the other columns, `ccols`, are copied): what a
        coupling layer needs for its identity features, without gathering them first."""
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), tcols, ccols, inverse, None)

    def _run(self, inputs, inverse):
        if inputs.dim() != 2 or inputs.shape[1] != self.unnormalized_widths.shape[0]:
            raise ValueError("expected inputs of shape [batch, {}]".format(self.unnormalized_widths.shape[0]))
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), None, None, inverse, None)

    def forward(self, inputs, context=None):
        return self._run(inputs, inverse=False)

    def inverse(self, inputs, context=None):
        return self._run(inputs, inverse=True)


class PiecewiseLinearCDF(Transform):
    """flowcon/transforms/nonlinearities.py:250-283: a piecewise-linear spline whose `unnormalized_pdf` [*shape, K] is a
    learnable tensor shared across the batch."""

    def __init__(self, shape, num_bins=10, tails=None, tail_bound=1.0):
        super().__init__()
        self.tail_bound = tail_bound
        self.tails = tails
        if isinstance(shape, int):
            shape = (shape,)
        shape = tuple(shape)
        if len(shape) != 1:
            raise NotImplementedError("image-shaped CDF layers are outside the B200 hot path")
        self.unnormalized_pdf = nn.Parameter(torch.randn(*shape, num_bins))
        self._spline = splines.LinearSplineSettings(num_bins, tails, tail_bound)

    def _shared_params(self, batch_size):
        return self.unnormalized_pdf.reshape(1, -1).expand(batch_size, -1)

    def apply_on_columns(self, inputs, tcols, ccols, inverse):
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), tcols, ccols, inverse)

    def _run(self, inputs, inverse):
        if inputs.dim() != 2 or inputs.shape[1] != self.unnormalized_pdf.shape[0]:
            raise ValueError("expected inputs of shape [batch, {}]".format(self.unnormalized_pdf.shape[0]))
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), None, None, inverse)

    def forward(self, inputs, context=None):
        return self._run(inputs, inverse=False)

    def inverse(self, inputs, context=None):
        return self._run(inputs, inverse=True)


class PiecewiseQuadraticCDF(Transform):
    """flowcon/transforms/nonlinearities.py:286-340: learnable `unnormalized_widths` [*shape, K] and
    `unnormalized_heights` [*shape, K+1] (K-1 with linear tails), shared across the batch."""

    def __init__(self, shape, num_bins=10, tails=None, tail_bound=1.0, min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH,
                 min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT):
        super().__init__()
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.tail_bound = tail_bound
        self.tails = tails
        if isinstance(shape, int):
            shape = (shape,)
        shape = tuple(shape)
        if len(shape) != 1:
            raise NotImplementedError("image-shaped CDF layers are outside the B200 hot path")
        self.unnormalized_widths = nn.Parameter(torch.randn(*shape, num_bins))
        self.unnormalized_heights = nn.Parameter(torch.randn(*shape, num_bins + 1 if tails is None else num_bins - 1))
        self._spline = splines.QuadraticSplineSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height)

    def _shared_params(self, batch_size):
        p = torch.cat((self.unnormalized_widths, self.unnormalized_heights), dim=-1)
        return p.reshape(1, -1).expand(batch_size, -1)

    def apply_on_columns(self, inputs, tcols, ccols, inverse):
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), tcols, ccols, inverse, None)

    def _run(self, inputs, inverse):
        if inputs.dim() != 2 or inputs.shape[1] != self.unnormalized_widths.shape[0]:
            raise ValueError("expected inputs of shape [batch, {}]".format(self.unnormalized_widths.shape[0]))
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), None, None, inverse, None)

    def forward(self, inputs, context=None):
        return self._run(inputs, inverse=False)

    def inverse(self, inputs, context=None):
        return self._run(inputs, inverse=True)


class PiecewiseCubicCDF(Transform):
    """flowcon/transforms/nonlinearities.py:342-404: learnable `unnormalized_widths` / `unnormalized_heights` [*shape, K]
    and `unnorm_derivatives_left` / `unnorm_derivatives_right` [*shape, 1], shared across the batch."""

    def __init__(self, shape, num_bins=10, tails=None, tail_bound=1.0, min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH,
                 min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT):
        super().__init__()
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.tail_bound = tail_bound
        self.tails = tails
        if isinstance(shape, int):
            shape = (shape,)
        shape = tuple(shape)
        if len(shape) != 1:
            raise NotImplementedError("image-shaped CDF layers are outside the B200 hot path")
        self.unnormalized_widths = nn.Parameter(torch.randn(*shape, num_bins))
        self.unnormalized_heights = nn.Parameter(torch.randn(*shape, num_bins))
        self.unnorm_derivatives_left = nn.Parameter(torch.randn(*shape, 1))
        self.unnorm_derivatives_right = nn.Parameter(torch.randn(*shape, 1))
        self._spline = splines.CubicSplineSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height)

    def _shared_params(self, batch_size):
        p = torch.cat((self.unnormalized_widths, self.unnormalized_heights, self.unnorm_derivatives_left,
                       self.unnorm_derivatives_right), dim=-1)
        return p.reshape(1, -1).expand(batch_size, -1)

    def apply_on_columns(self, inputs, tcols, ccols, inverse):
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), tcols, ccols, inverse, None)

    def _run(self, inputs, inverse):
        if inputs.dim() != 2 or inputs.shape[1] != self.unnormalized_widths.shape[0]:
            raise ValueError("expected inputs of shape [batch, {}]".format(self.unnormalized_widths.shape[0]))
        return self._spline.apply(inputs, self._shared_params(inputs.shape[0]), None, None, inverse, None)

    def forward(self, inputs, context=None):
        return self._run(inputs, inverse=False)

    def inverse(self, inputs, context=None):
        return self._run(inputs, inverse=True)
