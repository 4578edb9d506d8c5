"""Coupling layers on the hot path, API of flowcon/transforms/coupling.py (CouplingTransform :20-142,
AffineCouplingTransform :212-252, AdditiveCouplingTransform :255-269, PiecewiseRationalQuadraticCouplingTransform
:502-582).  Same constructor arguments, same buffers (`identity_features`, `transform_features`) and sub-module
names (`transform_net`), so reference state_dicts load.

What changed: the conditioner output goes straight into ONE kernel that evaluates the bijection on the
transform columns, copies the identity columns, and reduces the per-sample log-det — the reference's
gather / scatter / mask-dispatch / 40-op pointwise chain (coupling.py:82-98, rational_quadratic.py) is gone.
"""
import warnings

import torch

from .. import _cabi, ops
from ..nn import tensorcore
from . import splines
from .base import Transform
from .nonlinearities import (PiecewiseCubicCDF, PiecewiseLinearCDF, PiecewiseQuadraticCDF,
                            PiecewiseRationalQuadraticCDF)


class CouplingTransform(Transform):
    def __init__(self, mask, transform_net_create_fn, unconditional_transform=None):
        mask = torch.as_tensor(mask)
        if mask.dim() != 1:
            raise ValueError("Mask must be a 1-dim tensor.")
        if mask.numel() <= 0:
            raise ValueError("Mask can't be empty.")
        super().__init__()
        self.features = len(mask)
        index = torch.arange(self.features)
        self.register_buffer("identity_features", index.masked_select(mask <= 0))
        self.register_buffer("transform_features", index.masked_select(mask > 0))
        # int32 copies for the kernels; non-persistent so the state_dict equals the reference's
        self.register_buffer("_ccols", self.identity_features.to(torch.int32), persistent=False)
        self.register_buffer("_tcols", self.transform_features.to(torch.int32), persistent=False)
        assert self.num_identity_features + self.num_transform_features == self.features
        self.transform_net = transform_net_create_fn(
            self.num_identity_features, self.num_transform_features * self._transform_dim_multiplier())
        # coupling.py:59-64: an optional bijection on the identity features (e.g. an unconditional spline CDF)
        self.unconditional_transform = (None if unconditional_transform is None
                                        else unconditional_transform(features=self.num_identity_features))

    @property
    def num_identity_features(self):
        return len(self.identity_features)

    @property
    def num_transform_features(self):
        return len(self.transform_features)

    def _check(self, inputs):
        if inputs.dim() == 4:
            raise NotImplementedError("4-D (image) inputs are outside the B200 hot path")
        if inputs.dim() != 2:
            raise ValueError("Inputs must be a 2D or a 4D tensor.")
        if inputs.shape[1] != self.features:
            raise ValueError("Expected features = {}, got {}.".format(self.features, inputs.shape[1]))

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)
        self._ccols = self.identity_features.to(torch.int32)
        self._tcols = self.transform_features.to(torch.int32)

    def forward(self, inputs, context=None):
        self._check(inputs)
        return self._run_layer(inputs, context, inverse=False)

    def inverse(self, inputs, context=None):
        self._check(inputs)
        return self._run_layer(inputs, context, inverse=True)

    def _run_layer(self, inputs, context, inverse):
        ut = self.unconditional_transform
        if ut is None:
            return self._run_conditional(inputs, context, inverse)
        # coupling.py:90-94 / :116-120: the conditioner always sees the identity features on the DATA side, so the
        # unconditional transform runs after the layer in the forward direction and before it in the inverse
        if not inverse:
            outputs, logabsdet = self._run_conditional(inputs, context, False)
            outputs, lad_id = self._on_identity(ut, outputs, context, False)
            return outputs, logabsdet + lad_id
        inputs, lad_id = self._on_identity(ut, inputs, context, True)
        outputs, logabsdet = self._run_conditional(inputs, context, True)
        return outputs, lad_id + logabsdet

    def _on_identity(self, ut, full, context, inverse):
        """Apply `ut` to the identity columns of a full-width tensor; returns (full-width result, logabsdet)."""
        if hasattr(ut, "apply_on_columns"):  # our CDF layers: one kernel on the full-width tensor, no gather
            return ut.apply_on_columns(full, self._ccols, self._tcols, inverse)
        part, lad = (ut.inverse if inverse else ut)(full[:, self.identity_features], context)
        return full.index_copy(1, self.identity_features, part), lad

    def _run_conditional(self, inputs, context, inverse):
        if tensorcore.usable(self.transform_net, inputs, context):
            # inference: conditioner on the tensor cores; its first layer reads the full-width inputs through a
            # column-scattered weight, so the identity-column gather (coupling.py:82-86) disappears as well
            return self._tensorcore_layer(inputs, inverse, context)
        params = self.transform_net(inputs[:, self.identity_features], context)
        return self._coupling_layer(inputs, params, inverse)

    def _tensorcore_layer(self, inputs, inverse, context=None):
        params = tensorcore.params(self.transform_net, inputs, col_map=self._ccols, k_in=self.features, context=context)
        return self._coupling_layer(inputs, params, inverse)

    def _transform_dim_multiplier(self):
        raise NotImplementedError()

    def _coupling_layer(self, inputs, transform_params, inverse):
        """(full-width inputs, conditioner output) -> (full-width outputs, logabsdet[B]), one kernel."""
        raise NotImplementedError()


class AffineCouplingTransform(CouplingTransform):
    """Scale-and-shift coupling (Real NVP).  `scale_activation` must be one of the two predefined activations
    of the reference (coupling.py:224-225); they are selected by identity and evaluated inside the kernel."""

    DEFAULT_SCALE_ACTIVATION = "sigmoid(x + 2) + 1e-3"
    GENERAL_SCALE_ACTIVATION = "clamp(softplus(x) + 1e-3, 0, 3)"

    def __init__(self, mask, transform_net_create_fn, unconditional_transform=None,
                 scale_activation=DEFAULT_SCALE_ACTIVATION):
        if scale_activation == self.DEFAULT_SCALE_ACTIVATION:
            self._activation_code = _cabi.SCALE_SIGMOID2
        elif scale_activation == self.GENERAL_SCALE_ACTIVATION:
            self._activation_code = _cabi.SCALE_SOFTPLUS_CLAMP3
        else:
            raise NotImplementedError("scale_activation must be AffineCouplingTransform.DEFAULT_SCALE_ACTIVATION "
                                      "or GENERAL_SCALE_ACTIVATION (arbitrary callables cannot run in the kernel)")
        self.scale_activation = scale_activation
        super().__init__(mask, transform_net_create_fn, unconditional_transform)

    def _transform_dim_multiplier(self):
        return 2

    def _coupling_layer(self, inputs, transform_params, inverse):
        return ops.affine_layer(inputs, transform_params, self._tcols, self._ccols, _cabi.AFFINE_BLOCKED,
                                self._activation_code, bool(inverse))

    def _tensorcore_layer(self, inputs, inverse, context=None):
        net = self.transform_net
        if self._transform_dim_multiplier() != 2 or (context is not None and not tensorcore.affine_fusable(
                net, tensorcore.context_k_in(net, self.features, context), self.num_transform_features)):
            return super()._tensorcore_layer(inputs, inverse, context)
        # final layer + scale-and-shift in one kernel
        return tensorcore.affine_layer(net, inputs, inputs, self._tcols, self._ccols, _cabi.AFFINE_BLOCKED,
                                       self._activation_code, inverse, col_map=self._ccols, k_in=self.features,
                                       context=context)


class AdditiveCouplingTransform(AffineCouplingTransform):
    """Shift-only coupling (NICE, coupling.py:255-269): zero log-det, no kernel needed beyond an indexed add."""

    def _transform_dim_multiplier(self):
        return 1

    def _coupling_layer(self, inputs, transform_params, inverse):
        outputs = inputs.clone()
        cols = self.transform_features
        outputs[:, cols] = inputs[:, cols] - transform_params if inverse else inputs[:, cols] + transform_params
        return outputs, inputs.new_zeros(inputs.shape[0])


class PiecewiseRationalQuadraticCouplingTransform(CouplingTransform):
    def __init__(self, mask, transform_net_create_fn, num_bins=10, tails=None, tail_bound=1.0,
                 apply_unconditional_transform=False, img_shape=None,
                 min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH, min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT,
                 min_derivative=splines.DEFAULT_MIN_DERIVATIVE):
        if apply_unconditional_transform and img_shape:
            raise NotImplementedError("image-shaped inputs are outside the B200 hot path")
        self.num_bins = num_bins
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.min_derivative = min_derivative
        self.tails = tails
        self.tail_bound = tail_bound
        self._spline = splines.RationalQuadraticSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height,
                                                         min_derivative, identity_init=False,
                                                         constrained_box=(0.0, 1.0))
        unconditional = None
        if apply_unconditional_transform:  # coupling.py:524-535
            unconditional = lambda features: PiecewiseRationalQuadraticCDF(  # noqa: E731
                shape=[features], num_bins=num_bins, tails=tails, tail_bound=tail_bound, min_bin_width=min_bin_width,
                min_bin_height=min_bin_height, min_derivative=min_derivative)
        super().__init__(mask, transform_net_create_fn, unconditional_transform=unconditional)

    def _transform_dim_multiplier(self):
        return self._spline.params_per_feature()

    def _scaling_width(self):
        # coupling.py:554-563: widths and heights are divided by sqrt(hidden) when the net exposes it
        for attr in ("hidden_features", "hidden_channels"):
            if hasattr(self.transform_net, attr):
                return getattr(self.transform_net, attr)
        warnings.warn("Inputs to the softmax are not scaled down: initialization might be bad.")
        return None

    def _coupling_layer(self, inputs, transform_params, inverse):
        return self._spline.apply(inputs, transform_params, self._tcols, self._ccols, inverse, self._scaling_width())

    def _tensorcore_layer(self, inputs, inverse, context=None):
        net = self.transform_net
        if not tensorcore.rqs_fusable(self._spline, net.final_layer.weight.shape[0], self.num_transform_features, net,
                                      self.features, context):
            return super()._tensorcore_layer(inputs, inverse, context)
        # final layer + spline in one kernel: the [B, D_t*P] parameter tensor never reaches HBM
        return tensorcore.rqs_layer(net, inputs, inputs, self._spline, self._tcols, self._ccols, inverse,
                                    self._scaling_width(), col_map=self._ccols, k_in=self.features, context=context)


class PiecewiseLinearCouplingTransform(CouplingTransform):
    """coupling.py:299-352 (Mueller et al. 2018): K raw bin probabilities per transformed feature, no 1/sqrt(H)
    scaling; tails=None -> the unit box, tails="linear" -> identity outside [-tail_bound, tail_bound]."""

    def __init__(self, mask, transform_net_create_fn, num_bins=10, tails=None, tail_bound=1.0,
                 apply_unconditional_transform=False, img_shape=None):
        if apply_unconditional_transform and img_shape:
            raise NotImplementedError("image-shaped inputs are outside the B200 hot path")
        self.num_bins = num_bins
        self.tails = tails
        self.tail_bound = tail_bound
        self._spline = splines.LinearSplineSettings(num_bins, tails, tail_bound)
        unconditional = None
        if apply_unconditional_transform:  # coupling.py:319-327
            unconditional = lambda features: PiecewiseLinearCDF(  # noqa: E731
                shape=[features], num_bins=num_bins, tails=tails, tail_bound=tail_bound)
        super().__init__(mask, transform_net_create_fn, unconditional_transform=unconditional)

    def _transform_dim_multiplier(self):
        return self.num_bins

    def _coupling_layer(self, inputs, transform_params, inverse):
        return self._spline.apply(inputs, transform_params, self._tcols, self._ccols, inverse)


class PiecewiseQuadraticCouplingTransform(CouplingTransform):
    """coupling.py:355-427 (Mueller et al. 2018): per transformed feature K raw widths and K+1 raw knot heights (K-1 with
    linear tails), both divided by sqrt(hidden) when the conditioner exposes `hidden_features` (:409-411)."""

    def __init__(self, mask, transform_net_create_fn, num_bins=10, tails=None, tail_bound=1.0,
                 apply_unconditional_transform=False, img_shape=None, min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH,
                 min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT):
        if apply_unconditional_transform and img_shape:
            raise NotImplementedError("image-shaped inputs are outside the B200 hot path")
        self.num_bins = num_bins
        self.tails = tails
        self.tail_bound = tail_bound
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self._spline = splines.QuadraticSplineSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height)
        unconditional = None
        if apply_unconditional_transform:  # coupling.py:379-389
            unconditional = lambda features: PiecewiseQuadraticCDF(  # noqa: E731
                shape=[features], num_bins=num_bins, tails=tails, tail_bound=tail_bound, min_bin_width=min_bin_width,
                min_bin_height=min_bin_height)
        super().__init__(mask, transform_net_create_fn, unconditional_transform=unconditional)

    def _transform_dim_multiplier(self):
        return self._spline.params_per_feature()

    def _coupling_layer(self, inputs, transform_params, inverse):
        hidden = getattr(self.transform_net, "hidden_features", None)
        return self._spline.apply(inputs, transform_params, self._tcols, self._ccols, inverse, hidden)


class PiecewiseCubicCouplingTransform(CouplingTransform):
    """coupling.py:429-500: per transformed feature [K raw widths ; K raw heights ; raw left / right derivative]; widths
    and heights divided by sqrt(hidden) when the conditioner exposes `hidden_features` (:477-479)."""

    def __init__(self, mask, transform_net_create_fn, num_bins=10, tails=None, tail_bound=1.0,
                 apply_unconditional_transform=False, img_shape=None, min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH,
                 min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT):
        if apply_unconditional_transform and img_shape:
            raise NotImplementedError("image-shaped inputs are outside the B200 hot path")
        self.num_bins = num_bins
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.tails = tails
        self.tail_bound = tail_bound
        self._spline = splines.CubicSplineSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height)
        unconditional = None
        if apply_unconditional_transform:  # coupling.py:449-459
            unconditional = lambda features: PiecewiseCubicCDF(  # noqa: E731
                shape=[features], num_bins=num_bins, tails=tails, tail_bound=tail_bound, min_bin_width=min_bin_width,
                min_bin_height=min_bin_height)
        super().__init__(mask, transform_net_create_fn, unconditional_transform=unconditional)

    def _transform_dim_multiplier(self):
        return self.num_bins * 2 + 2

    def _coupling_layer(self, inputs, transform_params, inverse):
        hidden = getattr(self.transform_net, "hidden_features", None)
        return self._spline.apply(inputs, transform_params, self._tcols, self._ccols, inverse, hidden)
