"""Masked autoregressive layers on the hot path, API of
flowcon/transforms/autoregressive/autoregressive.py (AutoregressiveTransform :25-62,
MaskedAffineAutoregressiveTransform :65-129, MaskedSumOfSigmoidsTransform :266-318,
MaskedPiecewiseRationalQuadraticAutoregressiveTransform :529-621).  Sub-module name `autoregressive_net`
(a MADE) is kept so reference state_dicts load.
"""
import numpy as np
import torch
from torch.nn import functional as F

from .. import _cabi, made_inverse, ops
from ..nn import tensorcore
from . import made as made_module
from . import splines
from .base import Transform


class AutoregressiveTransform(Transform):
    """Forward: one conditioner pass + one element-wise kernel.  Inverse: where the layer supports it, ONE kernel that
    evaluates the MADE incrementally (`_incremental_inverse`, csrc/fc_made_inverse.cu); otherwise D passes, each re-running
    the conditioner on the partially inverted outputs (autoregressive.py:44-53) — D x the forward cost."""

    def __init__(self, autoregressive_net):
        super().__init__()
        self.autoregressive_net = autoregressive_net

    def forward(self, inputs, context=None):
        if tensorcore.usable(self.autoregressive_net, inputs, context):
            return self._tensorcore_layer(inputs, inputs, False, context)
        params = self.autoregressive_net(inputs, context)
        return self._elementwise_forward(inputs, params)

    def inverse(self, inputs, context=None):
        if made_inverse.usable(self.autoregressive_net, inputs, context):
            result = self._incremental_inverse(inputs, context)
            if result is not None:
                return result
        outputs = torch.zeros_like(inputs)
        logabsdet = None
        fast = tensorcore.usable(self.autoregressive_net, outputs, context, inputs)
        # the context terms do not depend on the partially inverted outputs: one launch for all D passes
        terms = tensorcore.context_terms(self.autoregressive_net, context) if fast and context is not None else None
        for _ in range(int(np.prod(inputs.shape[1:]))):
            if fast:
                outputs, logabsdet = self._tensorcore_layer(outputs, inputs, True, context, terms)
            else:
                params = self.autoregressive_net(outputs, context)
                outputs, logabsdet = self._elementwise_inverse(inputs, params)
        return outputs, logabsdet

    def _tensorcore_layer(self, conditioner_inputs, inputs, inverse, context=None, terms=None):
        """MADE on the tensor cores (inference); `conditioner_inputs` feeds the MADE, `inputs` the bijection; `terms`:
        the context terms of `context` when the caller has them already."""
        params = tensorcore.params(self.autoregressive_net, conditioner_inputs, context=context, terms=terms)
        if inverse:
            return self._elementwise_inverse(inputs, params)
        return self._elementwise_forward(inputs, params)

    def _incremental_inverse(self, inputs, context=None):
        """(outputs, logabsdet) from the incremental-MADE kernel, or None if this layer / network is not covered.
        `context`: the context of a conditional MADE (made_inverse.usable has checked it)."""
        return None

    def _output_dim_multiplier(self):
        raise NotImplementedError()

    def _elementwise_forward(self, inputs, autoregressive_params):
        raise NotImplementedError()

    def _elementwise_inverse(self, inputs, autoregressive_params):
        raise NotImplementedError()


def _made(layer, features, hidden_features, context_features, num_blocks, use_residual_blocks, random_mask,
          activation, dropout_probability, use_batch_norm):
    return made_module.MADE(features=features, hidden_features=hidden_features, context_features=context_features,
                            num_blocks=num_blocks, output_multiplier=layer._output_dim_multiplier(),
                            use_residual_blocks=use_residual_blocks, random_mask=random_mask, activation=activation,
                            dropout_probability=dropout_probability, use_batch_norm=use_batch_norm)


class MaskedAffineAutoregressiveTransform(AutoregressiveTransform):
    """MAF layer: params viewed [B, D, 2] = (raw scale, shift) pairs; scale = softplus(raw) + 1e-3."""

    def __init__(self, features, hidden_features, context_features=None, num_blocks=2, use_residual_blocks=True,
                 random_mask=False, activation=F.relu, dropout_probability=0.0, use_batch_norm=False):
        self.features = features
        self._epsilon = 1e-3
        super().__init__(_made(self, features, hidden_features, context_features, num_blocks, use_residual_blocks,
                               random_mask, activation, dropout_probability, use_batch_norm))

    def _output_dim_multiplier(self):
        return 2

    def _elementwise_forward(self, inputs, autoregressive_params):
        return ops.affine_layer(inputs, autoregressive_params, None, None, _cabi.AFFINE_INTERLEAVED,
                                _cabi.SCALE_SOFTPLUS_EPS, False)

    def _elementwise_inverse(self, inputs, autoregressive_params):
        return ops.affine_layer(inputs, autoregressive_params, None, None, _cabi.AFFINE_INTERLEAVED,
                                _cabi.SCALE_SOFTPLUS_EPS, True)

    def _incremental_inverse(self, inputs, context=None):
        prog = made_inverse.program_for(self.autoregressive_net, 2)
        if prog is None:
            return None
        return made_inverse.apply_affine(prog, inputs, _cabi.SCALE_SOFTPLUS_EPS, context)

    def _tensorcore_layer(self, conditioner_inputs, inputs, inverse, context=None, terms=None):
        net = self.autoregressive_net
        if context is not None and not tensorcore.affine_fusable(net, inputs.shape[1], inputs.shape[1]):
            return super()._tensorcore_layer(conditioner_inputs, inputs, inverse, context, terms)
        return tensorcore.affine_layer(net, conditioner_inputs, inputs, None, None, _cabi.AFFINE_INTERLEAVED,
                                       _cabi.SCALE_SOFTPLUS_EPS, inverse,
                                       allow_inplace=not inverse,  # the inverse re-reads `inputs` D times
                                       context=context, terms=terms)


class MaskedSumOfSigmoidsTransform(AutoregressiveTransform):
    """Autoregressive sum-of-sigmoids layer; forward output is shifted by -0.5 (autoregressive.py:309,313)."""

    def __init__(self, features, hidden_features, n_sigmoids=30, context_features=None, num_blocks=2,
                 use_residual_blocks=True, random_mask=False, activation=F.relu, dropout_probability=0.0,
                 use_batch_norm=False):
        self.features = features
        self.n_sigmoids = n_sigmoids
        super().__init__(_made(self, features, hidden_features, context_features, num_blocks, use_residual_blocks,
                               random_mask, activation, dropout_probability, use_batch_norm))

    def _output_dim_multiplier(self):
        return 3 * self.n_sigmoids + 1

    def _elementwise_forward(self, inputs, autoregressive_params):
        return ops.sos_layer(inputs, autoregressive_params, self.n_sigmoids, -0.5, False, 50, 120.0)

    def _elementwise_inverse(self, inputs, autoregressive_params):
        return ops.sos_layer(inputs, autoregressive_params, self.n_sigmoids, -0.5, True, 50, 120.0)

    def _incremental_inverse(self, inputs, context=None):
        prog = made_inverse.program_for(self.autoregressive_net, self._output_dim_multiplier())
        if prog is None:
            return None
        return made_inverse.apply_sos(prog, inputs, self.n_sigmoids, -0.5, 50, 120.0, context)

    def _tensorcore_layer(self, conditioner_inputs, inputs, inverse, context=None, terms=None):
        net = self.autoregressive_net
        if (not inverse and conditioner_inputs is inputs
                and tensorcore.sos_fusable(net, inputs.shape[1], self.n_sigmoids, inputs.shape[1])):
            return tensorcore.sos_layer(net, inputs, inputs, self.n_sigmoids, -0.5, context, terms)
        return super()._tensorcore_layer(conditioner_inputs, inputs, inverse, context, terms)


class MaskedPiecewiseRationalQuadraticAutoregressiveTransform(AutoregressiveTransform):
    """MAF-RQS layer.  Identity-init softplus (beta = ln2/(1-min_derivative)) is always on (autoregressive.py
    :611); tails=None means the box [-1.2, 1.2]^2 (:595); no 1/sqrt(H) pre-scale because MADE exposes no
    `hidden_features` (:589)."""

    def __init__(self, features, hidden_features, context_features=None, num_bins=10, tails=None, tail_bound=1.0,
                 num_blocks=2, use_residual_blocks=True, random_mask=False, activation=F.relu,
                 dropout_probability=0.0, use_batch_norm=False, min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH,
                 min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT, min_derivative=splines.DEFAULT_MIN_DERIVATIVE):
        self.num_bins = num_bins
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.min_derivative = min_derivative
        self.tails = tails
        self.tail_bound = tail_bound
        self._spline = splines.RationalQuadraticSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height,
                                                         min_derivative, identity_init=True,
                                                         constrained_box=(-1.2, 1.2))
        super().__init__(_made(self, features, hidden_features, context_features, num_blocks, use_residual_blocks,
                               random_mask, activation, dropout_probability, use_batch_norm))

    def _output_dim_multiplier(self):
        return self._spline.params_per_feature()

    def _elementwise(self, inputs, autoregressive_params, inverse=False):
        hidden = getattr(self.autoregressive_net, "hidden_features", None)
        return self._spline.apply(inputs, autoregressive_params, None, None, inverse, hidden)

    def _elementwise_forward(self, inputs, autoregressive_params):
        return self._elementwise(inputs, autoregressive_params)

    def _elementwise_inverse(self, inputs, autoregressive_params):
        return self._elementwise(inputs, autoregressive_params, inverse=True)

    def _incremental_inverse(self, inputs, context=None):
        prog = made_inverse.program_for(self.autoregressive_net, self._spline.params_per_feature())
        if prog is None:
            return None
        hidden = getattr(self.autoregressive_net, "hidden_features", None)
        cfg, tails = self._spline.config(True, hidden)
        status = torch.zeros((1,), dtype=torch.int32, device=inputs.device) if tails == _cabi.TAILS_NONE or splines.STRICT \
            else None
        outputs, logabsdet = made_inverse.apply_rqs(prog, inputs, cfg, status, context)
        if status is not None:
            splines.check_status(status, tails)
        return outputs, logabsdet

    def _tensorcore_layer(self, conditioner_inputs, inputs, inverse, context=None, terms=None):
        net = self.autoregressive_net
        if not tensorcore.rqs_fusable(self._spline, net.final_layer.weight.shape[0], inputs.shape[1], net, inputs.shape[1],
                                      context):
            return super()._tensorcore_layer(conditioner_inputs, inputs, inverse, context, terms)
        return tensorcore.rqs_layer(net, conditioner_inputs, inputs, self._spline, None, None, inverse,
                                    getattr(net, "hidden_features", None),
                                    allow_inplace=not inverse,  # the inverse re-reads `inputs` D times
                                    context=context, terms=terms)


def _status_for(inputs, tails):
    """Device status word when the reference would check the domain on the host (no tails / STRICT)."""
    if tails == _cabi.TAILS_NONE or splines.STRICT:
        return torch.zeros((1,), dtype=torch.int32, device=inputs.device)
    return None


class MaskedPiecewiseLinearAutoregressiveTransform(AutoregressiveTransform):
    """autoregressive.py:321-372: always the constrained unit box (`linear_spline` without tails).  Note the
    reference's argument order: `num_bins` comes first."""

    def __init__(self, num_bins, features, hidden_features, context_features=None, num_blocks=2,
                 use_residual_blocks=True, random_mask=False, activation=F.relu, dropout_probability=0.0,
                 use_batch_norm=False):
        self.num_bins = num_bins
        self.features = features
        self._spline = splines.LinearSplineSettings(num_bins, None, 1.0)
        super().__init__(_made(self, features, hidden_features, context_features, num_blocks, use_residual_blocks,
                               random_mask, activation, dropout_probability, use_batch_norm))

    def _output_dim_multiplier(self):
        return self.num_bins

    def _elementwise_forward(self, inputs, autoregressive_params):
        return self._spline.apply(inputs, autoregressive_params, None, None, False)

    def _elementwise_inverse(self, inputs, autoregressive_params):
        return self._spline.apply(inputs, autoregressive_params, None, None, True)

    def _incremental_inverse(self, inputs, context=None):
        prog = made_inverse.program_for(self.autoregressive_net, self._output_dim_multiplier())
        if prog is None:
            return None
        tails, lo, hi = self._spline.domain()
        status = _status_for(inputs, tails)
        out = made_inverse.apply_linspline(prog, inputs, self.num_bins, tails, lo, hi, status, context)
        if status is not None:
            splines.check_status(status, tails)
        return out


class MaskedPiecewiseQuadraticAutoregressiveTransform(AutoregressiveTransform):
    """autoregressive.py:375-457.  `transforms.made.MADE` has no `hidden_features`, so no pre-scale is applied (:426);
    the min_derivative argument is accepted and unused, as in the reference."""

    def __init__(self, features, hidden_features, context_features=None, num_bins=10, num_blocks=2, tails=None,
                 tail_bound=1.0, use_residual_blocks=True, random_mask=False, activation=F.relu,
                 dropout_probability=0.0, use_batch_norm=False, min_bin_width=splines.DEFAULT_MIN_BIN_WIDTH,
                 min_bin_height=splines.DEFAULT_MIN_BIN_HEIGHT, min_derivative=splines.DEFAULT_MIN_DERIVATIVE):
        self.num_bins = num_bins
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.min_derivative = min_derivative
        self.tails = tails
        self.tail_bound = tail_bound
        self.features = features
        if tails not in (None, "linear"):
            raise ValueError(tails)
        self._spline = splines.QuadraticSplineSettings(num_bins, tails, tail_bound, min_bin_width, min_bin_height)
        super().__init__(_made(self, features, hidden_features, context_features, num_blocks, use_residual_blocks,
                               random_mask, activation, dropout_probability, use_batch_norm))

    def _output_dim_multiplier(self):
        return self.num_bins * 2 - 1 if self.tails == "linear" else self.num_bins * 2 + 1

    def _elementwise_forward(self, inputs, autoregressive_params):
        return self._spline.apply(inputs, autoregressive_params, None, None, False, None)

    def _elementwise_inverse(self, inputs, autoregressive_params):
        return self._spline.apply(inputs, autoregressive_params, None, None, True, None)

    def _incremental_inverse(self, inputs, context=None):
        prog = made_inverse.program_for(self.autoregressive_net, self._output_dim_multiplier())
        if prog is None:
            return None
        cfg, tails = self._spline.config(True, None)
        status = _status_for(inputs, tails)
        out = made_inverse.apply_quadspline(prog, inputs, cfg, status, context)
        if status is not None:
            splines.check_status(status, tails)
        return out


class MaskedPiecewiseCubicAutoregressiveTransform(AutoregressiveTransform):
    """autoregressive.py:460-523: the constrained unit box (`cubic_spline` without tails); `num_bins` comes first as in
    the reference; MADE exposes no `hidden_features`, so no pre-scale (:507-509)."""

    def __init__(self, num_bins, features, hidden_features, context_features=None, num_blocks=2,
                 use_residual_blocks=True, random_mask=False, activation=F.relu, dropout_probability=0.0,
                 use_batch_norm=False):
        self.num_bins = num_bins
        self.features = features
        self._spline = splines.CubicSplineSettings(num_bins, None, 1.0)
        super().__init__(_made(self, features, hidden_features, context_features, num_blocks, use_residual_blocks,
                               random_mask, activation, dropout_probability, use_batch_norm))

    def _output_dim_multiplier(self):
        return self.num_bins * 2 + 2

    def _elementwise_forward(self, inputs, autoregressive_params):
        return self._spline.apply(inputs, autoregressive_params, None, None, False, None)

    def _elementwise_inverse(self, inputs, autoregressive_params):
        return self._spline.apply(inputs, autoregressive_params, None, None, True, None)

    def _incremental_inverse(self, inputs, context=None):
        prog = made_inverse.program_for(self.autoregressive_net, self._output_dim_multiplier())
        if prog is None:
            return None
        cfg, tails = self._spline.config(True, None)
        status = _status_for(inputs, tails)
        out = made_inverse.apply_cubicspline(prog, inputs, cfg, status, context)
        if status is not None:
            splines.check_status(status, tails)
        return out
