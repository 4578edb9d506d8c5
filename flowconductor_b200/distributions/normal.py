"""Gaussian base densities (flowcon/distributions/normal.py).  StandardNormal's `_log_prob` is one kernel:
-0.5 * sum z^2 - 0.5 D log(2 pi), optionally fused with the flow's `+ logabsdet` (flows/base.py:48).  DiagonalNormal and
ConditionalDiagonalNormal run their log-density, sampling and gradients on csrc/fc_diagnormal.cu."""
import numpy as np
import torch
from torch import nn

from .. import ops
from ..utils import torchutils
from .base import Distribution


class StandardNormal(Distribution):
    def __init__(self, shape):
        super().__init__()
        self._shape = torch.Size(shape)
        self.register_buffer("_log_z", torch.tensor(0.5 * np.prod(shape) * np.log(2 * np.pi), dtype=torch.float64),
                             persistent=False)

    def _check(self, inputs):
        if inputs.shape[1:] != self._shape:
            raise ValueError("Expected input of shape {}, got {}".format(self._shape, inputs.shape[1:]))

    def _log_prob(self, inputs, context):
        self._check(inputs)
        return ops.stdnormal_log_prob(inputs.reshape(inputs.shape[0], -1), None)

    def log_prob_plus(self, inputs, logabsdet):
        """log N(inputs) + logabsdet in one pass (the tail of Flow._log_prob)."""
        self._check(inputs)
        return ops.stdnormal_log_prob(inputs.reshape(inputs.shape[0], -1), logabsdet)

    def _sample(self, num_samples, context):
        if context is None:
            return torch.randn(num_samples, *self._shape, device=self._log_z.device)
        samples = torch.randn(context.shape[0] * num_samples, *self._shape, device=context.device)
        return torchutils.split_leading_dim(samples, [context.shape[0], num_samples])

    def _mean(self, context):
        if context is None:
            return self._log_z.new_zeros(self._shape)
        return context.new_zeros(context.shape[0], *self._shape)


class ConditionalDiagonalNormal(Distribution):
    """A diagonal Gaussian whose means and log standard deviations are functions of a context
    (flowcon/distributions/normal.py).  `context_encoder(context)` returns [C, 2D]: the means, then the log standard
    deviations; without an encoder the context itself is used.  The log-density and sampling read that tensor in place
    (`ops.diagnormal_log_prob`, `ops.diagnormal_sample`), and its gradient flows back as one [C, 2D] tensor."""

    def __init__(self, shape, context_encoder=None):
        super().__init__()
        self._shape = torch.Size(shape)
        if context_encoder is None:
            self._context_encoder = lambda x: x
        else:
            self._context_encoder = context_encoder
        self.register_buffer("_log_z", torch.tensor(0.5 * np.prod(shape) * np.log(2 * np.pi), dtype=torch.float64),
                             persistent=False)

    def _params(self, context):
        """The encoder output as [C, 2D], after the reference's checks."""
        if context is None:
            raise ValueError("Context can't be None.")
        params = self._context_encoder(context)
        if params.shape[-1] % 2 != 0:
            raise RuntimeError("The context encoder must return a tensor whose last dimension is even.")
        if params.shape[0] != context.shape[0]:
            raise RuntimeError("The batch dimension of the parameters is inconsistent with the input.")
        D = self._shape.numel()
        if params[0].numel() != 2 * D:
            raise RuntimeError("The context encoder returns {} parameters per row, expected {}.".format(
                params[0].numel(), 2 * D))
        return params.reshape(params.shape[0], 2 * D)

    def _compute_params(self, context):
        """Compute the means and log stds from the context (views of one tensor)."""
        params = self._params(context)
        D = self._shape.numel()
        means = params[..., :D].reshape(params.shape[0], *self._shape)
        log_stds = params[..., D:].reshape(params.shape[0], *self._shape)
        return means, log_stds

    def _check(self, inputs):
        if inputs.shape[1:] != self._shape:
            raise ValueError("Expected input of shape {}, got {}".format(self._shape, inputs.shape[1:]))

    def _log_prob(self, inputs, context):
        self._check(inputs)
        params = self._params(context)
        return ops.diagnormal_log_prob(inputs.reshape(inputs.shape[0], self._shape.numel()), params, 1, None)

    def log_prob_plus(self, inputs, logabsdet, context):
        """log N(inputs | context) + logabsdet in one pass (the tail of Flow._log_prob)."""
        if context is not None and inputs.shape[0] != context.shape[0]:
            raise ValueError("Number of input items must be equal to number of context items.")
        self._check(inputs)
        params = self._params(context)
        return ops.diagnormal_log_prob(inputs.reshape(inputs.shape[0], self._shape.numel()), params, 1, logabsdet)

    def _sample(self, num_samples, context):
        params = self._params(context)
        context_size = context.shape[0]
        noise = torch.randn(context_size * num_samples, *self._shape, device=params.device)
        samples = ops.diagnormal_sample(noise.reshape(noise.shape[0], self._shape.numel()), params, num_samples)
        return samples.reshape(context_size, num_samples, *self._shape)

    def _mean(self, context):
        means, _ = self._compute_params(context)
        return means


class DiagonalNormal(Distribution):
    """A diagonal Gaussian with learnable means and log standard deviations (flowcon/distributions/normal.py):
    parameters `mean_` and `log_std_`, both [1, D].  Unlike the reference, which raises NotImplementedError, it can be
    sampled from, with the kernel of ConditionalDiagonalNormal, so a flow trained with a learnable base can draw from it:
    `sample(n)` gives [n, *shape], `sample(n, context)` gives [C, n, *shape] (the context is ignored otherwise)."""

    def __init__(self, shape):
        super().__init__()
        self._shape = torch.Size(shape)
        self.mean_ = nn.Parameter(torch.zeros(shape).reshape(1, -1))
        self.log_std_ = nn.Parameter(torch.zeros(shape).reshape(1, -1))
        self.register_buffer("_log_z", torch.tensor(0.5 * np.prod(shape) * np.log(2 * np.pi), dtype=torch.float64),
                             persistent=False)

    def _params(self):
        return torch.cat([self.mean_, self.log_std_], 1)

    def _check(self, inputs):
        if inputs.shape[1:] != self._shape:
            raise ValueError("Expected input of shape {}, got {}".format(self._shape, inputs.shape[1:]))

    def _log_prob(self, inputs, context):
        self._check(inputs)
        rows = inputs.shape[0]
        return ops.diagnormal_log_prob(inputs.reshape(rows, self._shape.numel()), self._params(), max(rows, 1),
                                       None)

    def log_prob_plus(self, inputs, logabsdet, context=None):
        """log N(inputs) + logabsdet in one pass (the tail of Flow._log_prob); the context is not used."""
        self._check(inputs)
        rows = inputs.shape[0]
        return ops.diagnormal_log_prob(inputs.reshape(rows, self._shape.numel()), self._params(), max(rows, 1),
                                       logabsdet)

    def _sample(self, num_samples, context):
        rows = num_samples if context is None else context.shape[0] * num_samples
        noise = torch.randn(rows, *self._shape, device=self.mean_.device)
        samples = ops.diagnormal_sample(noise.reshape(rows, self._shape.numel()), self._params(), rows)
        if context is None:
            return samples.reshape(num_samples, *self._shape)
        return samples.reshape(context.shape[0], num_samples, *self._shape)
