"""`BatchNorm` and `ActNorm` with the API and state_dict of flowcon/transforms/normalization.py (2-D inputs).

`BatchNorm` normalises every feature with the statistics of the batch in training mode (mean and UNBIASED variance, also
folded into the running buffers with `momentum`) and with the running buffers in eval mode, then applies a learnable
positive scale and a shift; its inverse exists in eval mode only.  Statistics, forward / inverse and gradients run in
csrc/fc_batchnorm.cu.

`ActNorm` is a per-feature affine map whose scale and shift are learnable and, in training mode, initialised from the
first batch so that the outputs have zero mean and unit variance.  Forward / inverse / gradients run in csrc/fc_actnorm.cu
(SURVEY.md 8(f) n4)."""
import numpy as np
import torch
from torch import nn
from torch.nn import functional as F

from .. import ops
from ..utils import typechecks as check
from .base import InverseNotAvailable, Transform


class BatchNorm(Transform):
    """`affine` is accepted and unused, as in the reference."""

    def __init__(self, features, eps=1e-5, momentum=0.1, affine=True):
        if not check.is_positive_int(features):
            raise TypeError("Number of features must be a positive integer.")
        super().__init__()
        self.momentum = momentum
        self.eps = eps
        constant = np.log(np.exp(1 - eps) - 1)
        self.unconstrained_weight = nn.Parameter(constant * torch.ones(features))
        self.bias = nn.Parameter(torch.zeros(features))
        self.register_buffer("running_mean", torch.zeros(features))
        self.register_buffer("running_var", torch.zeros(features))

    @property
    def weight(self):
        return F.softplus(self.unconstrained_weight) + self.eps

    @staticmethod
    def _check(inputs):
        if inputs.dim() != 2:
            raise ValueError("Expected 2-dim inputs, got inputs of shape: {}".format(inputs.shape))

    def forward(self, inputs, context=None):
        self._check(inputs)
        if not self.training:
            return ops.batchnorm_eval(inputs, self.running_mean, self.running_var, self.unconstrained_weight, self.bias,
                                      self.eps, False)
        outputs, logabsdet, mean, var = ops.batchnorm_train(inputs, self.unconstrained_weight, self.bias, self.eps)
        # the reference's own in-place update, so the running buffers round exactly as there (six launches on [D])
        with torch.no_grad():
            self.running_mean.mul_(1 - self.momentum).add_(mean * self.momentum)
            self.running_var.mul_(1 - self.momentum).add_(var * self.momentum)
        return outputs, logabsdet

    def inverse(self, inputs, context=None):
        if self.training:
            raise InverseNotAvailable("Batch norm inverse is only available in eval mode, not in training mode.")
        self._check(inputs)
        return ops.batchnorm_eval(inputs, self.running_mean, self.running_var, self.unconstrained_weight, self.bias,
                                  self.eps, True)


class ActNorm(Transform):
    def __init__(self, features):
        if not check.is_positive_int(features):
            raise TypeError("Number of features must be a positive integer.")
        super().__init__()
        self.register_buffer("initialized", torch.tensor(False, dtype=torch.bool))
        self.log_scale = nn.Parameter(torch.zeros(features))
        self.shift = nn.Parameter(torch.zeros(features))

    @property
    def scale(self):
        return torch.exp(self.log_scale)

    @staticmethod
    def _check(inputs):
        if inputs.dim() not in [2, 4]:
            raise ValueError("Expecting inputs to be a 2D or a 4D tensor.")
        if inputs.dim() == 4:
            raise NotImplementedError("image-shaped (4-D) inputs are outside the B200 hot path")

    def forward(self, inputs, context=None):
        self._check(inputs)
        if self.training and not self.initialized:
            self._initialize(inputs)
        return ops.actnorm_layer(inputs, self.log_scale, self.shift, False)

    def inverse(self, inputs, context=None):
        self._check(inputs)
        return ops.actnorm_layer(inputs, self.log_scale, self.shift, True)

    def _initialize(self, inputs):
        """Data-dependent initialisation (normalization.py:204-218): one-off statistics of the first training batch."""
        with torch.no_grad():
            std = inputs.std(dim=0)
            mu = (inputs / std).mean(dim=0)
            self.log_scale.data = -torch.log(std)
            self.shift.data = -mu
            self.initialized.data = torch.tensor(True, dtype=torch.bool)
