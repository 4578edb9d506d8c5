"""`LULinear` with the API and state_dict of flowcon/transforms/lu.py (on top of flowcon/transforms/linear.py): an
invertible linear map y = W x + bias with W = L U, L unit lower triangular, U upper triangular with a positive diagonal
softplus(unconstrained_upper_diag) + eps, so log|det W| = Σ log(upper_diag).  Neural spline flows put one after every
coupling layer.

The factors are composed on the [D, D] matrices in fp64 and rounded once to fp32 — forward M = L U, c = bias; inverse
M = U⁻¹ L⁻¹ (two triangular solves on the identity), c = -M bias — and the rows run through one kernel y = x Mᵀ + c that
also writes the log-determinant on every row (csrc/fc_lulinear.cu, D < 64).  Wider maps are tensor-core GEMMs
(`nn.tc_autograd.linear`, the same MIN_K boundary the conditioners use).  The composition is differentiable, so autograd
takes the entries' gradients from the kernel's grad_M / grad_c / grad_logdet, in both directions.  Without autograd the
composed (M, c, logdet) are cached per direction and reused until a parameter changes (pointer + version counter, the rule
of `nn.tensorcore`)."""
import numpy as np
import torch
from torch import nn
from torch.nn import functional as F
from torch.nn import init

from .. import _cabi, ops
from ..nn import tc_autograd, tensorcore
from ..utils import typechecks as check
from .base import Transform


class LULinear(Transform):
    def __init__(self, features, using_cache=False, identity_init=True, eps=1e-3):
        if not check.is_positive_int(features):
            raise TypeError("Number of features must be a positive integer.")
        super().__init__()
        self.features = features
        self.bias = nn.Parameter(torch.zeros(features))
        self.using_cache = using_cache
        self.eps = eps
        self.lower_indices = np.tril_indices(features, k=-1)
        self.upper_indices = np.triu_indices(features, k=1)
        self.diag_indices = np.diag_indices(features)
        n_triangular_entries = ((features - 1) * features) // 2
        self.lower_entries = nn.Parameter(torch.zeros(n_triangular_entries))
        self.upper_entries = nn.Parameter(torch.zeros(n_triangular_entries))
        self.unconstrained_upper_diag = nn.Parameter(torch.zeros(features))
        self._fc_lu_cache = {}
        self._fc_lu_index = {}
        self._initialize(identity_init)

    def _initialize(self, identity_init):
        init.zeros_(self.bias)
        if identity_init:
            init.zeros_(self.lower_entries)
            init.zeros_(self.upper_entries)
            constant = np.log(np.exp(1 - self.eps) - 1)
            init.constant_(self.unconstrained_upper_diag, constant)
        else:
            stdv = 1.0 / np.sqrt(self.features)
            init.uniform_(self.lower_entries, -stdv, stdv)
            init.uniform_(self.upper_entries, -stdv, stdv)
            init.uniform_(self.unconstrained_upper_diag, -stdv, stdv)

    # ---- the reference's public helpers (parameter dtype) ----
    def _create_lower_upper(self):
        lower = self.lower_entries.new_zeros(self.features, self.features)
        lower[self.lower_indices[0], self.lower_indices[1]] = self.lower_entries
        lower[self.diag_indices[0], self.diag_indices[1]] = 1.0
        upper = self.upper_entries.new_zeros(self.features, self.features)
        upper[self.upper_indices[0], self.upper_indices[1]] = self.upper_entries
        upper[self.diag_indices[0], self.diag_indices[1]] = self.upper_diag
        return lower, upper

    @property
    def upper_diag(self):
        return F.softplus(self.unconstrained_upper_diag) + self.eps

    def weight(self):
        lower, upper = self._create_lower_upper()
        return lower @ upper

    def weight_inverse(self):
        lower, upper = self._create_lower_upper()
        return self._inverse_of(lower, upper)

    @staticmethod
    def _inverse_of(lower, upper):
        identity = torch.eye(lower.shape[0], dtype=lower.dtype, device=lower.device)
        lower_inverse = torch.linalg.solve_triangular(lower, identity, upper=False, unitriangular=True)
        return torch.linalg.solve_triangular(upper, lower_inverse, upper=True)

    def logabsdet(self):
        return torch.sum(torch.log(self.upper_diag))

    def use_cache(self, mode=True):
        if not check.is_bool(mode):
            raise TypeError("Mode must be boolean.")
        self.using_cache = mode

    def train(self, mode=True):
        if mode:
            self._fc_lu_cache.clear()
        return super().train(mode)

    # ---- the kernel operands ----
    def _factors64(self):
        """(L, U) in fp64, scattered with index tensors kept on the parameters' device: indexing with the numpy arrays
        copies them to the device on every call, which a CUDA graph capture (GraphedTrainStep) does not allow."""
        dev = self.bias.device
        idx = self._fc_lu_index.get(dev)
        if idx is None:
            idx = tuple(torch.as_tensor(np.asarray(a), dtype=torch.long).to(dev)
                        for a in (*self.lower_indices, *self.upper_indices, self.diag_indices[0]))
            self._fc_lu_index[dev] = idx
        lo_r, lo_c, up_r, up_c, dg = idx
        lower = torch.zeros(self.features, self.features, dtype=torch.float64, device=dev)
        lower = lower.index_put((lo_r, lo_c), self.lower_entries.to(torch.float64))
        lower = lower.index_put((dg, dg), lower.new_ones(self.features))
        upper = torch.zeros(self.features, self.features, dtype=torch.float64, device=dev)
        upper = upper.index_put((up_r, up_c), self.upper_entries.to(torch.float64))
        upper = upper.index_put((dg, dg), self.upper_diag.to(torch.float64))
        return lower, upper

    def _compose(self, inverse):
        """(M, c, logdet) in the parameters' dtype, composed in fp64: y = x Mᵀ + c, logabsdet = logdet."""
        dtype = self.bias.dtype
        lower, upper = self._factors64()
        bias = self.bias.to(torch.float64)
        logdet = torch.sum(torch.log(self.upper_diag.to(torch.float64)))
        if inverse:
            M = self._inverse_of(lower, upper)
            c = -(M @ bias)
            logdet = -logdet
        else:
            M, c = lower @ upper, bias
        return M.to(dtype), c.to(dtype), logdet.to(dtype)

    def _operands(self, inverse):
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return self._compose(inverse)
        key = tensorcore.module_param_key(self)
        hit = self._fc_lu_cache.get(inverse)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                hit = (key, self._compose(inverse))
            self._fc_lu_cache[inverse] = hit
            tensorcore._generation[0] += 1  # a recorded graph holding the old operands must record again
        return hit[1]

    def _run(self, inputs, inverse):
        if inputs.dim() != 2:
            raise NotImplementedError("LULinear on the B200 hot path takes [B, features] inputs")
        if inputs.shape[1] != self.features:
            raise ValueError("expected inputs with {} features, got {}".format(self.features, inputs.shape[1]))
        _cabi.require_cuda_f32(inputs, "inputs")
        M, c, logdet = self._operands(inverse)
        if self.features < tc_autograd.MIN_K:
            return ops.lulinear_layer(inputs, M, c, logdet)
        return tc_autograd.linear(inputs, M, c), logdet * inputs.new_ones(inputs.shape[0])

    def forward(self, inputs, context=None):
        return self._run(inputs, False)

    def inverse(self, inputs, context=None):
        return self._run(inputs, True)

    def forward_no_cache(self, inputs):
        return self._run(inputs, False)

    def inverse_no_cache(self, inputs):
        return self._run(inputs, True)
