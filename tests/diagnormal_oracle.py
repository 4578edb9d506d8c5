"""fp64-capable restatement of DiagonalNormal and ConditionalDiagonalNormal (flowcon/distributions/normal.py), written
literally from a state_dict: the log-density in the reference's order of operations, and sampling from given noise as
the reference composes it (repeat_rows of the means and standard deviations, then a multiply-add).  Flow-level helpers
hand every layer to `tests.bn_oracle` (and through it to `oracle.restated`)."""
import math

import torch
import torch.nn.functional as F

from tests import bn_oracle

PREFIX = "_distribution."


def log_z(D):
    return 0.5 * D * math.log(2 * math.pi)


def encode(state, context, prefix=PREFIX, dtype=None):
    """The context encoder of a workload base (nn.Linear), or the context itself when the state has none."""
    key = prefix + "_context_encoder.weight"
    dtype = dtype or context.dtype
    if key not in state:
        return context.to(dtype)
    return F.linear(context.to(dtype), state[key].to(dtype), state[prefix + "_context_encoder.bias"].to(dtype))


def params_from(params, D):
    """(means, log_stds) of an encoder output, as `_compute_params` splits it."""
    if params.shape[-1] % 2 != 0:
        raise RuntimeError("The context encoder must return a tensor whose last dimension is even.")
    split = params.shape[-1] // 2
    return params[..., :split].reshape(params.shape[0], D), params[..., split:].reshape(params.shape[0], D)


def normal_log_prob(inputs, means, log_stds):
    """The reference's `_log_prob`: means / log_stds [C, D] broadcast against inputs [B, D] (C = 1 or B)."""
    norm_inputs = (inputs - means) * torch.exp(-log_stds)
    log_prob = -0.5 * torch.sum(norm_inputs ** 2, dim=1)
    log_prob = log_prob - torch.sum(log_stds, dim=1)
    return log_prob - torch.tensor(log_z(inputs.shape[1]), dtype=torch.float64).to(inputs.dtype)


def sample_from_noise(means, log_stds, noise, num_samples):
    """The reference's `_sample` with its torch.randn draw given as `noise` [C n, D]: returns [C, n, D]."""
    stds = torch.exp(log_stds)
    means = torch.repeat_interleave(means, num_samples, dim=0)
    stds = torch.repeat_interleave(stds, num_samples, dim=0)
    samples = means + stds * noise
    return samples.reshape(-1, num_samples, noise.shape[1])


def base_params(state, base, D, context=None, dtype=torch.float64, prefix=PREFIX):
    """(means, log_stds) of a workload base: [1, D] for DiagonalNormal, [C, D] for ConditionalDiagonalNormal."""
    if base["kind"] == "diagonal_normal":
        return state[prefix + "mean_"].to(dtype), state[prefix + "log_std_"].to(dtype)
    return params_from(encode(state, context, prefix, dtype), D)


def base_log_prob(state, base, noise, context=None):
    if base is None:
        return bn_oracle.lu_oracle.restated.standard_normal_log_prob(noise)
    means, log_stds = base_params(state, base, noise.shape[1], context, noise.dtype)
    return normal_log_prob(noise, means, log_stds)


def flow_log_prob(state, specs, base, inputs, context=None):
    noise, lad = bn_oracle.composite(state, specs, inputs, context)
    return base_log_prob(state, base, noise, context) + lad


def flow_sample_from_noise(state, specs, noise, context=None):
    """Samples of the transform's inverse from base samples `noise` [R, D] (context repeated per row)."""
    return bn_oracle.composite(state, specs, noise, context, inverse=True)[0]
