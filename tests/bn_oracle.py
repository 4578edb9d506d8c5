"""fp64-capable restatement of BatchNorm (flowcon/transforms/normalization.py, 2-D inputs), written literally in both
modes: training mode normalises with the batch mean and unbiased variance, eval mode with the running buffers.  Flow-level
helpers hand every other layer kind to `tests.lu_oracle` (and through it to `oracle.restated`), so the maf_bn /
realnvp_bn workloads are evaluated the way `restated.flow_log_prob` evaluates the others."""
import torch
import torch.nn.functional as F

from tests import lu_oracle


def weight(state, prefix, dtype, eps=1e-5):
    return F.softplus(state[prefix + "unconstrained_weight"].to(dtype)) + eps


def batch_stats(inputs):
    """(mean, unbiased variance) over the batch, as the reference's forward computes them."""
    return inputs.mean(0), inputs.var(0)


def batch_norm(state, prefix, inputs, inverse=False, training=False, eps=1e-5):
    """(outputs, logabsdet[B]) of a BatchNorm with the state_dict entries under `prefix`."""
    w = weight(state, prefix, inputs.dtype, eps)
    bias = state[prefix + "bias"].to(inputs.dtype)
    if training:
        if inverse:
            raise ValueError("Batch norm inverse is only available in eval mode")
        mean, var = batch_stats(inputs)
    else:
        mean, var = state[prefix + "running_mean"].to(inputs.dtype), state[prefix + "running_var"].to(inputs.dtype)
    ones = inputs.new_ones(inputs.shape[0])
    if inverse:
        outputs = torch.sqrt(var + eps) * ((inputs - bias) / w) + mean
        return outputs, torch.sum(-torch.log(w) + 0.5 * torch.log(var + eps)) * ones
    outputs = w * ((inputs - mean) / torch.sqrt(var + eps)) + bias
    return outputs, torch.sum(torch.log(w) - 0.5 * torch.log(var + eps)) * ones


def update_running(state, prefix, inputs, momentum=0.1):
    """The training-mode update of the running buffers, in place on `state`, in the reference's arithmetic."""
    mean, var = batch_stats(inputs)
    for name, value in (("running_mean", mean), ("running_var", var)):
        state[prefix + name] = state[prefix + name].mul(1 - momentum).add(value.detach().to(state[prefix + name].dtype)
                                                                        * momentum)


def apply_layer(state, spec, inputs, context=None, inverse=False, training=False):
    if spec["kind"] == "batchnorm":
        return batch_norm(state, spec["prefix"], inputs, inverse, training, spec.get("eps", 1e-5))
    return lu_oracle.apply_layer(state, spec, inputs, context, inverse)


def composite(state, specs, inputs, context=None, inverse=False, training=False, update=False):
    """The layer cascade; `update` (training mode) also advances the BatchNorm running buffers in `state`."""
    total = inputs.new_zeros(inputs.shape[0])
    outputs = inputs
    for spec in (reversed(specs) if inverse else specs):
        if update and spec["kind"] == "batchnorm":
            update_running(state, spec["prefix"], outputs)
        outputs, lad = apply_layer(state, spec, outputs, context, inverse, training)
        total = total + lad
    return outputs, total


def flow_log_prob(state, specs, inputs, context=None, training=False, update=False):
    noise, lad = composite(state, specs, inputs, context, training=training, update=update)
    return lu_oracle.restated.standard_normal_log_prob(noise) + lad


def flow_sample_from_noise(state, specs, noise, context=None):
    return composite(state, specs, noise, context, inverse=True)[0]
