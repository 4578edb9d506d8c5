"""fp64-capable restatement of LULinear (flowcon/transforms/lu.py on top of flowcon/transforms/linear.py, forward_no_cache /
inverse_no_cache), written literally: two F.linear forward, two triangular solves inverse, dtype-generic.  Flow-level
helpers hand every other layer kind to `oracle.restated.apply_layer`, so stacks that mix LU layers with the bijections the
oracle restates (the nsf_lu workloads) are evaluated the way `restated.flow_log_prob` evaluates the others."""
import torch
import torch.nn.functional as F

from oracle import restated


def lu_linear(state, prefix, inputs, inverse=False, eps=1e-3):
    """(outputs, logabsdet[B]) of an LULinear with the state_dict entries under `prefix`."""
    D = inputs.shape[1]
    lower = inputs.new_zeros(D, D)
    rows, cols = torch.tril_indices(D, D, -1)
    lower[rows, cols] = state[prefix + "lower_entries"].to(inputs.dtype)
    lower[range(D), range(D)] = 1.0
    upper = inputs.new_zeros(D, D)
    rows, cols = torch.triu_indices(D, D, 1)
    upper[rows, cols] = state[prefix + "upper_entries"].to(inputs.dtype)
    upper_diag = F.softplus(state[prefix + "unconstrained_upper_diag"].to(inputs.dtype)) + eps
    upper[range(D), range(D)] = upper_diag
    bias = state[prefix + "bias"].to(inputs.dtype)
    logabsdet = torch.sum(torch.log(upper_diag)) * inputs.new_ones(inputs.shape[0])
    if inverse:
        outputs = torch.linalg.solve_triangular(lower, (inputs - bias).t(), upper=False, unitriangular=True)
        outputs = torch.linalg.solve_triangular(upper, outputs, upper=True)
        return outputs.t(), -logabsdet
    return F.linear(F.linear(inputs, upper), lower, bias), logabsdet


def apply_layer(state, spec, inputs, context=None, inverse=False):
    if spec["kind"] == "lu_linear":
        return lu_linear(state, spec["prefix"], inputs, inverse, spec.get("eps", 1e-3))
    return restated.apply_layer(state, spec, inputs, context, inverse)


def composite(state, specs, inputs, context=None, inverse=False):
    total = inputs.new_zeros(inputs.shape[0])
    outputs = inputs
    for spec in (reversed(specs) if inverse else specs):
        outputs, lad = apply_layer(state, spec, outputs, context, inverse)
        total = total + lad
    return outputs, total


def flow_log_prob(state, specs, inputs, context=None):
    noise, lad = composite(state, specs, inputs, context)
    return restated.standard_normal_log_prob(noise) + lad


def flow_sample_from_noise(state, specs, noise, context=None):
    return composite(state, specs, noise, context, inverse=True)[0]
