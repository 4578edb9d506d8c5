"""fp64-capable restatement of the element-wise squashing layers (flowcon/transforms/nonlinearities.py: Sigmoid, Logit,
Tanh, LeakyReLU, Exp, CauchyCDF, CauchyCDFInverse, CompositeCDFTransform), written literally in the reference's
formulas.  Each function maps [B, ...] to (outputs [B, ...], logabsdet [B]) and raises InputOutsideDomain where the
reference does.  `tanh_stable_logdet` is the exact forward log-det the kernel evaluates, for comparisons where the
literal log(1 − tanh² x) has rounded to −inf.  Flow-level helpers hand every other layer kind to `tests.bn_oracle` (and
through it to `oracle.restated`)."""
import math

import numpy as np
import torch
import torch.nn.functional as F

from flowconductor_b200.transforms.base import InputOutsideDomain
from tests import bn_oracle


def sum_except_batch(x):
    return x.reshape(x.shape[0], -1).sum(1)


def sigmoid(inputs, temperature, eps=1e-6, inverse=False):
    T = temperature.to(inputs.dtype)
    if not inverse:
        inputs = T * inputs
        outputs = torch.sigmoid(inputs)
        return outputs, sum_except_batch(torch.log(T) - F.softplus(-inputs) - F.softplus(inputs))
    if torch.min(inputs) < 0 or torch.max(inputs) > 1:
        raise InputOutsideDomain()
    inputs = torch.clamp(inputs, eps, 1 - eps)
    outputs = (1 / T) * (torch.log(inputs) - torch.log1p(-inputs))
    lad = -sum_except_batch(torch.log(T) - F.softplus(-T * outputs) - F.softplus(T * outputs))
    return outputs, lad


def tanh(inputs, inverse=False):
    if not inverse:
        outputs = torch.tanh(inputs)
        return outputs, sum_except_batch(torch.log(1 - outputs ** 2))
    if torch.min(inputs) <= -1 or torch.max(inputs) >= 1:
        raise InputOutsideDomain()
    outputs = 0.5 * torch.log((1 + inputs) / (1 - inputs))
    return outputs, -sum_except_batch(torch.log(1 - inputs ** 2))


def tanh_stable_logdet(inputs):
    """log(1 − tanh² x) = 2 (log 2 − |x| − softplus(−2|x|)), summed per row."""
    a = inputs.abs()
    return sum_except_batch(2 * (math.log(2) - a - F.softplus(-2 * a)))


def leaky_relu(inputs, negative_slope=1e-2, inverse=False):
    log_slope = torch.log(torch.as_tensor(negative_slope)).to(inputs.dtype)
    mask = (inputs < 0).to(inputs.dtype)
    if not inverse:
        return F.leaky_relu(inputs, negative_slope=negative_slope), sum_except_batch(log_slope * mask)
    return F.leaky_relu(inputs, negative_slope=1 / negative_slope), sum_except_batch(-log_slope * mask)


def exp(inputs, inverse=False):
    if not inverse:
        return torch.exp(inputs), sum_except_batch(inputs)
    if torch.min(inputs) <= 0.0:
        raise InputOutsideDomain()
    outputs = torch.log(inputs)
    return outputs, -sum_except_batch(outputs)


def cauchy_cdf(inputs, inverse=False):
    if not inverse:
        outputs = (1 / np.pi) * torch.atan(inputs) + 0.5
        return outputs, sum_except_batch(-np.log(np.pi) - torch.log(1 + inputs ** 2))
    if torch.min(inputs) < 0 or torch.max(inputs) > 1:
        raise InputOutsideDomain()
    outputs = torch.tan(np.pi * (inputs - 0.5))
    return outputs, -sum_except_batch(-np.log(np.pi) - torch.log(1 + outputs ** 2))


def composite_cdf(state, prefix, inputs, num_bins, inverse=False, eps=1e-6):
    """CompositeCDFTransform(Sigmoid(T), PiecewiseRationalQuadraticCDF([D], num_bins)): [squash, cdf, unsquash]."""
    T = state[prefix + "_transforms.0.temperature"]
    steps = [lambda x, inv: sigmoid(x, T, eps, inv),
             lambda x, inv: bn_oracle.lu_oracle.restated.rq_cdf(state, prefix + "_transforms.1.", x, num_bins, None,
                                                                1.0, inv),
             lambda x, inv: sigmoid(x, T, eps, not inv)]
    total = inputs.new_zeros(inputs.shape[0])
    for step in (reversed(steps) if inverse else steps):
        inputs, lad = step(inputs, inverse)
        total = total + lad
    return inputs, total


def apply_layer(state, spec, inputs, context=None, inverse=False):
    kind, p = spec["kind"], spec["prefix"]
    if kind == "logit":  # InverseTransform(Sigmoid)
        return sigmoid(inputs, state[p + "_transform.temperature"], 1e-6, not inverse)
    if kind == "composite_cdf":
        return composite_cdf(state, p, inputs, spec["num_bins"], inverse)
    return bn_oracle.apply_layer(state, spec, inputs, context, inverse)


def composite(state, specs, inputs, context=None, inverse=False):
    total = inputs.new_zeros(inputs.shape[0])
    outputs = inputs
    for spec in (reversed(specs) if inverse else specs):
        outputs, lad = apply_layer(state, spec, outputs, context, inverse)
        total = total + lad
    return outputs, total


def flow_log_prob(state, specs, inputs, context=None):
    noise, lad = composite(state, specs, inputs, context)
    return bn_oracle.lu_oracle.restated.standard_normal_log_prob(noise) + lad


def flow_sample_and_log_prob(state, specs, noise, context=None):
    """Flow.sample_and_log_prob with the base draw given as `noise`: (samples, log q(samples))."""
    samples, lad = composite(state, specs, noise, context, inverse=True)
    return samples, bn_oracle.lu_oracle.restated.standard_normal_log_prob(noise) - lad
