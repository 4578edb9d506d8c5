"""The flows named by BASELINE.json `configs`, with the sizes fixed in SURVEY.md §8, as plain data.

A workload is a dict: {"name", "features", "context_features", "batch", "layers": [layer dicts]}.
Layer dicts use the reference's own constructor vocabulary (`num_bins`, `tails`, `tail_bound`,
`hidden_features`, `num_blocks`, `n_sigmoids`).  `build_flow` instantiates the workload with this
package's drop-in classes; the same dict drives the reference builder in `oracle/make_golden.py`
and the oracle's layer spec, so all three describe the same model.
"""
import copy

import torch


def _prq_coupling_stack(features, num_layers, num_bins, hidden, tail_bound=3.0):
    return [
        {"kind": "prq_coupling", "mask": "alternating_even" if i % 2 == 0 else "alternating_odd",
         "num_bins": num_bins, "tails": "linear", "tail_bound": tail_bound,
         "hidden_features": hidden, "num_blocks": 2}
        for i in range(num_layers)
    ]


def _maf_prq_stack(features, num_layers, num_bins, hidden, tail_bound=3.0):
    layers = []
    for _ in range(num_layers):
        layers.append({"kind": "permutation", "mode": "random"})
        layers.append({"kind": "maf_prq", "num_bins": num_bins, "tails": "linear", "tail_bound": tail_bound,
                       "hidden_features": hidden, "num_blocks": 2})
    return layers


def _nsf_lu_stack(features, num_layers, num_bins, hidden, tail_bound=3.0):
    """Neural spline flow (Durkan et al. 2019): every coupling layer followed by LULinear(features, identity_init=True)."""
    layers = []
    for layer in _prq_coupling_stack(features, num_layers, num_bins, hidden, tail_bound):
        layers.append(layer)
        layers.append({"kind": "lu_linear", "identity_init": True})
    return layers


def _maf_bn_stack(num_layers, hidden, num_blocks=2):
    """flows.MaskedAutoregressiveFlow(..., batch_norm_between_layers=True): reverse permutation, MAF-affine, BatchNorm."""
    layers = []
    for _ in range(num_layers):
        layers.append({"kind": "permutation", "mode": "reverse"})
        layers.append({"kind": "maf_affine", "hidden_features": hidden, "num_blocks": num_blocks})
        layers.append({"kind": "batchnorm"})
    return layers


def _realnvp_bn_stack(num_layers, hidden, num_blocks=2):
    """flows.SimpleRealNVP(..., batch_norm_between_layers=True): affine couplings on the odd, then the even features
    (the reference's mask[::2] = -1, negated after every layer), each followed by BatchNorm."""
    layers = []
    for i in range(num_layers):
        layers.append({"kind": "affine_coupling", "mask": "alternating_odd" if i % 2 == 0 else "alternating_even",
                       "hidden_features": hidden, "num_blocks": num_blocks, "scale_activation": "sigmoid2"})
        layers.append({"kind": "batchnorm"})
    return layers


def _bounded_maf_stack(features, num_layers, num_bins, hidden, cdf_after=None, learn_logit_temperature=False):
    """Data on the unit box: a Logit in front of cfg 3's MAF-RQS stack; cdf_after = i puts
    CompositeCDFTransform(Sigmoid(learn_temperature=True), PiecewiseRationalQuadraticCDF([D], num_bins)) after layer i of
    that stack (the neural-spline-flow way to run a tails=None spline on unbounded features)."""
    layers = [{"kind": "logit", "learn_temperature": learn_logit_temperature}]
    for i, layer in enumerate(_maf_prq_stack(features, num_layers, num_bins, hidden)):
        layers.append(layer)
        if i == cdf_after:
            layers.append({"kind": "composite_cdf", "num_bins": 8, "learn_temperature": True})
    return layers


WORKLOADS = {
    # cfg 1: README.md:86-98 model (MAF(2, 4) + RandomPermutation), evaluated on 2-D toy batches
    "cfg1": {"features": 2, "context_features": None, "batch": 10000,
             "layers": [{"kind": "maf_affine", "hidden_features": 4, "num_blocks": 2},
                        {"kind": "permutation", "mode": "random"}]},
    # cfg 2 (headline): PRQ coupling D=64, K=8, 8 layers, H=256, linear tails at 3.0, batch 1M
    "cfg2": {"features": 64, "context_features": None, "batch": 1 << 20,
             "layers": _prq_coupling_stack(64, 8, 8, 256)},
    # cfg 3: MAF-RQS D=16, K=16, 5 layers, H=256; training step
    "cfg3": {"features": 16, "context_features": None, "batch": 262144,
             "layers": _maf_prq_stack(16, 5, 16, 256)},
    # cfg 4: conditional sum-of-sigmoids D=32, context 8, n=10, H=64, 3 layers, batch 256K
    "cfg4": {"features": 32, "context_features": 8, "batch": 262144,
             "layers": [{"kind": "cond_sos", "n_sigmoids": 10, "hidden_features": 64, "num_blocks": 2}
                        for _ in range(3)]},
    # cfg 5: cfg 2 at D=256, 100M rows streamed in 1M-row chunks
    "cfg5": {"features": 256, "context_features": None, "batch": 1 << 20, "total_rows": 100_000_000,
             "layers": _prq_coupling_stack(256, 8, 8, 256)},
    # reduced-size twins (same classes / masks / tails) used for committed golden vectors
    "cfg2_small": {"features": 64, "context_features": None, "batch": 128,
                   "layers": _prq_coupling_stack(64, 2, 8, 32)},
    # wide enough (H >= 64) for the tensor-core conditioner path; used by smoke() and the host tests
    "cfg2_tc_small": {"features": 64, "context_features": None, "batch": 512,
                      "layers": _prq_coupling_stack(64, 3, 8, 64)},
    "cfg3_small": {"features": 16, "context_features": None, "batch": 128,
                   "layers": _maf_prq_stack(16, 2, 16, 32)},
    "cfg4_small": {"features": 8, "context_features": 8, "batch": 128,
                   "layers": [{"kind": "cond_sos", "n_sigmoids": 10, "hidden_features": 16, "num_blocks": 2}
                              for _ in range(2)]},
    "affine_coupling_small": {"features": 10, "context_features": None, "batch": 64,
                              "layers": [{"kind": "affine_coupling", "mask": "mid_split", "hidden_features": 16,
                                          "num_blocks": 2, "scale_activation": "sigmoid2"},
                                         {"kind": "permutation", "mode": "reverse"},
                                         {"kind": "affine_coupling", "mask": "mid_split", "hidden_features": 16,
                                          "num_blocks": 2, "scale_activation": "softplus_clamp3"}]},
    "cond_prq_small": {"features": 6, "context_features": 4, "batch": 64,
                       "layers": [{"kind": "cond_prq", "num_bins": 8, "tails": "linear", "tail_bound": 3.0,
                                   "hidden_features": 16, "num_blocks": 2}]},
    "maf_sos_small": {"features": 5, "context_features": None, "batch": 64,
                      "layers": [{"kind": "maf_sos", "n_sigmoids": 6, "hidden_features": 16, "num_blocks": 2}]},
    # coupling.py:524-535 + nonlinearities.py:406-487: an unconditional RQ CDF on the identity features of every layer
    "prq_coupling_uncond_small": {"features": 6, "context_features": None, "batch": 64,
                                  "layers": [{"kind": "prq_coupling", "mask": "alternating_even", "num_bins": 5,
                                              "tails": "linear", "tail_bound": 3.0, "hidden_features": 16,
                                              "num_blocks": 2, "unconditional": True},
                                             {"kind": "prq_coupling", "mask": "alternating_odd", "num_bins": 5,
                                              "tails": "linear", "tail_bound": 3.0, "hidden_features": 16,
                                              "num_blocks": 2, "unconditional": True}]},
    # SURVEY 8f n4: ActNorm (normalization.py:144-218) between masked autoregressive layers
    "actnorm_maf_small": {"features": 6, "context_features": None, "batch": 96,
                          "layers": [{"kind": "actnorm"},
                                     {"kind": "maf_affine", "hidden_features": 16, "num_blocks": 2},
                                     {"kind": "permutation", "mode": "reverse"},
                                     {"kind": "actnorm"},
                                     {"kind": "maf_affine", "hidden_features": 16, "num_blocks": 2}]},
    # SURVEY 8f n3: the piecewise-linear family (coupling.py:299-352, autoregressive.py:321-372, nonlinearities.py:250-283)
    "plin_coupling_small": {"features": 6, "context_features": None, "batch": 64,
                            "layers": [{"kind": "plin_coupling", "mask": "alternating_even", "num_bins": 8,
                                        "tails": "linear", "tail_bound": 3.0, "hidden_features": 16, "num_blocks": 2,
                                        "unconditional": True},
                                       {"kind": "plin_coupling", "mask": "alternating_odd", "num_bins": 8,
                                        "tails": "linear", "tail_bound": 3.0, "hidden_features": 16, "num_blocks": 2}]},
    "maf_plin_small": {"features": 5, "context_features": None, "batch": 64,
                       "layers": [{"kind": "maf_plin", "num_bins": 10, "hidden_features": 16, "num_blocks": 2}]},
    # SURVEY 8f n3: the piecewise-quadratic family (coupling.py:355-427, autoregressive.py:375-457, nonlinearities.py:286-340)
    "pquad_coupling_small": {"features": 6, "context_features": None, "batch": 64,
                             "layers": [{"kind": "pquad_coupling", "mask": "alternating_even", "num_bins": 8,
                                         "tails": "linear", "tail_bound": 3.0, "hidden_features": 16, "num_blocks": 2,
                                         "unconditional": True},
                                        {"kind": "pquad_coupling", "mask": "alternating_odd", "num_bins": 8,
                                         "tails": "linear", "tail_bound": 3.0, "hidden_features": 16, "num_blocks": 2}]},
    "maf_pquad_small": {"features": 5, "context_features": None, "batch": 64,
                        "layers": [{"kind": "maf_pquad", "num_bins": 10, "tails": "linear", "tail_bound": 3.0,
                                    "hidden_features": 16, "num_blocks": 2}]},
    # cubic family (coupling.py:429-500, nonlinearities.py:342-404)
    "pcubic_coupling_small": {"features": 6, "context_features": None, "batch": 64,
                              "layers": [{"kind": "pcubic_coupling", "mask": "alternating_even", "num_bins": 8,
                                          "tails": "linear", "tail_bound": 3.0, "hidden_features": 16, "num_blocks": 2,
                                          "unconditional": True},
                                         {"kind": "pcubic_coupling", "mask": "alternating_odd", "num_bins": 8,
                                          "tails": "linear", "tail_bound": 3.0, "hidden_features": 16,
                                          "num_blocks": 2}]},
    # autoregressive.py:460-523: the constrained unit box (cubic_spline without tails), no pre-scale (MADE has no
    # hidden_features)
    "maf_pcubic_small": {"features": 5, "context_features": None, "batch": 64,
                         "layers": [{"kind": "maf_pcubic", "num_bins": 8, "hidden_features": 16, "num_blocks": 2}]},
    "prq_coupling_notails_small": {"features": 6, "context_features": None, "batch": 64,
                                   "layers": [{"kind": "prq_coupling", "mask": "mid_split", "num_bins": 5,
                                               "tails": None, "tail_bound": 1.0, "hidden_features": 16,
                                               "num_blocks": 2}]},
    # LU-factorised linear layers between the couplings (flowcon/transforms/lu.py): cfg 2's stack at D = 32
    "nsf_lu": {"features": 32, "context_features": None, "batch": 1 << 20, "layers": _nsf_lu_stack(32, 8, 8, 256)},
    "nsf_lu_small": {"features": 6, "context_features": None, "batch": 64, "layers": _nsf_lu_stack(6, 2, 8, 16)},
    # BatchNorm between layers (flowcon/flows/autoregressive.py, flowcon/flows/realnvp.py): the packaged flows'
    # layering; maf_bn is a MAF-affine training workload at D = 43, so the BatchNorm kernels take their unaligned path
    "maf_bn_small": {"features": 6, "context_features": None, "batch": 128, "layers": _maf_bn_stack(2, 16)},
    "realnvp_bn_small": {"features": 6, "context_features": None, "batch": 128, "layers": _realnvp_bn_stack(2, 16)},
    "maf_bn": {"features": 43, "context_features": None, "batch": 262144, "layers": _maf_bn_stack(5, 256)},
    # Gaussian bases with learned parameters (flowcon/distributions/normal.py): `base` names the base density, the
    # default being StandardNormal.  A conditional one reads its means and log standard deviations from a linear
    # encoder of the context (nn.Linear(context_features, 2 D)).
    "cond_prq_diag_small": {"features": 6, "context_features": 4, "batch": 64,
                            "layers": [{"kind": "cond_prq", "num_bins": 8, "tails": "linear", "tail_bound": 3.0,
                                        "hidden_features": 16, "num_blocks": 2}],
                            "base": {"kind": "conditional_diagonal_normal", "encoder": "linear"}},
    "maf_diag_small": {"features": 6, "context_features": None, "batch": 128,
                       "layers": [{"kind": "permutation", "mode": "reverse"},
                                  {"kind": "maf_affine", "hidden_features": 16, "num_blocks": 2},
                                  {"kind": "permutation", "mode": "reverse"},
                                  {"kind": "maf_affine", "hidden_features": 16, "num_blocks": 2}],
                       "base": {"kind": "diagonal_normal"}},
    # cfg 4's shape (D = 32, context 8, 262 144 rows) with a context-dependent base
    "cond_sos_diag": {"features": 32, "context_features": 8, "batch": 262144,
                      "layers": [{"kind": "cond_sos", "n_sigmoids": 10, "hidden_features": 64, "num_blocks": 2}
                                 for _ in range(3)],
                      "base": {"kind": "conditional_diagonal_normal", "encoder": "linear"}},
    # bounded data (drawn in (0, 1)): Logit in front, a squashed spline CDF inside (nonlinearities.py).  The small twin
    # learns its logit's temperature and has no layer that checks its domain in the sampling direction, so its sampler
    # and a training-by-sampling step can be recorded into CUDA graphs.
    "bounded_maf": {"features": 16, "context_features": None, "batch": 262144, "data": "unit_box",
                    "layers": _bounded_maf_stack(16, 5, 16, 256, cdf_after=1)},
    "bounded_maf_small": {"features": 6, "context_features": None, "batch": 128, "data": "unit_box",
                          "layers": _bounded_maf_stack(6, 2, 16, 32, learn_logit_temperature=True)},
}


def get_workload(name):
    wl = copy.deepcopy(WORKLOADS[name])
    wl["name"] = name
    return wl


def params_per_feature(layer):
    """Conditioner outputs per transformed feature (reference `_transform_dim_multiplier` /
    `_output_dim_multiplier`: coupling.py:543-547, autoregressive.py:94,296,570-576)."""
    kind = layer["kind"]
    if kind in ("prq_coupling", "maf_prq", "cond_prq"):
        return 3 * layer["num_bins"] - 1 if layer.get("tails") == "linear" else 3 * layer["num_bins"] + 1
    if kind in ("affine_coupling", "maf_affine"):
        return 2
    if kind in ("maf_sos", "cond_sos"):
        return 3 * layer["n_sigmoids"] + 1
    if kind in ("plin_coupling", "maf_plin"):
        return layer["num_bins"]
    if kind in ("pcubic_coupling", "maf_pcubic"):
        return 2 * layer["num_bins"] + 2
    if kind in ("pquad_coupling", "maf_pquad"):
        return 2 * layer["num_bins"] - 1 if layer.get("tails") == "linear" else 2 * layer["num_bins"] + 1
    raise ValueError(kind)


def layer_prefix(index):
    """state_dict prefix of layer `index` inside Flow(CompositeTransform([...]), ...)."""
    return "_transform._transforms.{}.".format(index)


def oracle_specs(workload):
    """Plain-data layer specs consumed by oracle/restated.py (adds the state_dict prefix)."""
    specs = []
    for i, layer in enumerate(workload["layers"]):
        spec = dict(layer)
        spec["prefix"] = layer_prefix(i)
        specs.append(spec)
    return specs


def make_mask(features, mode):
    """flowcon/utils/torchutils.py:102-128 mask builders (alternating / mid split)."""
    mask = torch.zeros(features, dtype=torch.uint8)
    if mode == "alternating_even":
        mask[0::2] = 1
    elif mode == "alternating_odd":
        mask[1::2] = 1
    elif mode == "mid_split":
        mask[: (features + 1) // 2] = 1
    else:
        raise ValueError(mode)
    return mask


def trained_like_(state, workload, seed=1, weight_gain=8.0):
    """SURVEY.md §8(d) 'trained-like' weights, applied IN PLACE to a state_dict: freshly
    initialised conditioners leave every spline near-uniform (residual blocks are zero-initialised),
    so scale each layer's final weight by `weight_gain` (8) and add a seeded random bias: std 16 on RQ width/height
    slots that are later divided by sqrt(H), std 1 elsewhere."""
    g = torch.Generator().manual_seed(seed)
    for i, layer in enumerate(workload["layers"]):
        kind = layer["kind"]
        if kind == "permutation":
            continue
        if kind in ("logit", "composite_cdf"):  # a learned temperature moves away from 1
            if layer.get("learn_temperature"):
                keys = ([layer_prefix(i) + "_transform.temperature"] if kind == "logit" else
                        [layer_prefix(i) + "_transforms.0.temperature", layer_prefix(i) + "_transforms.2._transform.temperature"])
                value = state[keys[0]] * torch.exp(0.3 * torch.randn(1, generator=g))
                for key in keys:  # CompositeCDFTransform holds its squashing layer twice
                    state[key] = value.clone()
            continue
        if kind == "actnorm":  # a trained ActNorm has non-trivial per-feature scales and shifts
            for name, std in (("log_scale", 0.4), ("shift", 0.7)):
                key = layer_prefix(i) + name
                state[key] = state[key] + std * torch.randn(state[key].numel(), generator=g, dtype=torch.float32).to(
                    state[key].dtype)
            continue
        if kind == "batchnorm":  # trained: weights away from 1, a shift, running statistics of a non-white input
            p = layer_prefix(i)
            for name, std in (("unconstrained_weight", 0.4), ("bias", 0.5), ("running_mean", 0.8)):
                state[p + name] = state[p + name] + std * torch.randn(state[p + name].numel(), generator=g)
            state[p + "running_var"] = torch.exp(0.6 * torch.randn(state[p + "running_var"].numel(), generator=g))
            continue
        if kind == "lu_linear":  # a trained LULinear is far from the identity: entries at the non-identity init scale
            for name in ("bias", "lower_entries", "upper_entries", "unconstrained_upper_diag"):
                key = layer_prefix(i) + name
                bound = 1.0 / workload["features"] ** 0.5
                u = torch.rand(state[key].numel(), generator=g, dtype=torch.float32) * 2.0 - 1.0
                state[key] = (bound * u).to(state[key].dtype)
            continue
        net = {"prq_coupling": "transform_net", "affine_coupling": "transform_net", "maf_affine": "autoregressive_net",
               "maf_prq": "autoregressive_net", "maf_sos": "autoregressive_net", "cond_sos": "conditional_net",
               "cond_prq": "conditional_net", "plin_coupling": "transform_net", "maf_plin": "autoregressive_net",
               "pquad_coupling": "transform_net", "maf_pquad": "autoregressive_net",
               "pcubic_coupling": "transform_net", "maf_pcubic": "autoregressive_net"}[kind]
        wkey = layer_prefix(i) + net + ".final_layer.weight"
        bkey = layer_prefix(i) + net + ".final_layer.bias"
        p = params_per_feature(layer)
        n_out = state[bkey].numel()
        noise = torch.randn(n_out, generator=g, dtype=torch.float32)
        std = torch.ones(n_out)
        if kind in ("pquad_coupling", "pcubic_coupling"):
            std = std * 4.0  # the width / height slots are divided by sqrt(H)
        if kind in ("prq_coupling", "cond_prq"):
            std = std.view(-1, p)
            std[:, : 2 * layer["num_bins"]] = 16.0
            std = std.reshape(-1)
        state[wkey] = state[wkey] * weight_gain
        state[bkey] = state[bkey] + (noise * std).to(state[bkey].dtype)
    base = workload.get("base", {}).get("kind")
    if base == "diagonal_normal":  # a trained base is shifted and scaled per feature
        for name, std in (("mean_", 0.5), ("log_std_", 0.3)):
            key = "_distribution." + name
            state[key] = state[key] + std * torch.randn(state[key].shape, generator=g)
    elif base == "conditional_diagonal_normal":
        key = "_distribution._context_encoder.bias"
        state[key] = state[key] + 0.3 * torch.randn(state[key].shape, generator=g)
    return state


def sample_data(workload, rows, seed=0):
    """Seeded data for a workload: in (0, 1) for `"data": "unit_box"` workloads, standard normal otherwise."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, workload["features"], generator=g)
    if workload.get("data") == "unit_box":
        return torch.sigmoid(x)
    return x


def build_base(workload):
    """The workload's base density: `base` {"kind": "diagonal_normal"} or {"kind": "conditional_diagonal_normal",
    "encoder": "linear"}; StandardNormal without one."""
    from . import distributions

    features = workload["features"]
    base = workload.get("base")
    if base is None:
        return distributions.StandardNormal([features])
    if base["kind"] == "diagonal_normal":
        return distributions.DiagonalNormal([features])
    if base["kind"] == "conditional_diagonal_normal":
        encoder = None
        if base.get("encoder") == "linear":
            encoder = torch.nn.Linear(workload["context_features"], 2 * features)
        return distributions.ConditionalDiagonalNormal([features], context_encoder=encoder)
    raise ValueError(base["kind"])


def build_flow(workload, seed=0):
    """Instantiate the workload with this package's drop-in classes (random init, CPU tensors;
    move with `.to('cuda')`)."""
    from . import flows, transforms
    from .nn import nets

    torch.manual_seed(seed)
    features = workload["features"]
    ctx = workload.get("context_features")
    layers = []
    for layer in workload["layers"]:
        kind = layer["kind"]
        if kind == "permutation":
            cls = transforms.RandomPermutation if layer["mode"] == "random" else transforms.ReversePermutation
            layers.append(cls(features))
        elif kind == "actnorm":
            layers.append(transforms.ActNorm(features))
        elif kind == "batchnorm":
            layers.append(transforms.BatchNorm(features))
        elif kind == "logit":
            if layer.get("learn_temperature"):  # Logit with its Sigmoid's temperature learned
                layers.append(transforms.InverseTransform(transforms.Sigmoid(learn_temperature=True)))
            else:
                layers.append(transforms.Logit())
        elif kind == "composite_cdf":
            layers.append(transforms.CompositeCDFTransform(
                transforms.Sigmoid(learn_temperature=layer.get("learn_temperature", False)),
                transforms.PiecewiseRationalQuadraticCDF([features], layer["num_bins"])))
        elif kind == "lu_linear":
            layers.append(transforms.LULinear(features, identity_init=layer.get("identity_init", True)))
        elif kind == "prq_coupling":
            hidden, blocks = layer["hidden_features"], layer["num_blocks"]
            layers.append(transforms.PiecewiseRationalQuadraticCouplingTransform(
                mask=make_mask(features, layer["mask"]),
                transform_net_create_fn=lambda i, o, h=hidden, b=blocks: nets.ResidualNet(
                    i, o, hidden_features=h, context_features=ctx, num_blocks=b),
                num_bins=layer["num_bins"], tails=layer["tails"], tail_bound=layer["tail_bound"],
                apply_unconditional_transform=layer.get("unconditional", False)))
        elif kind == "plin_coupling":
            hidden, blocks = layer["hidden_features"], layer["num_blocks"]
            layers.append(transforms.PiecewiseLinearCouplingTransform(
                mask=make_mask(features, layer["mask"]),
                transform_net_create_fn=lambda i, o, h=hidden, b=blocks: nets.ResidualNet(
                    i, o, hidden_features=h, context_features=ctx, num_blocks=b),
                num_bins=layer["num_bins"], tails=layer["tails"], tail_bound=layer["tail_bound"],
                apply_unconditional_transform=layer.get("unconditional", False)))
        elif kind == "pquad_coupling":
            hidden, blocks = layer["hidden_features"], layer["num_blocks"]
            layers.append(transforms.PiecewiseQuadraticCouplingTransform(
                mask=make_mask(features, layer["mask"]),
                transform_net_create_fn=lambda i, o, h=hidden, b=blocks: nets.ResidualNet(
                    i, o, hidden_features=h, context_features=ctx, num_blocks=b),
                num_bins=layer["num_bins"], tails=layer["tails"], tail_bound=layer["tail_bound"],
                apply_unconditional_transform=layer.get("unconditional", False)))
        elif kind == "pcubic_coupling":
            hidden, blocks = layer["hidden_features"], layer["num_blocks"]
            layers.append(transforms.PiecewiseCubicCouplingTransform(
                mask=make_mask(features, layer["mask"]),
                transform_net_create_fn=lambda i, o, h=hidden, b=blocks: nets.ResidualNet(
                    i, o, hidden_features=h, context_features=ctx, num_blocks=b),
                num_bins=layer["num_bins"], tails=layer["tails"], tail_bound=layer["tail_bound"],
                apply_unconditional_transform=layer.get("unconditional", False)))
        elif kind == "maf_pquad":
            layers.append(transforms.MaskedPiecewiseQuadraticAutoregressiveTransform(
                features=features, hidden_features=layer["hidden_features"], context_features=ctx,
                num_bins=layer["num_bins"], num_blocks=layer["num_blocks"], tails=layer["tails"],
                tail_bound=layer["tail_bound"]))
        elif kind == "maf_plin":
            layers.append(transforms.MaskedPiecewiseLinearAutoregressiveTransform(
                num_bins=layer["num_bins"], features=features, hidden_features=layer["hidden_features"],
                context_features=ctx, num_blocks=layer["num_blocks"]))
        elif kind == "maf_pcubic":
            layers.append(transforms.MaskedPiecewiseCubicAutoregressiveTransform(
                num_bins=layer["num_bins"], features=features, hidden_features=layer["hidden_features"],
                context_features=ctx, num_blocks=layer["num_blocks"]))
        elif kind == "affine_coupling":
            hidden, blocks = layer["hidden_features"], layer["num_blocks"]
            act = {"sigmoid2": transforms.AffineCouplingTransform.DEFAULT_SCALE_ACTIVATION,
                   "softplus_clamp3": transforms.AffineCouplingTransform.GENERAL_SCALE_ACTIVATION}[
                layer["scale_activation"]]
            layers.append(transforms.AffineCouplingTransform(
                mask=make_mask(features, layer["mask"]),
                transform_net_create_fn=lambda i, o, h=hidden, b=blocks: nets.ResidualNet(
                    i, o, hidden_features=h, context_features=ctx, num_blocks=b),
                scale_activation=act))
        elif kind == "maf_affine":
            layers.append(transforms.MaskedAffineAutoregressiveTransform(
                features=features, hidden_features=layer["hidden_features"], context_features=ctx,
                num_blocks=layer["num_blocks"]))
        elif kind == "maf_prq":
            layers.append(transforms.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(
                features=features, hidden_features=layer["hidden_features"], context_features=ctx,
                num_bins=layer["num_bins"], tails=layer["tails"], tail_bound=layer["tail_bound"],
                num_blocks=layer["num_blocks"]))
        elif kind == "maf_sos":
            layers.append(transforms.MaskedSumOfSigmoidsTransform(
                features=features, hidden_features=layer["hidden_features"], context_features=ctx,
                n_sigmoids=layer["n_sigmoids"], num_blocks=layer["num_blocks"]))
        elif kind == "cond_sos":
            layers.append(transforms.ConditionalSumOfSigmoidsTransform(
                features=features, hidden_features=layer["hidden_features"], context_features=ctx,
                n_sigmoids=layer["n_sigmoids"], num_blocks=layer["num_blocks"]))
        elif kind == "cond_prq":
            layers.append(transforms.ConditionalPiecewiseRationalQuadraticTransform(
                features=features, hidden_features=layer["hidden_features"], context_features=ctx,
                num_bins=layer["num_bins"], tails=layer["tails"], tail_bound=layer["tail_bound"],
                num_blocks=layer["num_blocks"]))
        else:
            raise ValueError(kind)
    return flows.Flow(transforms.CompositeTransform(layers), build_base(workload))
