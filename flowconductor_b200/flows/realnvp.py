"""`SimpleRealNVP` — flowcon/flows/realnvp.py:17-71 (Dinh et al. 2017): `num_layers` affine (or, volume preserving,
additive) coupling layers on alternating halves of the features, each conditioned by a ResidualNet and optionally followed
by `BatchNorm`, on a standard normal base."""
import torch
from torch.nn import functional as F

from ..distributions.normal import StandardNormal
from ..nn import nets
from ..transforms.base import CompositeTransform
from ..transforms.coupling import AdditiveCouplingTransform, AffineCouplingTransform
from ..transforms.normalization import BatchNorm
from .base import Flow

__all__ = ["SimpleRealNVP"]


class SimpleRealNVP(Flow):
    def __init__(self, features, hidden_features, num_layers, num_blocks_per_layer, use_volume_preserving=False,
                 activation=F.relu, dropout_probability=0.0, batch_norm_within_layers=False,
                 batch_norm_between_layers=False):
        coupling_constructor = AdditiveCouplingTransform if use_volume_preserving else AffineCouplingTransform
        mask = torch.ones(features)
        mask[::2] = -1

        def create_resnet(in_features, out_features):
            return nets.ResidualNet(in_features, out_features, hidden_features=hidden_features,
                                    num_blocks=num_blocks_per_layer, activation=activation,
                                    dropout_probability=dropout_probability, use_batch_norm=batch_norm_within_layers)

        layers = []
        for _ in range(num_layers):
            layers.append(coupling_constructor(mask=mask, transform_net_create_fn=create_resnet))
            mask *= -1
            if batch_norm_between_layers:
                layers.append(BatchNorm(features=features))
        super().__init__(transform=CompositeTransform(layers), distribution=StandardNormal([features]))
