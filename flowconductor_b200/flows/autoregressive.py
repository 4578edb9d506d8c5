"""`MaskedAutoregressiveFlow` — flowcon/flows/autoregressive.py:13-62 (Papamakarios et al. 2017): `num_layers` times a
permutation and an affine MADE layer, optionally followed by `BatchNorm`, on a standard normal base."""
from torch.nn import functional as F

from ..distributions.normal import StandardNormal
from ..transforms.autoregressive import MaskedAffineAutoregressiveTransform
from ..transforms.base import CompositeTransform
from ..transforms.normalization import BatchNorm
from ..transforms.permutations import RandomPermutation, ReversePermutation
from .base import Flow

__all__ = ["MaskedAutoregressiveFlow"]


class MaskedAutoregressiveFlow(Flow):
    def __init__(self, features, hidden_features, num_layers, num_blocks_per_layer, use_residual_blocks=True,
                 use_random_masks=False, use_random_permutations=False, activation=F.relu, dropout_probability=0.0,
                 batch_norm_within_layers=False, batch_norm_between_layers=False):
        permutation_constructor = RandomPermutation if use_random_permutations else ReversePermutation
        layers = []
        for _ in range(num_layers):
            layers.append(permutation_constructor(features))
            layers.append(MaskedAffineAutoregressiveTransform(
                features=features, hidden_features=hidden_features, num_blocks=num_blocks_per_layer,
                use_residual_blocks=use_residual_blocks, random_mask=use_random_masks, activation=activation,
                dropout_probability=dropout_probability, use_batch_norm=batch_norm_within_layers))
            if batch_norm_between_layers:
                layers.append(BatchNorm(features))
        super().__init__(transform=CompositeTransform(layers), distribution=StandardNormal([features]))
