"""`Flow(transform, distribution, embedding_net=None)` — flowcon/flows/base.py:11-119 with the same
attribute names (`_transform`, `_distribution`, `_embedding_net`), so state_dict keys match."""
from inspect import signature

import torch.nn

from ..distributions.base import Distribution
from ..distributions.normal import ConditionalDiagonalNormal, DiagonalNormal, StandardNormal
from ..utils import torchutils

__all__ = ["Flow"]


class Flow(Distribution):
    def __init__(self, transform, distribution, embedding_net=None):
        super().__init__()
        self._transform = transform
        self._distribution = distribution
        self._context_used_in_base = "context" in signature(self._distribution.log_prob).parameters.keys()
        if embedding_net is not None:
            assert isinstance(embedding_net, torch.nn.Module), (
                "embedding_net is not a nn.Module. If you want to use hard-coded summary features, "
                "please simply pass the encoded features and pass embedding_net=None")
            self._embedding_net = embedding_net
        else:
            self._embedding_net = torch.nn.Identity()

    def _log_prob(self, inputs, context):
        embedded = self._embedding_net(context)
        noise, logabsdet = self._transform(inputs, context=embedded)
        if type(self._distribution) is StandardNormal:
            return self._distribution.log_prob_plus(noise, logabsdet)  # fused base density + logabsdet
        if type(self._distribution) in (DiagonalNormal, ConditionalDiagonalNormal):
            return self._distribution.log_prob_plus(noise, logabsdet, context=embedded)
        if self._context_used_in_base:
            return self._distribution.log_prob(noise, context=embedded) + logabsdet
        return self._distribution.log_prob(noise) + logabsdet

    def _noise(self, num_samples, embedded, with_log_prob):
        draw = self._distribution.sample_and_log_prob if with_log_prob else self._distribution.sample
        if self._context_used_in_base:
            return draw(num_samples, context=embedded)
        if with_log_prob or embedded is None:
            return draw(num_samples)
        flat = draw(num_samples * embedded.shape[0])
        return torch.reshape(flat, (embedded.shape[0], -1, flat.shape[1]))

    def _sample(self, num_samples, context):
        embedded = self._embedding_net(context)
        noise = self._noise(num_samples, embedded, with_log_prob=False)
        if embedded is not None:
            noise = torchutils.merge_leading_dims(noise, num_dims=2)
            embedded = torchutils.repeat_rows(embedded, num_reps=num_samples)
        samples, _ = self._transform.inverse(noise, context=embedded)
        if embedded is not None:
            samples = torchutils.split_leading_dim(samples, shape=[-1, num_samples])
        return samples

    def sample_and_log_prob(self, num_samples, context=None):
        embedded = self._embedding_net(context)
        noise, log_prob = self._noise(num_samples, embedded, with_log_prob=True)
        if embedded is not None:
            noise = torchutils.merge_leading_dims(noise, num_dims=2)
            embedded = torchutils.repeat_rows(embedded, num_reps=num_samples)
        samples, logabsdet = self._transform.inverse(noise, context=embedded)
        if embedded is not None:
            samples = torchutils.split_leading_dim(samples, shape=[-1, num_samples])
            logabsdet = torchutils.split_leading_dim(logabsdet, shape=[-1, num_samples])
        return samples, log_prob - logabsdet

    def transform_to_noise(self, inputs, context=None):
        noise, _ = self._transform(inputs, context=self._embedding_net(context))
        return noise
