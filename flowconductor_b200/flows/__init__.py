from .autoregressive import MaskedAutoregressiveFlow  # noqa: F401
from .base import Flow  # noqa: F401
from .realnvp import SimpleRealNVP  # noqa: F401
