from .base import Distribution, NoMeanException  # noqa: F401
from .normal import ConditionalDiagonalNormal, DiagonalNormal, StandardNormal  # noqa: F401
