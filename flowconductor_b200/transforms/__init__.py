"""Drop-in subset of `flowcon.transforms` for the element-wise bijection hot path (SURVEY.md §8)."""
from .adaptive_sigmoids import SumOfSigmoids  # noqa: F401
from .autoregressive import (AutoregressiveTransform, MaskedAffineAutoregressiveTransform,  # noqa: F401
                             MaskedPiecewiseCubicAutoregressiveTransform,
                             MaskedPiecewiseLinearAutoregressiveTransform,
                             MaskedPiecewiseQuadraticAutoregressiveTransform,
                             MaskedPiecewiseRationalQuadraticAutoregressiveTransform,
                             MaskedSumOfSigmoidsTransform)
from .base import (CompositeTransform, InputOutsideDomain, InverseNotAvailable, InverseTransform,  # noqa: F401
                   Transform)
from .conditional import (ConditionalPiecewiseRationalQuadraticTransform,  # noqa: F401
                          ConditionalSumOfSigmoidsTransform, ConditionalTransform)
from .coupling import (AdditiveCouplingTransform, AffineCouplingTransform, CouplingTransform,  # noqa: F401
                       PiecewiseCubicCouplingTransform, PiecewiseLinearCouplingTransform,
                       PiecewiseQuadraticCouplingTransform,
                       PiecewiseRationalQuadraticCouplingTransform)
from .made import MADE, MaskedLinear  # noqa: F401
from .nonlinearities import (CauchyCDF, CauchyCDFInverse, CompositeCDFTransform, Exp, LeakyReLU,  # noqa: F401
                             Logit, PiecewiseCubicCDF, PiecewiseLinearCDF, PiecewiseQuadraticCDF,
                             PiecewiseRationalQuadraticCDF, Sigmoid, Tanh)
from .lu import LULinear  # noqa: F401
from .normalization import ActNorm, BatchNorm  # noqa: F401
from .permutations import Permutation, RandomPermutation, ReversePermutation  # noqa: F401
from . import splines  # noqa: F401
from .splines import (cubic_spline, linear_spline, quadratic_spline, rational_quadratic_spline,  # noqa: F401
                      unconstrained_cubic_spline, unconstrained_linear_spline, unconstrained_quadratic_spline,
                      unconstrained_rational_quadratic_spline)
