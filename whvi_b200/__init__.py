"""whvi_b200: B200-native (sm_100a) implementation of the WHVI hot path behind the
reference's Python surface.  See DESIGN.md for the path, INTEGRATION.md for the C ABI."""
from .fwht import FWHT, FWHTFunction, fwht_  # noqa: F401
from .layers import WHVI, WHVIConv2d, WHVILinear  # noqa: F401
from .likelihoods import CategoricalLikelihood, GaussianLikelihood, Likelihood  # noqa: F401
from .networks import WHVIClassification, WHVINetwork, WHVIRegression  # noqa: F401
from .optim import FlatAdam, FlatParams  # noqa: F401
from .utils import Cosine  # noqa: F401
from .weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix  # noqa: F401

__all__ = ["Cosine", "FWHT", "FWHTFunction", "fwht_", "WHVI", "WHVIConv2d", "WHVILinear", "CategoricalLikelihood", "GaussianLikelihood",
           "Likelihood", "WHVIClassification", "WHVINetwork", "WHVIRegression", "FlatAdam", "FlatParams", "WHVIColumnMatrix", "WHVISquarePow2Matrix", "WHVIStackedMatrix"]
