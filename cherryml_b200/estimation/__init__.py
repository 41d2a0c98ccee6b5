from ._engine import FitEngine, random_theta, theta_from_initialization  # noqa: F401
from ._jtt_ipw import jtt_ipw, jtt_ipw_from_counts  # noqa: F401
from ._quantized_transitions_mle import RateMatrixLearner, quantized_transitions_mle  # noqa: F401
from ._autograd import CherryLoss, RateMatrix  # noqa: F401
from ._tree_likelihood import (  # noqa: F401
    PairTreeLikelihoodData,
    TreeLikelihoodData,
    TreeLogLikelihood,
    coevolution_tree_likelihood_mle,
    tree_likelihood_mle,
)
