from ._engine import FitEngine, random_theta, theta_from_initialization  # noqa: F401
from ._jtt_ipw import jtt_ipw, jtt_ipw_from_counts  # noqa: F401
from ._quantized_transitions_mle import RateMatrixLearner, quantized_transitions_mle  # noqa: F401
from ._autograd import CherryLoss, RateMatrix  # noqa: F401
from ._tree_likelihood import TreeLikelihoodData, TreeLogLikelihood, tree_likelihood_mle  # noqa: F401
