"""Tree log-likelihoods on the GPU: drop-in for ``cherryml/evaluation/_likelihood.py``; the
rate-matrix distances of ``_metrics.py`` and the contact-map matching of ``_maximal_matching.py``."""
from .._public_api import create_maximal_matching_contact_map  # noqa: F401
from ._likelihood import (  # noqa: F401
    branch_length_gradient,
    compute_log_likelihoods,
    dp_likelihood_computation,
    log_likelihood_gradient,
    pair_log_likelihood_gradient,
)
from ._metrics import (  # noqa: F401
    l_infty_norm,
    mean_relative_error,
    mre,
    relative_error,
    relative_errors,
    rmse,
)
