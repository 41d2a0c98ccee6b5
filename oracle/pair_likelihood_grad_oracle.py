"""``pair_log_likelihood_gradient`` under its original module path; it is implemented, on the shared
inside/outside pass, in ``oracle/likelihood_grad_oracle.py`` (TEST INFRASTRUCTURE)."""
from oracle.likelihood_grad_oracle import pair_log_likelihood_gradient  # noqa: F401
