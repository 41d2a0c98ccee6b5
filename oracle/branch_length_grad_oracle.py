"""``branch_length_gradient`` under its original module path; it is implemented, on the shared inside/outside
pass, in ``oracle/likelihood_grad_oracle.py`` (TEST INFRASTRUCTURE)."""
from oracle.likelihood_grad_oracle import branch_length_gradient  # noqa: F401
