"""Tree estimation on the GPU: FastCherries (reference ``cherryml/phylogeny_estimation``) and
maximum-likelihood branch lengths on given topologies."""
from ._branch_length_mle import branch_length_mle  # noqa: F401
from ._fast_cherries import fast_cherries, fast_cherries_device  # noqa: F401
from ._gt_tree_estimator import gt_tree_estimator  # noqa: F401
from ._pipeline import fast_cherries_then_count_lg  # noqa: F401,E402
