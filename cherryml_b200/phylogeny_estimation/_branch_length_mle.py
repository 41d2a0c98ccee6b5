"""Maximum-likelihood branch lengths on given topologies: a stage with the tree estimators' interface that
keeps each family's tree and refits its branch lengths under a given rate matrix, so that
``lg_end_to_end_with_cherryml_optimizer`` can alternate re-estimating trees and re-fitting the rate matrix
on trees that come from elsewhere (FastTree, PhyML, simulations).

The gradient is exact: ``cherry_tree_ll_edge_derivatives`` gives ``d log L / d (length * rate)`` for every
edge and rate category in the same inside/outside pass that yields the log-likelihood
(``evaluation.branch_length_gradient`` is the one-family form of the same computation)."""
import os
import time
from typing import List, Optional

import numpy as np
import torch

from ..caching import cached_parallel_computation
from ..evaluation._likelihood import _expm_transposed, _exponent_union, _SiteFamily
from ..io import (Tree, read_msa, read_rate_matrix, read_site_rates, read_tree, write_log_likelihood,
                  write_site_rates, write_tree)
from ..markov_chain import compute_stationary_distribution

# cherry_expm_batched for S <= 32: thirty squarings of a Taylor step with t * ||Q||_1 <= 0.0376
_EXPM_MAX_T_NORM = 0.0376 * 2.0 ** 30


class _BranchLengthData:
    """The families on the device with their branch lengths as parameters: ``theta[f]`` holds the log of the
    length of every non-root node of family ``f`` in post order (the root has no branch)."""

    def __init__(self, trees, msas, site_rates, amino_acids, Q: np.ndarray, min_branch_length: float,
                 max_branch_length: float, dev):
        self.dev = dev
        self.fams = [_SiteFamily(t, m, r, amino_acids, dev) for t, m, r in zip(trees, msas, site_rates)]
        self.Q = np.array(Q, dtype=np.float64, order="C")
        self.d_Q = torch.from_numpy(self.Q).to(dev)
        self.d_pi = torch.from_numpy(np.ascontiguousarray(compute_stationary_distribution(self.Q))).to(dev)
        self.lo, self.hi = np.log(min_branch_length), np.log(max_branch_length)
        self.theta = [torch.from_numpy(np.log(np.clip(f.lengths[:-1], min_branch_length, max_branch_length)))
                      .requires_grad_() for f in self.fams]
        self.timing = {"expm": 0.0, "posterior": 0.0, "host": 0.0}

    def lengths(self, f: int) -> np.ndarray:
        """Branch lengths of family ``f`` at the current parameters, in post order (the root's is 0)."""
        return np.append(np.exp(self.theta[f].detach().numpy()), 0.0)

    def evaluate(self):
        """Per family (log-likelihood, per-site log-likelihoods [n_sites], branch lengths) at the current
        parameters, and sets ``theta[f].grad`` to the gradient of minus the mean per-site log-likelihood of
        family ``f``.  One expm pass over the union of the families' distinct exponents, one
        ``cherry_tree_ll_edge_derivatives`` launch per family."""
        t0 = time.perf_counter()
        lengths = [self.lengths(f) for f in range(len(self.fams))]
        for fam, ln in zip(self.fams, lengths):
            fam.set_lengths(ln)
        union, rows = _exponent_union(self.fams)
        t1 = time.perf_counter()
        P = _expm_transposed(self.Q, union, self.dev)
        torch.cuda.synchronize(self.dev)
        t2 = time.perf_counter()
        outs = []
        for fam, r in zip(self.fams, rows):
            P_f = P.index_select(0, torch.from_numpy(r).to(self.dev))
            ll, _, _, dtau = fam.edge_derivatives(P_f, self.d_pi, self.d_Q)
            outs.append((ll.cpu().numpy(), dtau.cpu().numpy()))  # the copies synchronise
        t3 = time.perf_counter()
        res = []
        for i, (fam, (lls, dtau)) in enumerate(zip(self.fams, outs)):
            dlen = dtau[:-1] @ fam.rates  # d ll / d length of every non-root node
            # d/d theta of -ll / n_sites, length = exp(theta)
            self.theta[i].grad = torch.from_numpy(-(dlen * lengths[i][:-1]) / max(1, fam.n_units))
            res.append((float(lls.sum()), lls, lengths[i]))
        t4 = time.perf_counter()
        self.timing["host"] += (t1 - t0) + (t4 - t3)
        self.timing["expm"] += t2 - t1
        self.timing["posterior"] += t3 - t2
        return res

    def clamp(self) -> None:
        with torch.no_grad():
            for th in self.theta:
                th.clamp_(self.lo, self.hi)


def _with_lengths(tree: Tree, length_of: dict) -> Tree:
    """``tree`` with the same nodes and edges in the same order, the edge above ``v`` of length ``length_of[v]``."""
    out = Tree()
    out.add_nodes(tree.nodes())
    out.add_edges([(u, v, float(length_of[v])) for u, v, _ in tree.edges()])
    return out


@cached_parallel_computation(
    parallel_arg="families",
    exclude_args=["num_processes", "device"],
    output_dirs=["output_tree_dir", "output_site_rates_dir", "output_likelihood_dir"],
    write_extra_log_files=True,
)
def branch_length_mle(
    tree_dir: str,
    site_rates_dir: str,
    msa_dir: str,
    families: List[str],
    rate_matrix_path: str,
    amino_acids: List[str],
    num_processes: int = 1,
    num_epochs: int = 200,
    learning_rate: float = 0.05,
    min_branch_length: float = 1e-6,
    max_branch_length: float = 10.0,
    device: str = "cuda",
    output_tree_dir: Optional[str] = None,
    output_site_rates_dir: Optional[str] = None,
    output_likelihood_dir: Optional[str] = None,
) -> None:
    """Maximum-likelihood branch lengths of the trees ``<tree_dir>/<family>.txt`` under the rate matrix at
    ``rate_matrix_path`` (root distribution: its stationary distribution), with the topology and the site
    rates (``<site_rates_dir>/<family>.txt``) held fixed.  Independent sites, up to 32 states; no CPU
    fallback.  ``functools.partial(branch_length_mle, tree_dir=..., site_rates_dir=..., amino_acids=...)``
    is a ``tree_estimator`` for ``lg_end_to_end_with_cherryml_optimizer``.

    The parameters are ``theta = log(clamp(length, min_branch_length, max_branch_length))`` per edge, and
    Adam (``learning_rate``, ``num_epochs`` steps) minimises the sum over families of minus the mean
    per-site log-likelihood, ``theta`` being clamped to the same bounds after every step.  Each family
    keeps the best of its own ``num_epochs + 1`` iterates.  Adam works elementwise and the loss is a sum
    of per-family terms, so a family's trajectory does not depend on which other families share the call.

    Defaults of the bounds:
    * ``min_branch_length = 1e-6``: the log parameterisation cannot reach 0.  The derivative of the
      log-likelihood at a zero-length branch is bounded by about ``n_sites * max rate * max |Q_ii|``, so
      the floor costs at most about ``1e-6`` times that, well under 0.01 nats for families of a few
      thousand sites.
    * ``max_branch_length = 10``: on a saturated branch the likelihood is flat and rises towards its
      limit, so the length would drift without end.  At 10 substitutions per site the slowest mode of LG
      (eigenvalue -0.267) has decayed to 7% at site rate 1 and to under 0.5% at rate 2; real trees have
      branches far shorter.
    ``max_branch_length * max site rate * ||Q||_1`` must stay within the expm's range (``0.0376 * 2^30``),
    which is checked on entry.

    Writes per family ``output_tree_dir/<family>.txt`` (the input tree, nodes and edges in the same order,
    only the lengths changed), ``output_site_rates_dir/<family>.txt`` (the input site rates),
    ``output_likelihood_dir/<family>.txt`` (log-likelihood and per-site values of the kept iterate) and
    ``output_tree_dir/<family>.profiling`` (a ``total_time:`` line; the stage's wall time is split evenly
    over the families).  ``num_processes`` is accepted and ignored: one GPU process does all families."""
    start = time.time()
    if not 0.0 < min_branch_length <= max_branch_length:
        raise ValueError(f"need 0 < min_branch_length <= max_branch_length ({min_branch_length}, "
                         f"{max_branch_length})")
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    Q_df = read_rate_matrix(rate_matrix_path)
    if list(Q_df.index) != list(amino_acids) or list(Q_df.columns) != list(amino_acids):
        raise ValueError(f"the rate matrix at {rate_matrix_path} is not over the states {amino_acids}")
    Q = Q_df.to_numpy()
    names = [f + ".txt" for f in families]
    trees = [read_tree(os.path.join(tree_dir, n)) for n in names]
    rates = [read_site_rates(os.path.join(site_rates_dir, n)) for n in names]
    msas = [read_msa(os.path.join(msa_dir, n)) for n in names]
    max_rate = max((max(r) for r in rates if r), default=0.0)
    norm = np.abs(Q).sum(axis=0).max()
    if max_branch_length * max_rate * norm > _EXPM_MAX_T_NORM:
        raise ValueError(f"max_branch_length * max site rate * ||Q||_1 = {max_branch_length * max_rate * norm:.3g} "
                         f"is beyond the expm's range ({_EXPM_MAX_T_NORM:.3g})")
    data = _BranchLengthData(trees, msas, rates, amino_acids, Q, min_branch_length, max_branch_length, dev)
    opt = torch.optim.Adam(data.theta, lr=learning_rate)
    best = None
    for epoch in range(num_epochs + 1):
        res = data.evaluate()
        best = res if best is None else [r if r[0] > b[0] else b for r, b in zip(res, best)]
        if epoch == num_epochs:
            break
        opt.step()
        data.clamp()
    for d in (output_tree_dir, output_site_rates_dir, output_likelihood_dir):
        os.makedirs(d, exist_ok=True)
    for f, n in enumerate(names):
        ll, lls, lengths = best[f]
        write_tree(_with_lengths(trees[f], dict(zip(data.fams[f].names, lengths))), os.path.join(output_tree_dir, n))
        write_site_rates(rates[f], os.path.join(output_site_rates_dir, n))
        write_log_likelihood((ll, [float(x) for x in lls]), os.path.join(output_likelihood_dir, n))
    share = (time.time() - start) / max(1, len(families))
    tm = data.timing
    for f in families:
        with open(os.path.join(output_tree_dir, f + ".profiling"), "w") as fh:
            fh.write(f"total_time: {share}\n")
            fh.write(f"(stage over {len(families)} families, {num_epochs} epochs: expm {tm['expm']} s, "
                     f"posterior {tm['posterior']} s, host {tm['host']} s)\n")
