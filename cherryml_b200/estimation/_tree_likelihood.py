"""Maximum-likelihood rate matrices on given trees: the exact tree log-likelihood of independent sites or of
contacting pairs as an autograd node (``TreeLogLikelihood``) and the ``tree_likelihood_mle`` and
``coevolution_tree_likelihood_mle`` stages around it.

The gradient is exact: the inside/outside pass ``cherry_tree_ll_posterior`` gives, per edge matrix
``P_m = expm(t_m Q)``, the posterior counts ``W_m`` of (parent state, child state); since
``d log L / d P_m = W_m / P_m``, ``d log L / d Q = sum_m d/dQ <W_m, log expm(t_m Q)>`` with ``W`` held
fixed, which is the fit's own loss gradient (``cherry_fit_loss_grad``) with ``C = W``.  The same check
a CherryML estimate is built around -- how close it comes to the full-likelihood estimate -- can
then be made on the same trees and MSAs.
"""
import logging
import os
import time
from typing import List, Optional

import numpy as np
import torch

from .. import caching
from ..evaluation._likelihood import (_expm_chunked, _expm_transposed, _exponent_union, _PairFamily, _q_gradient,
                                      _SiteFamily)
from ..io import (read_contact_map, read_mask_matrix, read_msa, read_rate_matrix, read_site_rates, read_tree,
                  write_rate_matrix)
from ._autograd import RateMatrix

logger = logging.getLogger(__name__)


class TreeLikelihoodData:
    """The families ``<tree_dir>/<family>.txt`` (with their MSAs and site rates), encoded once and resident
    on ``device``; every site is an independent unit.  ``exponents`` is the union of the families' distinct
    ``branch length * site rate`` values: one expm pass and one gradient pass per evaluation cover them all."""

    def __init__(self, tree_dir: str, msa_dir: str, site_rates_dir: str, families: List[str],
                 amino_acids: List[str], device="cuda"):
        dev = torch.device(device if str(device).startswith("cuda") else "cuda")
        self.device = dev
        self.amino_acids = list(amino_acids)
        self.families = list(families)
        self.fams = [
            _SiteFamily(read_tree(os.path.join(tree_dir, f + ".txt")), read_msa(os.path.join(msa_dir, f + ".txt")),
                        read_site_rates(os.path.join(site_rates_dir, f + ".txt")), amino_acids, dev)
            for f in families
        ]
        self.exponents, rows = _exponent_union(self.fams)
        self.t = torch.from_numpy(self.exponents).to(dev)
        self.rows = [torch.from_numpy(r).to(dev) for r in rows]
        self.n_sites = sum(f.n_units for f in self.fams)
        self.timing = {"expm": 0.0, "posterior": 0.0, "loss_grad": 0.0}

    def evaluate(self, Q: torch.Tensor, pi: torch.Tensor):
        """(total log-likelihood, d/dQ, d/dpi) at ``Q`` [S, S] and root distribution ``pi`` [S] (fp64, on the
        device); accumulated in family order, so repeated calls give identical results.  Adds the time of
        each phase (host clock around device-synchronised work) to ``self.timing``."""
        Q = Q.detach().to(self.device, torch.float64).contiguous()
        pi = pi.detach().to(self.device, torch.float64).contiguous()
        S = Q.shape[0]
        t0 = time.perf_counter()
        P = _expm_transposed(Q.cpu().numpy(), self.exponents, self.device)
        torch.cuda.synchronize(self.device)
        t1 = time.perf_counter()
        W = torch.zeros((len(self.exponents), S, S), dtype=torch.float64, device=self.device)
        root = torch.zeros(S, dtype=torch.float64, device=self.device)
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        for fam, rows in zip(self.fams, self.rows):
            ll, W_f, root_f = fam.posterior(P.index_select(0, rows), pi)
            W[rows] += W_f  # rows are distinct within a family: one add per entry
            root += root_f
            total += ll.sum()
        torch.cuda.synchronize(self.device)
        t2 = time.perf_counter()
        gQ = _q_gradient(Q, self.t, W)
        torch.cuda.synchronize(self.device)
        t3 = time.perf_counter()
        self.timing["expm"] += t1 - t0
        self.timing["posterior"] += t2 - t1
        self.timing["loss_grad"] += t3 - t2
        return total, gQ, root / pi


class PairTreeLikelihoodData:
    """The contacting pairs of the families ``<tree_dir>/<family>.txt`` (contact maps in ``contact_map_dir``, the
    pairs ``dp_likelihood_computation`` takes), encoded once and resident on ``device``; every pair is a unit on
    ``S^2`` states.  A family's distinct branch lengths need ``S^4`` doubles each (1.28 MB at S = 20), so the
    matrices are made, used and freed one family at a time."""

    def __init__(self, tree_dir: str, msa_dir: str, contact_map_dir: str, families: List[str],
                 amino_acids: List[str], device="cuda"):
        dev = torch.device(device if str(device).startswith("cuda") else "cuda")
        self.device = dev
        self.amino_acids = list(amino_acids)
        self.families = list(families)
        self.fams = [
            _PairFamily(read_tree(os.path.join(tree_dir, f + ".txt")), read_msa(os.path.join(msa_dir, f + ".txt")),
                        read_contact_map(os.path.join(contact_map_dir, f + ".txt")), amino_acids, dev)
            for f in families
        ]
        self.t = [torch.from_numpy(f.exponents).to(dev) for f in self.fams]
        self.n_pairs = sum(f.n_pairs for f in self.fams)
        self.n_exponents = sum(len(f.exponents) for f in self.fams)
        self.timing = {"expm": 0.0, "posterior": 0.0, "loss_grad": 0.0}

    def evaluate(self, Q: torch.Tensor, pi: torch.Tensor):
        """(total log-likelihood, d/dQ, d/dpi) at ``Q`` [S^2, S^2] and root distribution ``pi`` [S^2] (fp64, on the
        device); expm, posterior and gradient family by family, summed in family order, so repeated calls give
        identical results.  Adds the time of each phase (host clock around device-synchronised work) to
        ``self.timing``."""
        Q = Q.detach().to(self.device, torch.float64).contiguous()
        pi = pi.detach().to(self.device, torch.float64).contiguous()
        Su = Q.shape[0]
        Q_host = Q.cpu().numpy()
        gQ = torch.zeros((Su, Su), dtype=torch.float64, device=self.device)
        root = torch.zeros(Su, dtype=torch.float64, device=self.device)
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        for fam, t in zip(self.fams, self.t):
            if fam.n_pairs == 0:
                continue
            t0 = time.perf_counter()
            P = _expm_chunked(Q_host, fam.exponents, self.device, transpose=False)
            torch.cuda.synchronize(self.device)
            t1 = time.perf_counter()
            ll, W, root_f = fam.posterior(P, pi)
            del P
            root += root_f
            total += ll.sum()
            torch.cuda.synchronize(self.device)
            t2 = time.perf_counter()
            gQ += _q_gradient(Q, t, W)
            del W
            torch.cuda.synchronize(self.device)
            t3 = time.perf_counter()
            self.timing["expm"] += t1 - t0
            self.timing["posterior"] += t2 - t1
            self.timing["loss_grad"] += t3 - t2
        return total, gQ, root / pi


class TreeLogLikelihood(torch.autograd.Function):
    """``TreeLogLikelihood.apply(Q, pi, data)``: the total log-likelihood of the families of ``data`` under rate
    matrix ``Q`` and root distribution ``pi``, as a 0-dim fp64 tensor, with gradients to ``Q`` and ``pi`` (every
    entry a free variable).  ``data`` is a ``TreeLikelihoodData`` (independent sites, ``Q`` [S, S], ``pi`` [S])
    or a ``PairTreeLikelihoodData`` (contacting pairs, ``Q`` [S^2, S^2], ``pi`` [S^2])."""

    @staticmethod
    def forward(ctx, Q: torch.Tensor, pi: torch.Tensor, data) -> torch.Tensor:
        if not Q.is_cuda or Q.dtype != torch.float64:
            raise ValueError("TreeLogLikelihood needs an fp64 CUDA tensor Q (there is no CPU fallback)")
        total, gQ, gpi = data.evaluate(Q, pi)
        ctx.save_for_backward(gQ, gpi)
        return total

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        gQ, gpi = ctx.saved_tensors
        return grad_out * gQ, grad_out * gpi, None


def _adam_best_iterate(data, num_states: int, n_units: int, initialization_path: str, mask_path: Optional[str],
                       num_epochs: int, learning_rate: float, dev):
    """``RateMatrix`` (``pande_reversible``, pi learnt) from the rate matrix at ``initialization_path``, and
    ``num_epochs`` Adam steps on minus the log-likelihood of ``data`` per unit, pi being the model's own
    stationary distribution: (best log-likelihood, its rate matrix) over the ``num_epochs + 1`` iterates."""
    Q0 = read_rate_matrix(initialization_path).to_numpy()
    mask = read_mask_matrix(mask_path).to_numpy() if mask_path is not None else None
    model = RateMatrix(num_states=num_states, mask=mask, pi_requires_grad=True, initialization=Q0, device=dev)
    opt = torch.optim.Adam(model.parameters(), lr=learning_rate)
    best_ll, best_Q = -float("inf"), None
    for epoch in range(num_epochs + 1):
        opt.zero_grad()
        Q = model()
        ll = TreeLogLikelihood.apply(Q, model.stationary_distribution(), data)
        value = float(ll.item())
        if value > best_ll:
            best_ll, best_Q = value, Q.detach().cpu().numpy()
        logger.info(f"epoch {epoch}: log-likelihood {value}")
        if epoch == num_epochs:
            break
        (-ll / n_units).backward()
        opt.step()
    return best_ll, best_Q


def _write_stage_files(out_dir: str, states: List[str], best_Q: np.ndarray, best_ll: float, num_epochs: int,
                       n_families: int, units: str, start: float, t_setup: float, tm: dict) -> None:
    """A maximum-likelihood stage's ``result.txt`` (``best_Q`` labelled with ``states``), ``log_likelihood.txt``
    and ``profiling.txt``; ``units`` describes the data (units and distinct exponents), ``start`` is the
    stage's ``time.time()`` at entry and ``tm`` the data's phase timings."""
    os.makedirs(out_dir, exist_ok=True)
    write_rate_matrix(best_Q, states, os.path.join(out_dir, "result.txt"))
    with open(os.path.join(out_dir, "log_likelihood.txt"), "w") as f:
        f.write(f"{best_ll!r}\n")
    total = time.time() - start
    with open(os.path.join(out_dir, "profiling.txt"), "w") as f:
        f.write(f"Total time: {total} seconds for {num_epochs} epochs over {n_families} families ({units})\n"
                f"Set-up (read and encode): {t_setup}\nexpm: {tm['expm']}\nposterior: {tm['posterior']}\n"
                f"loss_grad: {tm['loss_grad']}\n"
                f"host and rest: {total - t_setup - tm['expm'] - tm['posterior'] - tm['loss_grad']}\n")


@caching.cached_computation(
    output_dirs=["output_rate_matrix_dir"],
    exclude_args=["device"],
    write_extra_log_files=True,
)
def tree_likelihood_mle(
    tree_dir: str,
    msa_dir: str,
    site_rates_dir: str,
    families: List[str],
    amino_acids: List[str],
    initialization_path: str,
    mask_path: Optional[str] = None,
    num_epochs: int = 100,
    learning_rate: float = 0.1,
    device: str = "cuda",
    output_rate_matrix_dir: Optional[str] = None,
):
    """Full-likelihood (ML) rate matrix of independent sites on the given trees, from the rate matrix at
    ``initialization_path``: ``RateMatrix`` (``pande_reversible``, pi learnt) and Adam on minus the mean
    per-site log-likelihood, pi being the model's own stationary distribution.  ``num_epochs`` steps; the
    best of the ``num_epochs + 1`` iterates is kept.  Writes ``result.txt`` (the rate matrix),
    ``log_likelihood.txt`` (its total log-likelihood over all families) and ``profiling.txt``."""
    start = time.time()
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    data = TreeLikelihoodData(tree_dir, msa_dir, site_rates_dir, families, amino_acids, dev)
    t_setup = time.time() - start
    best_ll, best_Q = _adam_best_iterate(data, len(amino_acids), data.n_sites, initialization_path, mask_path,
                                         num_epochs, learning_rate, dev)
    _write_stage_files(output_rate_matrix_dir, amino_acids, best_Q, best_ll, num_epochs, len(families),
                       f"{data.n_sites} sites, {len(data.exponents)} distinct exponents", start, t_setup, data.timing)


@caching.cached_computation(
    output_dirs=["output_rate_matrix_dir"],
    exclude_args=["device"],
    write_extra_log_files=True,
)
def coevolution_tree_likelihood_mle(
    tree_dir: str,
    msa_dir: str,
    contact_map_dir: str,
    families: List[str],
    amino_acids: List[str],
    initialization_path: str,
    mask_path: Optional[str] = None,
    num_epochs: int = 100,
    learning_rate: float = 0.1,
    device: str = "cuda",
    output_rate_matrix_dir: Optional[str] = None,
):
    """Full-likelihood (ML) co-evolution rate matrix on ``S^2`` pair states, from the contacting pairs of the
    given families on their trees (contact maps in ``contact_map_dir``, pairs as ``dp_likelihood_computation``
    takes them), starting from the rate matrix at ``initialization_path``: ``RateMatrix(S^2)``
    (``pande_reversible``, pi learnt) and Adam on minus the mean per-pair log-likelihood.  ``num_epochs``
    steps; the best of the ``num_epochs + 1`` iterates is kept.  Writes ``result.txt`` (the rate matrix,
    labelled with the pair states), ``log_likelihood.txt`` (its total pair log-likelihood over all families)
    and ``profiling.txt``.  The independent sites of the families are not part of this likelihood."""
    start = time.time()
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    data = PairTreeLikelihoodData(tree_dir, msa_dir, contact_map_dir, families, amino_acids, dev)
    t_setup = time.time() - start
    states = [a + b for a in amino_acids for b in amino_acids]
    best_ll, best_Q = _adam_best_iterate(data, len(states), data.n_pairs, initialization_path, mask_path,
                                         num_epochs, learning_rate, dev)
    _write_stage_files(output_rate_matrix_dir, states, best_Q, best_ll, num_epochs, len(families),
                       f"{data.n_pairs} pairs, {data.n_exponents} distinct branch lengths", start, t_setup, data.timing)
