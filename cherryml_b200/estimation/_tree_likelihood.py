"""Maximum-likelihood rate matrices on given trees: the exact tree log-likelihood of independent sites
as an autograd node (``TreeLogLikelihood``) and the ``tree_likelihood_mle`` stage around it.

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
from ..evaluation._likelihood import _expm_transposed, _q_gradient, _SiteFamily
from ..io import read_mask_matrix, read_msa, read_rate_matrix, read_site_rates, read_tree, write_rate_matrix
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
        self.exponents, inverse = np.unique(np.concatenate([f.exponents for f in self.fams]), return_inverse=True)
        self.t = torch.from_numpy(self.exponents).to(dev)
        # per family: the rows of the union its own exponents are (sorted, distinct)
        offs = np.cumsum([0] + [len(f.exponents) for f in self.fams])
        self.rows = [torch.from_numpy(inverse[offs[i]: offs[i + 1]]).to(dev) for i in range(len(self.fams))]
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


class TreeLogLikelihood(torch.autograd.Function):
    """``TreeLogLikelihood.apply(Q, pi, data)``: the total log-likelihood of the families of ``data``
    (a ``TreeLikelihoodData``) under rate matrix ``Q`` [S, S] and root distribution ``pi`` [S], as a
    0-dim fp64 tensor, with gradients to ``Q`` and ``pi`` (every entry a free variable)."""

    @staticmethod
    def forward(ctx, Q: torch.Tensor, pi: torch.Tensor, data: TreeLikelihoodData) -> torch.Tensor:
        if not Q.is_cuda or Q.dtype != torch.float64:
            raise ValueError("TreeLogLikelihood needs an fp64 CUDA tensor Q (there is no CPU fallback)")
        total, gQ, gpi = data.evaluate(Q, pi)
        ctx.save_for_backward(gQ, gpi)
        return total

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        gQ, gpi = ctx.saved_tensors
        return grad_out * gQ, grad_out * gpi, None


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
    Q0 = read_rate_matrix(initialization_path).to_numpy()
    mask = read_mask_matrix(mask_path).to_numpy() if mask_path is not None else None
    model = RateMatrix(num_states=len(amino_acids), mask=mask, pi_requires_grad=True, initialization=Q0, device=dev)
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
        (-ll / data.n_sites).backward()
        opt.step()
    os.makedirs(output_rate_matrix_dir, exist_ok=True)
    write_rate_matrix(best_Q, amino_acids, os.path.join(output_rate_matrix_dir, "result.txt"))
    with open(os.path.join(output_rate_matrix_dir, "log_likelihood.txt"), "w") as f:
        f.write(f"{best_ll!r}\n")
    total = time.time() - start
    tm = data.timing
    with open(os.path.join(output_rate_matrix_dir, "profiling.txt"), "w") as f:
        f.write(f"Total time: {total} seconds for {num_epochs} epochs over {len(families)} families "
                f"({data.n_sites} sites, {len(data.exponents)} distinct exponents)\n"
                f"Set-up (read and encode): {t_setup}\nexpm: {tm['expm']}\nposterior: {tm['posterior']}\n"
                f"loss_grad: {tm['loss_grad']}\n"
                f"host and rest: {total - t_setup - tm['expm'] - tm['posterior'] - tm['loss_grad']}\n")
