"""``compute_log_likelihoods`` with the reference's signature, caching behaviour and output
files (``cherryml/evaluation/_likelihood.py:436-590``), and ``dp_likelihood_computation``
(:47-326) on the GPU: the transition matrices of all edges come from ``cherry_expm_batched``
(one matrix per DISTINCT ``branch length * site rate``), the dynamic programme is
``cherry_tree_log_likelihood`` (one launch per model: independent sites, contacting pairs).

No CPU fallback: the functions raise if the CUDA library or a GPU is missing.
"""
import os
import time
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from .. import _lib
from ..caching import cached_parallel_computation
from ..io import (Tree, read_contact_map, read_msa, read_probability_distribution, read_rate_matrix, read_site_rates,
                  read_tree, write_log_likelihood)
from ..markov_chain import LARGE_MAX_K, expm_batched

_PAIR_EXPM_CHUNK = 128  # 400 x 400 exponentials per cherry_expm_batched call (bounds its workspace)


def _contact_pairs(contact_map: Optional[np.ndarray]) -> List[Tuple[int, int]]:
    """The contacting pairs ``(i, j)``, ``i < j``, in ``np.where`` order; every site in at most one pair."""
    if contact_map is None:
        return []
    ii, jj = np.where(contact_map == 1)
    pairs = [(int(i), int(j)) for i, j in zip(ii, jj) if i < j]
    flat = [s for p in pairs for s in p]
    if len(set(flat)) != len(flat):
        raise Exception(
            f"Each site can only be in contact with one other site. The contacting sites were: {pairs}"
        )
    return pairs


def _tree_arrays(tree: Tree, with_names: bool = False):
    """Post-order node table for the kernel + per node branch length (one iterative walk; the
    order is ``tree.postorder_traversal()``'s: children in edge order, then their parent).  With
    ``with_names`` the node names in that order come fifth."""
    kids_of = {v: tree.children(v) for v in tree.nodes()}
    depths: List[int] = []
    flags: List[int] = []
    obs_rows: List[int] = []
    lengths: List[float] = []
    leaves: List[str] = []
    names: List[str] = []
    stack = [(tree.root(), 0, 0.0, 0, False)]
    while stack:
        v, d, length, first, expanded = stack.pop()
        kids = kids_of[v]
        if kids and not expanded:
            stack.append((v, d, length, first, True))
            for j in range(len(kids) - 1, -1, -1):
                stack.append((kids[j][0], d + 1, kids[j][1], 2 if j == 0 else 0, False))
            continue
        depths.append(d)
        lengths.append(length)
        names.append(v)
        if kids:
            flags.append(first)
            obs_rows.append(-1)
        else:
            flags.append(first | 1)
            obs_rows.append(len(leaves))
            leaves.append(v)
    nodes = np.zeros(len(depths), dtype=_lib.LL_NODE_DTYPE)
    nodes["depth"] = depths
    nodes["flags"] = flags
    nodes["obs_row"] = obs_rows
    if with_names:
        return nodes, np.array(lengths, dtype=np.float64), leaves, max(depths), names
    return nodes, np.array(lengths, dtype=np.float64), leaves, max(depths)


def _encode_leaves(msa: Dict[str, str], leaves: List[str], amino_acids: List[str]) -> np.ndarray:
    """uint8 [n_leaves, n_sites]: index in ``amino_acids``, S for any other character."""
    S = len(amino_acids)
    lut = np.full(256, S, dtype=np.uint8)
    for i, ch in enumerate(amino_acids):
        lut[ord(ch)] = i
    n_sites = len(msa[leaves[0]])
    seqs = [msa[v] for v in leaves]
    if any(len(q) != n_sites for q in seqs):
        raise ValueError("the sequences of the MSA have different lengths")
    flat = np.frombuffer("".join(seqs).encode("latin-1"), dtype=np.uint8)
    return lut[flat].reshape(len(leaves), n_sites)


def _matrices(Q: np.ndarray, exponents: np.ndarray, device) -> Tuple[torch.Tensor, np.ndarray]:
    """One expm per distinct exponent -> (the TRANSPOSED matrices [n_distinct, S, S] on the device, as the
    pruning kernel reads them, and the index of every exponent)."""
    uniq, inverse = np.unique(exponents, return_inverse=True)
    return _expm_transposed(Q, uniq, device), inverse.astype(np.int32)


def _expm_transposed(Q, exponents: np.ndarray, device) -> torch.Tensor:
    """``[K, S, S]``: ``expm(exponents[k] * Q)`` TRANSPOSED, as the pruning kernels read it (``Q``: numpy or a
    device tensor)."""
    return _expm_chunked(Q, exponents, device, transpose=True)


def _expm_chunked(Q, exponents: np.ndarray, device, transpose: bool) -> torch.Tensor:
    """``[K, S, S]``: ``expm(exponents[k] * Q)``, transposed or not, in ``cherry_expm_batched`` calls of at most
    ``_PAIR_EXPM_CHUNK`` exponents for S > 32."""
    lib = _lib.load()
    S = Q.shape[0]
    chunk = _PAIR_EXPM_CHUNK if S > 32 else 1 << 16
    dev = torch.device(device)
    out = torch.empty((len(exponents), S, S), dtype=torch.float64, device=dev)
    for i in range(0, len(exponents), chunk):
        part = expm_batched(Q, exponents[i: i + chunk], dev)
        if not transpose:
            out[i: i + chunk].copy_(part)
            continue
        with torch.cuda.device(dev):
            _lib.check(lib.cherry_tree_ll_transpose(_lib.ptr(part), part.shape[0], S, _lib.ptr(out[i: i + chunk]),
                                                    _lib.current_stream_ptr()), "cherry_tree_ll_transpose")
    return out


def _prune(nodes, max_depth, p_index, n_cats, P, obs, unit_cat, pi, S, c, device) -> np.ndarray:
    lib = _lib.load()
    n_units = obs.shape[1]
    dev = torch.device(device)
    with torch.cuda.device(dev):
        d_nodes = torch.from_numpy(nodes.view(np.uint8).reshape(-1)).to(dev)
        d_pidx = torch.from_numpy(np.ascontiguousarray(p_index, dtype=np.int32)).to(dev)
        d_obs = torch.from_numpy(np.ascontiguousarray(obs, dtype=np.uint8)).to(dev)
        d_cat = torch.from_numpy(np.ascontiguousarray(unit_cat, dtype=np.int32)).to(dev)
        d_pi = torch.from_numpy(np.array(pi, dtype=np.float64).reshape(-1)).to(dev)
        nbytes = int(lib.cherry_tree_ll_scratch_bytes(S, c, n_units, max_depth))
        scratch = torch.empty(max(8, nbytes), dtype=torch.uint8, device=dev)
        out = torch.empty(n_units, dtype=torch.float64, device=dev)
        _lib.check(
            lib.cherry_tree_log_likelihood(_lib.ptr(d_nodes), len(nodes), _lib.ptr(d_pidx), n_cats, _lib.ptr(P),
                                           _lib.ptr(d_obs), _lib.ptr(d_cat), _lib.ptr(d_pi), S, c, n_units,
                                           max_depth, _lib.ptr(scratch), nbytes, _lib.ptr(out),
                                           _lib.current_stream_ptr()),
            "cherry_tree_log_likelihood",
        )
        return out.cpu().numpy()


def dp_likelihood_computation(
    tree: Tree,
    msa: Dict[str, str],
    contact_map: Optional[np.ndarray],
    site_rates: List[float],
    amino_acids: List[str],
    pi_1: np.ndarray,
    Q_1: np.ndarray,
    fact_1=None,
    reversible_1: bool = False,
    device_1: str = "cuda",
    pi_2: Optional[np.ndarray] = None,
    Q_2: Optional[np.ndarray] = None,
    fact_2=None,
    reversible_2: Optional[bool] = None,
    device_2: Optional[str] = None,
    output_profiling_path: Optional[str] = None,
) -> Tuple[float, List[float]]:
    """Data log-likelihood and its per-site split, like the reference function.  ``fact_*``,
    ``reversible_*`` select among the reference's expm back ends, which all compute the same
    matrices; here they are accepted and ignored.  ``device_*`` other than a CUDA device name
    means "cuda"."""
    st_all = time.time()
    S = len(amino_acids)
    num_sites = len(site_rates)
    pairs = _contact_pairs(contact_map)
    in_contact = set(s for p in pairs for s in p)
    independent = [i for i in range(num_sites) if i not in in_contact]
    device = device_1 if str(device_1).startswith("cuda") else "cuda"

    nodes, lengths, leaves, max_depth = _tree_arrays(tree)
    enc = _encode_leaves(msa, leaves, amino_acids)
    lls = [0] * num_sites
    t_expm = t_dp = 0.0
    if independent:
        t0 = time.time()
        cats = sorted(set(site_rates))
        cat_of = {r: k for k, r in enumerate(cats)}
        exps = (lengths[:, None] * np.array(cats)[None, :]).reshape(-1)  # length * site_rate, as the reference
        P, p_index = _matrices(np.asarray(Q_1, dtype=np.float64), exps, device)
        t_expm += time.time() - t0
        t0 = time.time()
        res = _prune(nodes, max_depth, p_index, len(cats), P, enc[:, independent][:, :, None],
                     [cat_of[site_rates[i]] for i in independent], pi_1, S, 1, device)
        t_dp += time.time() - t0
        for k, i in enumerate(independent):
            lls[i] = float(res[k])
    if pairs:
        t0 = time.time()
        P, p_index = _matrices(np.asarray(Q_2, dtype=np.float64), lengths.copy(), device)
        t_expm += time.time() - t0
        t0 = time.time()
        obs = np.stack([enc[:, [i for i, _ in pairs]], enc[:, [j for _, j in pairs]]], axis=2)
        res = _prune(nodes, max_depth, p_index, 1, P, obs, [0] * len(pairs), pi_2, S, 2, device)
        t_dp += time.time() - t0
        for k, (i, j) in enumerate(pairs):
            lls[i] = float(res[k]) / 2.0
            lls[j] = float(res[k]) / 2.0
    if output_profiling_path is not None:
        with open(output_profiling_path, "w") as f:
            f.write(f"Time to populate_transition_mats: {t_expm}\nTime for dp: {t_dp}\n"
                    f"Total time: {time.time() - st_all}\n")
    return sum(lls), lls


_GRAD_CHUNK = 1 << 16  # exponents per cherry_fit_loss_grad call (one S x S gradient piece each)


class _SiteFamily:
    """One family's independent sites on the device, for the posterior pass: the node table, the leaf
    residues, the distinct ``branch length * site rate`` exponents and, on the host, which of them
    each (node, rate category) uses and the category of every site.  ``names`` are the nodes in the
    table's (post) order, ``lengths`` their branch lengths (the root's is not read) and ``rates`` the
    sorted distinct site rates; ``set_lengths`` rebuilds the exponents for new branch lengths."""

    def __init__(self, tree: Tree, msa: Dict[str, str], site_rates: List[float], amino_acids: List[str], device):
        nodes, lengths, leaves, self.max_depth, self.names = _tree_arrays(tree, with_names=True)
        self.S = len(amino_acids)
        if self.S > 32:
            raise ValueError(f"the likelihood gradient supports up to 32 states ({self.S} given)")
        cats = sorted(set(site_rates))
        cat_of = {r: k for k, r in enumerate(cats)}
        self.rates = np.array(cats, dtype=np.float64)
        self.set_lengths(lengths)
        self.unit_cat = np.array([cat_of[r] for r in site_rates], dtype=np.int32)
        self.n_nodes, self.n_cats, self.n_units = len(nodes), len(cats), len(site_rates)
        dev = torch.device(device)
        self.device = dev
        self.nodes = torch.from_numpy(nodes.view(np.uint8).reshape(-1)).to(dev)
        self.obs = torch.from_numpy(np.ascontiguousarray(_encode_leaves(msa, leaves, amino_acids))).to(dev)

    def set_lengths(self, lengths: np.ndarray) -> None:
        """New branch lengths [n_nodes] in ``names`` order: ``exponents`` and ``p_index`` from them."""
        self.lengths = np.asarray(lengths, dtype=np.float64)
        exps = (self.lengths[:, None] * self.rates[None, :]).reshape(-1)  # as dp_likelihood_computation
        self.exponents, inverse = np.unique(exps, return_inverse=True)
        self.p_index = np.ascontiguousarray(inverse, dtype=np.int32)

    def posterior(self, P: torch.Tensor, pi: torch.Tensor):
        """``cherry_tree_ll_posterior`` with the transposed matrices ``P`` of ``self.exponents`` and the root
        distribution ``pi`` (device fp64): (per-site log-likelihoods [n_units], W [n_exponents, S, S],
        root posterior sums [S])."""
        return self._run(P, pi, None)

    def edge_derivatives(self, P: torch.Tensor, pi: torch.Tensor, Q: torch.Tensor):
        """``cherry_tree_ll_edge_derivatives``: ``posterior``'s outputs and ``dtau`` [n_nodes, n_cats], the
        derivative of the log-likelihood with respect to ``length * rate`` of every (edge, rate category);
        ``Q`` [S, S] (device fp64) is the rate matrix of ``P``."""
        return self._run(P, pi, Q)

    def _run(self, P: torch.Tensor, pi: torch.Tensor, Q: Optional[torch.Tensor]):
        lib = _lib.load()
        S, n_m = self.S, len(self.exponents)
        with torch.cuda.device(self.device):
            sizes = (S, self.n_nodes, self.max_depth, self.n_cats, n_m, self.n_units, _lib.ptr(self.unit_cat))
            if Q is None:
                nbytes = int(lib.cherry_tree_ll_posterior_scratch_bytes(*sizes))
            else:
                nbytes = int(lib.cherry_tree_ll_edge_derivatives_scratch_bytes(*sizes))
            scratch = torch.empty(max(8, nbytes), dtype=torch.uint8, device=self.device)
            f64 = dict(dtype=torch.float64, device=self.device)
            ll = torch.empty(max(1, self.n_units), **f64)
            W = torch.empty((n_m, S, S), **f64)
            root = torch.empty(S, **f64)
            head = (_lib.ptr(self.nodes), self.n_nodes, self.max_depth, _lib.ptr(self.p_index), self.n_cats,
                    _lib.ptr(P), n_m, _lib.ptr(self.obs), _lib.ptr(self.unit_cat), _lib.ptr(pi))
            tail = (S, self.n_units, _lib.ptr(scratch), nbytes, _lib.ptr(ll), _lib.ptr(W), _lib.ptr(root))
            if Q is None:
                _lib.check(lib.cherry_tree_ll_posterior(*head, *tail, _lib.current_stream_ptr()),
                           "cherry_tree_ll_posterior")
                return ll[: self.n_units], W, root
            dtau = torch.empty((self.n_nodes, self.n_cats), **f64)
            Q = Q.contiguous()
            _lib.check(lib.cherry_tree_ll_edge_derivatives(*head, _lib.ptr(Q), *tail, _lib.ptr(dtau),
                                                           _lib.current_stream_ptr()),
                       "cherry_tree_ll_edge_derivatives")
        return ll[: self.n_units], W, root, dtau


def _exponent_union(fams: List[_SiteFamily]) -> Tuple[np.ndarray, List[np.ndarray]]:
    """The sorted distinct exponents of all ``fams``, and per family the rows of that union its own
    (sorted, distinct) exponents are."""
    union, inverse = np.unique(np.concatenate([f.exponents for f in fams]), return_inverse=True)
    offs = np.cumsum([0] + [len(f.exponents) for f in fams])
    return union, [inverse[offs[i]: offs[i + 1]] for i in range(len(fams))]


class _PairFamily:
    """One family's contacting pairs on the device, for the pair posterior pass: the node table, the leaf
    residues of both sites of every pair (``dp_likelihood_computation``'s pair order), the distinct branch
    lengths and, on the host, which of them each node uses."""

    def __init__(self, tree: Tree, msa: Dict[str, str], contact_map: Optional[np.ndarray], amino_acids: List[str],
                 device):
        nodes, lengths, leaves, self.max_depth = _tree_arrays(tree)
        self.S = len(amino_acids)
        if self.S > 32:
            raise ValueError(f"the pair likelihood gradient supports up to 32 states per site ({self.S} given)")
        self.pairs = _contact_pairs(contact_map)
        self.exponents, inverse = np.unique(lengths, return_inverse=True)
        self.p_index = np.ascontiguousarray(inverse, dtype=np.int32)
        self.nodes_host = nodes
        self.n_nodes, self.n_pairs = len(nodes), len(self.pairs)
        enc = _encode_leaves(msa, leaves, amino_acids)
        obs = np.stack([enc[:, [i for i, _ in self.pairs]], enc[:, [j for _, j in self.pairs]]], axis=2)
        dev = torch.device(device)
        self.device = dev
        self.obs = torch.from_numpy(np.ascontiguousarray(obs, dtype=np.uint8)).to(dev)

    def posterior(self, P: torch.Tensor, pi: torch.Tensor):
        """``cherry_tree_ll_pair_posterior`` with the (not transposed) matrices ``P`` of ``self.exponents`` and the
        root distribution ``pi`` [S^2] (device fp64): (per-pair log-likelihoods [n_pairs], W [n_exponents, S^2,
        S^2], root posterior sums [S^2])."""
        lib = _lib.load()
        Su, n_m = self.S * self.S, len(self.exponents)
        with torch.cuda.device(self.device):
            nbytes = int(lib.cherry_tree_ll_pair_posterior_scratch_bytes(self.S, self.n_nodes, self.max_depth,
                                                                        self.n_pairs, n_m))
            scratch = torch.empty(max(8, nbytes), dtype=torch.uint8, device=self.device)
            f64 = dict(dtype=torch.float64, device=self.device)
            ll = torch.empty(max(1, self.n_pairs), **f64)
            W = torch.empty((n_m, Su, Su), **f64)
            root = torch.empty(Su, **f64)
            _lib.check(
                lib.cherry_tree_ll_pair_posterior(self.nodes_host.ctypes.data, self.n_nodes, self.max_depth,
                                                  self.p_index.ctypes.data, _lib.ptr(P), n_m, _lib.ptr(self.obs),
                                                  _lib.ptr(pi), self.S, self.n_pairs, _lib.ptr(scratch), nbytes,
                                                  _lib.ptr(ll), _lib.ptr(W), _lib.ptr(root),
                                                  _lib.current_stream_ptr()),
                "cherry_tree_ll_pair_posterior",
            )
        return ll[: self.n_pairs], W, root


def _q_gradient(Q: torch.Tensor, t: torch.Tensor, W: torch.Tensor) -> torch.Tensor:
    """``d/dQ sum_m <W_m, log expm(t_m Q)>`` with ``W`` held fixed: minus the summed output of
    ``cherry_fit_loss_grad`` with ``C = W``, in calls of at most ``_GRAD_CHUNK`` exponents that share one
    set of buffers.  (``W_m / P_m = d log L / d P_m``, so this is the gradient of the log-likelihood.)"""
    import ctypes

    from ..estimation._engine import FitArgs

    lib = _lib.load()
    S, K = int(Q.shape[-1]), int(t.numel())
    dev = Q.device
    f64 = dict(dtype=torch.float64, device=dev)
    grad = torch.zeros((S, S), **f64)
    if K == 0:
        return grad
    # S > 32: at most CHERRY_LARGE_FIT_MAX_K exponents per call, and only dQ_part[0] (the sum over them) is written
    small = S <= 32
    kc = min(K, _GRAD_CHUNK if small else LARGE_MAX_K)
    nbytes = ctypes.c_size_t(0)
    _lib.check(lib.cherry_fit_workspace_bytes(S, kc, 1, ctypes.byref(nbytes)), "cherry_fit_workspace_bytes")
    ws = torch.empty(max(8, nbytes.value), dtype=torch.uint8, device=dev)
    dQ = torch.empty((kc if small else 1, S, S), **f64)
    lp = torch.empty(kc, **f64)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    Qc = Q.detach().contiguous()
    a = FitArgs()
    a.S, a.n_problems = S, 1
    a.Q, a.dQ_part, a.loss_part = _lib.ptr(Qc), _lib.ptr(dQ), _lib.ptr(lp)
    a.workspace, a.workspace_bytes, a.status_flag = _lib.ptr(ws), nbytes.value, _lib.ptr(flag)
    with torch.cuda.device(dev):
        for k0 in range(0, K, kc):
            k = min(kc, K - k0)
            a.K, a.t, a.C = k, _lib.ptr(t[k0:]), _lib.ptr(W[k0:])
            _lib.check(lib.cherry_fit_loss_grad(ctypes.byref(a), _lib.current_stream_ptr()), "cherry_fit_loss_grad")
            grad -= dQ[:k].sum(dim=0) if small else dQ[0]
    if int(flag.item()) != 0:
        raise _lib.CherryError(f"cherry_fit_loss_grad reported status {int(flag.item())}: exponent * rate beyond "
                               "the supported range")
    return grad


def log_likelihood_gradient(
    tree: Tree,
    msa: Dict[str, str],
    site_rates: List[float],
    amino_acids: List[str],
    pi: np.ndarray,
    Q: np.ndarray,
    device: str = "cuda",
) -> Tuple[float, List[float], np.ndarray, np.ndarray]:
    """Exact log-likelihood of one family of independent sites and its gradient:
    ``(ll, lls, d ll / d Q [S, S], d ll / d pi [S])``, every entry of ``Q`` and ``pi`` taken as a free
    variable.  ``lls`` equals ``dp_likelihood_computation``'s per-site values bit for bit.  Edge posteriors
    come from the inside/outside pass ``cherry_tree_ll_posterior``, the ``Q`` gradient from the fit's exact
    expm adjoint (``cherry_fit_loss_grad``) with the posteriors as counts.  S <= 32; no CPU fallback."""
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    fam = _SiteFamily(tree, msa, site_rates, amino_acids, dev)
    Q = np.asarray(Q, dtype=np.float64)
    P = _expm_transposed(Q, fam.exponents, dev)
    d_pi = torch.from_numpy(np.array(pi, dtype=np.float64).reshape(-1)).to(dev)
    ll, W, root = fam.posterior(P, d_pi)
    t = torch.from_numpy(fam.exponents).to(dev)
    gQ = _q_gradient(torch.from_numpy(Q).to(dev), t, W)
    lls = [float(x) for x in ll.cpu().numpy()]
    return sum(lls), lls, gQ.cpu().numpy(), (root / d_pi).cpu().numpy()


def branch_length_gradient(
    tree: Tree,
    msa: Dict[str, str],
    site_rates: List[float],
    amino_acids: List[str],
    pi: np.ndarray,
    Q: np.ndarray,
    device: str = "cuda",
) -> Tuple[float, List[float], Dict[str, float]]:
    """Exact log-likelihood of one family of independent sites and its derivative with respect to every
    branch length: ``(ll, lls, {child node: d ll / d length of the edge above it})``.  ``lls`` equals
    ``dp_likelihood_computation``'s per-site values bit for bit.  One pass of
    ``cherry_tree_ll_edge_derivatives`` gives ``d ll / d (length * rate_k)`` per edge and rate category;
    the length derivative is their sum weighted by the rates.  S <= 32; no CPU fallback."""
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    fam = _SiteFamily(tree, msa, site_rates, amino_acids, dev)
    Q = np.array(Q, dtype=np.float64, order="C")  # the kernel reads Q row-major (a DataFrame's array is not)
    P = _expm_transposed(Q, fam.exponents, dev)
    d_pi = torch.from_numpy(np.array(pi, dtype=np.float64).reshape(-1)).to(dev)
    ll, _, _, dtau = fam.edge_derivatives(P, d_pi, torch.from_numpy(Q).to(dev))
    dlen = dtau.cpu().numpy() @ fam.rates
    lls = [float(x) for x in ll.cpu().numpy()]
    return sum(lls), lls, {v: float(dlen[i]) for i, v in enumerate(fam.names[:-1])}


def pair_log_likelihood_gradient(
    tree: Tree,
    msa: Dict[str, str],
    contact_map: np.ndarray,
    amino_acids: List[str],
    pi_2: np.ndarray,
    Q_2: np.ndarray,
    device: str = "cuda",
) -> Tuple[float, List[float], np.ndarray, np.ndarray]:
    """Exact log-likelihood of the contacting pairs of one family under the co-evolution model ``(Q_2, pi_2)``
    on ``S^2`` pair states, and its gradient: ``(ll, lls_per_pair, d ll / d Q_2 [S^2, S^2], d ll / d pi_2
    [S^2])``.  Pairs are ``dp_likelihood_computation``'s (``i < j`` in ``np.where(contact_map == 1)`` order);
    the independent sites of the family are not included (``log_likelihood_gradient`` gives them).  Edge
    posteriors come from ``cherry_tree_ll_pair_posterior``, the ``Q_2`` gradient from the fit's exact expm
    adjoint with the posteriors as counts.  S <= 32 per site; no CPU fallback."""
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    fam = _PairFamily(tree, msa, contact_map, amino_acids, dev)
    Q = np.array(Q_2, dtype=np.float64)
    P = _expm_chunked(Q, fam.exponents, dev, transpose=False)
    d_pi = torch.from_numpy(np.array(pi_2, dtype=np.float64).reshape(-1)).to(dev)
    ll, W, root = fam.posterior(P, d_pi)
    del P
    gQ = _q_gradient(torch.from_numpy(Q).to(dev), torch.from_numpy(fam.exponents).to(dev), W)
    lls = [float(x) for x in ll.cpu().numpy()]
    return sum(lls), lls, gQ.cpu().numpy(), (root / d_pi).cpu().numpy()


@cached_parallel_computation(
    parallel_arg="families",
    exclude_args=[
        "device_1",
        "device_2",
        "num_processes",
        "use_cpp_implementation",
        "OMP_NUM_THREADS",
        "OPENBLAS_NUM_THREADS",
        "process_group",
    ],
    output_dirs=["output_likelihood_dir"],
    write_extra_log_files=True,
)
def compute_log_likelihoods(
    tree_dir: str,
    msa_dir: str,
    site_rates_dir: str,
    contact_map_dir: Optional[str],
    families: List[str],
    amino_acids: List[str],
    pi_1_path: str,
    Q_1_path: str,
    reversible_1: bool,
    device_1: str,
    pi_2_path: Optional[str],
    Q_2_path: Optional[str],
    reversible_2: Optional[bool],
    device_2: Optional[str],
    output_likelihood_dir: Optional[str],
    num_processes: int,
    use_cpp_implementation: bool = False,
    OMP_NUM_THREADS: Optional[int] = 1,
    OPENBLAS_NUM_THREADS: Optional[int] = 1,
    process_group=None,
) -> None:
    """Per family ``<output_likelihood_dir>/<family>.txt`` (total, then the per-site values) and
    ``<family>.profiling``.  Model validation as in the reference (:377-416).

    ``process_group`` (a torch.distributed group, one process per GPU): families are independent,
    so rank r evaluates ``families[r::world]`` -- the striping of the reference's worker processes
    (``get_process_args``, :565-575) -- and a barrier makes every file exist before any rank
    returns.  No data-path collective."""
    if use_cpp_implementation:
        raise NotImplementedError
    rank, world = 0, 1
    if process_group is not None:
        import torch.distributed as dist

        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        try:
            _compute_log_likelihoods_local(
                tree_dir, msa_dir, site_rates_dir, contact_map_dir, families[rank::world], amino_acids, pi_1_path,
                Q_1_path, reversible_1, device_1, pi_2_path, Q_2_path, reversible_2, device_2, output_likelihood_dir,
                write_total=rank == 0)
        finally:
            dist.barrier(process_group)
        return
    _compute_log_likelihoods_local(
        tree_dir, msa_dir, site_rates_dir, contact_map_dir, families, amino_acids, pi_1_path, Q_1_path, reversible_1,
        device_1, pi_2_path, Q_2_path, reversible_2, device_2, output_likelihood_dir, write_total=True)


def _compute_log_likelihoods_local(tree_dir, msa_dir, site_rates_dir, contact_map_dir, families, amino_acids,
                                   pi_1_path, Q_1_path, reversible_1, device_1, pi_2_path, Q_2_path, reversible_2,
                                   device_2, output_likelihood_dir, write_total: bool) -> None:
    os.makedirs(output_likelihood_dir, exist_ok=True)
    st = time.time()
    pi_1_df = read_probability_distribution(pi_1_path)
    Q_1_df = read_rate_matrix(Q_1_path)
    pi_2_df = read_probability_distribution(pi_2_path) if pi_2_path is not None else None
    Q_2_df = read_rate_matrix(Q_2_path) if Q_2_path is not None else None
    pairs_of_amino_acids = [a + b for a in amino_acids for b in amino_acids]
    if list(pi_1_df.index) != amino_acids:
        raise Exception(f"pi_1 index is:\n{list(pi_1_df.index)}\nbut expected amino acids:\n{amino_acids}")
    if pi_2_df is not None and list(pi_2_df.index) != pairs_of_amino_acids:
        raise Exception(
            f"pi_2 index is:\n{list(pi_2_df.index)}\nbut expected pairs of amino acids:\n{pairs_of_amino_acids}")
    if list(Q_1_df.index) != amino_acids:
        raise Exception(f"Q_1 index is:\n{list(Q_1_df.index)}\n\nbut expected amino acids:\n{amino_acids}")
    if list(Q_1_df.columns) != amino_acids:
        raise Exception(f"Q_1 columns are:\n{list(Q_1_df.columns)}\n\nbut expected amino acids:\n{amino_acids}")
    if Q_2_df is not None and list(Q_2_df.index) != pairs_of_amino_acids:
        raise Exception(
            f"Q_2 index is:\n{list(Q_2_df.index)}\n\nbut expected pairs of amino acids:\n{pairs_of_amino_acids}")
    if Q_2_df is not None and list(Q_2_df.columns) != pairs_of_amino_acids:
        raise Exception(
            f"Q_1 columns are:\n{list(Q_2_df.columns)}\n\nbut expected pairs of amino acids:\n{pairs_of_amino_acids}")
    for family in families:
        contact_map = (read_contact_map(os.path.join(contact_map_dir, family + ".txt"))
                       if contact_map_dir is not None else None)
        ll, lls = dp_likelihood_computation(
            tree=read_tree(os.path.join(tree_dir, family + ".txt")),
            msa=read_msa(os.path.join(msa_dir, family + ".txt")),
            contact_map=contact_map,
            site_rates=read_site_rates(os.path.join(site_rates_dir, family + ".txt")),
            amino_acids=amino_acids,
            pi_1=pi_1_df.to_numpy(), Q_1=Q_1_df.to_numpy(), reversible_1=reversible_1, device_1=device_1,
            pi_2=pi_2_df.to_numpy() if pi_2_df is not None else None,
            Q_2=Q_2_df.to_numpy() if Q_2_df is not None else None, reversible_2=reversible_2, device_2=device_2,
            output_profiling_path=os.path.join(output_likelihood_dir, family + ".profiling"),
        )
        write_log_likelihood((ll, lls), os.path.join(output_likelihood_dir, family + ".txt"))
    if write_total:
        with open(os.path.join(output_likelihood_dir, "profiling.txt"), "w") as f:
            f.write(f"Total time: {time.time() - st}\n")
