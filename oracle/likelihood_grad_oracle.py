"""CPU references for the exact derivatives of the tree log-likelihood (TEST INFRASTRUCTURE).

One numpy inside and outside pass in log space, per unit (an independent site on S states, or a pair of
contacting sites on S^2 states):
    h_v        inside vector (leaf: log of the observation vector, all-compatible for a character
               outside the alphabet; internal node: the sum of its children's messages),
    M_v(a)     = log sum_b P_v[a][b] exp(h_v(b)), the message of v to its parent,
    A_root     = log pi,  O_v = A_p + sum over the OTHER children j of p of M_j,
    A_v(b)     = log sum_a exp(O_v(a)) P_v[a][b],
so that d log L / d P_v[a][b] = exp(O_v(a) + h_v(b) - log L) =: G_v[a][b] (the outside vector times the
inside vector over the likelihood), and d log L / d pi = sum over units of exp(h_root - log L).  Then
    d log L / d Q   = sum over edges and rate categories of t r * expm_frechet(t r Q^T, G),
    d log L / d tau = sum_ab G[a][b] (dP/dtau)[a][b],  dP/dtau = expm_frechet(tau Q, Q),  tau = length * rate,
with P_v = scipy.linalg.expm(t r Q).  These routes use the Frechet derivative directly; the GPU path never
does (it goes through the edge posteriors W = P * G and the fit's expm adjoint, and dP/dtau = QP), so the
two are independent derivations.  The sum over siblings is recomputed per child (quadratic in the number
of children, which is fine at test sizes).
"""
from typing import Dict, List

import numpy as np


def _inside_outside(tree, obs: Dict[str, np.ndarray], P: Dict[str, np.ndarray], unit_cat, pi: np.ndarray):
    """The pass above for the units of ``obs`` (leaf -> observation vectors [n_units, Su]).  ``P``: per
    non-root node, its matrices per rate category [n_cats, Su, Su] with ``unit_cat`` [n_units] the category of
    each unit, or one matrix [Su, Su] shared by every unit with ``unit_cat`` None.  Returns ``(lls, R, edges)``:
    the per-unit log-likelihoods, the per-unit d log L_u / d pi [n_units, Su], and a generator of
    ``(v, G_v [n_units, Su, Su])`` over the non-root nodes, parents before children."""
    n, Su = next(iter(obs.values())).shape
    root = tree.root()
    post = tree.postorder_traversal()

    def lse_matvec(v, x, transpose):  # log sum_b P_v[u, a, b] exp(x[u, b]) (or P_v^T), per-unit maximum
        mx = np.max(x, axis=1, keepdims=True)
        mx[~np.isfinite(mx)] = 0.0
        with np.errstate(divide="ignore"):
            if unit_cat is None:
                return np.log(np.exp(x - mx) @ (P[v] if transpose else P[v].T)) + mx
            Pu = P[v][unit_cat]
            if transpose:
                Pu = np.transpose(Pu, (0, 2, 1))
            return np.log(np.einsum("uab,ub->ua", Pu, np.exp(x - mx))) + mx

    h, M = {}, {}
    for v in post:
        if tree.is_leaf(v):
            with np.errstate(divide="ignore"):
                h[v] = np.log(obs[v])
        else:
            h[v] = np.zeros((n, Su))
            for c, _ in tree.children(v):
                h[v] = h[v] + M[c]
        if v != root:
            M[v] = lse_matvec(v, h[v], False)
    mx = np.max(h[root], axis=1, keepdims=True)
    mx[~np.isfinite(mx)] = 0.0
    with np.errstate(divide="ignore"):
        lls = np.log(np.exp(h[root] - mx) @ pi) + mx[:, 0]
        A = {root: np.broadcast_to(np.log(pi), (n, Su)).copy()}

    def edges():
        for v in reversed(post):  # a parent before its children
            if v == root:
                continue
            p = tree.parent(v)[0]
            O = A[p].copy()
            for c, _ in tree.children(p):
                if c != v:
                    O = O + M[c]
            A[v] = lse_matvec(v, O, True)
            with np.errstate(over="ignore"):
                G = np.exp(O[:, :, None] + h[v][:, None, :] - lls[:, None, None])
            yield v, G

    return lls, np.exp(h[root] - lls[:, None]), edges()


def _site_units(tree, msa: Dict[str, str], site_rates: List[float], amino_acids: List[str], Q: np.ndarray):
    """Sites as units: the rate categories in sorted order, each site's category, per non-root node
    expm(length * rate * Q) per category [n_cats, S, S], and per leaf the observation vectors [n_sites, S]."""
    from scipy.linalg import expm

    S = len(amino_acids)
    aa = {a: i for i, a in enumerate(amino_acids)}
    cats = sorted(set(site_rates))
    site_cat = np.array([cats.index(r) for r in site_rates])
    root = tree.root()
    P, obs = {}, {}
    for v in tree.postorder_traversal():
        if v != root:
            P[v] = np.stack([expm(tree.parent(v)[1] * r * Q) for r in cats])
        if tree.is_leaf(v):
            obs[v] = np.zeros((len(site_rates), S))
            for i, ch in enumerate(msa[v]):
                if ch in aa:
                    obs[v][i, aa[ch]] = 1.0
                else:
                    obs[v][i] = 1.0
    return cats, site_cat, P, obs


def log_likelihood_gradient(tree, msa: Dict[str, str], site_rates: List[float], amino_acids: List[str],
                            pi: np.ndarray, Q: np.ndarray) -> dict:
    """{"ll", "lls" [n], "grad_Q" [S, S], "grad_pi" [S], "root" [S] (summed root posterior),
    "W": {branch length * rate: summed edge posterior [S, S] (parent state, child state)},
    "edge_mass": {node: [n] total posterior mass of the edge above it per unit (1 in exact arithmetic)}}
    for every site as an independent unit."""
    from scipy.linalg import expm_frechet

    Q = np.asarray(Q, dtype=np.float64)
    pi = np.asarray(pi, dtype=np.float64).reshape(-1)
    cats, site_cat, P, obs = _site_units(tree, msa, site_rates, amino_acids, Q)
    lls, R, edges = _inside_outside(tree, obs, P, site_cat, pi)
    grad_Q = np.zeros_like(Q)
    W: Dict[float, np.ndarray] = {}
    edge_mass = {}
    for v, G in edges:
        for k, r in enumerate(cats):
            Gk = G[site_cat == k].sum(axis=0)
            t = tree.parent(v)[1] * r
            grad_Q += t * expm_frechet(t * Q.T, Gk, compute_expm=False)
            W[t] = W.get(t, 0.0) + P[v][k] * Gk
        edge_mass[v] = np.einsum("uab,uab->u", P[v][site_cat], G)
    return {"ll": float(lls.sum()), "lls": lls, "grad_Q": grad_Q, "grad_pi": R.sum(axis=0),
            "root": (R * pi[None, :]).sum(axis=0), "W": W, "edge_mass": edge_mass}


def branch_length_gradient(tree, msa: Dict[str, str], site_rates: List[float], amino_acids: List[str],
                           pi: np.ndarray, Q: np.ndarray) -> dict:
    """{"ll", "lls" [n], "dtau": {node: [n_cats] d log L / d (length * rate_k) of the edge above it},
    "grad_length": {node: d log L / d length of the edge above it}} for every site as an independent unit,
    categories in sorted rate order."""
    from scipy.linalg import expm_frechet

    Q = np.asarray(Q, dtype=np.float64)
    pi = np.asarray(pi, dtype=np.float64).reshape(-1)
    cats, site_cat, P, obs = _site_units(tree, msa, site_rates, amino_acids, Q)
    lls, _, edges = _inside_outside(tree, obs, P, site_cat, pi)
    dtau, grad_length = {}, {}
    for v, G in edges:
        length = tree.parent(v)[1]
        d = np.zeros(len(cats))
        for k, r in enumerate(cats):
            dP = expm_frechet(length * r * Q, Q, compute_expm=False)
            d[k] = np.sum(G[site_cat == k].sum(axis=0) * dP)
        dtau[v] = d
        grad_length[v] = float(np.dot(d, cats))
    return {"ll": float(lls.sum()), "lls": lls, "dtau": dtau, "grad_length": grad_length}


def pair_log_likelihood_gradient(tree, msa: Dict[str, str], contact_map: np.ndarray, amino_acids: List[str],
                                 pi_2: np.ndarray, Q_2: np.ndarray) -> dict:
    """Log-likelihood and gradient of the contacting pairs of ``contact_map`` (``i < j`` in ``np.where`` order)
    as units on S^2 states (state S*a + b), with no rate categories: the observation vector of a leaf is the
    product of the two sites' compatibility sets, P_v = scipy.linalg.expm(t Q_2).  Returns
    {"ll", "lls" [n_pairs], "grad_Q" [S^2, S^2], "grad_pi" [S^2], "root" [S^2],
     "W": {branch length: summed edge posterior [S^2, S^2]}}."""
    from scipy.linalg import expm, expm_frechet

    S = len(amino_acids)
    Su = S * S
    aa = {a: i for i, a in enumerate(amino_acids)}
    ii, jj = np.where(np.asarray(contact_map) == 1)
    pairs = [(int(i), int(j)) for i, j in zip(ii, jj) if i < j]
    Q = np.asarray(Q_2, dtype=np.float64)
    pi = np.asarray(pi_2, dtype=np.float64).reshape(-1)
    root = tree.root()
    P = {v: expm(tree.parent(v)[1] * Q) for v in tree.postorder_traversal() if v != root}

    def site_set(ch):
        x = np.zeros(S)
        if ch in aa:
            x[aa[ch]] = 1.0
        else:
            x[:] = 1.0
        return x

    obs = {v: np.stack([np.outer(site_set(msa[v][i]), site_set(msa[v][j])).reshape(-1) for i, j in pairs])
           if pairs else np.zeros((0, Su)) for v in tree.leaves()}
    lls, R, edges = _inside_outside(tree, obs, P, None, pi)
    grad_Q = np.zeros((Su, Su))
    W: Dict[float, np.ndarray] = {}
    for v, G in edges:
        G = G.sum(axis=0)
        t = tree.parent(v)[1]
        grad_Q += t * expm_frechet(t * Q.T, G, compute_expm=False)
        W[t] = W.get(t, 0.0) + P[v] * G
    return {"ll": float(lls.sum()), "lls": lls, "grad_Q": grad_Q, "grad_pi": R.sum(axis=0),
            "root": (R * pi[None, :]).sum(axis=0), "W": W}
