"""CPU reference for the exact gradient of the tree log-likelihood of independent sites (TEST INFRASTRUCTURE).

Numpy inside and outside passes in log space, per unit (site):
    h_v        inside vector (leaf: log of the observation vector, all-compatible for a character
               outside the alphabet; internal node: the sum of its children's messages),
    M_v(a)     = log sum_b P_v[a][b] exp(h_v(b)), the message of v to its parent,
    A_root     = log pi,  O_v = A_p + sum over the OTHER children j of p of M_j,
    A_v(b)     = log sum_a exp(O_v(a)) P_v[a][b],
so that d log L / d P_v[a][b] = exp(O_v(a) + h_v(b) - log L) =: G_v[a][b] (the outside vector times the
inside vector over the likelihood).  Then
    d log L / d Q  = sum over edges and rate categories of t r * expm_frechet(t r Q^T, G),
    d log L / d pi = sum over units of exp(h_root - log L),
with P_v = scipy.linalg.expm(t r Q).  This route uses the Frechet derivative directly; the GPU path never
does (it goes through the edge posteriors W = P * G and the fit's expm adjoint), so the two are
independent derivations.  The sum over siblings is recomputed per child (quadratic in the number of
children, which is fine at test sizes).
"""
from typing import Dict, List

import numpy as np


def log_likelihood_gradient(tree, msa: Dict[str, str], site_rates: List[float], amino_acids: List[str],
                            pi: np.ndarray, Q: np.ndarray) -> dict:
    """{"ll", "lls" [n], "grad_Q" [S, S], "grad_pi" [S], "root" [S] (summed root posterior),
    "W": {branch length * rate: summed edge posterior [S, S] (parent state, child state)},
    "edge_mass": {node: [n] total posterior mass of the edge above it per unit (1 in exact arithmetic)}}
    for every site as an independent unit."""
    from scipy.linalg import expm, expm_frechet

    S = len(amino_acids)
    aa = {a: i for i, a in enumerate(amino_acids)}
    n = len(site_rates)
    Q = np.asarray(Q, dtype=np.float64)
    pi = np.asarray(pi, dtype=np.float64).reshape(-1)
    cats = sorted(set(site_rates))
    site_cat = np.array([cats.index(r) for r in site_rates])
    root = tree.root()
    post = tree.postorder_traversal()
    P = {}  # node -> [n_cats, S, S]
    for v in post:
        if v != root:
            P[v] = np.stack([expm(tree.parent(v)[1] * r * Q) for r in cats])

    def lse_matvec(Pu, x):  # log sum_b Pu[u, a, b] exp(x[u, b]), scaled by the per-unit maximum
        mx = np.max(x, axis=1, keepdims=True)
        mx[~np.isfinite(mx)] = 0.0
        with np.errstate(divide="ignore"):
            return np.log(np.einsum("uab,ub->ua", Pu, np.exp(x - mx))) + mx

    h, M = {}, {}
    for v in post:
        if tree.is_leaf(v):
            obs = np.zeros((n, S))
            for i, ch in enumerate(msa[v]):
                if ch in aa:
                    obs[i, aa[ch]] = 1.0
                else:
                    obs[i] = 1.0
            with np.errstate(divide="ignore"):
                h[v] = np.log(obs)
        else:
            h[v] = np.zeros((n, S))
            for c, _ in tree.children(v):
                h[v] = h[v] + M[c]
        if v != root:
            M[v] = lse_matvec(P[v][site_cat], h[v])
    mx = np.max(h[root], axis=1, keepdims=True)
    lls = np.log(np.exp(h[root] - mx) @ pi) + mx[:, 0]
    with np.errstate(divide="ignore"):
        A = {root: np.broadcast_to(np.log(pi), (n, S)).copy()}
    grad_Q = np.zeros((S, S))
    W: Dict[float, np.ndarray] = {}
    edge_mass = {}
    for v in reversed(post):  # a parent before its children
        if v == root:
            continue
        p = tree.parent(v)[0]
        O = A[p].copy()
        for c, _ in tree.children(p):
            if c != v:
                O = O + M[c]
        Pt = np.transpose(P[v][site_cat], (0, 2, 1))
        A[v] = lse_matvec(Pt, O)
        with np.errstate(over="ignore"):
            G = np.exp(O[:, :, None] + h[v][:, None, :] - lls[:, None, None])  # d log L_u / d P_v[a][b]
        for k, r in enumerate(cats):
            Gk = G[site_cat == k].sum(axis=0)
            t = tree.parent(v)[1] * r
            grad_Q += t * expm_frechet(t * Q.T, Gk, compute_expm=False)
            W[t] = W.get(t, 0.0) + P[v][k] * Gk
        edge_mass[v] = np.einsum("uab,uab->u", P[v][site_cat], G)
    R = np.exp(h[root] - lls[:, None])  # d log L_u / d pi
    return {"ll": float(lls.sum()), "lls": lls, "grad_Q": grad_Q, "grad_pi": R.sum(axis=0),
            "root": (R * pi[None, :]).sum(axis=0), "W": W, "edge_mass": edge_mass}
