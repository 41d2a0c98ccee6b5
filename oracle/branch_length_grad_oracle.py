"""CPU reference for the exact derivative of the tree log-likelihood of independent sites with respect to
every branch length (TEST INFRASTRUCTURE).

The same numpy inside and outside passes as ``oracle/likelihood_grad_oracle.py`` (per unit, in log space):
G_v[a][b] = exp(O_v(a) + h_v(b) - log L) = d log L / d P_v[a][b] for the edge above v, and then
    d log L / d tau = sum_ab G_v[a][b] (dP_v / dtau)[a][b],  tau = length * rate,
with dP/dtau = scipy.linalg.expm_frechet(tau Q, Q), the Frechet derivative of expm at tau Q in the direction
Q.  The GPU uses dP/dtau = QP instead, so the two are independent derivations.
"""
from typing import Dict, List

import numpy as np


def branch_length_gradient(tree, msa: Dict[str, str], site_rates: List[float], amino_acids: List[str],
                           pi: np.ndarray, Q: np.ndarray) -> dict:
    """{"ll", "lls" [n], "dtau": {node: [n_cats] d log L / d (length * rate_k) of the edge above it},
    "grad_length": {node: d log L / d length of the edge above it}} for every site as an independent unit,
    categories in sorted rate order.  The same inside/outside pass as ``log_likelihood_gradient``, with
    d log L / d tau = sum_ab G[a][b] (dP/dtau)[a][b] and dP/dtau = scipy.linalg.expm_frechet(tau Q, Q),
    the Frechet derivative of expm at tau Q in the direction Q (the GPU uses QP instead)."""
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
    P = {v: np.stack([expm(tree.parent(v)[1] * r * Q) for r in cats]) for v in post if v != root}

    def lse_matvec(Pu, x):
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
    dtau, grad_length = {}, {}
    for v in reversed(post):
        if v == root:
            continue
        p, length = tree.parent(v)
        O = A[p].copy()
        for c, _ in tree.children(p):
            if c != v:
                O = O + M[c]
        A[v] = lse_matvec(np.transpose(P[v][site_cat], (0, 2, 1)), O)
        with np.errstate(over="ignore"):
            G = np.exp(O[:, :, None] + h[v][:, None, :] - lls[:, None, None])
        d = np.zeros(len(cats))
        for k, r in enumerate(cats):
            dP = expm_frechet(length * r * Q, Q, compute_expm=False)
            d[k] = np.sum(G[site_cat == k].sum(axis=0) * dP)
        dtau[v] = d
        grad_length[v] = float(np.dot(d, cats))
    return {"ll": float(lls.sum()), "lls": lls, "dtau": dtau, "grad_length": grad_length}
