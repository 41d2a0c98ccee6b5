"""CPU reference for the exact gradient of the log-likelihood of contacting pairs (TEST INFRASTRUCTURE).

The inside and outside passes of ``likelihood_grad_oracle.log_likelihood_gradient`` for pairs of contacting
sites as units on S^2 states (state S*a + b), with no rate categories, and the gradient through
``scipy.linalg.expm_frechet`` -- never through the edge posteriors W and the fit's expm adjoint that the GPU
path uses, so the two routes are independent derivations.
"""
from typing import Dict, List

import numpy as np


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
    n = len(pairs)
    Q = np.asarray(Q_2, dtype=np.float64)
    pi = np.asarray(pi_2, dtype=np.float64).reshape(-1)
    root = tree.root()
    post = tree.postorder_traversal()
    P = {v: expm(tree.parent(v)[1] * Q) for v in post if v != root}

    def site_set(ch):
        x = np.zeros(S)
        if ch in aa:
            x[aa[ch]] = 1.0
        else:
            x[:] = 1.0
        return x

    def lse_matvec(Pm, x):  # log sum_b Pm[a, b] exp(x[u, b]), scaled by the per-unit maximum
        mx = np.max(x, axis=1, keepdims=True)
        mx[~np.isfinite(mx)] = 0.0
        with np.errstate(divide="ignore"):
            return np.log(np.exp(x - mx) @ Pm.T) + mx

    h, M = {}, {}
    for v in post:
        if tree.is_leaf(v):
            obs = np.stack([np.outer(site_set(msa[v][i]), site_set(msa[v][j])).reshape(-1) for i, j in pairs]
                           ) if n else np.zeros((0, Su))
            with np.errstate(divide="ignore"):
                h[v] = np.log(obs)
        else:
            h[v] = np.zeros((n, Su))
            for c, _ in tree.children(v):
                h[v] = h[v] + M[c]
        if v != root:
            M[v] = lse_matvec(P[v], h[v])
    mx = np.max(h[root], axis=1, keepdims=True)
    mx[~np.isfinite(mx)] = 0.0
    with np.errstate(divide="ignore"):
        lls = np.log(np.exp(h[root] - mx) @ pi) + mx[:, 0]
        A = {root: np.broadcast_to(np.log(pi), (n, Su)).copy()}
    grad_Q = np.zeros((Su, Su))
    W: Dict[float, np.ndarray] = {}
    for v in reversed(post):  # a parent before its children
        if v == root:
            continue
        p, t = tree.parent(v)
        O = A[p].copy()
        for c, _ in tree.children(p):
            if c != v:
                O = O + M[c]
        A[v] = lse_matvec(P[v].T, O)
        with np.errstate(over="ignore"):
            G = np.exp(O[:, :, None] + h[v][:, None, :] - lls[:, None, None]).sum(axis=0)  # d log L / d P_v
        grad_Q += t * expm_frechet(t * Q.T, G, compute_expm=False)
        W[t] = W.get(t, 0.0) + P[v] * G
    R = np.exp(h[root] - lls[:, None])  # d log L_u / d pi
    return {"ll": float(lls.sum()), "lls": lls, "grad_Q": grad_Q, "grad_pi": R.sum(axis=0),
            "root": (R * pi[None, :]).sum(axis=0), "W": W}
