"""Extended-precision and complex-step references of the likelihood kernels (shared by the likelihood coverage
tests), and thin calls of the kernels through the package's own Python entry points.

Everything works on the kernels' node table (``evaluation._likelihood._tree_arrays``: post-order, the root last,
``depth``, ``flags`` bit 0 = leaf, bit 1 = first child, ``obs_row``), so the references see exactly the tree the
kernel sees.  Matrices are given as fp64 ``P[m][a][b]`` (parent state a, child state b, NOT transposed); the
long-double pass converts exactly those entries, so what it measures is the kernel's own arithmetic.
"""
import numpy as np

U64 = 2.0 ** -53
LD = np.longdouble
# exp(x) is 0 in fp64 below x = -745: the largest |v - max v| whose rounding can still reach a summed term
EXP_RANGE = 745


def tree_links(nodes):
    """(parent [n_nodes] with -1 at the root, children [n_nodes] lists in tree order) from a post-order table."""
    n = len(nodes)
    parent = np.full(n, -1, dtype=np.int64)
    children = [[] for _ in range(n)]
    pending = {}
    for v in range(n):
        d = int(nodes["depth"][v])
        if not nodes["flags"][v] & 1:
            children[v] = pending.pop(d + 1)
            for c in children[v]:
                parent[c] = v
        pending.setdefault(d, []).append(v)
    assert list(pending) == [0] and pending[0] == [n - 1]
    return parent, children


def obs_vectors(obs, S, c):
    """[n_leaves, n_units, c] residue bytes (S = any state) -> 0/1 observation vectors [n_leaves, n_units, S^c]."""
    one = np.zeros(obs.shape + (S,))
    idx = obs.astype(np.int64)
    known = idx < S
    one[known, idx[known]] = 1.0
    one[~known] = 1.0
    if c == 1:
        return one[..., 0, :]
    return (one[..., 0, :, None] * one[..., 1, None, :]).reshape(obs.shape[:2] + (S * S,))


def _lse_rows(x, M):
    """log(exp(x - mx) @ M) + mx per row, the per-unit maximum of the kernels (-inf rows stay -inf)."""
    mx = np.max(x, axis=1, keepdims=True)
    mx[~np.isfinite(mx)] = 0
    with np.errstate(divide="ignore", under="ignore"):
        return np.log(np.exp(x - mx) @ M) + mx


def _finite_max_abs(x):
    f = np.abs(x[np.isfinite(x)])
    return float(f.max()) if f.size else 0.0


def inside_outside_ld(nodes, p_index, P, obs, unit_cat, pi, S, c, Q=None, posterior=True):
    """The inside/outside pass in np.longdouble on the fp64 inputs of the kernels.

    p_index [n_nodes, n_cats] (or [n_nodes] for one category), P [n_m, Su, Su] fp64 not transposed,
    obs [n_leaves, n_units, c] uint8, unit_cat [n_units], pi [Su], Q [Su, Su] (for dtau) or None.
    Returns a dict with ``ll`` [n_units] and ``bound`` [n_units], the a-priori bound on the kernels' error of
    ``ll`` (tests/test_gpu_likelihood_coverage.py derives it); with ``posterior`` also ``W`` [n_m, Su, Su],
    ``root`` [Su], ``dtau`` [n_nodes, n_cats] and ``dmass`` [n_nodes, n_cats] (the sum of the absolute values of
    the terms of dtau in the kernel's factored form sum_s (Q^T e_O)(s) (P e_h)(s): sum_ab G (|Q| P))."""
    n_nodes = len(nodes)
    p_index = np.asarray(p_index).reshape(n_nodes, -1)
    n_cats = p_index.shape[1]
    unit_cat = np.asarray(unit_cat, dtype=np.int64)
    n_units = len(unit_cat)
    Su = S ** c
    PL = np.asarray(P, dtype=np.float64).astype(LD)
    piL = np.asarray(pi, dtype=np.float64).astype(LD)
    ov = obs_vectors(obs, S, c).astype(LD)
    parent, children = tree_links(nodes)
    root = n_nodes - 1
    by_cat = [np.flatnonzero(unit_cat == k) for k in range(n_cats)]

    def matvec(v, x, transpose):
        out = np.empty_like(x)
        for k, us in enumerate(by_cat):
            if len(us):
                M = PL[p_index[v, k]]
                out[us] = _lse_rows(x[us], M if transpose else M.T)
        return out

    h, M = [None] * n_nodes, [None] * n_nodes
    scale = np.zeros(n_units)  # per unit: the largest finite |value| met
    for v in range(n_nodes):
        if nodes["flags"][v] & 1:
            with np.errstate(divide="ignore"):
                h[v] = np.log(ov[nodes["obs_row"][v]])
        else:
            h[v] = sum(M[ch] for ch in children[v])
        if v != root:
            M[v] = matvec(v, h[v], False)
    with np.errstate(divide="ignore", under="ignore"):
        mx = np.max(h[root], axis=1, keepdims=True)
        mx[~np.isfinite(mx)] = 0
        ll = np.log(np.exp(h[root] - mx) @ piL) + mx[:, 0]
    out = {"ll": ll}
    A, O = {root: np.broadcast_to(np.log(piL), (n_units, Su)).copy()}, {}
    if posterior:
        W = np.zeros((len(P), Su, Su), dtype=LD)
        dtau = np.zeros((n_nodes, n_cats), dtype=LD)
        dmass = np.zeros((n_nodes, n_cats), dtype=LD)
        QL = None if Q is None else np.asarray(Q, dtype=np.float64).astype(LD)
        for v in range(n_nodes - 2, -1, -1):  # a parent before its children
            p = parent[v]
            o = A[p] + sum((M[ch] for ch in children[p] if ch != v), np.zeros((n_units, Su), dtype=LD))
            O[v] = o
            if not nodes["flags"][v] & 1:
                A[v] = matvec(v, o, True)
            mo = np.max(o, axis=1, keepdims=True)
            mo[~np.isfinite(mo)] = 0
            mh = np.max(h[v], axis=1, keepdims=True)
            mh[~np.isfinite(mh)] = 0
            with np.errstate(under="ignore"):
                U = np.exp(o - mo)
                V = np.exp(h[v] - mh) * np.exp(mo + mh - ll[:, None])
            for k, us in enumerate(by_cat):
                if not len(us):
                    continue
                G = U[us].T @ V[us]  # sum over the units of d log L_u / d P[a][b]
                m = p_index[v, k]
                W[m] += PL[m] * G
                if QL is not None:
                    dtau[v, k] = np.sum(G * (QL @ PL[m]))
                    dmass[v, k] = np.sum(G * (np.abs(QL) @ PL[m]))
        with np.errstate(under="ignore"):
            out["root"] = (np.exp(h[root] - ll[:, None]) * piL[None, :]).sum(axis=0)
        out.update(W=W, dtau=dtau, dmass=dmass)
    for v in range(n_nodes):
        for x in (h[v], M[v], A.get(v), O.get(v)):
            if x is not None:
                scale = np.maximum(scale, [_finite_max_abs(r) for r in x])
    # per node: Su products and sums, exp/log/rounding of the shift (a few ulp), the shifted exponent's rounding
    # (at most EXP_RANGE ulp) and the rounding of three additions of values up to `scale`
    out["bound"] = n_nodes * U64 * (Su + 8 + EXP_RANGE + 3 * np.maximum(scale, np.abs(ll.astype(np.float64))))
    return out


# ------------------------------------------------------------------ complex step (complex128, torch.matrix_exp)

def complex_ll(nodes, exps, n_cats, obs, unit_cat, pi, Q, S, c):
    """Total log-likelihood in complex128: P = torch.matrix_exp(exps[v, k] Q) per (non-root node, category).
    ``exps`` [n_nodes, n_cats] complex, ``Q`` [Su, Su] complex, ``pi`` [Su] complex (numpy).  Analytic in every
    input, so Im(f(x + i h e)) / h is the directional derivative to within O(h^2)."""
    import torch

    n_nodes = len(nodes)
    _, children = tree_links(nodes)
    unit_cat = np.asarray(unit_cat)
    Qt = torch.from_numpy(np.asarray(Q, dtype=np.complex128))
    ov = torch.from_numpy(obs_vectors(obs, S, c).astype(np.complex128))
    t = torch.from_numpy(np.asarray(exps, dtype=np.complex128).reshape(n_nodes, n_cats))
    P = torch.matrix_exp(t[:, :, None, None] * Qt)  # [n_nodes, n_cats, Su, Su]
    cat = torch.from_numpy(unit_cat.astype(np.int64))
    # linear-space messages with a real per-unit scale (log(z / s) + log s = log z for any real s > 0)
    lin, logs = [None] * n_nodes, [None] * n_nodes
    for v in range(n_nodes):
        if nodes["flags"][v] & 1:
            x, ls = ov[nodes["obs_row"][v]], torch.zeros(len(unit_cat), dtype=torch.float64)
        else:
            x, ls = None, torch.zeros(len(unit_cat), dtype=torch.float64)
            for ch in children[v]:
                x = lin[ch] if x is None else x * lin[ch]
                ls = ls + logs[ch]
        if v == n_nodes - 1:
            Pi = torch.from_numpy(np.asarray(pi, dtype=np.complex128))
            return complex((torch.log(x @ Pi) + ls).sum())
        m = torch.einsum("uab,ub->ua", P[v][cat], x)
        s = m.real.abs().amax(dim=1).clamp_min(1e-300)
        lin[v], logs[v] = m / s[:, None], ls + torch.log(s)


def complex_step(f, x, direction, h=1e-30):
    """d f(x + s direction) / ds at s = 0 by complex step."""
    return f(np.asarray(x, dtype=np.complex128) + 1j * h * np.asarray(direction)).imag / h


# ------------------------------------------------------------------ the kernels, through the package's entry points

def gpu_forward(nodes, max_depth, p_index, P, obs, unit_cat, pi, S, c):
    """cherry_tree_log_likelihood (evaluation._likelihood._prune) on fp64 P [n_m, Su, Su] (not transposed)."""
    import torch

    from cherryml_b200.evaluation._likelihood import _prune

    p_index = np.asarray(p_index, dtype=np.int32).reshape(len(nodes), -1)
    Pt = torch.from_numpy(np.ascontiguousarray(np.swapaxes(P, 1, 2))).cuda()
    return _prune(nodes, max_depth, p_index, p_index.shape[1], Pt, obs, unit_cat, pi, S, c, "cuda")


def site_family(nodes, max_depth, p_index, n_m, obs, unit_cat, S):
    """An ``evaluation._likelihood._SiteFamily`` over a given node table, matrix index and leaf residues."""
    import torch

    from cherryml_b200.evaluation._likelihood import _SiteFamily

    fam = object.__new__(_SiteFamily)
    fam.S, fam.max_depth = S, int(max_depth)
    fam.p_index = np.ascontiguousarray(np.asarray(p_index, dtype=np.int32).reshape(len(nodes), -1))
    fam.unit_cat = np.ascontiguousarray(unit_cat, dtype=np.int32)
    fam.n_nodes, fam.n_cats, fam.n_units = len(nodes), fam.p_index.shape[1], len(unit_cat)
    fam.exponents = np.zeros(n_m)  # only its length is read
    fam.device = torch.device("cuda")
    fam.nodes = torch.from_numpy(nodes.view(np.uint8).reshape(-1)).cuda()
    fam.obs = torch.from_numpy(np.ascontiguousarray(obs[:, :, 0], dtype=np.uint8)).cuda()
    return fam


def pair_family(nodes, max_depth, p_index, n_m, obs, S):
    """An ``evaluation._likelihood._PairFamily`` over a given node table, matrix index and leaf residue pairs."""
    import torch

    from cherryml_b200.evaluation._likelihood import _PairFamily

    fam = object.__new__(_PairFamily)
    fam.S, fam.max_depth = S, int(max_depth)
    fam.p_index = np.ascontiguousarray(np.asarray(p_index, dtype=np.int32).reshape(-1))
    fam.nodes_host = nodes
    fam.n_nodes, fam.n_pairs = len(nodes), obs.shape[1]
    fam.exponents = np.zeros(n_m)
    fam.device = torch.device("cuda")
    fam.obs = torch.from_numpy(np.ascontiguousarray(obs, dtype=np.uint8)).cuda()
    return fam
