"""Likelihood kernels (likelihood.cu, pair_posterior.cu) against extended-precision references, at every launch
shape the hosts can select from the sizes: the forward pass (tree_ll_kernel), the site posterior and edge
derivatives (tree_ll_post_*), the pair posterior (pair_*_kernel) and the matrix transpose.

Isolation from expm.  Each kernel gets fp64 matrices P built here (scipy expm of a dense reversible Q at zero,
short and long exponents, clipped at 0; for pairs the Kronecker product expm(t Q1) (x) expm(t Q2), which is
expm(t (Q1 (+) Q2)) exactly, so Su = 1024 needs no 1024 x 1024 expm).  The reference (tests/_ll_precise.py)
prunes in np.longdouble with exactly those fp64 entries, so any difference is the kernel's own arithmetic.

Tolerances, a priori (u = 2^-53, x87 long double carries 11 more bits, so the reference's error is negligible):
- log-likelihood, absolute: every message is log(sum of Su non-negative terms P[s][k] exp(v_k - max v)).  With
  relative errors of at most u per product, exp and log, and (Su - 1) u for the sequential or tensor-core sum,
  the sum carries (Su + 2) u relative error; the rounded shift v_k - max v adds u |v_k - max v| <= 745 u relative
  to a term that is not flushed to zero (exp underflows below -745); the log and the additions of the shift, of
  the message into its parent's running sum and of the maximum add u |value| each.  An error E on every entry
  of a child's inside vector is an error of at most E on its message (a relative error E on every term), so the
  errors of the nodes add up: |d log L_u| <= n_nodes u (Su + 8 + 745 + 3 V_u) =: T_u, V_u the largest finite
  |value| (inside, outside, message, log L_u) of unit u.  inside_outside_ld computes T_u from its own values.
- edge posteriors W and root posteriors, relative per entry: a term of W is exp(O(a) - max O) exp(h(b) - max h)
  exp(max O + max h - log L) P[a][b]; O carries the forward and the outside pass's errors (2 T), h and log L one
  T each, the exps and products a few u, and the sums over units, CTAs and edges add (n_units + n_cats n_nodes) u
  (all terms non-negative).  So rtol_W = 5 max T_u + (n_units + n_cats n_nodes + 800) u; entries below 1e-290
  (near fp64 underflow) are compared absolutely at that level.
- dtau, absolute: the kernel sums (Q^T e_O)(s) (P e_h)(s) over s, and Q^T e_O sums terms of both signs (the rows
  of Q sum to zero).  Every product Q[a][s] e_O(a) P[s][b] e_h(b) is within the relative error above, so
  |d dtau| <= (5 max T_u + (2 S + n_units + 800) u) * sum_ab G[a][b] (|Q| P)[a][b] (the reference's dmass),
  the sum of the absolute values of those products.
- gradients end to end (log_likelihood_gradient, branch_length_gradient, pair_log_likelihood_gradient, each
  through the package's expm and the fit's adjoint): complex step in complex128 (h = 1e-30, torch.matrix_exp),
  whose error is O(h^2) plus the rounding of complex128 expm and pruning, a few hundred u relative; the tests
  use the 1e-9 relative tolerance of the existing gradient tests.  At Su = 1024 the reference is
  oracle.likelihood_grad_oracle (scipy expm_frechet), also at 1e-9.
- invariants, exact in real arithmetic and checked at the W tolerance: sum_m sum_ab W_m = n_units (n_nodes - 1),
  the root posterior sums to n_units; and bitwise: two calls give the same bits, the posterior pass's log L
  equals the forward pass's, the edge-derivative pass's W equals the posterior pass's, the transpose equals
  np.swapaxes.
"""
import numpy as np
import pytest

from cherryml_b200 import _lib
from cherryml_b200.io import Tree
from tests._ll_cases import AA, DNA, _caterpillar, _random_reversible, _random_tree
from tests._ll_precise import (U64, complex_ll, complex_step, gpu_forward, inside_outside_ld, pair_family,
                               site_family)

# ------------------------------------------------------------------ the host's path selection, mirrored
# likelihood.cu: kLlBatch, the 227 KB dynamic shared memory limit, G = max(1, 256 / Su)
LL_BATCH, SMEM_LIMIT = 16, 227 * 1024
# pair_posterior.cu: kPairSpAlign, kPairNpAlign, kNodeTN, kEdgeT, kPrepThreads, kPrepPerThread
PAIR_SP_ALIGN, PAIR_NP_ALIGN, NODE_TN, EDGE_T, PREP_THREADS, PREP_PER_THREAD = 64, 16, 128, 64, 128, 8
# markov_chain.LARGE_MAX_K = CHERRY_LARGE_FIT_MAX_K: exponents per cherry_fit_loss_grad call for S > 32
LARGE_MAX_K = 811


def fwd_layout(S, c):
    """cherry_tree_log_likelihood's launch: G, threads, shared bytes, staged, batches, tail, dead threads."""
    Su = S ** c
    G = max(1, 256 // Su)
    threads = (G * Su + 31) // 32 * 32
    smem = G * (Su + 32) * 8
    staging = 2 * LL_BATCH * threads * 8
    staged = Su > 64 and smem + staging <= SMEM_LIMIT
    return dict(Su=Su, G=G, threads=threads, smem=smem + (staging if staged else 0), staged=staged,
                two_stage_max=Su > 64, batches=-(-Su // LL_BATCH), tail=Su % LL_BATCH != 0, dead=threads > G * Su)


def post_layout(S, counts):
    """tree_ll_post_launch: G, threads, CTAs per category, padded last CTAs, bwd<true> shared bytes."""
    G = 256 // S
    threads = (G * S + 31) // 32 * 32
    ctas = [-(-n // G) for n in counts]
    return dict(G=G, threads=threads, dead=threads > G * S, ctas=ctas,
                padded=any(n % G for n in counts), smem_dtau=(2 * S * S + 3 * G * S + 2 * G) * 8)


def pair_layout(S, n_pairs):
    """cherry_tree_ll_pair_posterior: Sp, Np, state tiles of the node products (partial last tile), edge tiles,
    whether the outside prep's last register slot holds states, and the gradient's path."""
    Su = S * S
    Sp = -(-Su // PAIR_SP_ALIGN) * PAIR_SP_ALIGN
    Np = -(-max(n_pairs, 1) // PAIR_NP_ALIGN) * PAIR_NP_ALIGN
    return dict(Su=Su, Sp=Sp, Np=Np, np_rem=n_pairs % PAIR_NP_ALIGN, n_stile=-(-Sp // NODE_TN),
                partial_stile=Sp % NODE_TN != 0, edge_tiles=Sp // EDGE_T, padded_states=Sp > Su,
                last_register=Sp > (PREP_PER_THREAD - 1) * PREP_THREADS, small_grad=Su <= 32)


# ------------------------------------------------------------------ the cases (the coverage test reads these)

def _units(S, c):
    G = fwd_layout(S, c)["G"]
    return sorted({n for n in (G - 1, G, G + 1, 2 * G + 1) if n > 0})


# forward: (S, c, n_units, tree, n_cats)
FWD_CASES = ([(S, 2, n, "random", 1) for S in (8, 9, 11, 16, 17, 20, 29, 30, 32) for n in _units(S, 2)] +
             [(S, 1, n, "random", 1) for S in (2, 33, 64, 65, 100, 255) for n in _units(S, 1)] +
             [(20, 1, 7, "single", 1), (20, 2, 9, "single", 1), (21, 1, 30, "caterpillar", 3),
              (9, 2, 7, "caterpillar", 1), (65, 1, 5, "star", 2), (11, 2, 4, "star", 1), (9, 2, 11, "random", 3),
              (30, 2, 2, "random", 2)])
# site posterior: (S, per-category unit counts as multiples/offsets of G, tree)
POST_CASES = ([(S, "G", "random") for S in (2, 3, 5, 8, 16, 31, 32)] +
              [(8, "20cats", "random"), (20, "G", "caterpillar"), (5, "empty", "random"), (31, "G", "single")])
# pair posterior: (S, n_pairs, tree, model)
PAIR_CASES = [(3, 15, "random", "product"), (5, 16, "cherries", "coupled"), (6, 17, "multi", "product"),
              (8, 32, "random", "coupled"), (9, 33, "cherries", "product"), (11, 16, "multi", "coupled"),
              (16, 15, "random", "product"), (24, 17, "small", "product"), (29, 16, "small", "product"),
              (32, 33, "cherries_small", "product")]
TRANSPOSE_CASES = [(3, 7), (33, 5), (81, 3), (3, 65537)]
BIG_K_PAIR = (6, 430)  # Su = 36 on a random tree of 430 leaves: more than LARGE_MAX_K distinct branch lengths


def _post_counts(kind, G, rng):
    if kind == "G":
        return [1, G - 1, G, G + 1]
    if kind == "20cats":
        return [int(x) for x in rng.integers(1, 2 * G + 2, 20)]
    return [G + 1, 0, 3]  # "empty": category 1 has no units


# ------------------------------------------------------------------ 0. the cases reach every host path (CPU)

def test_cases_reach_every_host_path():
    """If a constant of likelihood.cu or pair_posterior.cu moves, this names the path no case reaches any more."""
    fwd = [fwd_layout(S, c) | dict(n=n, tree=t) for S, c, n, t, _ in FWD_CASES]
    big = [(L["staged"], L["tail"], L["G"] > 1, L["dead"]) for L in fwd if L["Su"] > 64]
    need = {"staged, tail": (True, True), "staged, no tail": (True, False), "direct, tail": (False, True),
            "direct, no tail": (False, False)}
    for name, (st, tl) in need.items():
        assert any(b[0] == st and b[1] == tl for b in big), f"Su > 64 {name} not reached"
    for name, key in (("staged G > 1", (True, 2, True)), ("staged G = 1", (True, 2, False)),
                      ("staged, dead threads", (True, 3, True)), ("staged, no dead threads", (True, 3, False)),
                      ("direct, dead threads", (False, 3, True)), ("direct, no dead threads", (False, 3, False))):
        assert any(b[0] == key[0] and b[key[1]] == key[2] for b in big), f"{name} not reached"
    small = [L for L in fwd if L["Su"] <= 64]
    assert any(L["dead"] for L in small) and any(not L["dead"] for L in small), "Su <= 64 dead threads"
    assert any(L["G"] > 1 for L in small) and not any(L["two_stage_max"] for L in small)
    assert all(L["two_stage_max"] == (L["Su"] > 64) for L in fwd)
    # the documented sizes: c = 1 at S = 65, 100 staged with dead threads, S = 33, 64 not staged; S = 255 staged
    # with one dead thread; the last staged pair size S = 29 (228 168 of 232 448 bytes); S = 30..32 direct
    assert fwd_layout(65, 1)["staged"] and fwd_layout(65, 1)["dead"] and fwd_layout(100, 1)["staged"]
    assert fwd_layout(100, 1)["dead"] and not fwd_layout(33, 1)["staged"] and not fwd_layout(64, 1)["staged"]
    L = fwd_layout(255, 1)
    assert L["staged"] and L["threads"] - L["Su"] == 1
    L = fwd_layout(29, 2)
    assert L["staged"] and L["smem"] == 228168 and SMEM_LIMIT == 232448
    assert not any(fwd_layout(S, 2)["staged"] for S in (30, 31, 32))
    assert {(S, c) for S, c, *_ in FWD_CASES} >= {(29, 2), (30, 2), (32, 2), (255, 1)}
    for S, c in {(S, c) for S, c, _, t, _ in FWD_CASES if t == "random"}:  # units G - 1, G, G + 1, 2 G + 1
        ns = {n for s, cc, n, t, k in FWD_CASES if (s, cc, t, k) == (S, c, "random", 1)}
        assert ns == set(_units(S, c)), (S, c, ns)
    trees = {(c, t) for _, c, _, t, _ in FWD_CASES}
    assert {(1, "single"), (2, "single"), (1, "caterpillar"), (2, "caterpillar"), (1, "star"), (2, "star")} <= trees
    assert any(c == 2 and k > 1 for _, c, _, _, k in FWD_CASES), "a pair case with several categories"

    rng = np.random.default_rng(0)
    posts = [(S, post_layout(S, _post_counts(k, 256 // S, rng)), k) for S, k, _ in POST_CASES]
    assert {S for S, _, _ in posts} >= {2, 3, 5, 8, 16, 31, 32}
    assert any(L["dead"] for _, L, _ in posts) and any(not L["dead"] for _, L, _ in posts)
    assert any(L["padded"] for _, L, _ in posts) and any(1 in L["ctas"] for _, L, _ in posts)
    assert any(0 in L["ctas"] for _, L, _ in posts), "a category without units"
    assert any(len(L["ctas"]) == 20 for _, L, _ in posts)
    assert post_layout(2, [1])["G"] == 128 and post_layout(3, [1])["G"] == 85 and post_layout(31, [1])["G"] == 8
    assert post_layout(32, [1])["smem_dtau"] == 22656

    pairs = [pair_layout(S, n) for S, n, _, _ in PAIR_CASES]
    assert {L["Su"] for L in pairs} >= {9, 25, 36, 64, 81, 121, 256, 576, 841, 1024}
    assert {n for _, n, _, _ in PAIR_CASES} >= {15, 16, 17, 32, 33}
    for rem in {L["np_rem"] for L in pairs}:
        for partial in (True, False):
            assert any(L["np_rem"] == rem and L["partial_stile"] == partial for L in pairs), (rem, partial)
    assert {L["np_rem"] for L in pairs} >= {0, 1, 15}
    assert any(L["last_register"] for L in pairs) and any(not L["padded_states"] for L in pairs)
    assert any(L["small_grad"] for L in pairs) and any(not L["small_grad"] for L in pairs)
    assert {t for _, _, t, _ in PAIR_CASES} >= {"cherries", "multi"}
    S, n_leaves = BIG_K_PAIR
    assert 2 * n_leaves - 2 > LARGE_MAX_K and S * S > 32

    assert any(Su % 32 for Su, _ in TRANSPOSE_CASES) and any(n > 65535 for _, n in TRANSPOSE_CASES)


def test_size_functions_without_gpu():
    lib = _lib.load()
    for S in range(1, 257):
        for c in (1, 2):
            if S ** c > 1024 and c == 2:
                continue
            L = fwd_layout(S, c)
            assert lib.cherry_tree_ll_units_per_block(S, c) == L["G"], (S, c)
            for n_units, depth in ((1, 0), (L["G"] + 1, 3), (1000, 250)):
                blocks = -(-n_units // L["G"])
                want = blocks * (depth + 1) * L["G"] * L["Su"] * 8
                assert lib.cherry_tree_ll_scratch_bytes(S, c, n_units, depth) == want, (S, c, n_units, depth)


# ------------------------------------------------------------------ case builders

def _star(n, rng):
    t = Tree()
    t.add_node("root")
    names = [f"L{i}" for i in range(n)]
    t.add_nodes(names)
    t.add_edges([("root", v, float(rng.lognormal(-2, 1))) for v in names])
    return t


def _cherries(n, rng, grid=(0.02, 0.1, 0.4)):
    """FastCherries-shaped: root -> internal -> two leaves at d / 2, d from a small quantized grid."""
    t = Tree()
    t.add_node("root")
    for k in range(n):
        p, a, b = f"c{k}", f"c{k}a", f"c{k}b"
        d = float(rng.choice(grid))
        t.add_nodes([p, a, b])
        t.add_edges([("root", p, float(rng.choice(grid))), (p, a, d / 2), (p, b, d / 2)])
    return t


def _single():
    t = Tree()
    t.add_node("only")
    return t


def _make_tree(kind, rng):
    if kind == "random":
        return _random_tree(6, rng, zero_branch=True)
    if kind == "small":
        return _random_tree(4, rng)
    if kind == "multi":
        return _random_tree(9, rng, root_children=5, zero_branch=True)
    if kind == "single":
        return _single()
    if kind == "caterpillar":
        return _caterpillar(201, rng)
    if kind == "star":
        return _star(300, rng)
    if kind == "cherries":
        return _cherries(24, rng)
    if kind == "cherries_small":
        return _cherries(3, rng)
    raise ValueError(kind)


def _table(tree, long_every=4):
    """Node table, max depth, and branch lengths with every `long_every`-th branch made long (rows near pi)."""
    from cherryml_b200.evaluation._likelihood import _tree_arrays

    nodes, lengths, leaves, max_depth = _tree_arrays(tree)
    lengths = lengths.copy()
    lengths[::long_every] *= 40.0
    return nodes, max_depth, lengths, len(leaves)


def _obs(rng, n_leaves, n_units, S, c, gap=0.2):
    """Residues with gaps (byte S); unit 0 cycles through every gap pattern of a pair across the leaves."""
    obs = rng.integers(0, S, (n_leaves, n_units, c)).astype(np.uint8)
    obs[rng.random(obs.shape) < gap] = S
    if c == 2 and n_units:
        for j in range(n_leaves):
            x, y = rng.integers(0, S, 2)
            obs[j, 0] = [(x, y), (S, y), (x, S), (S, S)][j % 4]
    return obs


def _expm_clip(Q, t):
    from scipy.linalg import expm

    if t == 0.0:
        return np.eye(Q.shape[0])
    return np.maximum(expm(t * Q), 0.0)


def _matrices(S, c, exps, seed, coupled=False):
    """fp64 P [n, Su, Su] (not transposed) for the distinct exponents: a dense reversible model on S states
    (c = 1), a Kronecker product of two (c = 2), or a coupled reversible model on S^2 states.  Also (Q, pi)."""
    if c == 1 or coupled:
        Q, pi = _random_reversible(S ** c, seed)
        return np.stack([_expm_clip(Q, t) for t in exps]), Q, pi
    Q1, p1 = _random_reversible(S, seed)
    Q2, p2 = _random_reversible(S, seed + 1)
    P = np.stack([np.kron(_expm_clip(Q1, t), _expm_clip(Q2, t)) for t in exps])
    Q = np.kron(Q1, np.eye(S)) + np.kron(np.eye(S), Q2)
    return P, Q, np.kron(p1, p2)


def _site_case(S, c, n_units, tree_kind, n_cats, seed, counts=None):
    rng = np.random.default_rng(seed)
    nodes, max_depth, lengths, n_leaves = _table(_make_tree(tree_kind, rng))
    rates = np.array([1.0] if n_cats == 1 else [0.25] + sorted(rng.uniform(0.5, 3.0, n_cats - 1)))
    exps, p_index = np.unique((lengths[:, None] * rates[None, :]).reshape(-1), return_inverse=True)
    P, Q, pi = _matrices(S, c, exps, seed)
    if counts is not None:
        unit_cat = np.concatenate([np.full(n, k) for k, n in enumerate(counts)]).astype(np.int32)
        rng.shuffle(unit_cat)
    else:
        unit_cat = rng.integers(0, n_cats, n_units).astype(np.int32)
    obs = _obs(rng, n_leaves, len(unit_cat), S, c)
    return dict(nodes=nodes, max_depth=max_depth, p_index=p_index.reshape(len(nodes), n_cats).astype(np.int32),
                P=P, Q=Q, pi=pi, obs=obs, unit_cat=unit_cat, S=S, c=c, exps=exps)


def _check_close(got, ref, rtol, what):
    ref = np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref)
    lim = rtol * np.abs(ref) + 1e-290
    bad = err > lim
    assert not bad.any(), f"{what}: {bad.sum()} entries off, worst {np.max(err / np.maximum(lim, 1e-300)):.3g} x tol"


# ------------------------------------------------------------------ 1. reference self-checks (CPU)

def test_long_double_reference_matches_the_fp64_oracle():
    """inside_outside_ld against oracle.likelihood_grad_oracle (fp64, its own tree walk and expm) on Tree inputs."""
    from scipy.linalg import expm

    from cherryml_b200.evaluation._likelihood import _encode_leaves, _tree_arrays
    from oracle.likelihood_grad_oracle import log_likelihood_gradient, pair_log_likelihood_gradient

    rng = np.random.default_rng(1)
    tree = _random_tree(7, rng, root_children=3, zero_branch=True)
    Q, pi = _random_reversible(4, 3)
    rates = [0.5, 1.0, 2.0, 1.0, 0.5, 2.0]
    msa = {v: "".join(rng.choice(DNA + ["-"], 6)) for v in tree.leaves()}
    ref = log_likelihood_gradient(tree, msa, rates, DNA, pi, Q)
    nodes, lengths, leaves, _ = _tree_arrays(tree)
    cats = np.array(sorted(set(rates)))
    exps, p_index = np.unique((lengths[:, None] * cats[None, :]).reshape(-1), return_inverse=True)
    P = np.stack([expm(t * Q) for t in exps])
    obs = _encode_leaves(msa, leaves, DNA)[:, :, None]
    unit_cat = np.searchsorted(cats, rates)
    got = inside_outside_ld(nodes, p_index.reshape(len(nodes), -1), P, obs, unit_cat, pi, 4, 1, Q=Q)
    np.testing.assert_allclose(got["ll"].astype(float), ref["lls"], rtol=1e-13)
    for k, t in enumerate(exps):
        if t in ref["W"]:
            np.testing.assert_allclose(got["W"][k].astype(float), ref["W"][t], rtol=1e-11, atol=1e-14)
    np.testing.assert_allclose(got["root"].astype(float), ref["root"], rtol=1e-12)
    assert np.all(got["bound"] > 0) and np.all(got["bound"] < 1e-10)
    # pairs: the same pass on S^2 states
    S = 3
    cmap = np.zeros((4, 4))
    cmap[0, 1] = cmap[1, 0] = cmap[2, 3] = cmap[3, 2] = 1
    Q2, pi2 = _random_reversible(S * S, 5)
    msa = {v: "".join(rng.choice(DNA[:S] + ["-"], 4)) for v in tree.leaves()}
    ref = pair_log_likelihood_gradient(tree, msa, cmap, DNA[:S], pi2, Q2)
    enc = _encode_leaves(msa, leaves, DNA[:S])
    obs = np.stack([enc[:, [0, 2]], enc[:, [1, 3]]], axis=2)
    exps, p_index = np.unique(lengths, return_inverse=True)
    P = np.stack([expm(t * Q2) for t in exps])
    got = inside_outside_ld(nodes, p_index, P, obs, np.zeros(2), pi2, S, 2)
    np.testing.assert_allclose(got["ll"].astype(float), ref["lls"], rtol=1e-13)
    for k, t in enumerate(exps):
        if t in ref["W"]:
            np.testing.assert_allclose(got["W"][k].astype(float), ref["W"][t], rtol=1e-11, atol=1e-14)


def test_kronecker_matrices_are_the_pair_model_expm():
    from scipy.linalg import expm

    P, Q, pi = _matrices(4, 2, np.array([0.0, 0.03, 2.0]), seed=2)
    for k, t in enumerate((0.0, 0.03, 2.0)):
        np.testing.assert_allclose(P[k], expm(t * Q), rtol=1e-12, atol=1e-15)
    assert np.allclose(pi @ Q, 0.0, atol=1e-14)


def test_complex_step_matches_finite_differences():
    from cherryml_b200.evaluation._likelihood import _tree_arrays

    rng = np.random.default_rng(4)
    tree = _random_tree(6, rng, root_children=3)
    nodes, lengths, leaves, _ = _tree_arrays(tree)
    S, n_units = 4, 5
    obs = _obs(rng, len(leaves), n_units, S, 1)
    unit_cat = rng.integers(0, 2, n_units)
    rates = np.array([0.5, 2.0])
    Q, pi = _random_reversible(S, 6)
    exps = lengths[:, None] * rates[None, :]
    f = lambda Qx: complex_ll(nodes, exps, 2, obs, unit_cat, pi, Qx, S, 1)  # noqa: E731
    E = rng.standard_normal((S, S))
    h = 1e-6
    fd = (f(Q + h * E).real - f(Q - h * E).real) / (2 * h)
    cs = complex_step(f, Q, E)
    assert abs(cs - fd) <= 1e-7 * abs(cs), (cs, fd)
    g = lambda e: complex_ll(nodes, e, 2, obs, unit_cat, pi, Q, S, 1)  # noqa: E731
    D = np.zeros_like(exps)
    D[2] = rates
    fd = (g(exps + h * D).real - g(exps - h * D).real) / (2 * h)
    assert abs(complex_step(g, exps, D) - fd) <= 1e-7 * abs(fd)
    # against the long-double pass's log-likelihood
    from scipy.linalg import expm

    ue, p_index = np.unique(exps.reshape(-1), return_inverse=True)
    ref = inside_outside_ld(nodes, p_index.reshape(len(nodes), 2), np.stack([expm(t * Q) for t in ue]), obs,
                            unit_cat, pi, S, 1, posterior=False)
    assert abs(f(Q).real - float(ref["ll"].sum())) <= 1e-12 * abs(f(Q).real)


# ------------------------------------------------------------------ 2. forward pass

@pytest.mark.gpu
@pytest.mark.parametrize("S,c,n_units,tree,n_cats", FWD_CASES)
def test_forward_against_long_double(S, c, n_units, tree, n_cats):
    k = _site_case(S, c, n_units, tree, n_cats, seed=1000 * c + S + n_units)
    args = (k["nodes"], k["max_depth"], k["p_index"], k["P"], k["obs"], k["unit_cat"], k["pi"], S, c)
    got = gpu_forward(*args)
    ref = inside_outside_ld(k["nodes"], k["p_index"], k["P"], k["obs"], k["unit_cat"], k["pi"], S, c,
                            posterior=False)
    err = np.abs(got - ref["ll"].astype(np.float64))
    assert np.all(np.isfinite(got))
    assert np.all(err <= ref["bound"]), (err.max(), ref["bound"][np.argmax(err / ref["bound"])])
    assert np.array_equal(got, gpu_forward(*args))


# ------------------------------------------------------------------ 3. site posterior and edge derivatives

def _post_case(S, kind, tree, seed):
    rng = np.random.default_rng(seed)
    counts = _post_counts(kind, 256 // S, rng)
    return _site_case(S, 1, sum(counts), tree, len(counts), seed, counts=counts), counts


@pytest.mark.gpu
@pytest.mark.parametrize("S,kind,tree", POST_CASES)
def test_site_posterior_and_edge_derivatives_against_long_double(S, kind, tree):
    import torch

    k, counts = _post_case(S, kind, tree, seed=77 + S)
    n_units, n_nodes = len(k["unit_cat"]), len(k["nodes"])
    fam = site_family(k["nodes"], k["max_depth"], k["p_index"], len(k["P"]), k["obs"], k["unit_cat"], S)
    Pt = torch.from_numpy(np.ascontiguousarray(np.swapaxes(k["P"], 1, 2))).cuda()
    pi, Q = torch.from_numpy(k["pi"]).cuda(), torch.from_numpy(k["Q"]).cuda()
    ll, W, root, dtau = (x.cpu().numpy() for x in fam.edge_derivatives(Pt, pi, Q))
    ll0, W0, root0 = (x.cpu().numpy() for x in fam.posterior(Pt, pi))
    assert np.array_equal(ll, ll0) and np.array_equal(W, W0) and np.array_equal(root, root0)
    fwd = gpu_forward(k["nodes"], k["max_depth"], k["p_index"], k["P"], k["obs"], k["unit_cat"], k["pi"], S, 1)
    assert np.array_equal(ll, fwd)
    again = [x.cpu().numpy() for x in fam.edge_derivatives(Pt, pi, Q)]
    assert all(np.array_equal(a, b) for a, b in zip((ll, W, root, dtau), again))

    ref = inside_outside_ld(k["nodes"], k["p_index"], k["P"], k["obs"], k["unit_cat"], k["pi"], S, 1, Q=k["Q"])
    T = float(ref["bound"].max())
    assert np.all(np.abs(ll - ref["ll"].astype(float)) <= ref["bound"])
    rtol = 5 * T + (n_units + len(counts) * n_nodes + 800) * U64
    _check_close(W, ref["W"], rtol, "W")
    _check_close(root, ref["root"], 2 * T + (n_units + 800) * U64, "root")
    dtol = (5 * T + (2 * S + n_units + 800) * U64) * ref["dmass"].astype(float)
    assert np.all(np.abs(dtau - ref["dtau"].astype(float)) <= dtol + 1e-300), np.max(np.abs(dtau - ref["dtau"]))
    assert np.all(dtau[-1] == 0.0)
    for cat, n in enumerate(counts):
        if n == 0:  # a category with no units contributes nothing
            assert np.all(dtau[:, cat] == 0.0)
    assert abs(W.sum() - n_units * (n_nodes - 1)) <= rtol * n_units * n_nodes
    assert abs(root.sum() - n_units) <= rtol * n_units


@pytest.mark.gpu
def test_empty_category_adds_exactly_nothing_to_w():
    """The units of categories 0 and 2 alone, with and without an empty category 1 between them, share every
    matrix: W and dtau of categories 0 and 2 are bitwise those of the call without the empty category."""
    import torch

    S = 5
    k, counts = _post_case(S, "empty", "random", seed=5)
    assert counts[1] == 0
    Pt = torch.from_numpy(np.ascontiguousarray(np.swapaxes(k["P"], 1, 2))).cuda()
    pi, Q = torch.from_numpy(k["pi"]).cuda(), torch.from_numpy(k["Q"]).cuda()
    fam = site_family(k["nodes"], k["max_depth"], k["p_index"], len(k["P"]), k["obs"], k["unit_cat"], S)
    ll, W, root, dtau = (x.cpu().numpy() for x in fam.edge_derivatives(Pt, pi, Q))
    # the same data with category 1 dropped from the table: its matrix index column goes away
    uc = np.where(k["unit_cat"] == 2, 1, k["unit_cat"]).astype(np.int32)
    fam2 = site_family(k["nodes"], k["max_depth"], k["p_index"][:, [0, 2]], len(k["P"]), k["obs"], uc, S)
    ll2, W2, root2, dtau2 = (x.cpu().numpy() for x in fam2.edge_derivatives(Pt, pi, Q))
    assert np.array_equal(ll, ll2) and np.array_equal(root, root2)
    assert np.array_equal(dtau[:, [0, 2]], dtau2) and np.all(dtau[:, 1] == 0.0)
    # matrices used only by the empty category get exactly zero
    only1 = set(k["p_index"][:-1, 1]) - set(k["p_index"][:-1, 0]) - set(k["p_index"][:-1, 2])
    for m in only1:
        assert np.all(W[m] == 0.0)
    assert np.array_equal(W, W2)


# ------------------------------------------------------------------ 4. pair posterior

def _pair_case(S, n_pairs, tree_kind, model, seed):
    rng = np.random.default_rng(seed)
    nodes, max_depth, lengths, n_leaves = _table(_make_tree(tree_kind, rng), long_every=5)
    exps, p_index = np.unique(lengths, return_inverse=True)
    P, Q, pi = _matrices(S, 2, exps, seed, coupled=model == "coupled")
    obs = _obs(rng, n_leaves, n_pairs, S, 2)
    return dict(nodes=nodes, max_depth=max_depth, p_index=p_index.astype(np.int32), P=P, Q=Q, pi=pi, obs=obs, S=S)


@pytest.mark.gpu
@pytest.mark.parametrize("S,n_pairs,tree,model", PAIR_CASES)
def test_pair_posterior_against_long_double(S, n_pairs, tree, model):
    import torch

    k = _pair_case(S, n_pairs, tree, model, seed=S * 100 + n_pairs)
    n_nodes = len(k["nodes"])
    fam = pair_family(k["nodes"], k["max_depth"], k["p_index"], len(k["P"]), k["obs"], S)
    P, pi = torch.from_numpy(k["P"]).cuda(), torch.from_numpy(k["pi"]).cuda()
    ll, W, root = (x.cpu().numpy() for x in fam.posterior(P, pi))
    again = [x.cpu().numpy() for x in fam.posterior(P, pi)]
    assert all(np.array_equal(a, b) for a, b in zip((ll, W, root), again))
    unit_cat = np.zeros(n_pairs, dtype=np.int32)
    ref = inside_outside_ld(k["nodes"], k["p_index"], k["P"], k["obs"], unit_cat, k["pi"], S, 2)
    T = float(ref["bound"].max())
    assert np.all(np.abs(ll - ref["ll"].astype(float)) <= ref["bound"])
    fwd = gpu_forward(k["nodes"], k["max_depth"], k["p_index"], k["P"], k["obs"], unit_cat, k["pi"], S, 2)
    assert np.all(np.abs(fwd - ref["ll"].astype(float)) <= ref["bound"])
    rtol = 5 * T + (n_pairs + n_nodes + 800) * U64
    _check_close(W, ref["W"], rtol, "W")
    _check_close(root, ref["root"], 2 * T + (n_pairs + 800) * U64, "root")
    assert abs(W.sum() - n_pairs * (n_nodes - 1)) <= rtol * n_pairs * n_nodes
    assert abs(root.sum() - n_pairs) <= rtol * n_pairs


# ------------------------------------------------------------------ 5. gradients end to end

def _grad_family(S, n_leaves, L, seed, tree=None):
    rng = np.random.default_rng(seed)
    alphabet = (AA + list("BJOUZ") + list("abcdefg"))[:S]
    tree = tree or _random_tree(n_leaves, rng, root_children=3, zero_branch=True)
    msa = {v: "".join(rng.choice(alphabet + ["-"], L)) for v in tree.leaves()}
    return tree, msa, alphabet, rng


def _complex_inputs(tree, msa, alphabet, rates):
    from cherryml_b200.evaluation._likelihood import _encode_leaves, _tree_arrays

    nodes, lengths, leaves, _, names = _tree_arrays(tree, with_names=True)
    cats = np.array(sorted(set(rates)))
    return nodes, lengths, names, cats, _encode_leaves(msa, leaves, alphabet), np.searchsorted(cats, rates)


def _rate_direction(rng, S):
    R = rng.random((S, S))
    np.fill_diagonal(R, 0.0)
    np.fill_diagonal(R, -R.sum(axis=1))
    return R


@pytest.mark.gpu
@pytest.mark.parametrize("S", [3, 8, 20, 31])
def test_site_gradients_against_complex_step(S):
    from cherryml_b200.evaluation import branch_length_gradient, log_likelihood_gradient

    tree, msa, alphabet, rng = _grad_family(S, 9, 40, seed=S)
    rates = [float(x) for x in rng.choice([0.3, 1.0, 2.2], 40)]
    Q, pi = _random_reversible(S, S + 1)
    ll, lls, gQ, gpi = log_likelihood_gradient(tree, msa, rates, alphabet, pi, Q)
    _, _, dlen = branch_length_gradient(tree, msa, rates, alphabet, pi, Q)
    nodes, lengths, names, cats, enc, cat = _complex_inputs(tree, msa, alphabet, rates)
    obs = enc[:, :, None]
    exps = lengths[:, None] * cats[None, :]
    fQ = lambda Qx: complex_ll(nodes, exps, len(cats), obs, cat, pi, Qx, S, 1)  # noqa: E731
    for E in (rng.standard_normal((S, S)), _rate_direction(rng, S)):
        ref = complex_step(fQ, Q, E)
        assert abs(np.sum(gQ * E) - ref) <= 1e-9 * abs(ref), (np.sum(gQ * E), ref)
    fpi = lambda p: complex_ll(nodes, exps, len(cats), obs, cat, p, Q, S, 1)  # noqa: E731
    e = rng.standard_normal(S)
    ref = complex_step(fpi, pi, e)
    assert abs(np.dot(gpi, e) - ref) <= 1e-9 * max(abs(ref), np.abs(gpi).max()), (np.dot(gpi, e), ref)
    fe = lambda x: complex_ll(nodes, x, len(cats), obs, cat, pi, Q, S, 1)  # noqa: E731
    for i in range(0, len(nodes) - 1, 3):
        D = np.zeros_like(exps)
        D[i] = cats
        ref = complex_step(fe, exps, D)
        assert abs(dlen[names[i]] - ref) <= 1e-9 * max(1.0, abs(ref)), (names[i], dlen[names[i]], ref)


def _pair_msa(tree, alphabet, n_pairs, rng):
    L = 2 * n_pairs
    msa = {v: "".join(rng.choice(alphabet + ["-"], L)) for v in tree.leaves()}
    cmap = np.zeros((L, L))
    for j in range(n_pairs):
        cmap[2 * j, 2 * j + 1] = cmap[2 * j + 1, 2 * j] = 1
    return msa, cmap


@pytest.mark.gpu
@pytest.mark.parametrize("S,n_leaves,n_pairs", [(3, 9, 17), (5, 7, 16), (6, BIG_K_PAIR[1], 17), (9, 6, 15)])
def test_pair_gradient_against_complex_step(S, n_leaves, n_pairs):
    """Su = 9, 25 (small adjoint path), 36 on a tree with more than 811 distinct branch lengths (large path, in
    chunks), 81; a coupled (non-product) model."""
    from cherryml_b200.evaluation import pair_log_likelihood_gradient
    from cherryml_b200.evaluation._likelihood import _encode_leaves, _tree_arrays
    from cherryml_b200.markov_chain import compute_stationary_distribution

    rng = np.random.default_rng(S)
    alphabet = (AA + ["X"])[:S]
    tree = _random_tree(n_leaves, rng, root_children=3, zero_branch=True)
    msa, cmap = _pair_msa(tree, alphabet, n_pairs, rng)
    Q, _ = _random_reversible(S * S, S + 2)
    pi = compute_stationary_distribution(Q)
    ll, lls, gQ, gpi = pair_log_likelihood_gradient(tree, msa, cmap, alphabet, pi, Q)
    nodes, lengths, leaves, _ = _tree_arrays(tree)
    if S == BIG_K_PAIR[0]:
        assert len(np.unique(lengths[:-1])) > LARGE_MAX_K
    enc = _encode_leaves(msa, leaves, alphabet)
    obs = np.stack([enc[:, 0::2], enc[:, 1::2]], axis=2)
    zeros = np.zeros(n_pairs, dtype=np.int64)
    fQ = lambda Qx: complex_ll(nodes, lengths[:, None], 1, obs, zeros, pi, Qx, S, 2)  # noqa: E731
    assert abs(fQ(Q).real - ll) <= 1e-10 * abs(ll)
    for E in (rng.standard_normal((S * S, S * S)), _rate_direction(rng, S * S)):
        ref = complex_step(fQ, Q, E)
        assert abs(np.sum(gQ * E) - ref) <= 1e-9 * abs(ref), (np.sum(gQ * E), ref)
    fpi = lambda p: complex_ll(nodes, lengths[:, None], 1, obs, zeros, p, Q, S, 2)  # noqa: E731
    e = rng.standard_normal(S * S)
    ref = complex_step(fpi, pi, e)
    assert abs(np.dot(gpi, e) - ref) <= 1e-9 * max(abs(ref), np.abs(gpi).max())


@pytest.mark.gpu
@pytest.mark.parametrize("S,model", [(24, "coupled"), (32, "product")])
def test_large_pair_gradient_against_frechet_oracle(S, model):
    """Su = 576 under a coupled model and Su = 1024 under a Kronecker sum, on a FastCherries-shaped tree with few
    distinct lengths, against oracle.likelihood_grad_oracle (scipy expm and expm_frechet in fp64)."""
    from cherryml_b200.evaluation import pair_log_likelihood_gradient
    from cherryml_b200.markov_chain import chain_product, compute_stationary_distribution
    from oracle.likelihood_grad_oracle import pair_log_likelihood_gradient as oracle_gradient

    rng = np.random.default_rng(S)
    alphabet = (AA + list("BJOUZXabcdef"))[:S]
    tree = _cherries(2, rng, grid=(0.05, 0.3))
    msa, cmap = _pair_msa(tree, alphabet, 17, rng)
    if model == "coupled":
        Q, _ = _random_reversible(S * S, 9)
    else:
        Q = chain_product(*(_random_reversible(S, s)[0] for s in (3, 3)))
    pi = compute_stationary_distribution(Q)
    ll, lls, gQ, gpi = pair_log_likelihood_gradient(tree, msa, cmap, alphabet, pi, Q)
    ref = oracle_gradient(tree, msa, cmap, alphabet, pi, Q)
    assert abs(ll - ref["ll"]) <= 1e-10 * abs(ref["ll"])
    np.testing.assert_allclose(gQ, ref["grad_Q"], rtol=1e-9, atol=1e-9 * np.abs(ref["grad_Q"]).max())
    np.testing.assert_allclose(gpi, ref["grad_pi"], rtol=1e-9, atol=1e-9 * np.abs(ref["grad_pi"]).max())


# ------------------------------------------------------------------ 6. transpose

@pytest.mark.gpu
@pytest.mark.parametrize("Su,n", TRANSPOSE_CASES)
def test_transpose_is_bitwise_swapaxes(Su, n):
    import torch

    lib = _lib.load()
    x = torch.from_numpy(np.random.default_rng(Su).standard_normal((n, Su, Su))).cuda()
    out = torch.full_like(x, np.nan)
    _lib.check(lib.cherry_tree_ll_transpose(_lib.ptr(x), n, Su, _lib.ptr(out), _lib.current_stream_ptr()),
               "cherry_tree_ll_transpose")
    assert np.array_equal(out.cpu().numpy(), np.swapaxes(x.cpu().numpy(), 1, 2))
