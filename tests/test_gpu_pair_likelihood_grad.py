"""Exact gradient of the log-likelihood of contacting pairs (cherry_tree_ll_pair_posterior + the fit's expm
adjoint) and the co-evolution maximum-likelihood stage built on it (coevolution_tree_likelihood_mle).

CPU: the numpy pair oracle against central finite differences of the likelihood oracle and against the site
oracle under product models, and the new C entry points' argument checks.
GPU: per-pair log-likelihoods against cherry_tree_log_likelihood (c = 2), edge posteriors and both gradients
against the oracle (1e-9 relative), the reference's pair goldens, a full-size demo family, determinism,
gradcheck of the autograd node, and the stage's fit, files and cache."""
import ctypes
import os
import tarfile

import numpy as np
import pytest

from cherryml_b200 import _lib
from cherryml_b200.io import Tree
from tests._ll_cases import (AA, DNA, _caterpillar, _random_reversible, _random_tree, _star_of_cherries, golden_cases,
                             rate_matrix)
from tests.conftest import GOLDEN


# ------------------------------------------------------------------ fixtures

def _coupled(S, seed):
    """A random reversible pair model on S^2 states that is not a product of two site models."""
    from cherryml_b200.markov_chain import compute_stationary_distribution

    Q, _ = _random_reversible(S * S, seed)
    return Q, compute_stationary_distribution(Q)


def _two_leaves(rng):
    t = Tree()
    t.add_nodes(["r", "a", "b"])
    t.add_edges([("r", "a", float(rng.lognormal(-2, 1))), ("r", "b", float(rng.lognormal(-2, 1)))])
    return t


def _single_leaf():
    t = Tree()
    t.add_node("only")
    return t


def _pair_msa(tree, alphabet, n_pairs, rng, gap_frac=0.15):
    """Sites 2k and 2k+1 form pair k (contact map returned too).  With more than one pair, pair 0 is gapped in
    both sites at every leaf (an all-gap pair column); the other pairs have random gaps in one or both sites."""
    L = 2 * n_pairs
    msa = {}
    for v in tree.leaves():
        s = rng.choice(alphabet, L)
        s[rng.random(L) < gap_frac] = "-"
        if n_pairs > 1:
            s[0] = s[1] = "-"
        msa[v] = "".join(s)
    cmap = np.zeros((L, L))
    for k in range(n_pairs):
        cmap[2 * k, 2 * k + 1] = cmap[2 * k + 1, 2 * k] = 1
    return msa, cmap


def _scratch_formula(S, n_nodes, n_pairs, n_matrices):
    Sp = -(-S * S // 64) * 64
    Np = -(-max(n_pairs, 1) // 16) * 16
    return 8 * (3 * n_nodes * Np * Sp + 2 * n_nodes * Np) + 4 * (8 * n_nodes + n_matrices + 2)


# ------------------------------------------------------------------ CPU: oracle and ABI

@pytest.mark.parametrize("S", [2, 3, 4])
def test_pair_oracle_matches_finite_differences(S):
    from oracle.likelihood_grad_oracle import pair_log_likelihood_gradient
    from oracle.likelihood_oracle import log_likelihood

    rng = np.random.default_rng(S)
    alphabet = DNA[:S]
    tree = _random_tree(5, rng, zero_branch=S == 3)
    msa, cmap = _pair_msa(tree, alphabet, 3, rng, gap_frac=0.3)
    Q, pi = _coupled(S, seed=10 + S)
    Su = S * S
    res = pair_log_likelihood_gradient(tree, msa, cmap, alphabet, pi, Q)
    Q1, pi1 = _random_reversible(S, 1)  # no independent site: the site model is unused

    def ll(Qx, pix):
        return log_likelihood(tree, msa, cmap, [1.0] * len(cmap), alphabet, pi1, Q1, pix, Qx)[0]

    assert abs(res["ll"] - ll(Q, pi)) <= 1e-12 * abs(res["ll"])
    h = 1e-5
    fd_Q = np.zeros((Su, Su))
    for i in range(Su):
        for j in range(Su):
            E = np.zeros((Su, Su))
            E[i, j] = h
            fd_Q[i, j] = (ll(Q + E, pi) - ll(Q - E, pi)) / (2 * h)
    fd_pi = np.zeros(Su)
    for i in range(Su):
        e = np.zeros(Su)
        e[i] = h * pi[i]
        fd_pi[i] = (ll(Q, pi + e) - ll(Q, pi - e)) / (2 * h * pi[i])
    np.testing.assert_allclose(res["grad_Q"], fd_Q, rtol=1e-6, atol=1e-6 * np.abs(fd_Q).max())
    np.testing.assert_allclose(res["grad_pi"], fd_pi, rtol=1e-6, atol=1e-6 * np.abs(fd_pi).max())
    assert abs(res["root"].sum() - 3) <= 1e-12 * 3


def _block_sums(G2, S):
    """d/dQ of f(Q (+) Q) from G2 = d f / d Q2: sum_j G2[(a,j),(b,j)] + sum_i G2[(i,a),(i,b)]."""
    G = G2.reshape(S, S, S, S)
    return np.einsum("ajbj->ab", G) + np.einsum("iaib->ab", G)


def _pi_block_sums(g2, pi, S):
    g = g2.reshape(S, S)
    return g @ pi + g.T @ pi


def test_pair_oracle_reduces_to_sites_under_product_model():
    from cherryml_b200.markov_chain import chain_product
    from oracle.likelihood_grad_oracle import log_likelihood_gradient, pair_log_likelihood_gradient

    rng = np.random.default_rng(3)
    S = 4
    tree = _random_tree(6, rng, root_children=3)
    msa, cmap = _pair_msa(tree, DNA, 4, rng)
    Q, pi = _random_reversible(S, 5)
    pair = pair_log_likelihood_gradient(tree, msa, cmap, DNA, np.kron(pi, pi), chain_product(Q, Q))
    site = log_likelihood_gradient(tree, msa, [1.0] * len(cmap), DNA, pi, Q)
    np.testing.assert_allclose(pair["lls"], site["lls"][0::2] + site["lls"][1::2], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(_block_sums(pair["grad_Q"], S), site["grad_Q"], rtol=1e-10,
                               atol=1e-12 * np.abs(site["grad_Q"]).max())
    np.testing.assert_allclose(_pi_block_sums(pair["grad_pi"], pi, S), site["grad_pi"], rtol=1e-10)


def test_pair_posterior_entry_arguments_without_gpu():
    lib = _lib.load()
    assert lib.cherry_tree_ll_pair_posterior(0, 3, 1, 0, 0, 2, 0, 0, 20, 4, 0, 0, 0, 0, 0, 0) == -1
    assert b"null pointer" in lib.cherry_last_error()
    buf = (ctypes.c_int32 * 64)()
    p = ctypes.addressof(buf)
    # more than 32 states per site: checked before anything is read or launched
    assert lib.cherry_tree_ll_pair_posterior(p, 3, 1, p, p, 2, p, p, 33, 4, p, 1 << 30, p, p, p, 0) == -3
    assert b"S <= 32" in lib.cherry_last_error()
    assert lib.cherry_tree_ll_pair_posterior(p, 3, 1, p, p, 2, p, p, 20, -1, p, 1 << 30, p, p, p, 0) == -1
    nodes = np.zeros(3, dtype=_lib.LL_NODE_DTYPE)
    nodes["depth"] = [1, 1, 0]
    nodes["flags"] = [3, 1, 0]
    nodes["obs_row"] = [0, 1, -1]
    # p_index out of range (host array, checked before any launch)
    pidx = np.array([0, 5, 0], dtype=np.int32)
    assert lib.cherry_tree_ll_pair_posterior(nodes.ctypes.data, 3, 1, pidx.ctypes.data, p, 2, p, p, 20, 4, p,
                                             1 << 30, p, p, p, 0) == -1
    assert b"p_index" in lib.cherry_last_error()
    pidx[1] = 1
    assert lib.cherry_tree_ll_pair_posterior(nodes.ctypes.data, 3, 1, pidx.ctypes.data, p, 2, p, p, 20, 4, p, 16,
                                             p, p, p, 0) == -1
    assert b"scratch too small" in lib.cherry_last_error()
    # a node table that is not a post-order of one tree
    bad = nodes.copy()
    bad["depth"] = [1, 2, 0]
    assert lib.cherry_tree_ll_pair_posterior(bad.ctypes.data, 3, 2, pidx.ctypes.data, p, 2, p, p, 20, 4, p,
                                             1 << 30, p, p, p, 0) == -1
    for S, n_nodes, depth, n_pairs, n_m in ((20, 2047, 30, 65, 2044), (20, 2047, 60, 187, 2045), (2, 5, 2, 1, 3),
                                            (21, 3, 1, 81, 2), (32, 1, 0, 0, 1), (3, 9, 4, 7, 5)):
        got = lib.cherry_tree_ll_pair_posterior_scratch_bytes(S, n_nodes, depth, n_pairs, n_m)
        assert got == _scratch_formula(S, n_nodes, n_pairs, n_m)
    assert lib.cherry_tree_ll_pair_posterior_scratch_bytes(33, 5, 2, 3, 3) == 0
    assert lib.cherry_tree_ll_pair_posterior_scratch_bytes(20, 5, 2, -1, 3) == 0


# ------------------------------------------------------------------ GPU

def _oracle_cases():
    """(id, tree, alphabet, n_pairs, model): Su in {4, 16, 49, 400, 441}, n_pairs in {1, 7, 80, 81}."""
    rng = np.random.default_rng(17)
    aa7 = AA[:7]
    aa21 = AA + ["X"]  # "-" stays outside the alphabet
    return [
        ("su4_p7_random_zero_branch", _random_tree(9, rng, zero_branch=True), DNA[:2], 7, "coupled"),
        ("su16_p80_star_512_cherries", _star_of_cherries(512, rng), DNA, 80, "coupled"),
        ("su49_p81_caterpillar_60", _caterpillar(60, rng), aa7, 81, "coupled"),
        ("su400_p1_random", _random_tree(7, rng, root_children=3), AA, 1, "lg_x_lg"),
        ("su400_p80_random_zero_branch", _random_tree(6, rng, zero_branch=True), AA, 80, "coupled"),
        ("su441_p7_two_leaves", _two_leaves(rng), aa21, 7, "coupled"),
        ("su400_p7_single_leaf", _single_leaf(), AA, 7, "coupled"),
    ]


def _pair_model(kind, S):
    from cherryml_b200.markov_chain import chain_product, compute_stationary_distribution

    if kind == "lg_x_lg":
        Q = chain_product(rate_matrix("lg"), rate_matrix("lg"))
        return Q, compute_stationary_distribution(Q)
    return _coupled(S, seed=S)


def _gpu_pair_posterior(tree, msa, cmap, alphabet, pi, Q):
    import torch

    from cherryml_b200.evaluation._likelihood import _expm_chunked, _PairFamily

    fam = _PairFamily(tree, msa, cmap, alphabet, "cuda")
    P = _expm_chunked(Q, fam.exponents, "cuda", transpose=False)
    ll, W, root = fam.posterior(P, torch.from_numpy(np.asarray(pi, dtype=np.float64)).cuda())
    return fam.exponents, ll.cpu().numpy(), W.cpu().numpy(), root.cpu().numpy()


def _forward_pair_lls(tree, msa, cmap, alphabet, pi, Q):
    """cherry_tree_log_likelihood with c = 2, through dp_likelihood_computation (every site is paired)."""
    from cherryml_b200.evaluation import dp_likelihood_computation

    S = len(alphabet)
    Q1, pi1 = _random_reversible(S, 0)
    _, lls = dp_likelihood_computation(tree=tree, msa=msa, contact_map=cmap, site_rates=[1.0] * len(cmap),
                                       amino_acids=alphabet, pi_1=pi1, Q_1=Q1, pi_2=pi, Q_2=Q)
    ii, jj = np.where(cmap == 1)
    return np.array([lls[i] + lls[j] for i, j in zip(ii, jj) if i < j])


def _rel(a, b):
    """Relative difference; absolute for values below 1 in magnitude (an all-gap pair has log-likelihood 0)."""
    return np.abs(a - b) / np.maximum(np.abs(b), 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _oracle_cases(), ids=lambda c: c[0])
def test_pair_posterior_and_gradient_against_oracle(case):
    from cherryml_b200.evaluation import pair_log_likelihood_gradient
    from oracle.likelihood_grad_oracle import pair_log_likelihood_gradient as oracle_gradient

    _, tree, alphabet, n_pairs, kind = case
    rng = np.random.default_rng(n_pairs)
    S = len(alphabet)
    Su = S * S
    msa, cmap = _pair_msa(tree, alphabet, n_pairs, rng)
    Q, pi = _pair_model(kind, S)
    exps, lls_post, W, root = _gpu_pair_posterior(tree, msa, cmap, alphabet, pi, Q)
    ll, lls, gQ, gpi = pair_log_likelihood_gradient(tree, msa, cmap, alphabet, pi, Q)
    assert np.array_equal(np.array(lls), lls_post)
    fwd = _forward_pair_lls(tree, msa, cmap, alphabet, pi, Q)
    assert np.all(_rel(np.array(lls), fwd) <= 1e-12), (np.array(lls), fwd)
    ref = oracle_gradient(tree, msa, cmap, alphabet, pi, Q)
    assert abs(ll - ref["ll"]) <= 1e-10 * max(1.0, abs(ref["ll"]))
    W_ref = np.stack([ref["W"].get(t, np.zeros((Su, Su))) for t in exps])
    np.testing.assert_allclose(W, W_ref, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(W_ref).max()))
    np.testing.assert_allclose(root, ref["root"], rtol=1e-9, atol=1e-12 * n_pairs)
    np.testing.assert_allclose(gQ, ref["grad_Q"], rtol=1e-9, atol=1e-9 * np.abs(ref["grad_Q"]).max())
    np.testing.assert_allclose(gpi, ref["grad_pi"], rtol=1e-9, atol=1e-9 * np.abs(ref["grad_pi"]).max())


@pytest.mark.gpu
def test_reference_pair_goldens():
    """The pair cases of the reference's goldens ("product" and "perturbed" 400-state models): each half of a
    pair's log-likelihood is the reference's value of its two sites."""
    from cherryml_b200.evaluation import pair_log_likelihood_gradient

    n = 0
    for c in golden_cases():
        cm = c["contact_map"]
        if c["Q2"] is None or cm is None or not np.any(cm - np.diag(np.diag(cm))):
            continue
        ll, lls, gQ, gpi = pair_log_likelihood_gradient(c["tree"], c["msa"], cm, AA, c["pi2"], c["Q2"])
        ii, jj = np.where(cm == 1)
        pairs = [(i, j) for i, j in zip(ii, jj) if i < j]
        assert len(lls) == len(pairs)
        for x, (i, j) in zip(lls, pairs):
            for site in (i, j):
                assert abs(x / 2 - c["lls"][site]) <= 1e-7 * abs(c["lls"][site])
        assert np.all(np.isfinite(gQ)) and np.all(np.isfinite(gpi))
        n += 1
    assert n == 5


def _demo_family(tmp_dir, fam="13gs_1_A"):
    from cherryml_b200._public_api import maximal_matching_pairs
    from cherryml_b200.io import read_contact_map, read_msa, read_tree

    with tarfile.open(os.path.join(GOLDEN, "demo_data.tar.xz")) as tf:
        tf.extractall(tmp_dir, members=[tf.getmember(f"{d}/{fam}.txt") for d in ("msas", "trees", "contact_maps")])
    cm = read_contact_map(os.path.join(tmp_dir, "contact_maps", f"{fam}.txt"))
    matched = np.zeros_like(cm)
    for i, j in maximal_matching_pairs(cm, 7):
        matched[i, j] = matched[j, i] = 1
    return (read_tree(os.path.join(tmp_dir, "trees", f"{fam}.txt")), read_msa(os.path.join(tmp_dir, "msas", f"{fam}.txt")),
            matched)


@pytest.mark.gpu
def test_demo_family_product_model_equals_sites(tmp_path):
    """13gs_1_A (1 024 leaves, 65 pairs, Su = 400) under LG (+) LG: the pair values and the block sums of the
    pair gradients are those of the 130 paired sites at rate 1 under LG."""
    from cherryml_b200.evaluation import log_likelihood_gradient, pair_log_likelihood_gradient
    from cherryml_b200.markov_chain import chain_product, compute_stationary_distribution

    tree, msa, cmap = _demo_family(str(tmp_path))
    lg = rate_matrix("lg")
    pi = compute_stationary_distribution(lg)
    ll, lls, gQ, gpi = pair_log_likelihood_gradient(tree, msa, cmap, AA, np.kron(pi, pi), chain_product(lg, lg))
    assert len(lls) == 65
    ii, jj = np.where(cmap == 1)
    pairs = [(i, j) for i, j in zip(ii, jj) if i < j]
    sites = [s for p in pairs for s in p]
    sub = {v: "".join(seq[s] for s in sites) for v, seq in msa.items()}
    ll1, lls1, gQ1, gpi1 = log_likelihood_gradient(tree, sub, [1.0] * len(sites), AA, pi, lg)
    assert abs(ll - ll1) <= 1e-10 * abs(ll1)
    np.testing.assert_allclose(lls, np.array(lls1)[0::2] + np.array(lls1)[1::2], rtol=1e-10)
    np.testing.assert_allclose(_block_sums(gQ, 20), gQ1, rtol=1e-8, atol=1e-8 * np.abs(gQ1).max())
    np.testing.assert_allclose(_pi_block_sums(gpi, pi, 20), gpi1, rtol=1e-8, atol=1e-8 * np.abs(gpi1).max())


def _masked_coupled_400(seed):
    """Random reversible 400 x 400 model: every single substitution and 5 % of the double ones allowed."""
    rng = np.random.default_rng(seed)
    a, b = np.divmod(np.arange(400), 20)
    changes = (a[:, None] != a[None, :]).astype(int) + (b[:, None] != b[None, :]).astype(int)
    extra = rng.random((400, 400)) < 0.05
    extra = extra | extra.T
    mask = ((changes == 1) | ((changes == 2) & extra)).astype(float)
    from cherryml_b200.markov_chain import compute_stationary_distribution

    Q, _ = _random_reversible(400, seed, mask=mask)
    return Q, compute_stationary_distribution(Q), mask


@pytest.mark.gpu
def test_demo_family_directional_derivatives_and_determinism(tmp_path):
    """13gs_1_A under a coupled, masked random 400 x 400 model: central differences of the forward pass
    (cherry_tree_log_likelihood, c = 2) along three random directions match <dQ, D>; two calls are bitwise
    identical."""
    from cherryml_b200.evaluation import pair_log_likelihood_gradient

    tree, msa, cmap = _demo_family(str(tmp_path))
    Q, pi, mask = _masked_coupled_400(4)
    ll, lls, gQ, gpi = pair_log_likelihood_gradient(tree, msa, cmap, AA, pi, Q)
    fwd = _forward_pair_lls(tree, msa, cmap, AA, pi, Q)
    assert np.all(_rel(np.array(lls), fwd) <= 1e-12)
    rng = np.random.default_rng(8)
    h = 1e-5
    for _ in range(3):
        D = rng.standard_normal((400, 400)) * mask * np.abs(Q)
        np.fill_diagonal(D, 0.0)
        np.fill_diagonal(D, -D.sum(axis=1))
        fd = (_forward_pair_lls(tree, msa, cmap, AA, pi, Q + h * D).sum()
              - _forward_pair_lls(tree, msa, cmap, AA, pi, Q - h * D).sum()) / (2 * h)
        exact = float(np.sum(gQ * D))
        assert abs(fd - exact) <= 1e-6 * abs(exact), (fd, exact)
    a = _gpu_pair_posterior(tree, msa, cmap, AA, pi, Q)
    b = _gpu_pair_posterior(tree, msa, cmap, AA, pi, Q)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    g2 = pair_log_likelihood_gradient(tree, msa, cmap, AA, pi, Q)
    assert g2[0] == ll and np.array_equal(g2[2], gQ) and np.array_equal(g2[3], gpi)


def _write_pair_families(root, fams, alphabet):
    """fams: {name: (tree, msa, contact_map)} -> (tree_dir, msa_dir, contact_map_dir)."""
    from cherryml_b200.io import write_contact_map, write_msa, write_tree

    dirs = [os.path.join(root, d) for d in ("trees", "msas", "contact_maps")]
    for d in dirs:
        os.makedirs(d, exist_ok=True)
    for name, (tree, msa, cmap) in fams.items():
        write_tree(tree, os.path.join(dirs[0], name + ".txt"))
        write_msa(msa, os.path.join(dirs[1], name + ".txt"))
        write_contact_map(cmap, os.path.join(dirs[2], name + ".txt"))
    return dirs


@pytest.mark.gpu
def test_autograd_gradcheck_pairs(tmp_path):
    import torch

    from cherryml_b200.estimation import PairTreeLikelihoodData, TreeLogLikelihood

    rng = np.random.default_rng(7)
    alphabet = DNA[:3]
    fams = {}
    for f in ("f", "g"):
        t = _random_tree(6, rng)
        fams[f] = (t, *_pair_msa(t, alphabet, 9, rng))
    dirs = _write_pair_families(str(tmp_path), fams, alphabet)
    data = PairTreeLikelihoodData(*dirs, ["f", "g"], alphabet)
    assert data.n_pairs == 18
    Q0, pi0 = _coupled(3, seed=9)
    Q = torch.tensor(Q0, dtype=torch.float64, device="cuda", requires_grad=True)
    pi = torch.tensor(pi0, dtype=torch.float64, device="cuda", requires_grad=True)
    assert torch.autograd.gradcheck(lambda q, p: TreeLogLikelihood.apply(q, p, data), (Q, pi), eps=1e-6, atol=1e-6,
                                    rtol=1e-5)
    a, b = data.evaluate(Q, pi), data.evaluate(Q, pi)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def _simulate_pairs(Q2, pi2, alphabet, n_leaves, n_pairs, rng):
    from scipy.linalg import expm

    S = len(alphabet)
    tree = _random_tree(n_leaves, rng)
    states = {tree.root(): rng.choice(len(pi2), n_pairs, p=pi2)}
    for v in reversed(tree.postorder_traversal()):
        if v == tree.root():
            continue
        p, length = tree.parent(v)
        cdf = np.cumsum(expm(length * Q2), axis=1)[states[p]]
        states[v] = np.minimum((rng.random(n_pairs)[:, None] > cdf).sum(axis=1), len(pi2) - 1)
    msa = {v: "".join(alphabet[x // S] + alphabet[x % S] for x in states[v]) for v in tree.leaves()}
    cmap = np.zeros((2 * n_pairs, 2 * n_pairs))
    for k in range(n_pairs):
        cmap[2 * k, 2 * k + 1] = cmap[2 * k + 1, 2 * k] = 1
    return tree, msa, cmap


@pytest.mark.gpu
def test_coevolution_mle_recovers_simulated_model(tmp_path):
    """Su = 9: data simulated under a coupled model; the ML estimate scores at least the true model and lies
    close to it (mean relative error below 0.25 and below half the start's)."""
    import torch

    from cherryml_b200 import caching
    from cherryml_b200.estimation import PairTreeLikelihoodData, coevolution_tree_likelihood_mle
    from cherryml_b200.evaluation import mean_relative_error
    from cherryml_b200.io import read_rate_matrix, write_rate_matrix

    alphabet = list("ACG")
    states = [a + b for a in alphabet for b in alphabet]
    rng = np.random.default_rng(2025)
    Q_true, pi_true = _coupled(3, seed=77)
    fams = {f"sim{i}": _simulate_pairs(Q_true, pi_true, alphabet, 48, 60, rng) for i in range(24)}
    dirs = _write_pair_families(str(tmp_path), fams, alphabet)
    Q0, _ = _coupled(3, seed=5)
    write_rate_matrix(Q0, states, str(tmp_path / "init.txt"))
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        out = coevolution_tree_likelihood_mle(tree_dir=dirs[0], msa_dir=dirs[1], contact_map_dir=dirs[2],
                                              families=sorted(fams), amino_acids=alphabet,
                                              initialization_path=str(tmp_path / "init.txt"), num_epochs=300,
                                              learning_rate=0.05)["output_rate_matrix_dir"]
    finally:
        caching.set_cache_dir(None)
    Q_ml = read_rate_matrix(os.path.join(out, "result.txt"))
    assert list(Q_ml.index) == states and list(Q_ml.columns) == states
    best = float(open(os.path.join(out, "log_likelihood.txt")).read())
    data = PairTreeLikelihoodData(*dirs, sorted(fams), alphabet)
    true_ll = float(data.evaluate(torch.tensor(Q_true, device="cuda"), torch.tensor(pi_true, device="cuda"))[0])
    before, after = mean_relative_error(Q_true, Q0), mean_relative_error(Q_true, Q_ml.to_numpy())
    print(f"\nlog-likelihood: true model {true_ll}, ML {best}; mean relative error: start {before:.4f}, ML {after:.4f}")
    assert best >= true_ll
    assert after <= 0.25 and after <= before / 2


@pytest.mark.gpu
def test_coevolution_mle_demo_families_files_and_cache(tmp_path):
    """Two demo families, 3 epochs at Su = 400 from LG x LG: the log-likelihood rises, the output files are
    labelled with the 400 pair states, and a second call is a cache hit (no launch)."""
    from cherryml_b200 import caching
    from cherryml_b200.estimation import coevolution_tree_likelihood_mle
    from cherryml_b200.evaluation import pair_log_likelihood_gradient
    from cherryml_b200.io import read_rate_matrix, write_contact_map
    from cherryml_b200.markov_chain import compute_stationary_distribution, get_lg_x_lg_path

    fams = ["13gs_1_A", "1a92_1_A"]
    data = {}
    os.makedirs(tmp_path / "matched")
    for f in fams:
        tree, msa, cmap = _demo_family(str(tmp_path), f)
        write_contact_map(cmap, str(tmp_path / "matched" / f"{f}.txt"))  # the maximal matching
        data[f] = (tree, msa, cmap)
    kw = dict(tree_dir=str(tmp_path / "trees"), msa_dir=str(tmp_path / "msas"),
              contact_map_dir=str(tmp_path / "matched"), families=fams, amino_acids=AA,
              initialization_path=get_lg_x_lg_path(), num_epochs=3)
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        out = coevolution_tree_likelihood_mle(**kw)["output_rate_matrix_dir"]
        before = _lib.launch_count()
        assert coevolution_tree_likelihood_mle(**kw)["output_rate_matrix_dir"] == out
        assert _lib.launch_count() == before
    finally:
        caching.set_cache_dir(None)
    assert {"log_likelihood.txt", "profiling.txt", "result.txt"} <= set(os.listdir(out))
    Q = read_rate_matrix(os.path.join(out, "result.txt"))
    states = [a + b for a in AA for b in AA]
    assert list(Q.index) == states and list(Q.columns) == states
    best = float(open(os.path.join(out, "log_likelihood.txt")).read())
    assert "posterior" in open(os.path.join(out, "profiling.txt")).read()
    Q0 = read_rate_matrix(get_lg_x_lg_path()).to_numpy()

    def total(Qx):
        pi = compute_stationary_distribution(Qx)
        return sum(pair_log_likelihood_gradient(*data[f], AA, pi, Qx)[0] for f in fams)

    start = total(Q0)
    assert best > start
    assert abs(total(Q.to_numpy()) - best) <= 1e-9 * abs(best)
