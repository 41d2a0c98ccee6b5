"""Exact gradient of the tree log-likelihood (cherry_tree_ll_posterior + the fit's expm adjoint) and the
maximum-likelihood stage built on it (tree_likelihood_mle).

CPU: the numpy oracle (oracle/likelihood_grad_oracle.py) against central finite differences of the
likelihood oracle, its posterior identities, and the new C entry points' argument checks.
GPU: per-site log-likelihoods bitwise equal to cherry_tree_log_likelihood's, edge posteriors, root
posteriors and both gradients against the oracle (1e-9 relative), determinism, gradcheck of the autograd
node, the stage's files and cache, and recovery of WAG from data simulated under it."""
import ctypes
import os
import tarfile

import numpy as np
import pytest

from cherryml_b200 import _lib
from tests._ll_cases import (AA, DNA, _demo_family, _model, _random_msa, _random_reversible, _random_tree, _rates,
                             _scratch_formula, _simulate_family, _synthetic_cases, _write_families, rate_matrix)
from tests.conftest import GOLDEN


# ------------------------------------------------------------------ CPU: oracle and ABI

def _fd_cases():
    rng = np.random.default_rng(5)
    out = []
    t = _random_tree(5, rng)
    out.append(("five_leaves", t, _random_msa(t, DNA, 6, rng, gap_frac=0.0), _rates(6, 2, rng), DNA))
    t = _random_tree(6, rng, root_children=4)
    out.append(("multifurcating_root", t, _random_msa(t, DNA, 5, rng, gap_frac=0.0), _rates(5, 1, rng), DNA))
    t = _random_tree(5, rng, zero_branch=True)
    out.append(("zero_length_branch", t, _random_msa(t, DNA, 5, rng, gap_frac=0.0), _rates(5, 2, rng), DNA))
    t = _random_tree(5, rng)
    out.append(("gaps", t, _random_msa(t, DNA, 6, rng, gap_frac=0.3, all_gap_column=True), _rates(6, 3, rng), DNA))
    return out


@pytest.mark.parametrize("case", _fd_cases(), ids=lambda c: c[0])
def test_oracle_gradient_matches_finite_differences(case):
    from oracle.likelihood_grad_oracle import log_likelihood_gradient
    from oracle.likelihood_oracle import log_likelihood

    _, tree, msa, rates, alphabet = case
    S = len(alphabet)
    Q, pi = _random_reversible(S, seed=3)
    res = log_likelihood_gradient(tree, msa, rates, alphabet, pi, Q)

    def ll(Qx, pix):
        return log_likelihood(tree, msa, None, rates, alphabet, pix, Qx, None, None)[0]

    assert abs(res["ll"] - ll(Q, pi)) <= 1e-12 * abs(res["ll"])
    h = 1e-5
    fd_Q = np.zeros((S, S))
    for i in range(S):
        for j in range(S):
            E = np.zeros((S, S))
            E[i, j] = h
            fd_Q[i, j] = (ll(Q + E, pi) - ll(Q - E, pi)) / (2 * h)
    fd_pi = np.zeros(S)
    for i in range(S):
        e = np.zeros(S)
        e[i] = h * pi[i]
        fd_pi[i] = (ll(Q, pi + e) - ll(Q, pi - e)) / (2 * h * pi[i])
    np.testing.assert_allclose(res["grad_Q"], fd_Q, rtol=1e-6, atol=1e-6 * np.abs(fd_Q).max())
    np.testing.assert_allclose(res["grad_pi"], fd_pi, rtol=1e-6, atol=1e-6 * np.abs(fd_pi).max())


@pytest.mark.parametrize("case", _fd_cases(), ids=lambda c: c[0])
def test_oracle_posterior_identities(case):
    from oracle.likelihood_grad_oracle import log_likelihood_gradient

    _, tree, msa, rates, alphabet = case
    Q, pi = _random_reversible(len(alphabet), seed=4)
    res = log_likelihood_gradient(tree, msa, rates, alphabet, pi, Q)
    for v, mass in res["edge_mass"].items():
        np.testing.assert_allclose(mass, 1.0, rtol=1e-12, err_msg=v)
    assert abs(res["root"].sum() - len(rates)) <= 1e-12 * len(rates)
    np.testing.assert_allclose(res["root"], res["grad_pi"] * pi, rtol=1e-14)


def test_posterior_entry_arguments_without_gpu():
    lib = _lib.load()
    assert lib.cherry_tree_ll_posterior(0, 3, 1, 0, 1, 0, 2, 0, 0, 0, 20, 4, 0, 0, 0, 0, 0, 0) == -1
    assert b"null pointer" in lib.cherry_last_error()
    buf = (ctypes.c_int32 * 64)()
    p = ctypes.addressof(buf)
    # more than 32 states: checked before anything is read or launched
    assert lib.cherry_tree_ll_posterior(p, 3, 1, p, 1, p, 2, p, p, p, 33, 4, p, 1 << 20, p, p, p, 0) == -3
    # p_index out of range (host array, checked before any launch)
    pidx = np.array([0, 5, 0], dtype=np.int32)
    cat = np.zeros(4, dtype=np.int32)
    assert lib.cherry_tree_ll_posterior(p, 3, 1, pidx.ctypes.data, 1, p, 2, p, cat.ctypes.data, p, 20, 4, p, 1 << 30,
                                        p, p, p, 0) == -1
    assert b"p_index" in lib.cherry_last_error()
    pidx[1] = 1
    cat[2] = 3  # category beyond n_cats
    assert lib.cherry_tree_ll_posterior(p, 3, 1, pidx.ctypes.data, 1, p, 2, p, cat.ctypes.data, p, 20, 4, p, 1 << 30,
                                        p, p, p, 0) == -1
    cat[2] = 0
    assert lib.cherry_tree_ll_posterior(p, 3, 1, pidx.ctypes.data, 1, p, 2, p, cat.ctypes.data, p, 20, 4, p, 16,
                                        p, p, p, 0) == -1
    assert b"scratch too small" in lib.cherry_last_error()
    for S, n_nodes, depth, n_cats, n_m, n_units in ((20, 2047, 30, 4, 7000, 210), (4, 5, 2, 1, 3, 1),
                                                    (21, 1537, 2, 20, 9000, 300), (32, 1, 0, 1, 1, 9)):
        unit_cat = np.random.default_rng(S).integers(0, n_cats, n_units).astype(np.int32)
        got = lib.cherry_tree_ll_posterior_scratch_bytes(S, n_nodes, depth, n_cats, n_m, n_units, unit_cat.ctypes.data)
        assert got == _scratch_formula(S, n_nodes, depth, n_cats, n_m, unit_cat)
    bad = np.array([0, 1, 2], dtype=np.int32)
    assert lib.cherry_tree_ll_posterior_scratch_bytes(20, 5, 2, 2, 3, 3, bad.ctypes.data) == 0
    assert lib.cherry_tree_ll_posterior_scratch_bytes(33, 5, 2, 3, 3, 3, bad.ctypes.data) == 0


# ------------------------------------------------------------------ GPU

def _gpu_posterior(tree, msa, rates, alphabet, pi, Q):
    import torch

    from cherryml_b200.evaluation._likelihood import _expm_transposed, _SiteFamily

    fam = _SiteFamily(tree, msa, rates, alphabet, "cuda")
    P = _expm_transposed(Q, fam.exponents, "cuda")
    ll, W, root = fam.posterior(P, torch.from_numpy(np.asarray(pi, dtype=np.float64)).cuda())
    return fam.exponents, ll.cpu().numpy(), W.cpu().numpy(), root.cpu().numpy()


def _check_against_oracle(tree, msa, rates, alphabet, Q, pi):
    from cherryml_b200.evaluation import dp_likelihood_computation, log_likelihood_gradient
    from oracle.likelihood_grad_oracle import log_likelihood_gradient as oracle_gradient

    S = len(alphabet)
    exps, lls_post, W, root = _gpu_posterior(tree, msa, rates, alphabet, pi, Q)
    ll, lls, gQ, gpi = log_likelihood_gradient(tree, msa, rates, alphabet, pi, Q)
    _, lls_fwd = dp_likelihood_computation(tree=tree, msa=msa, contact_map=None, site_rates=rates,
                                           amino_acids=alphabet, pi_1=pi, Q_1=Q)
    # bitwise: the same per-unit arithmetic as cherry_tree_log_likelihood
    assert np.array_equal(np.array(lls), np.array(lls_fwd)) and np.array_equal(lls_post, np.array(lls_fwd))
    ref = oracle_gradient(tree, msa, rates, alphabet, pi, Q)
    assert abs(ll - ref["ll"]) <= 1e-10 * abs(ref["ll"])
    W_ref = np.stack([ref["W"].get(t, np.zeros((S, S))) for t in exps])
    np.testing.assert_allclose(W, W_ref, rtol=1e-9, atol=1e-12 * max(1.0, np.abs(W_ref).max()))
    np.testing.assert_allclose(root, ref["root"], rtol=1e-9, atol=1e-12 * len(rates))
    np.testing.assert_allclose(gQ, ref["grad_Q"], rtol=1e-9, atol=1e-9 * np.abs(ref["grad_Q"]).max())
    np.testing.assert_allclose(gpi, ref["grad_pi"], rtol=1e-9, atol=1e-9 * np.abs(ref["grad_pi"]).max())


@pytest.mark.gpu
@pytest.mark.parametrize("case", _synthetic_cases(), ids=lambda c: c[0])
def test_posterior_and_gradient_against_oracle(case):
    _, tree, msa, rates, alphabet, model = case
    Q, pi = _model(model, len(alphabet))
    _check_against_oracle(tree, msa, rates, alphabet, Q, pi)


@pytest.mark.gpu
def test_demo_family_against_oracle_and_deterministic(tmp_path):
    """13gs_1_A: 1024 leaves x 210 sites, its FastTree tree and site-rate categories, LG."""
    from cherryml_b200.evaluation import log_likelihood_gradient

    tree, msa, rates = _demo_family(str(tmp_path))
    Q, pi = _model("lg", 20)
    _check_against_oracle(tree, msa, rates, AA, Q, pi)
    a = _gpu_posterior(tree, msa, rates, AA, pi, Q)
    b = _gpu_posterior(tree, msa, rates, AA, pi, Q)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    g1 = log_likelihood_gradient(tree, msa, rates, AA, pi, Q)
    g2 = log_likelihood_gradient(tree, msa, rates, AA, pi, Q)
    assert g1[0] == g2[0] and np.array_equal(g1[2], g2[2]) and np.array_equal(g1[3], g2[3])


@pytest.mark.gpu
def test_autograd_gradcheck(tmp_path):
    import torch

    from cherryml_b200.estimation import TreeLikelihoodData, TreeLogLikelihood

    rng = np.random.default_rng(7)
    t = _random_tree(6, rng)
    dirs = _write_families(str(tmp_path), {"f": (t, _random_msa(t, DNA, 20, rng), _rates(20, 2, rng))})
    data = TreeLikelihoodData(*dirs, ["f"], DNA)
    Q0, pi0 = _random_reversible(4, seed=9)
    Q = torch.tensor(Q0, dtype=torch.float64, device="cuda", requires_grad=True)
    pi = torch.tensor(pi0, dtype=torch.float64, device="cuda", requires_grad=True)
    assert torch.autograd.gradcheck(lambda q, p: TreeLogLikelihood.apply(q, p, data), (Q, pi), eps=1e-6, atol=1e-6,
                                    rtol=1e-5)


@pytest.mark.gpu
def test_tree_likelihood_mle_demo_families(tmp_path):
    from cherryml_b200 import caching
    from cherryml_b200.estimation import tree_likelihood_mle
    from cherryml_b200.evaluation import compute_log_likelihoods
    from cherryml_b200.io import read_rate_matrix, write_probability_distribution, write_rate_matrix
    from cherryml_b200.markov_chain import _rate_matrix_path, compute_stationary_distribution

    with tarfile.open(os.path.join(GOLDEN, "demo_data.tar.xz")) as tf:
        fams = sorted(n.split("/")[1][:-4] for n in tf.getnames() if n.startswith("trees/") and n.endswith(".txt"))[:8]
        tf.extractall(tmp_path, members=[tf.getmember(f"{d}/{f}.txt") for d in ("msas", "trees", "site_rates")
                                         for f in fams])
    dirs = dict(tree_dir=str(tmp_path / "trees"), msa_dir=str(tmp_path / "msas"),
                site_rates_dir=str(tmp_path / "site_rates"))
    lg = _rate_matrix_path("lg")
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        kw = dict(**dirs, families=fams, amino_acids=AA, initialization_path=lg, num_epochs=10)
        out = tree_likelihood_mle(**kw)["output_rate_matrix_dir"]
        before = _lib.launch_count()
        assert tree_likelihood_mle(**kw)["output_rate_matrix_dir"] == out and _lib.launch_count() == before
        best = float(open(os.path.join(out, "log_likelihood.txt")).read())
        Q = read_rate_matrix(os.path.join(out, "result.txt")).to_numpy()

        def total(Q_path, pi_path):
            d = compute_log_likelihoods(**dirs, contact_map_dir=None, families=fams, amino_acids=AA,
                                        pi_1_path=pi_path, Q_1_path=Q_path, reversible_1=True, device_1="cuda",
                                        pi_2_path=None, Q_2_path=None, reversible_2=None, device_2=None,
                                        num_processes=1)["output_likelihood_dir"]
            return sum(float(open(os.path.join(d, f + ".txt")).readline()) for f in fams)

        write_probability_distribution(compute_stationary_distribution(Q), AA, str(tmp_path / "pi_ml.txt"))
        write_rate_matrix(Q, AA, str(tmp_path / "Q_ml.txt"))
        Q_lg = read_rate_matrix(lg).to_numpy()
        write_probability_distribution(compute_stationary_distribution(Q_lg), AA, str(tmp_path / "pi_lg.txt"))
        start = total(lg, str(tmp_path / "pi_lg.txt"))
        assert best >= start
        assert abs(total(str(tmp_path / "Q_ml.txt"), str(tmp_path / "pi_ml.txt")) - best) <= 1e-9 * abs(best)
    finally:
        caching.set_cache_dir(None)


@pytest.mark.gpu
def test_recovers_wag_from_lg_start(tmp_path):
    from cherryml_b200 import caching
    from cherryml_b200.estimation import tree_likelihood_mle
    from cherryml_b200.evaluation import mean_relative_error
    from cherryml_b200.io import read_rate_matrix
    from cherryml_b200.markov_chain import _rate_matrix_path, compute_stationary_distribution

    rng = np.random.default_rng(2024)
    wag, lg = rate_matrix("wag"), rate_matrix("lg")
    pi = compute_stationary_distribution(wag)
    fams = {f"sim{i}": _simulate_family(wag, pi, 64, 100, rng) for i in range(64)}
    dirs = _write_families(str(tmp_path), fams)
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        out = tree_likelihood_mle(tree_dir=dirs[0], msa_dir=dirs[1], site_rates_dir=dirs[2], families=sorted(fams),
                                  amino_acids=AA, initialization_path=_rate_matrix_path("lg"),
                                  num_epochs=150)["output_rate_matrix_dir"]
    finally:
        caching.set_cache_dir(None)
    Q = read_rate_matrix(os.path.join(out, "result.txt")).to_numpy()
    before, after = mean_relative_error(wag, lg), mean_relative_error(wag, Q)
    print(f"\nmean relative error to WAG: LG {before:.4f}, ML from LG {after:.4f}")
    assert after <= before / 2
