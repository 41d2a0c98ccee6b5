"""Exact branch-length gradient of the tree log-likelihood (cherry_tree_ll_edge_derivatives) and the
maximum-likelihood branch-length stage built on it (phylogeny_estimation.branch_length_mle).

CPU: the numpy oracle (oracle.likelihood_grad_oracle.branch_length_gradient) against central finite
differences of the likelihood oracle and the pulley principle, and the new C entry point's argument checks
and scratch formula.
GPU: dtau and the length gradient against the oracle (1e-9 relative), ll / W / root bitwise equal to
cherry_tree_ll_posterior's, determinism, the pulley principle, the scaling identity against the Q
gradient, and the stage: recovery of simulated lengths, its files, per-family independence, its cache and a
two-iteration CherryML run on refitted demo trees."""
import ctypes
import functools
import os
import tarfile

import numpy as np
import pytest

from cherryml_b200 import _lib
from cherryml_b200.io import Tree
from tests._ll_cases import (AA, DNA, _demo_family, _model, _random_msa, _random_reversible, _random_tree, _rates,
                             _scratch_formula, _simulate_family, _synthetic_cases, _write_families, rate_matrix)
from tests.conftest import GOLDEN


def _with_length(tree: Tree, child: str, length: float) -> Tree:
    out = Tree()
    out.add_nodes(tree.nodes())
    out.add_edges([(u, v, length if v == child else d) for u, v, d in tree.edges()])
    return out


# ------------------------------------------------------------------ CPU: oracle and ABI

def _fd_cases():
    """(id, tree, msa, site_rates, alphabet, model): 4 and 20 states, 1 and 4 rate categories."""
    rng = np.random.default_rng(17)
    out = []
    for S_name, alphabet, model in (("dna", DNA, "random"), ("aa", AA, "lg")):
        for n_cats in (1, 4):
            t = _random_tree(5, rng, root_children=3 if n_cats == 4 else 2)
            out.append((f"{S_name}_{n_cats}cat", t, _random_msa(t, alphabet, 6, rng, gap_frac=0.15),
                        _rates(6, n_cats, rng), alphabet, model))
    return out


@pytest.mark.parametrize("case", _fd_cases(), ids=lambda c: c[0])
def test_oracle_length_gradient_matches_finite_differences(case):
    from oracle.likelihood_grad_oracle import branch_length_gradient
    from oracle.likelihood_oracle import log_likelihood

    _, tree, msa, rates, alphabet, model = case
    Q, pi = _model(model, len(alphabet))
    res = branch_length_gradient(tree, msa, rates, alphabet, pi, Q)

    def ll(t):
        return log_likelihood(t, msa, None, rates, alphabet, pi, Q, None, None)[0]

    assert abs(res["ll"] - ll(tree)) <= 1e-12 * abs(res["ll"])
    cats = sorted(set(rates))
    for u, v, length in tree.edges():
        h = 1e-5 * length
        fd = (ll(_with_length(tree, v, length + h)) - ll(_with_length(tree, v, length - h))) / (2 * h)
        g = res["grad_length"][v]
        assert abs(g - fd) <= 1e-6 * max(1.0, abs(fd)), (v, g, fd)
        assert g == pytest.approx(float(np.dot(res["dtau"][v], cats)), rel=1e-15)


def _pulley_case(S, seed):
    rng = np.random.default_rng(seed)
    t = _random_tree(9, rng, root_children=2)
    alphabet = DNA if S == 4 else AA
    return t, _random_msa(t, alphabet, 40, rng), _rates(40, 4, rng), alphabet


@pytest.mark.parametrize("S", [4, 20])
def test_oracle_pulley_principle(S):
    """Reversible Q, pi stationary: moving the root along its two edges does not change L, so the two
    edges under a root of degree two have equal derivatives."""
    from oracle.likelihood_grad_oracle import branch_length_gradient

    tree, msa, rates, alphabet = _pulley_case(S, seed=S)
    Q, pi = _random_reversible(S, seed=31)
    g = branch_length_gradient(tree, msa, rates, alphabet, pi, Q)["grad_length"]
    a, b = [c for c, _ in tree.children(tree.root())]
    assert g[a] == pytest.approx(g[b], rel=1e-10)


def test_edge_derivatives_entry_arguments_without_gpu():
    lib = _lib.load()
    buf = (ctypes.c_int32 * 64)()
    p = ctypes.addressof(buf)
    args = [p, 3, 1, p, 1, p, 2, p, p, p, p, 20, 4, p, 1 << 20, p, p, p, p, 0]
    assert lib.cherry_tree_ll_edge_derivatives(*[0 if i not in (1, 2, 4, 6, 11, 12, 14, 19) else a
                                                 for i, a in enumerate(args)]) == -1
    assert b"null pointer" in lib.cherry_last_error()
    for i in (10, 18):  # Q, dtau_out
        bad = list(args)
        bad[i] = 0
        assert lib.cherry_tree_ll_edge_derivatives(*bad) == -1
        assert b"null pointer" in lib.cherry_last_error()
    big = list(args)
    big[11] = 33
    assert lib.cherry_tree_ll_edge_derivatives(*big) == -3  # more than 32 states
    pidx = np.array([0, 5, 0], dtype=np.int32)
    cat = np.zeros(4, dtype=np.int32)
    args[3], args[8], args[14] = pidx.ctypes.data, cat.ctypes.data, 1 << 30
    assert lib.cherry_tree_ll_edge_derivatives(*args) == -1
    assert b"p_index" in lib.cherry_last_error()
    pidx[1] = 1
    cat[2] = 3  # category beyond n_cats
    assert lib.cherry_tree_ll_edge_derivatives(*args) == -1
    cat[2] = 0
    args[14] = 16
    assert lib.cherry_tree_ll_edge_derivatives(*args) == -1
    assert b"scratch too small" in lib.cherry_last_error()


def test_edge_derivatives_scratch_formula():
    lib = _lib.load()
    for S, n_nodes, depth, n_cats, n_m, n_units in ((20, 2047, 30, 4, 7000, 210), (4, 5, 2, 1, 3, 1),
                                                    (21, 1537, 2, 20, 9000, 300), (32, 1, 0, 1, 1, 9)):
        unit_cat = np.random.default_rng(S).integers(0, n_cats, n_units).astype(np.int32)
        G = max(1, 256 // S)
        ctas = int(sum((c + G - 1) // G for c in np.bincount(unit_cat, minlength=n_cats)))
        got = lib.cherry_tree_ll_edge_derivatives_scratch_bytes(S, n_nodes, depth, n_cats, n_m, n_units,
                                                                unit_cat.ctypes.data)
        # the posterior pass's scratch plus one double per (CTA, node)
        assert got == _scratch_formula(S, n_nodes, depth, n_cats, n_m, unit_cat) + 8 * ctas * n_nodes
    bad = np.array([0, 1, 2], dtype=np.int32)
    assert lib.cherry_tree_ll_edge_derivatives_scratch_bytes(20, 5, 2, 2, 3, 3, bad.ctypes.data) == 0
    assert lib.cherry_tree_ll_edge_derivatives_scratch_bytes(33, 5, 2, 3, 3, 3, bad.ctypes.data) == 0


# ------------------------------------------------------------------ GPU: the entry point

def _gpu_both(tree, msa, rates, alphabet, pi, Q):
    """(names, rates, posterior outputs, edge-derivative outputs) as numpy, on the same matrices."""
    import torch

    from cherryml_b200.evaluation._likelihood import _expm_transposed, _SiteFamily

    fam = _SiteFamily(tree, msa, rates, alphabet, "cuda")
    P = _expm_transposed(Q, fam.exponents, "cuda")
    d_pi = torch.from_numpy(np.asarray(pi, dtype=np.float64)).cuda()
    post = [x.cpu().numpy() for x in fam.posterior(P, d_pi)]
    d_Q = torch.from_numpy(np.ascontiguousarray(Q, dtype=np.float64)).cuda()
    der = [x.cpu().numpy() for x in fam.edge_derivatives(P, d_pi, d_Q)]
    return fam.names, fam.rates, post, der


def _check_against_oracle(tree, msa, rates, alphabet, Q, pi):
    from cherryml_b200.evaluation import branch_length_gradient, dp_likelihood_computation
    from oracle.likelihood_grad_oracle import branch_length_gradient as oracle_gradient

    names, cats, post, der = _gpu_both(tree, msa, rates, alphabet, pi, Q)
    for x, y in zip(post, der[:3]):  # ll, W, root: the posterior pass's, bit for bit
        assert np.array_equal(x, y)
    dtau = der[3]
    assert dtau.shape == (len(names), len(cats)) and np.all(dtau[-1] == 0.0)
    ll, lls, grad = branch_length_gradient(tree, msa, rates, alphabet, pi, Q)
    _, lls_fwd = dp_likelihood_computation(tree=tree, msa=msa, contact_map=None, site_rates=rates,
                                           amino_acids=alphabet, pi_1=pi, Q_1=Q)
    assert np.array_equal(np.array(lls), np.array(lls_fwd))
    assert sorted(grad) == sorted(names[:-1])
    ref = oracle_gradient(tree, msa, rates, alphabet, pi, Q)
    assert abs(ll - ref["ll"]) <= 1e-10 * abs(ref["ll"])
    if len(names) == 1:
        return
    d_ref = np.stack([ref["dtau"][v] for v in names[:-1]])
    np.testing.assert_allclose(dtau[:-1], d_ref, rtol=1e-9, atol=1e-9 * np.abs(d_ref).max())
    g_ref = np.array([ref["grad_length"][v] for v in names[:-1]])
    g = np.array([grad[v] for v in names[:-1]])
    np.testing.assert_allclose(g, g_ref, rtol=1e-9, atol=1e-9 * np.abs(g_ref).max())


def _two_leaves():
    rng = np.random.default_rng(3)
    t = Tree()
    t.add_nodes(["r", "a", "b"])
    t.add_edges([("r", "a", 0.3), ("r", "b", 0.05)])
    return ("two_leaves", t, _random_msa(t, AA, 33, rng), _rates(33, 4, rng), AA, "lg")


@pytest.mark.gpu
@pytest.mark.parametrize("case", _synthetic_cases() + [_two_leaves()], ids=lambda c: c[0])
def test_edge_derivatives_against_oracle(case):
    _, tree, msa, rates, alphabet, model = case
    Q, pi = _model(model, len(alphabet))
    _check_against_oracle(tree, msa, rates, alphabet, Q, pi)


@pytest.mark.gpu
def test_demo_family_against_oracle_deterministic_and_scaling_identity(tmp_path):
    """13gs_1_A (1024 leaves x 210 sites, 13 rate categories, LG).  Scaling identity: L(cQ, t) = L(Q, ct),
    so sum_i length_i d ll / d length_i = sum_ab Q_ab (d ll / d Q)_ab."""
    from cherryml_b200.evaluation import branch_length_gradient, log_likelihood_gradient

    tree, msa, rates = _demo_family(str(tmp_path))
    Q, pi = _model("lg", 20)
    _check_against_oracle(tree, msa, rates, AA, Q, pi)
    a = _gpu_both(tree, msa, rates, AA, pi, Q)[3]
    b = _gpu_both(tree, msa, rates, AA, pi, Q)[3]
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    _, _, grad = branch_length_gradient(tree, msa, rates, AA, pi, Q)
    lhs = sum(tree.parent(v)[1] * g for v, g in grad.items())
    gQ = log_likelihood_gradient(tree, msa, rates, AA, pi, Q)[2]
    rhs = float(np.sum(Q * gQ))
    assert abs(lhs - rhs) <= 1e-9 * abs(rhs), (lhs, rhs)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [4, 20])
def test_pulley_principle_on_gpu(S):
    from cherryml_b200.evaluation import branch_length_gradient

    tree, msa, rates, alphabet = _pulley_case(S, seed=S)
    Q, pi = _random_reversible(S, seed=31)
    g = branch_length_gradient(tree, msa, rates, alphabet, pi, Q)[2]
    a, b = [c for c, _ in tree.children(tree.root())]
    assert g[a] == pytest.approx(g[b], rel=1e-9)


# ------------------------------------------------------------------ GPU: the stage

def _scaled(tree, rng, sigma):
    """`tree` with every length multiplied by exp(N(0, sigma))."""
    out = Tree()
    out.add_nodes(tree.nodes())
    out.add_edges([(u, v, d * float(np.exp(rng.normal(0, sigma)))) for u, v, d in tree.edges()])
    return out


def _read(d, f):
    from cherryml_b200.io import read_log_likelihood, read_site_rates, read_tree

    return (read_tree(os.path.join(d["output_tree_dir"], f + ".txt")),
            read_site_rates(os.path.join(d["output_site_rates_dir"], f + ".txt")),
            read_log_likelihood(os.path.join(d["output_likelihood_dir"], f + ".txt")))


N_SITES = 2000


@pytest.fixture(scope="module")
def simulated(tmp_path_factory):
    """Three families simulated under LG down known 16-leaf trees (2000 sites, rates 0.5 / 1 / 2), each
    written with its lengths perturbed by a factor exp(N(0, 0.5))."""
    from cherryml_b200.markov_chain import compute_stationary_distribution

    root = str(tmp_path_factory.mktemp("blmle"))
    rng = np.random.default_rng(2026)
    Q = rate_matrix("lg")
    pi = compute_stationary_distribution(Q)
    truth, fams = {}, {}
    for i in range(3):
        t, msa, rates = _simulate_family(Q, pi, 16, N_SITES, rng)
        truth[f"sim{i}"] = t
        fams[f"sim{i}"] = (_scaled(t, rng, 0.5), msa, rates)
    dirs = _write_families(root, fams)
    from cherryml_b200.markov_chain import _rate_matrix_path

    return dict(root=root, truth=truth, fams=fams, tree_dir=dirs[0], msa_dir=dirs[1], site_rates_dir=dirs[2],
                Q=Q, pi=pi, lg=_rate_matrix_path("lg"))


def _run(sim, families, out, **kw):
    from cherryml_b200.phylogeny_estimation import branch_length_mle

    dirs = {k: os.path.join(sim["root"], out, k) for k in ("output_tree_dir", "output_site_rates_dir",
                                                           "output_likelihood_dir")}
    branch_length_mle(tree_dir=sim["tree_dir"], site_rates_dir=sim["site_rates_dir"], msa_dir=sim["msa_dir"],
                      families=families, rate_matrix_path=sim["lg"], amino_acids=AA, num_processes=1,
                      num_epochs=kw.pop("num_epochs", 300), **dirs, **kw)
    return dirs


@pytest.mark.gpu
def test_stage_recovers_simulated_lengths(simulated):
    """ML lengths from perturbed starts score at least as well as the true lengths, and the lengths above
    0.05 are within 7 sqrt(t / n) of the truth.  For a pendant branch of length t with n sites the number of
    substitutions on it is about Poisson(n t), so the ML length has a standard error of about sqrt(t / n):
    at n = 2000 that is 5% of a 0.1 branch.  An internal branch has both end states inferred and carries
    less information, up to about twice that error on trees like these; 7 is 3.5 such errors, for the few
    dozen branches checked.  The root has two children, and with a reversible model whose root distribution is
    stationary only the sum of their lengths is identifiable, so that sum is checked as one branch."""
    from cherryml_b200.evaluation import dp_likelihood_computation

    sim = simulated
    fams = sorted(sim["fams"])
    dirs = _run(sim, fams, "recover")
    worst = 0.0
    for f in fams:
        tree, rates, (ll, _) = _read(dirs, f)
        msa = sim["fams"][f][1]
        true_ll, _ = dp_likelihood_computation(tree=sim["truth"][f], msa=msa, contact_map=None, site_rates=rates,
                                               amino_acids=AA, pi_1=sim["pi"], Q_1=sim["Q"])
        assert ll >= true_ll, (f, ll, true_ll)
        true = {v: d for _, v, d in sim["truth"][f].edges()}
        got = {v: d for _, v, d in tree.edges()}
        # pulley principle: only the sum of the root's two branches is identifiable
        a, b = [c for c, _ in tree.children(tree.root())]
        true[a], got[a] = true.pop(a) + true.pop(b), got.pop(a) + got.pop(b)
        for v, t in true.items():
            if t < 0.05:
                continue
            z = abs(got[v] - t) / np.sqrt(t / N_SITES)
            worst = max(worst, z)
            assert z <= 7.0, (f, v, t, got[v])
    print(f"\nlargest error of a length >= 0.05, in units of sqrt(t / n): {worst:.2f}")


@pytest.mark.gpu
def test_stage_files(simulated):
    """Topology and site rates unchanged; the likelihood file is dp_likelihood_computation's on the written
    tree (1e-12 relative); the profiling files hold total_time lines."""
    from cherryml_b200.evaluation import dp_likelihood_computation
    from cherryml_b200.io import read_site_rates, read_tree

    sim = simulated
    fams = sorted(sim["fams"])
    dirs = _run(sim, fams, "files", num_epochs=30)
    for f in fams:
        tree, rates, (ll, lls) = _read(dirs, f)
        given = read_tree(os.path.join(sim["tree_dir"], f + ".txt"))
        assert tree.nodes() == given.nodes()
        assert [(u, v) for u, v, _ in tree.edges()] == [(u, v) for u, v, _ in given.edges()]
        assert [d for _, _, d in tree.edges()] != [d for _, _, d in given.edges()]
        assert rates == read_site_rates(os.path.join(sim["site_rates_dir"], f + ".txt"))
        ref, ref_lls = dp_likelihood_computation(tree=tree, msa=sim["fams"][f][1], contact_map=None,
                                                 site_rates=rates, amino_acids=AA, pi_1=sim["pi"], Q_1=sim["Q"])
        assert abs(ll - ref) <= 1e-12 * abs(ref)
        np.testing.assert_allclose(lls, ref_lls, rtol=1e-12)
        lines = open(os.path.join(dirs["output_tree_dir"], f + ".profiling")).read().splitlines()
        assert lines[0].startswith("total_time: ") and float(lines[0].split()[1]) > 0


@pytest.mark.gpu
def test_stage_family_alone_equals_family_in_batch(simulated):
    """A family's trajectory does not depend on the other families of the call (Adam is elementwise, the
    loss a sum of per-family terms): the same lengths alone as in a batch of three, to 1e-9 relative."""
    sim = simulated
    alone = _run(sim, ["sim1"], "alone", num_epochs=50)
    batch = _run(sim, sorted(sim["fams"]), "batch", num_epochs=50)
    a, b = _read(alone, "sim1")[0], _read(batch, "sim1")[0]
    la = np.array([d for _, _, d in a.edges()])
    lb = np.array([d for _, _, d in b.edges()])
    np.testing.assert_allclose(la, lb, rtol=1e-9)
    print(f"\nalone vs batch: bitwise equal {np.array_equal(la, lb)}, "
          f"largest relative difference {np.max(np.abs(la - lb) / la):.3g}")


@pytest.mark.gpu
def test_stage_cache(simulated, tmp_path):
    from cherryml_b200 import caching
    from cherryml_b200.phylogeny_estimation import branch_length_mle

    sim = simulated
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        kw = dict(tree_dir=sim["tree_dir"], site_rates_dir=sim["site_rates_dir"], msa_dir=sim["msa_dir"],
                  families=["sim0", "sim2"], rate_matrix_path=sim["lg"], amino_acids=AA, num_processes=4,
                  num_epochs=5)
        first = branch_length_mle(**kw)
        before = _lib.launch_count()
        again = branch_length_mle(**dict(kw, num_processes=1, device="cuda:0"))
        assert again == first and _lib.launch_count() == before
        for d in first.values():
            assert os.path.exists(os.path.join(d, "sim0.txt")) and os.path.exists(os.path.join(d, "sim2.txt"))
    finally:
        caching.set_cache_dir(None)


@pytest.mark.gpu
def test_two_cherryml_iterations_on_refitted_demo_trees(tmp_path):
    """lg_end_to_end_with_cherryml_optimizer on FastTree trees of the demo data: iteration 0 counts on the
    given trees, iteration 1 refits their branch lengths under iteration 0's rate matrix and counts on
    those -- the same counts as a count pass run by hand on the refitted trees."""
    from cherryml_b200 import caching
    from cherryml_b200._public_api import _quantization_points, lg_end_to_end_with_cherryml_optimizer
    from cherryml_b200.counting import count_transitions
    from cherryml_b200.markov_chain import _rate_matrix_path
    from cherryml_b200.phylogeny_estimation import branch_length_mle

    fams = ["13gs_1_A", "19hc_1_A", "1a0b_1_A"]
    with tarfile.open(os.path.join(GOLDEN, "demo_data.tar.xz")) as tf:
        tf.extractall(tmp_path, members=[tf.getmember(f"{d}/{f}.txt") for d in ("msas", "trees", "site_rates")
                                         for f in fams])
    trees, rates, msas = (str(tmp_path / d) for d in ("trees", "site_rates", "msas"))
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        est = functools.partial(branch_length_mle, tree_dir=trees, site_rates_dir=rates, amino_acids=AA,
                                num_epochs=20)
        res = lg_end_to_end_with_cherryml_optimizer(
            msa_dir=msas, families=fams, tree_estimator=est, initial_tree_estimator_rate_matrix_path=_rate_matrix_path(
                "lg"), num_iterations=2, tree_dir=trees, site_rates_dir=rates, num_epochs=20,
            use_cpp_counting_implementation=False)
        refit = res["tree_estimator_output_dirs_1"]
        assert refit["output_tree_dir"] != trees
        by_hand = count_transitions(
            tree_dir=refit["output_tree_dir"], msa_dir=msas, site_rates_dir=refit["output_site_rates_dir"],
            families=fams, amino_acids=AA, quantization_points=_quantization_points(0.03, 1.1, 64),
            edge_or_cherry="cherry++", num_processes=1, use_cpp_implementation=False)["output_count_matrices_dir"]
    finally:
        caching.set_cache_dir(None)

    def counts(d):
        return open(os.path.join(d, "result.txt")).read()

    assert counts(res["count_matrices_dir_1"]) == counts(by_hand)
    assert counts(res["count_matrices_dir_1"]) != counts(res["count_matrices_dir_0"])
    assert res["time_tree_estimation"] > 0
