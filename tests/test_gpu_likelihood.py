"""Tree log-likelihood on the GPU (cherry_expm_batched + cherry_tree_log_likelihood) against the
FastTree-verified constants of the reference's tests, outputs of the unmodified reference
function (tests/golden/likelihood) and the oracle on seeded trees.  Tolerance: 1e-6 relative
(the north star's bound for fp64 log-likelihoods); observed differences are ~1e-12 against
the oracle and ~1e-9 against the reference's eigendecomposition back end."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from cherryml_b200.evaluation import compute_log_likelihoods, dp_likelihood_computation
from cherryml_b200.io import (Tree, write_msa, write_probability_distribution, write_rate_matrix, write_site_rates,
                              write_tree)
from tests._ll_cases import AA, _caterpillar, fasttree_kats, golden_cases


@pytest.mark.parametrize("kat", fasttree_kats(), ids=lambda k: k[0])
def test_fasttree_verified_constants(kat):
    name, tree, msa, cmap, rates, pi1, Q1, pi2, Q2, ll_exp, lls_exp, dec = kat
    if Q2 is None:
        cmap = np.eye(len(rates))
    ll, lls = dp_likelihood_computation(tree=tree, msa=msa, contact_map=cmap, site_rates=rates, amino_acids=AA,
                                        pi_1=pi1, Q_1=Q1, pi_2=pi2, Q_2=Q2)
    np.testing.assert_almost_equal(ll, ll_exp, decimal=dec)
    if lls_exp is not None:
        np.testing.assert_almost_equal(lls, lls_exp, decimal=dec)


@pytest.mark.parametrize("i", range(len(golden_cases())))
def test_matches_reference_function_and_oracle(i):
    from oracle.likelihood_oracle import log_likelihood

    c = golden_cases()[i]
    ll, lls = dp_likelihood_computation(tree=c["tree"], msa=c["msa"], contact_map=c["contact_map"],
                                        site_rates=c["site_rates"], amino_acids=AA, pi_1=c["pi1"], Q_1=c["Q1"],
                                        pi_2=c["pi2"], Q_2=c["Q2"])
    assert abs(ll - c["ll"]) <= 1e-7 * abs(c["ll"])
    np.testing.assert_allclose(lls, c["lls"], rtol=1e-6, atol=1e-9)
    ll_o, lls_o = log_likelihood(c["tree"], c["msa"], c["contact_map"], c["site_rates"], AA, c["pi1"], c["Q1"],
                                 c["pi2"], c["Q2"])
    assert abs(ll - ll_o) <= 1e-10 * abs(ll_o)
    np.testing.assert_allclose(lls, lls_o, rtol=1e-9, atol=1e-11)


def test_deep_tree_many_sites_against_oracle():
    from oracle.likelihood_oracle import log_likelihood
    from tests._ll_cases import rate_matrix
    from cherryml_b200.markov_chain import chain_product, compute_stationary_distribution

    rng = np.random.default_rng(3)
    tree = _caterpillar(60, rng)
    L = 77
    msa = {}
    for v in tree.leaves():
        s = rng.choice(AA, L)
        s[rng.random(L) < 0.2] = "-"
        msa[v] = "".join(s)
    cmap = np.zeros((L, L))
    sites = rng.permutation(L)[:14]
    for a, b in zip(sites[0::2], sites[1::2]):
        cmap[a, b] = cmap[b, a] = 1
    rates = [float(r) for r in rng.choice([0.2, 0.7, 1.0, 2.5], L)]
    Q1 = rate_matrix("lg")
    Q2 = chain_product(Q1, Q1)
    pi1, pi2 = compute_stationary_distribution(Q1), compute_stationary_distribution(Q2)
    ll, lls = dp_likelihood_computation(tree=tree, msa=msa, contact_map=cmap, site_rates=rates, amino_acids=AA,
                                        pi_1=pi1, Q_1=Q1, pi_2=pi2, Q_2=Q2)
    ll_o, lls_o = log_likelihood(tree, msa, cmap, rates, AA, pi1, Q1, pi2, Q2)
    assert abs(ll - ll_o) <= 1e-10 * abs(ll_o)
    np.testing.assert_allclose(lls, lls_o, rtol=1e-9, atol=1e-11)


def test_stage_function_files_and_cache(tmp_path):
    from cherryml_b200 import _lib, caching
    from cherryml_b200.io import read_msa
    from tests._ll_cases import LL_DIR, rate_matrix
    from cherryml_b200.markov_chain import compute_stationary_distribution
    from cherryml_b200.io import read_site_rates, read_tree

    d = os.path.join(LL_DIR, "1a92")
    for sub in ("trees", "msas", "rates"):
        (tmp_path / sub).mkdir()
    for fam in ("a", "b"):
        write_tree(read_tree(os.path.join(d, "tree_4_cat.txt")), str(tmp_path / "trees" / f"{fam}.txt"))
        write_msa(read_msa(os.path.join(d, "msa.txt")), str(tmp_path / "msas" / f"{fam}.txt"))
        write_site_rates(read_site_rates(os.path.join(d, "site_rates_4_cat.txt")), str(tmp_path / "rates" / f"{fam}.txt"))
    wag = rate_matrix("wag")
    write_rate_matrix(wag, AA, str(tmp_path / "Q1.txt"))
    write_probability_distribution(compute_stationary_distribution(wag), AA, str(tmp_path / "pi1.txt"))
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        kw = dict(tree_dir=str(tmp_path / "trees"), msa_dir=str(tmp_path / "msas"),
                  site_rates_dir=str(tmp_path / "rates"), contact_map_dir=None, families=["a", "b"], amino_acids=AA,
                  pi_1_path=str(tmp_path / "pi1.txt"), Q_1_path=str(tmp_path / "Q1.txt"), reversible_1=True,
                  device_1="cpu", pi_2_path=None, Q_2_path=None, reversible_2=None, device_2=None, num_processes=2)
        out = compute_log_likelihoods(**kw)["output_likelihood_dir"]
        before = _lib.launch_count()
        assert compute_log_likelihoods(**kw)["output_likelihood_dir"] == out and _lib.launch_count() == before
    finally:
        caching.set_cache_dir(None)
    lines = open(os.path.join(out, "a.txt")).read().split("\n")
    np.testing.assert_almost_equal(float(lines[0]), -4337.8688, decimal=4)  # FastTree, likelihood_test.py:913
    n = int(lines[1].split()[0])
    assert lines[1].split()[1] == "sites" and len(lines[2].split()) == n
    assert abs(sum(float(x) for x in lines[2].split()) - float(lines[0])) < 1e-8
    assert os.path.exists(os.path.join(out, "b.success")) and os.path.exists(os.path.join(out, "a.profiling"))


def test_pfam_sized_family_against_oracle(tmp_path):
    """1024 leaves x 210 sites, the demo family 13gs_1_A with its FastTree tree and 4 site-rate
    categories... (tests/golden/demo_data.tar.xz), LG model, independent sites only."""
    import tarfile
    import time

    from oracle.likelihood_oracle import log_likelihood
    from cherryml_b200.io import read_msa, read_site_rates, read_tree
    from cherryml_b200.markov_chain import compute_stationary_distribution
    from tests._ll_cases import rate_matrix
    from tests.conftest import GOLDEN

    fam = "13gs_1_A"
    with tarfile.open(os.path.join(GOLDEN, "demo_data.tar.xz")) as tf:
        tf.extractall(tmp_path, members=[tf.getmember(f"{d}/{fam}.txt") for d in ("msas", "trees", "site_rates")])
    tree = read_tree(str(tmp_path / "trees" / f"{fam}.txt"))
    msa = read_msa(str(tmp_path / "msas" / f"{fam}.txt"))
    rates = read_site_rates(str(tmp_path / "site_rates" / f"{fam}.txt"))
    Q1 = rate_matrix("lg")
    pi1 = compute_stationary_distribution(Q1)
    dp_likelihood_computation(tree=tree, msa=msa, contact_map=None, site_rates=rates, amino_acids=AA, pi_1=pi1, Q_1=Q1)
    t0 = time.time()
    ll, lls = dp_likelihood_computation(tree=tree, msa=msa, contact_map=None, site_rates=rates, amino_acids=AA,
                                        pi_1=pi1, Q_1=Q1)
    t_gpu = time.time() - t0
    t0 = time.time()
    ll_o, lls_o = log_likelihood(tree, msa, None, rates, AA, pi1, Q1, None, None)
    t_cpu = time.time() - t0
    print(f"\nlikelihood {fam}: {len(tree.leaves())} leaves x {len(rates)} sites, {len(set(rates))} rate categories: "
          f"GPU {t_gpu:.3f} s (host set-up included), numpy oracle {t_cpu:.1f} s, ll {ll:.4f}")
    assert abs(ll - ll_o) <= 1e-10 * abs(ll_o)
    np.testing.assert_allclose(lls, lls_o, rtol=1e-9, atol=1e-10)


@pytest.mark.parametrize("num_cats,ll_expected", [(1, -4649.6146), (2, -4397.8184), (4, -4337.8688), (20, -4307.0638)])
def test_real_data_pair_site_medium_fasttree_constants(num_cats, ll_expected):
    """The reference's Test_real_data_pair_site_medium (likelihood_test.py:996-1068): half of the sites
    with the median site rate are coupled in pairs under the WAG x WAG product model (tree and rates
    rescaled so that the coupled sites evolve at rate 1); the total must equal FastTree's single-site
    log-likelihood to 4 decimals.  Exercises the 400-state kernel path on real data."""
    from cherryml_b200.io import Tree, read_msa, read_site_rates, read_tree
    from cherryml_b200.markov_chain import chain_product, compute_stationary_distribution
    from tests._ll_cases import LL_DIR, rate_matrix

    d = os.path.join(LL_DIR, "1a92")
    tree = read_tree(os.path.join(d, f"tree_{num_cats}_cat.txt"))
    msa = read_msa(os.path.join(d, "msa.txt"))
    site_rates = read_site_rates(os.path.join(d, f"site_rates_{num_cats}_cat.txt"))
    median = np.median(site_rates)
    places = [i for i, r in enumerate(site_rates) if r == median]
    np.random.seed(1)
    np.random.shuffle(places)
    cmap = np.eye(len(site_rates))
    for i in range(len(places) // 4):
        j, k = places[2 * i], places[2 * i + 1]
        cmap[j, k] = cmap[k, j] = 1
    scaled = Tree()
    scaled.add_nodes(tree.nodes())
    for u, v, length in tree.edges():
        scaled.add_edge(u, v, length * median)
    rates_scaled = [r / median for r in site_rates]
    wag = rate_matrix("wag")
    wag2 = chain_product(wag, wag)
    ll, lls = dp_likelihood_computation(
        tree=scaled, msa=msa, contact_map=cmap, site_rates=rates_scaled, amino_acids=AA,
        pi_1=compute_stationary_distribution(wag), Q_1=wag, pi_2=compute_stationary_distribution(wag2), Q_2=wag2)
    np.testing.assert_almost_equal(ll, ll_expected, decimal=4)
    assert len(lls) == len(site_rates)
