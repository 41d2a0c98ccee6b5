"""The rate-matrix data getters of cherryml.markov_chain: shipped matrices, and the files derived
from them (stationary distributions, product chains)."""
import os

import numpy as np
import pytest

from cherryml_b200 import io
from cherryml_b200 import markov_chain as mc
from cherryml_b200.utils import amino_acids

REF_DATA = "/root/reference/data/rate_matrices"
# byte copies of the reference's data/rate_matrices/lg.txt and equ.txt (tests/golden/make_golden_fit.py)
REF_COPIES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fit", "inputs")
PAIRS = [a + b for a in amino_acids for b in amino_acids]


def test_derived_files_are_consistent_with_their_matrices():
    for q_path, pi_path, states in ((mc.get_lg_path(), mc.get_lg_stationary_path(), list(amino_acids)),
                                    (mc.get_wag_path(), mc.get_wag_stationary_path(), list(amino_acids)),
                                    (mc.get_lg_x_lg_path(), mc.get_lg_x_lg_stationary_path(), PAIRS)):
        Q = io.read_rate_matrix(q_path)
        pi = io.read_probability_distribution(pi_path)
        assert list(Q.index) == states and list(Q.columns) == states and list(pi.index) == states
        p = pi.to_numpy().reshape(-1)
        assert abs(p.sum() - 1.0) < 1e-12 and (p > 0).all()
        assert np.abs(p @ Q.to_numpy()).max() < 1e-12
        assert np.abs(Q.to_numpy().sum(axis=1)).max() < 1e-12
    lg = io.read_rate_matrix(mc.get_lg_path()).to_numpy()
    lg2 = io.read_rate_matrix(mc.get_lg_x_lg_path()).to_numpy()
    assert np.array_equal(lg2, mc.chain_product(lg, lg))
    # product chain: (i, j) -> (k, j) at rate Q[i, k], (i, j) -> (i, l) at rate Q[j, l], nothing else off the diagonal
    assert lg2[20 * 3 + 5, 20 * 7 + 5] == lg[3, 7] and lg2[20 * 3 + 5, 20 * 3 + 9] == lg[5, 9]
    assert lg2[20 * 3 + 5, 20 * 7 + 9] == 0.0 and lg2[20 * 3 + 5, 20 * 3 + 5] == lg[3, 3] + lg[5, 5]
    pi2 = io.read_probability_distribution(mc.get_lg_x_lg_stationary_path()).to_numpy().reshape(-1)
    pi1 = io.read_probability_distribution(mc.get_lg_stationary_path()).to_numpy().reshape(-1)
    assert np.abs(pi2 - np.outer(pi1, pi1).reshape(-1)).max() < 1e-15
    assert mc.equ_matrix().shape == (20, 20) and list(mc.wag_matrix().index) == list(amino_acids)
    w = mc.wag_matrix().to_numpy()
    assert abs(mc.compute_mutation_rate(w) - 1.0) < 1e-12
    assert abs(float(mc.wag_stationary_distribution().to_numpy().sum()) - 1.0) < 1e-12


def test_values_equal_stored_copies_of_the_reference_data_files():
    for mine, ref in ((mc.get_lg_path(), "lg.txt"), (mc.get_equ_path(), "equ.txt")):
        a, b = io.read_rate_matrix(mine), io.read_rate_matrix(os.path.join(REF_COPIES, ref))
        assert list(a.index) == list(b.index) and list(a.columns) == list(b.columns)
        assert np.array_equal(a.to_numpy(), b.to_numpy())


@pytest.mark.skipif(not os.path.isdir(REF_DATA), reason="the reference checkout is only present in the build container")
def test_values_equal_the_reference_data_files():
    for mine, ref, is_q in ((mc.get_lg_path(), "lg.txt", True), (mc.get_wag_path(), "wag.txt", True),
                            (mc.get_equ_path(), "equ.txt", True),
                            (mc.get_lg_stationary_path(), "lg_stationary.txt", False),
                            (mc.get_wag_stationary_path(), "wag_stationary.txt", False),
                            (mc.get_lg_x_lg_path(), "lg_x_lg.txt", True),
                            (mc.get_lg_x_lg_stationary_path(), "lg_x_lg_stationary.txt", False),
                            (mc.get_equ_x_equ_path(), "equ_x_equ.txt", True)):
        read = io.read_rate_matrix if is_q else io.read_probability_distribution
        a, b = read(mine), read(os.path.join(REF_DATA, ref))
        assert list(a.index) == list(b.index)
        tol = 0.0 if ref in ("lg.txt", "wag.txt", "equ.txt") else 1e-15  # shipped: exact; derived: recomputed
        assert np.abs(a.to_numpy() - b.to_numpy()).max() <= tol
