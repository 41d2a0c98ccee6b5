"""``matrix_exponential`` and friends: drop-in for the part of the reference's
``cherryml/markov_chain/_markov_chain.py`` that sits on the hot path (:22-168).

``matrix_exponential(exponents, Q, fact, reversible, device)`` returns the fp64 numpy array
``[len(exponents), S, S]`` with ``res[i] = expm(exponents[i] * Q)``.  Both of the reference's
back ends (``torch.matrix_exp`` and the eigendecomposition of a reversible model) compute the
same mathematical object; here both are served by the CUDA expm of the fit
(``cherry_expm_batched``: Taylor + scaling-and-squaring on the FP64 tensor pipe).  ``device`` is
accepted for compatibility; the computation always runs on a CUDA device.
"""
import ctypes
import os
from typing import List, Optional

import numpy as np
import torch

from .. import _lib
from ..estimation._engine import FitArgs, solve_stationary_dist


def compute_stationary_distribution(rate_matrix: np.ndarray) -> np.ndarray:
    return solve_stationary_dist(np.asarray(rate_matrix, dtype=np.float64))


def compute_mutation_rate(rate_matrix: np.ndarray) -> float:
    pi = compute_stationary_distribution(rate_matrix)
    return float(pi @ -np.diag(rate_matrix))


def normalized(rate_matrix: np.ndarray) -> np.ndarray:
    return rate_matrix / compute_mutation_rate(rate_matrix)


class FactorizedReversibleModel:
    """Same factorisation object as the reference's (``_markov_chain.py:56-89``):
    ``exp(tQ) = P2 @ U @ diag(exp(t D)) @ U_t @ P1``."""

    def __init__(self, Q: np.ndarray) -> None:
        Q = np.asarray(Q, dtype=np.float64)
        pi = compute_stationary_distribution(Q)
        P1 = np.diag(np.sqrt(pi))
        P2 = np.diag(np.sqrt(1 / pi))
        D, U = np.linalg.eigh(P1 @ Q @ P2)
        self.P2, self.U, self.D, self.U_t, self.P1 = P2, U, D, U.transpose(), P1

    def get_factorization(self):
        return (self.P2, self.U, self.D, self.U_t, self.P1)

    def rate_matrix(self) -> np.ndarray:
        return self.P2 @ self.U @ np.diag(self.D) @ self.U_t @ self.P1


# Exponents per cherry_expm_batched call for S > 32 (CHERRY_LARGE_FIT_MAX_K in include/cherryml_b200.h)
LARGE_MAX_K = 811
_SMALL_MAX_S = 32


def expm_batched(Q, exponents, device="cuda") -> torch.Tensor:
    """``[K, S, S]`` CUDA fp64 tensor of ``expm(exponents[k] * Q)``, for any number of exponents."""
    lib = _lib.load()
    dev = torch.device(device if str(device).startswith("cuda") else "cuda")
    Qt = torch.from_numpy(np.array(Q, dtype=np.float64)).to(dev).contiguous()
    t = torch.from_numpy(np.array(exponents, dtype=np.float64).reshape(-1)).to(dev).contiguous()
    S, K = int(Qt.shape[-1]), int(t.numel())
    out = torch.empty((K, S, S), dtype=torch.float64, device=dev)
    chunk = LARGE_MAX_K if S > _SMALL_MAX_S else max(K, 1)
    for k0 in range(0, K, chunk):
        _expm_call(lib, Qt, t[k0: k0 + chunk], out[k0: k0 + chunk], dev)
    return out


def _expm_call(lib, Qt, t, out, dev) -> None:
    S, K = int(Qt.shape[-1]), int(t.numel())
    nbytes = ctypes.c_size_t(0)
    _lib.check(lib.cherry_fit_workspace_bytes(S, K, 1, ctypes.byref(nbytes)), "cherry_fit_workspace_bytes")
    ws = torch.empty(max(8, nbytes.value), dtype=torch.uint8, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    a = FitArgs()
    a.S, a.K, a.n_problems = S, K, 1
    a.t, a.Q = _lib.ptr(t), _lib.ptr(Qt)
    a.workspace, a.workspace_bytes = _lib.ptr(ws), nbytes.value
    a.status_flag = _lib.ptr(flag)
    with torch.cuda.device(dev):
        _lib.check(lib.cherry_expm_batched(ctypes.byref(a), _lib.ptr(out), _lib.current_stream_ptr()),
                   "cherry_expm_batched")
    status = int(flag.item())
    if status == 3:
        raise _lib.CherryError("expm: internal scheduling timeout of the squaring kernels (status 3)")
    if status != 0:
        if S > _SMALL_MAX_S:  # eight squarings of a Taylor step with t * max|Q_ii| <= 2.2
            bound = "t * max|Q_ii| > 2.2 * 2^8 = 563.2"
        else:  # thirty squarings of a Taylor step with t * ||Q||_1 <= 0.0376
            bound = "t * ||Q||_1 > 0.0376 * 2^30 = 4.0e7"
        raise _lib.CherryError(f"expm: exponent * rate is beyond the supported range ({bound})")


def matrix_exponential_pytorch(exponents: List[float], Q: np.ndarray, device: str) -> np.ndarray:
    return expm_batched(Q, exponents, device).cpu().numpy()


def matrix_exponential_reversible(exponents: List[float], fact: FactorizedReversibleModel, device: str) -> np.ndarray:
    return expm_batched(fact.rate_matrix(), exponents, device).cpu().numpy()


def matrix_exponential(exponents, Q: Optional[np.ndarray], fact: Optional[FactorizedReversibleModel],
                       reversible: bool, device) -> np.ndarray:
    if reversible:
        return matrix_exponential_reversible(exponents, fact, device)
    return matrix_exponential_pytorch(exponents, Q, device)


def chain_product(rate_matrix_1: np.ndarray, rate_matrix_2: np.ndarray) -> np.ndarray:
    """Rate matrix of two independent sites, state (i, j) -> index i*n + j
    (reference ``_markov_chain.py:216-239``): Q1 (+) Q2 = Q1 x I + I x Q2."""
    n = rate_matrix_1.shape[0]
    eye = np.eye(n)
    return np.kron(rate_matrix_1, eye) + np.kron(eye, rate_matrix_2)


_DATA_FILE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "data", "rate_matrices.npz")
_MATERIALISED = {}


def _rate_matrix_path(name: str) -> str:
    """Published 20 x 20 amino-acid rate matrices ship as one compressed array file
    (data/rate_matrices.npz: LG, WAG and the uniform-exchangeability matrix in the alphabet order of
    ``utils.amino_acids``); the reference's path-based API wants labelled text files, which are
    written on first use (floats as repr, so they parse back to the stored doubles)."""
    if name not in _MATERIALISED:
        import tempfile

        from ..io import write_rate_matrix
        from ..utils import amino_acids

        out_dir = os.path.join(tempfile.gettempdir(), f"cherryml_b200_data_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, name + ".txt")
        with np.load(_DATA_FILE) as z:
            matrix = z[name]
        tmp = f"{path}.{os.getpid()}.tmp"
        write_rate_matrix(matrix, amino_acids, tmp)
        os.replace(tmp, path)
        _MATERIALISED[name] = path
    return _MATERIALISED[name]


def get_lg_path() -> str:
    """The LG rate matrix (Le & Gascuel 2008) as a labelled text file (reference ``get_lg_path``)."""
    return _rate_matrix_path("lg")


def get_equ_path() -> str:
    """The uniform-exchangeability rate matrix (reference ``get_equ_path``)."""
    return _rate_matrix_path("equ")


def get_wag_path() -> str:
    """The WAG rate matrix (Whelan & Goldman 2001) (reference ``get_wag_path``)."""
    return _rate_matrix_path("wag")


def _stored_matrix(name: str) -> np.ndarray:
    with np.load(_DATA_FILE) as z:
        return z[name]


def _derived_path(name: str, build) -> str:
    """A file derived from the shipped matrices (stationary distribution, product chain), written on
    first use next to them.  The reference ships these as data files computed once by its authors;
    the values here come from ``compute_stationary_distribution`` / ``chain_product`` and agree with
    those files to ~1e-16 (checked in tests/test_markov_chain_data.py where the reference is present)."""
    if name not in _MATERIALISED:
        import tempfile

        out_dir = os.path.join(tempfile.gettempdir(), f"cherryml_b200_data_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, name + ".txt")
        tmp = f"{path}.{os.getpid()}.tmp"
        build(tmp)
        os.replace(tmp, path)
        _MATERIALISED[name] = path
    return _MATERIALISED[name]


def _stationary_path(name: str, matrix_name: str, product: bool) -> str:
    from ..io import write_probability_distribution
    from ..utils import amino_acids

    def build(path):
        Q = _stored_matrix(matrix_name)
        states = list(amino_acids)
        if product:
            Q = chain_product(Q, Q)
            states = [a + b for a in amino_acids for b in amino_acids]
        write_probability_distribution(compute_stationary_distribution(Q), states, path)

    return _derived_path(name, build)


def _product_path(name: str, matrix_name: str) -> str:
    from ..io import write_rate_matrix
    from ..utils import amino_acids

    def build(path):
        Q = _stored_matrix(matrix_name)
        write_rate_matrix(chain_product(Q, Q), [a + b for a in amino_acids for b in amino_acids], path)

    return _derived_path(name, build)


def get_lg_stationary_path() -> str:
    """Stationary distribution of LG (reference ``get_lg_stationary_path``)."""
    return _stationary_path("lg_stationary", "lg", product=False)


def get_wag_stationary_path() -> str:
    """Stationary distribution of WAG (reference ``get_wag_stationary_path``)."""
    return _stationary_path("wag_stationary", "wag", product=False)


def get_lg_x_lg_path() -> str:
    """The 400 x 400 chain of two independent LG sites (reference ``get_lg_x_lg_path``)."""
    return _product_path("lg_x_lg", "lg")


def get_lg_x_lg_stationary_path() -> str:
    """Stationary distribution of the LG x LG chain (reference ``get_lg_x_lg_stationary_path``)."""
    return _stationary_path("lg_x_lg_stationary", "lg", product=True)


def get_equ_x_equ_path() -> str:
    """The 400 x 400 chain of two independent uniform-exchangeability sites (reference ``get_equ_x_equ_path``)."""
    return _product_path("equ_x_equ", "equ")


def equ_matrix():
    """The uniform-exchangeability matrix as a labelled table (reference ``equ_matrix``)."""
    from ..io import read_rate_matrix

    return read_rate_matrix(get_equ_path())


def wag_matrix():
    """WAG rescaled to one expected mutation per unit time (reference ``wag_matrix``,
    _markov_chain.py:171-184; the shipped matrix already is, so this is a no-op up to rounding)."""
    from ..io import read_rate_matrix

    wag = read_rate_matrix(get_wag_path())
    pi = compute_stationary_distribution(wag.to_numpy())
    return wag / np.dot(-np.diag(wag.to_numpy()), pi)


def wag_stationary_distribution():
    """Reference ``wag_stationary_distribution`` (_markov_chain.py:187-191)."""
    import pandas as pd

    wag = wag_matrix()
    return pd.DataFrame(compute_stationary_distribution(wag.to_numpy()), index=wag.index)
