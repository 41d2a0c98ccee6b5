"""Large-S fit and expm (S > 32, fit_large.cu) against extended-precision references, at every padded size, Taylor
pass variant, tail split and squaring count the host can select.

References (all in this file):
- expm, entrywise relative: uniformization, P(t) = sum_n Pois(n; t mu) (B / mu)^n with B = Q + mu I >= 0.  Every
  term is non-negative, so every entry keeps its relative accuracy.  Small matrices run it in np.longdouble; a
  Kronecker sum Q1 (+) Q2 (markov_chain.chain_product) uses expm(t (Q1 (+) Q2)) = expm(t Q1) (x) expm(t Q2) with
  longdouble factors, which is exact entry by entry, so S = 400..530 at t mu = 563 get a relative reference too.
  Dense large S run it in fp64 on BLAS: n products of non-negative matrices, so each entry is within n * S * u
  relative of the exact one (u = 2^-53), and that bound is added to the tolerance.
- gradient: complex step, D_E L = Im L(Q + i h E) / h with torch.matrix_exp in complex128, h = 1e-30.
- fits: oracle.fit_oracle in fp64.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from cherryml_b200 import _lib
from cherryml_b200.estimation import FitEngine, random_theta
from cherryml_b200.estimation._engine import FitArgs
from cherryml_b200.markov_chain import LARGE_MAX_K, chain_product, expm_batched, matrix_exponential
from oracle.fit_oracle import fit_oracle
from tests.test_gpu_fit import REL_FP64, random_rate_matrix

U64 = 2.0 ** -53

# ------------------------------------------------------------------ the host's path selection, mirrored
# Constants of fit_large.cu: kTheta, kSStore, kDeg, BT, kTaylorThreads, kTaylorStagesS, kTaylorTailUnits.
THETA, S_STORE, DEG, BT = 2.2, 8, 24, 80
TAYLOR_THREADS, TAYLOR_STAGES_S, TAIL_UNITS = 256, 16, 512
X_MAX = THETA * 2 ** S_STORE  # 563.2: largest t * mu with at most kSStore squarings


def padded(S):
    """make_plan: Sp = S rounded up to a multiple of the 80 x 80 GEMM tile."""
    return (S + BT - 1) // BT * BT


def squarings(x):
    """coef_kernel: s = ceil(log2(t ||B||_inf / theta)), ||B||_inf = mu for a rate matrix; > kSStore is an error."""
    return 0 if x <= THETA else int(math.ceil(math.log2(x / THETA)))


def register_taylor(K):
    """fit_large_impl, two_ctas_fit: the shared-memory Taylor pass runs two CTAs per SM while their weight tables,
    bucket lists, count ring and staged powers fit 227 KB; beyond (K >= 157) the register variant runs."""
    smem = 8 * K * (DEG + 1) + 12 * K + 8 + 8 * (TAYLOR_STAGES_S + DEG) * TAYLOR_THREADS + 1024
    return 2 * smem > 227 * 1024


def tail_parts(S, sym, sms):
    """fit_large_impl: the chunks of the shared-memory Taylor pass beyond a multiple of 2 * SMs, when they fill at
    most half a round, run split over 16, 8, 4 or 2 bucket shares (the largest that fits the round and the
    512-unit tail buffer); 1 = no split.  The symmetric form visits (Sp / 2) (Sp + 1) elements, so on 148 SMs its
    2- and 4-part splits need Sp >= 720 and no case here reaches them."""
    return _tail(S, sym, sms)[0]


def _tail(S, sym, sms):
    Sp = padded(S)
    n_visit = (Sp // 2) * (Sp + 1) if sym else Sp * Sp
    n_chunks, slots = -(-n_visit // TAYLOR_THREADS), 2 * sms
    tail = n_chunks % slots
    if n_chunks > slots and tail and tail <= slots // 2:
        for cand in (16, 8, 4, 2):
            if cand * tail <= slots and cand * tail <= TAIL_UNITS:
                return cand, np.arange((n_chunks - tail) * TAYLOR_THREADS, n_visit)
    return 1, np.arange(0)


def tail_has_real_elements(S, sym, sms):
    """Whether the split tail visits any element of the S x S matrix: a tail of padding rows only adds nothing
    to the loss or the gradient, so a wrong split would pass unseen.  taylor_visit maps visit slots to elements."""
    Sp = padded(S)
    v = _tail(S, sym, sms)[1]
    if sym:
        f, q = v // (Sp + 1), v % (Sp + 1)
        row = np.where(q < Sp - f, f, Sp - 1 - f)
        col = np.where(q < Sp - f, f + q, Sp - 1 - f + q - (Sp - f))
    else:
        row, col = v // Sp, v % Sp
    return bool(np.any((row < S) & (col < S)))


# ------------------------------------------------------------------ the cases (the coverage test reads these)
# (S, Kronecker factors or None for a dense matrix)
EXPM_CASES = [(33, (3, 11)), (36, (6, 6)), (79, None), (80, (8, 10)), (81, (9, 9)), (161, (7, 23)), (241, None),
              (300, None), (320, (16, 20)), (400, (20, 20)), (441, (21, 21)), (500, (20, 25))]
# t * mu of the expm exponents: every squaring count 0..8, each just below and just above its threshold
EXPM_X = sorted([THETA * 2 ** k * (1 - 1e-3) for k in range(S_STORE + 1)] +
                [THETA * 2 ** k * (1 + 1e-3) for k in range(S_STORE)])
# loss and gradient, general form: (S, factors, K)
# (441 and 500 would reach the 16- and 4-part splits with padding rows only: 480 and 560 fill their tails)
LOSS_CASES = [(81, (9, 9), 8), (241, None, 8), (400, (20, 20), 8), (480, (20, 24), 8), (560, (20, 28), 8),
              (81, (9, 9), 160), (81, (9, 9), 300)]
# symmetric form against the general form: (S, K)
SYM_CASES = [(80, 6), (400, 5), (530, 5), (36, 160), (36, 300)]
SYM_X_MAX = 400.0  # t_max * mu of the initial model: 8 squarings with room for 3 epochs of Adam to move mu
BIG_K = [300, LARGE_MAX_K]  # expm beyond the 256 buckets one CTA of coef_kernel once held
FIT_BIG_K = 300


def _rate(S, factors, seed):
    rng = np.random.default_rng(seed)
    if factors is None:
        return random_rate_matrix(S, rng), None
    n1, n2 = factors
    Q1, Q2 = random_rate_matrix(n1, rng), random_rate_matrix(n2, rng)
    # Q1 (+) Q2 = Q1 x I + I x Q2; chain_product (the reference's) takes two matrices of one size
    Q = chain_product(Q1, Q2) if n1 == n2 else np.kron(Q1, np.eye(n2)) + np.kron(np.eye(n1), Q2)
    return Q, (Q1, Q2)


def _mu(Q):
    return float(np.max(-np.diag(Q)))


def uniformized(Q, times, dtype):
    """expm(t Q) for every t by uniformization in `dtype`; also the number of terms summed.  The sum stops when
    the Poisson mass left, which bounds the error of every entry, is below 1e-20 of the smallest entry formed."""
    S = Q.shape[0]
    mu = dtype(_mu(Q))
    A = (np.asarray(Q, dtype=dtype) + mu * np.eye(S, dtype=dtype)) / mu
    lam = np.asarray(times, dtype=dtype) * mu
    w = np.exp(-lam)
    M = np.eye(S, dtype=dtype)
    P = np.zeros((len(lam), S, S), dtype=dtype)
    n = 0
    while True:
        P += w[:, None, None] * M
        w = w * lam / (n + 1)
        n += 1
        ratio = lam / (n + 1)
        if np.all(ratio < 1):
            tail = w / (1 - ratio)  # the remaining weights are below a geometric series of this ratio
            if np.all(tail <= dtype(1e-20)):
                smallest = np.array([p[p > 0].min() if np.any(p > 0) else 1.0 for p in P], dtype=dtype)
                if np.all(tail <= dtype(1e-20) * smallest):
                    return P, n
        M = M @ A


def reference_expm(Q, factors, times):
    """(P, relative error bound of P) for Q with its Kronecker factors (or None)."""
    if factors is not None:
        P1, _ = uniformized(factors[0], times, np.longdouble)
        P2, _ = uniformized(factors[1], times, np.longdouble)
        return np.stack([np.kron(a, b) for a, b in zip(P1, P2)]), 0.0
    S = Q.shape[0]
    if S <= 80:
        return uniformized(Q, times, np.longdouble)[0], 0.0
    P, n = uniformized(Q, times, np.float64)
    return P.astype(np.longdouble), n * S * U64


def _torch_expm(Q, times):
    t = torch.tensor(np.asarray(times, dtype=np.float64), device="cuda")
    return torch.matrix_exp(t[:, None, None] * torch.tensor(Q, device="cuda")[None]).cpu().numpy()


def _check_expm(got, Q, factors, times):
    ref, bound = reference_expm(Q, factors, times)
    S = Q.shape[0]
    assert np.abs(got.sum(axis=2) - 1.0).max() <= 1e-13
    absd = np.abs(got - _torch_expm(Q, times)).max()
    assert absd <= 1e-12, absd
    pos = ref > 1e-280
    rel = float(np.max(np.abs((got[pos] - ref[pos]) / ref[pos])))
    # 1e-11: the Taylor truncation (2e-17) and the rounding of each squaring, amplified by up to 2^8 over 8
    # squarings; plus the reference's own bound
    assert rel <= 1e-11 + bound, (rel, bound)
    print(f"S={S}: max abs vs torch {absd:.2e}, max rel vs reference {rel:.2e} (reference bound {bound:.1e})")


# ------------------------------------------------------------------ 0. the parametrization reaches every path
def test_cases_reach_every_host_path():
    """If a constant of fit_large.cu moves, this names the path no case reaches any more."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sps = {padded(S) for S, _ in EXPM_CASES} | {padded(S) for S, _, _ in LOSS_CASES} | {padded(S) for S, _ in SYM_CASES}
    missing = {80, 160, 240, 320, 400, 480, 560} - sps
    assert not missing, f"padded sizes not reached: {missing}"
    assert any(S == padded(S) for S, _ in EXPM_CASES) and any(S < padded(S) for S, _ in EXPM_CASES)
    s_seen = {squarings(x) for x in [0.0] + EXPM_X}
    assert s_seen >= set(range(S_STORE + 1)), f"squaring counts not reached: {set(range(S_STORE + 1)) - s_seen}"
    assert squarings(X_MAX * 1.001) > S_STORE
    assert squarings(SYM_X_MAX) == S_STORE and squarings(SYM_X_MAX * 1.35) == S_STORE
    general = [(S, K) for S, _, K in LOSS_CASES] + [(36, FIT_BIG_K)]
    sym = list(SYM_CASES) + [(36, FIT_BIG_K)]
    gparts = {tail_parts(S, False, sms) for S, K in general
              if not register_taylor(K) and (tail_parts(S, False, sms) == 1 or tail_has_real_elements(S, False, sms))}
    sparts = {tail_parts(S, True, sms) for S, K in sym
              if not register_taylor(K) and (tail_parts(S, True, sms) == 1 or tail_has_real_elements(S, True, sms))}
    assert gparts >= {1, 2, 4, 8, 16}, f"general-form tail splits not reached: {({1, 2, 4, 8, 16} - gparts)} on {sms} SMs"
    assert sparts >= {1, 8, 16}, f"symmetric-form tail splits not reached: {({1, 8, 16} - sparts)} on {sms} SMs"
    assert any(register_taylor(K) for _, K in general) and any(register_taylor(K) for _, K in sym)
    assert max(BIG_K) > 256 and FIT_BIG_K > 256


# ------------------------------------------------------------------ 1. expm across shapes and squarings
@pytest.mark.parametrize("S,factors", EXPM_CASES)
def test_expm_relative_accuracy_at_every_squaring_count(S, factors):
    Q, fac = _rate(S, factors, seed=S)
    mu = _mu(Q)
    times = np.array([0.0, 1e-7] + [x / mu for x in EXPM_X])
    got = expm_batched(Q, times).cpu().numpy()
    assert np.array_equal(got[0], np.eye(S))
    _check_expm(got, Q, fac, times)
    with pytest.raises(_lib.CherryError, match=r"563\.2"):
        expm_batched(Q, [1.0 / mu, X_MAX * 1.001 / mu])


# ------------------------------------------------------------------ 2. K beyond one CTA's worth of buckets
@pytest.mark.parametrize("K", BIG_K)
def test_expm_with_many_exponents(K):
    Q, fac = _rate(36, (6, 6), seed=7)
    mu = _mu(Q)
    rng = np.random.default_rng(K)
    times = np.concatenate([[0.0, 1e-7], np.array(EXPM_X) / mu, rng.uniform(0, X_MAX / mu, K - 2 - len(EXPM_X))])
    got = expm_batched(Q, times).cpu().numpy()
    assert np.array_equal(got[0], np.eye(36))
    _check_expm(got, Q, fac, times)


def test_more_exponents_than_the_limit():
    lib = _lib.load()
    Q, fac = _rate(36, (6, 6), seed=8)
    K = LARGE_MAX_K + 1
    t = torch.full((K,), 0.1, dtype=torch.float64, device="cuda")
    Qt = torch.tensor(Q, device="cuda")
    out = torch.empty((K, 36, 36), dtype=torch.float64, device="cuda")
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    a = FitArgs()
    a.S, a.K, a.n_problems = 36, K, 1
    a.t, a.Q, a.status_flag = _lib.ptr(t), _lib.ptr(Qt), _lib.ptr(flag)
    a.workspace, a.workspace_bytes = _lib.ptr(ws), ws.numel()
    assert lib.cherry_expm_batched(ctypes.byref(a), _lib.ptr(out), _lib.current_stream_ptr()) == -3  # CHERRY_ELIMIT
    assert b"limit of %d" % LARGE_MAX_K in lib.cherry_last_error()
    with pytest.raises(_lib.CherryError, match="limit"):
        FitEngine(np.full(K, 0.1), np.ones((K, 36, 36)), random_theta(36), num_epochs=1)
    # the drop-in for the reference splits any number of exponents into calls within the limit
    times = np.random.default_rng(3).uniform(0, 40.0 / _mu(Q), 1000)
    got = matrix_exponential(times, Q, None, False, "cuda")
    assert got.shape == (1000, 36, 36)
    _check_expm(got, Q, fac, times)


def _symmetric_counts(rng, K, S):
    half = rng.integers(0, 40, size=(K, S, S)).astype(np.float64)
    half[rng.random(half.shape) < 0.4] = 0.0
    return half + half.transpose(0, 2, 1)


def _fit(times, counts, theta0, n, sym, monkeypatch):
    if sym:
        monkeypatch.delenv("CHERRY_FIT_SYMMETRIC", raising=False)
    else:
        monkeypatch.setenv("CHERRY_FIT_SYMMETRIC", "0")
    eng = FitEngine(times, counts, theta0.copy(), num_epochs=n)
    assert eng.symmetric_form == sym
    eng.run()
    return eng.results()


@pytest.mark.parametrize("sym", [True, False])
def test_fit_with_300_buckets_matches_the_oracle(sym, monkeypatch):
    rng = np.random.default_rng(11)
    S, K, n = 36, FIT_BIG_K, 3
    times = np.exp(rng.uniform(np.log(1e-3), np.log(20.0), K))
    counts = _symmetric_counts(rng, K, S)
    res = _fit(times, counts, random_theta(S), n, sym, monkeypatch)
    ref = fit_oracle(times, counts, None, None, 0.1, n, dtype=torch.float64)
    rel = np.max(np.abs(res["loss"] - ref["loss"]) / np.abs(ref["loss"]))
    qd = np.max(np.abs(res["Q_last"] - ref["Q_last"])) / np.max(np.abs(ref["Q_last"]))
    print(f"K={K} sym={sym}: loss rel {rel:.2e}, Q_last rel {qd:.2e}")
    assert rel < REL_FP64 and qd < REL_FP64


# ------------------------------------------------------------------ 3. loss and gradient, general form
def _complex_step(Q, times, counts, E, h=1e-30):
    dev = "cuda"
    Qc = torch.tensor(Q, device=dev).to(torch.complex128) + 1j * h * torch.tensor(E, device=dev)
    t = torch.tensor(np.asarray(times, dtype=np.float64), device=dev)
    C = torch.tensor(counts, device=dev)
    P = torch.matrix_exp(t[:, None, None].to(torch.complex128) * Qc[None])
    L = -(torch.log(P) * C).sum() / C.sum()
    return float(L.imag.item()) / h


def _autograd(Q, times, counts):
    """oracle.fit_oracle.loss_and_grad_oracle on the GPU (the same expression)."""
    Qt = torch.tensor(Q, device="cuda", requires_grad=True)
    t = torch.tensor(np.asarray(times, dtype=np.float64), device="cuda")
    C = torch.tensor(counts, device="cuda")
    loss = -(torch.log(torch.matrix_exp(t[:, None, None] * Qt)) * C).sum() / C.sum()
    loss.backward()
    return Qt.grad.cpu().numpy()


@pytest.mark.parametrize("S,factors,K", LOSS_CASES)
def test_loss_and_directional_derivatives_per_taylor_variant(S, factors, K):
    Q, fac = _rate(S, factors, seed=S + K)
    mu = _mu(Q)
    rng = np.random.default_rng(S * K)
    times = np.exp(np.linspace(np.log(1e-6), np.log(500.0 / mu), K))
    counts = rng.integers(0, 50, size=(K, S, S)).astype(np.float64)
    counts[rng.random(counts.shape) < 0.5] = 0.0
    eng = FitEngine(times, counts, random_theta(S), num_epochs=0)
    eng.Q.copy_(torch.from_numpy(Q)[None])
    loss, grad = eng.loss_and_grad()
    g = grad[0].cpu().numpy()
    ref, bound = reference_expm(Q, fac, times)
    C = counts.astype(np.longdouble)
    exp_loss = float(-(C * np.log(ref)).sum() / C.sum())
    lrel = abs(float(loss[0]) - exp_loss) / abs(exp_loss)
    # the dense case's reference entries are within `bound` relative, so its log within `bound` absolute
    assert lrel <= 1e-12 + bound, (lrel, bound)
    R = rng.random((S, S))  # along the rate matrices
    np.fill_diagonal(R, 0.0)
    np.fill_diagonal(R, -R.sum(axis=1))
    unit = np.zeros((S, S))
    unit[np.unravel_index(np.argmax(np.abs(g)), g.shape)] = 1.0  # the largest entry of the gradient on its own
    directions = [rng.standard_normal((S, S)), (rng.random((S, S)) < 0.05) * rng.standard_normal((S, S)),
                  np.diag(rng.standard_normal(S)), R, unit]
    drel = 0.0
    for E in directions:
        d_ref = _complex_step(Q, times, counts, E)
        drel = max(drel, abs(float((g * E).sum()) - d_ref) / abs(d_ref))
    print(f"S={S} K={K}: loss rel {lrel:.2e}, directional derivative rel {drel:.2e}")
    assert drel <= 1e-9, drel
    if factors is None:
        # The max-abs check of test_gpu_fit.test_large_loss_and_gradient_match_the_oracle.  Autograd through
        # torch.matrix_exp is good to ~1e-10 on dense matrices; on a Kronecker sum, whose entries first reached in
        # two steps make |dL/dP| ~ 1e6 at small t, it misses the complex step by ~6e-6 relative, so it is no
        # reference there.
        g_ag = _autograd(Q, times, counts)
        assert np.max(np.abs(g - g_ag)) < 1e-7 * np.max(np.abs(g_ag))


# ------------------------------------------------------------------ 4. symmetric form, the form the fits use
@pytest.mark.parametrize("S,K", SYM_CASES)
def test_symmetric_form_equals_general_form_and_oracle(S, K, monkeypatch):
    """Same losses and iterates as the general evaluation and as the fp64 oracle (the tolerances of
    test_gpu_fit.test_symmetric_form_equals_the_general_evaluation), with the longest time at 8 squarings."""
    rng = np.random.default_rng(S + K)
    theta0 = random_theta(S)
    counts = _symmetric_counts(rng, K, S)
    probe = FitEngine(np.ones(K), counts, theta0.copy(), num_epochs=0)
    mu0 = _mu(probe.Q[0].cpu().numpy())
    tmax = SYM_X_MAX / mu0
    times = np.exp(rng.uniform(np.log(1e-5 * tmax), np.log(tmax), K))
    times[0], times[-1] = 1e-5 * tmax, tmax
    n = 3
    a = _fit(times, counts, theta0, n, True, monkeypatch)
    b = _fit(times, counts, theta0, n, False, monkeypatch)
    assert squarings(tmax * _mu(a["Q_last"])) == S_STORE
    lab = np.max(np.abs(a["loss"] - b["loss"]) / np.abs(b["loss"]))
    qab = max(np.max(np.abs(a[k] - b[k])) / np.max(np.abs(b[k])) for k in ("Q_best", "Q_last"))
    ref = fit_oracle(times, counts, None, None, 0.1, n, dtype=torch.float64)
    lref = np.max(np.abs(a["loss"] - ref["loss"]) / np.abs(ref["loss"]))
    qref = np.max(np.abs(a["Q_last"] - ref["Q_last"])) / np.max(np.abs(ref["Q_last"]))
    print(f"S={S} K={K}: sym vs general loss {lab:.2e} Q {qab:.2e}; vs oracle loss {lref:.2e} Q {qref:.2e}")
    assert lab < 1e-11 and qab < 1e-9
    assert lref < REL_FP64 and qref < REL_FP64
