"""Small-S fit and expm (S <= 32, fit_small.cu) against extended-precision references, at every launch shape, tile
count, Taylor degree, squaring count and spill boundary the host can select.

The kernel evaluates expm(tQ) as X_0 = sum_{k<=m} B^k / k! (Horner, B = tQ / 2^s), then squares s times.  The
degree m and the count s come from ||tQ||_1 (choose_degree in fit_common.cuh); the documented truncation bound is
||B||_1^(m+1) / (m+1)! <= 1.1e-19 ||B||_1.

Tolerance of an entry, a-priori (not fitted to the measured error):
- rounding: X_0 is built by m products of length spad = 8 ceil(S / 8), so its entries (non-negative, little
  cancellation for ||B||_1 <= 0.04) carry at most (2m + 2)(spad + 2) u relative error; each squaring of a
  non-negative matrix at most doubles the relative error and adds (spad + 2) u.  So rel(s) = 2^s (2m + 2)(spad + 2) u.
- truncation: at s = 0 the error of entry (i, j) is at most R_ij = sum_{k>m} (|B|^k)_ij / k!, which for a banded or
  masked Q is zero or tiny exactly where the top term c_m B^m is the only one reaching the entry (so a wrong c_m,
  or a wrong degree, shows).  The series is evaluated in long double with the degree the documented bound asks
  for, not the kernel's table.  After s squarings the error E obeys ||E_{k+1}||_inf <= 2 ||E_k||_inf +
  ||E_k||_inf^2 (every exact power is stochastic), so it is at most 2^s max_i sum_j R_ij of the scaled B.
References (all in this file or in test_gpu_fit_large_coverage):
- uniformization in np.longdouble (entries non-negative, each within 1e-20 relative) while ||tQ||_1 <= 300;
- Kronecker sums of 2-state chains with dyadic rates (the fp64 Q is exact), whose expm is the Kronecker product
  of closed forms evaluated with expm1 in long double: exact at every exponent up to 30 squarings;
- for a reversible Q and ||tQ||_1 > 300, the stationary distribution solved in long double, P = 1 pi^T, plus the
  bound sqrt(pi_max / pi_min) exp(-gap t) of the spectral gap (below 1e-30 at these exponents);
- gradients: complex step, in complex128 through torch.matrix_exp for dense Q, through the long-double stationary
  solve at the largest exponents (along rate matrices), and for banded Q at s = 0 in np.clongdouble through the
  degree-m Taylor polynomial itself, whose exact adjoint the kernel computes;
- fits: oracle.fit_oracle and oracle.siterm_oracle.fit_sites in fp64.
"""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from cherryml_b200 import _lib
from cherryml_b200.estimation import FitEngine, random_theta
from cherryml_b200.estimation._engine import FitArgs
from cherryml_b200.markov_chain import expm_batched
from cherryml_b200.siterm import quantized_transitions_mle_vectorized_over_sites
from oracle.fit_oracle import fit_oracle
from oracle.siterm_oracle import fit_sites
from tests.test_gpu_fit import REL_FP64, random_rate_matrix
from tests.test_gpu_fit_large_coverage import U64, _complex_step, uniformized

LD, CLD = np.longdouble, np.clongdouble

# ------------------------------------------------------------------ the host's choices, mirrored from the source
_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cherryml_b200", "csrc")


def _source(name):
    with open(os.path.join(_CSRC, name)) as f:
        return f.read()


def _const(text, pattern):
    m = re.search(pattern, text)
    assert m, f"constant not found: {pattern}"
    return m.group(1)


_SMALL, _COMMON = _source("fit_small.cu"), _source("fit_common.cuh")
LAT_THREADS = int(_const(_SMALL, r"kSmallThreads = (\d+)"))
TP_THREADS = int(_const(_SMALL, r"kThroughputThreads = (\d+)"))
TP_SLOTS = int(_const(_SMALL, r"kThroughputSlots = (\d+)"))
TP_MAX_S = int(_const(_SMALL, r"return S <= (\d+) && grid > sm_count\(\)"))
SLOT_BUDGET = int(_const(_SMALL, r"budget = (\d+) \* 1024")) * 1024
MAX_DEG = int(_const(_COMMON, r"kMaxDegree = (\d+)"))
MAX_SQ = int(_const(_COMMON, r"kMaxSquarings = (\d+)"))
THETA = [float(x) for x in _const(_COMMON, r"theta\[kMaxDegree \+ 1\] = \{([^}]*)\}").split(",")]
TRUNC = 1.1e-19  # documented: theta_m^m / (m+1)! <= 1.1e-19


def ntl(S):
    return (S + 7) // 8


def throughput(S, grid, sms):
    return S <= TP_MAX_S and grid > sms


def resident_slots(S, tp):
    """fit_small_workspace: slots of 8 ntl x (8 ntl + 4) doubles in the shared-memory budget, at most the
    m + s + 4 the deepest evaluation uses, at most kThroughputSlots in the throughput shape."""
    spad = 8 * ntl(S)
    ns = min(SLOT_BUDGET // (spad * (spad + 4) * 8), MAX_DEG + MAX_SQ + 4)
    return min(ns, TP_SLOTS) if tp else ns


def first_spills(S, tp):
    """Smallest s at which (backward slots G0, G1, Bbar; forward result X_s) live in global memory (degree m = 9
    whenever s > 0): Bbar is slot m + s + 3, X_s is slot m + s."""
    ns = resident_slots(S, tp)
    return ns - MAX_DEG - 3, ns - MAX_DEG


def choose_degree(norm):
    """(m, s, in range) as choose_degree computes them."""
    for m in range(1, MAX_DEG + 1):
        if norm <= THETA[m]:
            return m, 0, True
    if not norm < 1e300:
        return MAX_DEG, 0, True
    s = max(0, math.ceil(math.log2(norm / THETA[MAX_DEG])))
    return MAX_DEG, min(s, MAX_SQ), s <= MAX_SQ


def documented_degree(norm):
    """Smallest degree whose truncation ||B||^(m+1)/(m+1)! stays within 1.1e-19 ||B||: the degree the tolerance
    assumes, independent of the kernel's table."""
    for m in range(1, 30):
        if norm ** m / math.factorial(m + 1) <= TRUNC:
            return m
    raise AssertionError(norm)


def col_norm(Q):
    """max column abs sum, added in row order as the kernel does"""
    cs = np.zeros(Q.shape[0])
    for i in range(Q.shape[0]):
        cs = cs + np.abs(Q[i])
    return float(cs.max())


# ------------------------------------------------------------------ the cases (fixed: the coverage test reads them)
THETA_DOC = (0.0, 2.2e-19, 8.1e-10, 1.38e-6, 6.0e-5, 6.0e-4, 2.8e-3, 8.4e-3, 0.0195, 0.0376)
S_CAP = 30
# ||tQ||_1 of the exponents: just below and above each degree threshold; just below 2^k theta_9 (s = k) and just
# above (s = k + 1) for every squaring count up to 30; a sweep of 16 per octave from 1e-20 to 0.04
DEGREE_NORMS = [th * f for th in THETA_DOC[1:] for f in (1 - 1e-3, 1 + 1e-3)]
SQUARING_NORMS = [THETA_DOC[9] * 2.0 ** k * (1 - 1e-3) for k in range(1, S_CAP + 1)] + \
                 [THETA_DOC[9] * 2.0 ** k * (1 + 1e-3) for k in range(1, S_CAP)]
SWEEP_NORMS = list(2.0 ** (np.arange(math.floor(16 * math.log2(1e-20)), math.ceil(16 * math.log2(0.04)) + 1) / 16))
UNIF_MAX = 300.0  # uniformization reference up to this ||tQ||_1 (s <= 14): bounded long-double work
OUT_OF_RANGE = THETA_DOC[9] * 2.0 ** S_CAP  # 4.0e7

EXPM_S = [1, 2, 7, 8, 9, 16, 17, 20, 24, 25, 31, 32]
# (S, kind): every S with a dense, a tridiagonal and a masked Q up to UNIF_MAX; beyond, Kronecker sums (S = 2^d)
# and reversible Q with their stationary distribution
EXPM_CASES = [(S, kind) for S in EXPM_S for kind in ("dense", "tridiagonal", "masked")] + \
             [(2, "kron"), (8, "kron"), (16, "kron"), (32, "kron"), (17, "reversible"), (20, "reversible"),
              (24, "reversible")]

# loss and gradient, dense reversible Q: (S, shape, squaring counts); both sides of each backward and X_s spill
LOSS_CASES = [(8, "throughput", (0, 7, 8, 10, 11)), (16, "throughput", (0, 7, 8, 10, 11)),
              (24, "throughput", (0, 7, 8, 10, 11)), (8, "latency", (0, 6)), (16, "latency", (0, 6)),
              (24, "latency", (0, 6, 28, 29)), (32, "latency", (0, 11, 12, 14, 15))]
# loss and gradient at s = 0 on a birth-death Q, one exponent just below each degree threshold
BANDED_CASES = [(8, "throughput"), (16, "throughput"), (24, "throughput"), (8, "latency"), (16, "latency"),
                (24, "latency"), (32, "latency")]
# the two shapes on one problem: S and the squaring counts (the throughput shape spills from s = 8 on)
SHAPE_CASES = [(8, 13), (16, 13), (24, 13)]
# fused update vs fit_oracle: (S, K); K = None means SMs + 13 (throughput for S <= 24, a 20-bucket batch ends
# after one bucket); K > S * S for S = 3
FUSED_CASES = [(3, 24), (3, None), (8, 21), (8, 41), (8, None), (20, 41), (20, None), (28, 41)]
SITE_S = [4, 12, 20, 28]


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _shape_of(name):
    return name == "throughput"


# ------------------------------------------------------------------ matrices and references
def _matrix(S, kind, seed):
    rng = np.random.default_rng(seed)
    if S == 1:
        return np.zeros((1, 1)), None
    if kind == "dense":
        return random_rate_matrix(S, rng), None
    if kind == "tridiagonal":  # birth-death, births dominant: the entries m steps up come from c_m B^m alone
        Q = np.diag(rng.uniform(0.5, 1.5, S - 1), 1) + np.diag(0.01 * rng.uniform(0.5, 1.5, S - 1), -1)
    elif kind == "masked":  # a sparse mask with a cycle through every state
        mask = rng.random((S, S)) < 0.12
        mask[np.arange(S), (np.arange(S) + 1) % S] = True
        Q = mask * rng.uniform(0.5, 1.5, (S, S))
    elif kind == "kron":  # Kronecker sum of 2-state chains, dyadic rates: exact in fp64
        d = int(round(math.log2(S)))
        rates = rng.choice(np.arange(1, 13) / 8.0, size=(d, 2))
        Q = np.zeros((1, 1))
        for a, b in rates:
            f = np.array([[-a, a], [b, -b]])
            Q = np.kron(Q, np.eye(2)) + np.kron(np.eye(Q.shape[0]), f)
        return Q, rates
    elif kind == "reversible":  # Q_ij = s_ij pi_j, s symmetric
        pi = rng.uniform(0.5, 1.5, S)
        pi /= pi.sum()
        s = rng.uniform(0.2, 1.0, (S, S))
        Q = (s + s.T) * pi[None, :]
    else:
        raise ValueError(kind)
    np.fill_diagonal(Q, 0.0)
    np.fill_diagonal(Q, -Q.sum(axis=1))
    return Q, None


def _kron_expm(rates, times):
    t = np.asarray(times, dtype=LD)
    P = np.ones((len(t), 1, 1), dtype=LD)
    for a, b in rates:
        a, b = LD(a), LD(b)
        e = -np.expm1(-(a + b) * t)
        f = np.empty((len(t), 2, 2), dtype=LD)
        f[:, 0, 1], f[:, 1, 0] = a / (a + b) * e, b / (a + b) * e
        f[:, 0, 0], f[:, 1, 1] = 1 - f[:, 0, 1], 1 - f[:, 1, 0]
        P = np.einsum("kab,kcd->kacbd", P, f).reshape(len(t), P.shape[1] * 2, P.shape[2] * 2)
    return P


def _solve(A, b):
    """Gaussian elimination with partial pivoting in A's dtype (long double or complex long double)."""
    A, b = A.copy(), b.copy()
    n = len(b)
    for c in range(n):
        p = c + int(np.argmax(np.abs(A[c:, c])))
        A[[c, p]], b[[c, p]] = A[[p, c]], b[[p, c]]
        f = A[c + 1:, c] / A[c, c]
        A[c + 1:] -= f[:, None] * A[c][None, :]
        b[c + 1:] -= f * b[c]
    x = np.zeros_like(b)
    for r in range(n - 1, -1, -1):
        x[r] = (b[r] - np.sum(A[r, r + 1:] * x[r + 1:])) / A[r, r]
    return x


def _stationary(Q, dtype=LD):
    S = Q.shape[0]
    A = np.asarray(Q).T.astype(dtype)
    A[-1, :] = 1
    b = np.zeros(S, dtype=dtype)
    b[-1] = 1
    return _solve(A, b)


def _stationary_bound(Q, pi, times):
    """|P_ij(t) - pi_j| <= sqrt(pi_j / pi_i) exp(-gap t) for a reversible Q"""
    p = np.asarray(pi, dtype=np.float64)
    A = np.sqrt(p)[:, None] * Q / np.sqrt(p)[None, :]
    gap = -np.sort(np.linalg.eigvalsh((A + A.T) / 2))[-2]
    return math.sqrt(p.max() / p.min()) * np.exp(-gap * np.asarray(times, dtype=np.float64))


def _unif(Q, times):
    if Q.shape[0] == 1 or not np.any(Q):
        return np.ones((len(times), 1, 1), dtype=LD) if Q.shape[0] == 1 else np.stack([np.eye(Q.shape[0], dtype=LD)] * len(times))
    out = np.zeros((len(times), Q.shape[0], Q.shape[0]), dtype=LD)
    lam = np.asarray(times) * float(np.max(-np.diag(Q)))
    for sel in (lam <= 1.0, lam > 1.0):  # converge the small exponents without the long series of the large ones
        if np.any(sel):
            out[sel] = uniformized(Q, np.asarray(times)[sel], LD)[0]
    return out


def reference_expm(Q, kind, rates, times):
    """(P in long double, absolute bound of the reference itself)"""
    times = np.asarray(times, dtype=np.float64)
    bound = np.zeros(len(times))
    if kind == "kron":
        return _kron_expm(rates, times), bound
    ref = np.zeros((len(times), Q.shape[0], Q.shape[0]), dtype=LD)
    norms = np.abs(times) * col_norm(Q)
    small = norms <= UNIF_MAX
    if np.any(small):
        ref[small] = _unif(Q, times[small])
    if np.any(~small):
        assert kind == "reversible", kind
        pi = _stationary(Q)
        ref[~small] = pi[None, None, :]
        bound[~small] = _stationary_bound(Q, pi, times[~small])
        assert bound.max() < 1e-30
    return ref, bound


def truncation_bound(Q, taus, degrees):
    """R = sum_{k > m} |tau Q|^k / k! entrywise, in long double, for every tau with its degree m."""
    S = Q.shape[0]
    kmax = S + MAX_DEG + 24
    A = np.abs(np.asarray(Q, dtype=LD))
    pw = [np.eye(S, dtype=LD)]
    for _ in range(kmax):
        pw.append(pw[-1] @ A)
    flat = np.stack(pw).reshape(kmax + 1, S * S)
    k = np.arange(kmax + 1)
    logw = np.array([[LD(j) * np.log(LD(abs(tau))) - LD(math.lgamma(j + 1)) if tau != 0 else -np.inf for j in k]
                     for tau in taus], dtype=LD)
    W = np.where(k[None, :] > np.asarray(degrees)[:, None], np.exp(logw), LD(0))
    R = (W @ flat).reshape(len(taus), S, S)
    # what the series leaves beyond kmax: each entry of |B|^k is below ||B||_1^k
    x = np.array([abs(tau) * col_norm(Q) for tau in taus])
    R += np.array(x, dtype=LD)[:, None, None] ** (kmax + 1) / LD(math.factorial(kmax + 1)) * 2
    return R


def expm_tolerance(Q, times, ref):
    """Entrywise a-priori tolerance of the kernel's result (module docstring)."""
    S = Q.shape[0]
    spad = 8 * ntl(S)
    cn = col_norm(Q)
    ms, ss = [], []
    for t in times:
        _, s, _ = choose_degree(abs(t) * cn)
        s = min(s, S_CAP)
        ms.append(documented_degree(abs(t) * cn / 2.0 ** s))
        ss.append(s)
    ms, ss = np.array(ms), np.array(ss)
    R = truncation_bound(Q, np.asarray(times) / 2.0 ** ss, ms)
    slack = np.where(ss[:, None, None] == 0, R, (2.0 ** ss * R.sum(axis=2).max(axis=1))[:, None, None])
    rel = 2.0 ** ss * (2 * ms + 2) * (spad + 2) * U64
    return rel[:, None, None] * ref + 2 * slack


# ------------------------------------------------------------------ raw calls
def _expm_raw(Qs, t):
    """cherry_expm_batched with n_problems = len(Qs), t [P, K]: (P_out [P, K, S, S] on the device, status)."""
    lib = _lib.load()
    P, K = t.shape
    S = Qs.shape[-1]
    nbytes = ctypes.c_size_t(0)
    _lib.check(lib.cherry_fit_workspace_bytes(S, K, P, ctypes.byref(nbytes)), "cherry_fit_workspace_bytes")
    ws = torch.empty(max(8, nbytes.value), dtype=torch.uint8, device="cuda")
    Qt = torch.tensor(np.ascontiguousarray(Qs), device="cuda")
    tt = torch.tensor(np.ascontiguousarray(t, dtype=np.float64), device="cuda")
    out = torch.empty((P, K, S, S), dtype=torch.float64, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    a = FitArgs()
    a.S, a.K, a.n_problems = S, K, P
    a.t, a.Q, a.status_flag = _lib.ptr(tt), _lib.ptr(Qt), _lib.ptr(flag)
    a.workspace, a.workspace_bytes = _lib.ptr(ws), nbytes.value
    _lib.check(lib.cherry_expm_batched(ctypes.byref(a), _lib.ptr(out), _lib.current_stream_ptr()), "expm")
    return out, int(flag.item())


def _expm_both_shapes(Q, times, sms):
    """The same exponents once in calls of at most SMs CTAs (latency shape) and once in one call of more than SMs
    (throughput shape for S <= 24); returns both results and the exponents of the second call."""
    lat = np.concatenate([expm_batched(Q, times[i:i + sms]).cpu().numpy() for i in range(0, len(times), sms)])
    big = np.resize(times, max(len(times), sms + 1))
    tp = expm_batched(Q, big).cpu().numpy()
    return lat, tp, big


def _expm_norms(kind):
    norms = DEGREE_NORMS + SQUARING_NORMS + SWEEP_NORMS
    if kind in ("dense", "tridiagonal", "masked"):
        norms = [x for x in norms if x <= UNIF_MAX]
    return norms


def _loss_norms(S, shape, s_list):
    return [THETA_DOC[9] * 2.0 ** s * (1 - 1e-3) if s > 0 else THETA_DOC[9] * (1 - 1e-3) for s in s_list] + \
           [THETA_DOC[9] * 2.0 ** s * (1 - 0.3) for s in s_list if s > 1]


_WORST = {}


def _report(section, value, tol):
    w = _WORST.get(section, (0.0, tol))
    _WORST[section] = (max(w[0], value), tol)
    print(f"WORST {section}: {_WORST[section][0]:.2e} (tolerance {tol})")


# ------------------------------------------------------------------ 0. the cases reach every host path
def test_cases_reach_every_host_path():
    """If a constant of fit_small.cu or fit_common.cuh moves, this names what no case reaches any more."""
    sms = _sms()
    for m in range(1, MAX_DEG + 1):
        assert THETA[m] ** m / math.factorial(m + 1) <= TRUNC * 1.001, f"theta[{m}] = {THETA[m]} breaks the bound"
    inst, degrees, squarings, fwd, bwd = set(), set(), set(), set(), set()
    for S, kind in EXPM_CASES:
        Q, _ = _matrix(S, kind, seed=S)
        cn = col_norm(Q)
        times = [x / cn for x in _expm_norms(kind)] if cn > 0 else [1.0]
        for tp in {False, throughput(S, max(len(times), sms + 1), sms)}:
            inst.add((tp, ntl(S)))
            for t in times:
                m, s, ok = choose_degree(abs(t) * cn)
                if ok:
                    degrees.add(m)
                    squarings.add(s)
                    fwd.add((tp, ntl(S), s))
    for S, shape, s_list in LOSS_CASES:
        tp = _shape_of(shape)
        assert throughput(S, sms + 1 if tp else 1, sms) == tp
        inst.add((tp, ntl(S)))
        for x in _loss_norms(S, shape, s_list):
            m, s, ok = choose_degree(x)
            assert ok
            bwd.add((tp, ntl(S), s))
            fwd.add((tp, ntl(S), s))
    for S, K in FUSED_CASES:
        inst.add((throughput(S, K or sms + 13, sms), ntl(S)))
    for S in SITE_S:
        inst.add((throughput(S, 4 * (sms // 4 + 3), sms), ntl(S)))
    want = {(True, n) for n in range(1, ntl(TP_MAX_S) + 1)} | {(False, n) for n in range(1, 5)}
    assert inst >= want, f"instantiations not reached: {sorted(want - inst)} on {sms} SMs"
    assert degrees >= set(range(1, MAX_DEG + 1)), f"degrees not reached: {set(range(1, MAX_DEG + 1)) - degrees}"
    assert squarings >= set(range(MAX_SQ + 1)), f"squaring counts not reached: {sorted(set(range(MAX_SQ + 1)) - squarings)}"
    for m in range(1, MAX_DEG + 1):
        near = [x for x in DEGREE_NORMS if abs(x / THETA[m] - 1) <= 2e-3]
        assert any(x <= THETA[m] for x in near) and any(x > THETA[m] for x in near), f"degree threshold {m} not bracketed"
    missing = []
    for tp, n in sorted(want):
        S = 8 * n
        sb, sx = first_spills(S, tp)
        if 0 < sb <= MAX_SQ and not {(tp, n, sb - 1), (tp, n, sb)} <= bwd:
            missing.append(f"backward spill at s = {sb} ({'throughput' if tp else 'latency'}, NTL = {n})")
        if 0 < sx <= MAX_SQ and not {(tp, n, sx - 1), (tp, n, sx)} <= fwd:
            missing.append(f"X_s spill at s = {sx} ({'throughput' if tp else 'latency'}, NTL = {n})")
    assert not missing, f"spill boundaries not reached: {missing}"

    # what actually launched: the kernel's template arguments, one call per instantiation
    from torch.profiler import ProfilerActivity, profile

    seen = {}
    for tp, n in sorted(want):
        S = 8 * n
        Q, _ = _matrix(S, "dense", seed=1)
        K = sms + 1 if tp else 2
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            expm_batched(Q, np.full(K, 0.1))
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if "expm_loss_grad_small" in e.name]
        if not names:
            print("no CUDA kernel activity recorded by torch.profiler: launch shapes not confirmed by name")
            return
        seen[(tp, n)] = {tuple(int(v) for v in re.search(r"expm_loss_grad_small<(\d+), (\d+), (\d+)>", x).groups())
                         for x in names}
    for (tp, n), got in seen.items():
        assert got == {(TP_THREADS, 2, n) if tp else (LAT_THREADS, 1, n)}, (tp, n, got)


# ------------------------------------------------------------------ 1. expm, every S, kind, degree and squaring
@pytest.mark.parametrize("S,kind", EXPM_CASES)
def test_expm_entrywise_against_extended_precision(S, kind):
    sms = _sms()
    Q, rates = _matrix(S, kind, seed=S)
    cn = col_norm(Q)
    times = np.array([0.0] + ([x / cn for x in _expm_norms(kind)] if cn > 0 else [1.0]))
    lat, tp, big = _expm_both_shapes(Q, times, sms)
    assert np.array_equal(lat[0], np.eye(S))
    assert np.array_equal(tp[:len(times)], lat), "latency and throughput shapes differ"
    ref, rbound = reference_expm(Q, kind, rates, times)
    tol = expm_tolerance(Q, times, ref) + rbound[:, None, None]
    err = np.abs(lat.astype(LD) - ref)
    bad = err > tol
    ratio = np.where(tol > 0, err / np.where(tol > 0, tol, 1), np.where(err > 0, np.inf, 0))
    assert not np.any(bad), (
        f"{int(bad.sum())} entries beyond tolerance, worst ratio {float(ratio.max()):.3g} "
        f"at exponent {times[np.argwhere(bad)[0][0]]!r} entry {tuple(np.argwhere(bad)[0][1:])}")
    s_of = np.array([choose_degree(abs(t) * cn)[1] for t in times])
    pos = ref > 1e-250
    rel = np.zeros(len(times))
    for i in range(len(times)):
        rel[i] = float(np.max(np.where(pos[i], err[i] / np.where(pos[i], ref[i], 1), 0)))
    for s in sorted(set(s_of)):
        _report(f"expm rel error at s = {s:2d}", float(rel[s_of == s].max()),
                f"{2.0 ** s * (2 * 9 + 2) * (8 * ntl(S) + 2) * U64:.1e} + truncation")
    _report("expm max error / tolerance", float(ratio.max()), 1.0)


# ------------------------------------------------------------------ 2. the two shapes agree
@pytest.mark.parametrize("S,s_max", SHAPE_CASES)
def test_latency_and_throughput_shapes_agree_bitwise(S, s_max):
    sms = _sms()
    rng = np.random.default_rng(S)
    Q = random_rate_matrix(S, rng)
    cn = col_norm(Q)
    times = np.array([THETA_DOC[9] * 2.0 ** s * f / cn for s in range(s_max + 1) for f in (0.3, 0.999)])
    K = len(times)
    P = sms // K + 1
    assert not throughput(S, K, sms) and throughput(S, P * K, sms)
    one, f1 = _expm_raw(Q[None], times[None])
    many, f2 = _expm_raw(np.repeat(Q[None], P, 0), np.repeat(times[None], P, 0))
    assert f1 == 0 and f2 == 0
    one, many = one.cpu().numpy(), many.cpu().numpy()
    for p in range(P):
        assert np.array_equal(many[p], one[0]), f"P_out of problem {p} differs between the shapes"
    counts = rng.integers(0, 30, size=(K, S, S)).astype(np.float64)

    def parts(n):
        eng = FitEngine(np.repeat(times[None], n, 0), np.repeat(counts[None], n, 0),
                        np.repeat(random_theta(S)[None], n, 0), num_epochs=0)
        eng.Q.copy_(torch.from_numpy(np.repeat(Q[None], n, 0)))
        eng.loss_and_grad()
        return (eng.dQ_part.view(n, K, S, S).cpu().numpy(), eng.loss_part.view(n, K).cpu().numpy())

    (g1, l1), (gp, lp) = parts(1), parts(P)
    worst = 0.0
    for p in range(P):
        assert np.array_equal(gp[p], g1[0]), f"dQ_part of problem {p} differs between the shapes"
        worst = max(worst, float(np.max(np.abs(lp[p] - l1[0]) / np.abs(l1[0]))))
    # positive terms summed in another order: within 2 S^2 u relative
    _report("shapes: loss_part rel", worst, f"{2 * S * S * U64:.1e}")
    assert worst <= 2 * S * S * U64, worst


# ------------------------------------------------------------------ 3. loss and gradient
def _stationary_loss(Q, E, counts, h=1e-30):
    """(-sum C log pi, and its directional derivative along E by the complex step), long double"""
    C = counts.sum(axis=0).astype(LD)
    pi = _stationary(Q)
    pic = _stationary(np.asarray(Q, dtype=CLD) + 1j * LD(h) * np.asarray(E, dtype=CLD), CLD)
    return -(C * np.log(pi)[None, :]).sum(), -(C * np.log(pic)[None, :]).sum().imag / LD(h)


def _directions(S, g, rng, band=None):
    R = rng.random((S, S))
    np.fill_diagonal(R, 0.0)
    np.fill_diagonal(R, -R.sum(axis=1))
    unit = np.zeros((S, S))
    unit[np.unravel_index(np.argmax(np.abs(g)), g.shape)] = 1.0
    dirs = [rng.standard_normal((S, S)), np.diag(rng.standard_normal(S)), R, unit]
    if band is not None:
        dirs.append(band * rng.standard_normal((S, S)))
    return dirs


@pytest.mark.parametrize("S,shape,s_list", LOSS_CASES)
def test_loss_and_directional_derivatives_across_spills(S, shape, s_list):
    sms = _sms()
    Q, _ = _matrix(S, "reversible", seed=100 + S)
    cn = col_norm(Q)
    norms = _loss_norms(S, shape, s_list)
    times = np.array(norms) / cn
    if _shape_of(shape):
        times = np.resize(times, sms + 1)
    K = len(times)
    rng = np.random.default_rng(S * 7 + len(s_list))
    counts = rng.integers(0, 40, size=(K, S, S)).astype(np.float64)
    counts[rng.random(counts.shape) < 0.4] = 0.0
    eng = FitEngine(times, counts, random_theta(S), num_epochs=0)
    eng.Q.copy_(torch.from_numpy(Q)[None])
    loss, grad = eng.loss_and_grad()
    g = grad[0].cpu().numpy()
    sumC = counts.sum()
    small = np.abs(times) * cn <= UNIF_MAX * 5
    ref, _ = reference_expm(Q, "reversible", None, times[small]) if np.any(small) else (None, None)
    exp_loss = LD(0)
    if np.any(small):
        exp_loss += -(counts[small].astype(LD) * np.log(ref)).sum()
    if np.any(~small):
        exp_loss += _stationary_loss(Q, np.zeros((S, S)), counts[~small])[0]
    exp_loss = float(exp_loss / LD(sumC))
    s_max = max(choose_degree(x)[1] for x in np.abs(times) * cn)
    ltol = 2.0 ** s_max * (2 * 9 + 2) * (8 * ntl(S) + 2) * U64
    lrel = abs(float(loss[0]) - exp_loss) / abs(exp_loss)
    _report("loss rel", lrel, "2^s (2m+2)(spad+2) u")
    assert lrel <= ltol, (lrel, ltol)
    dtol = max(1e-9, 2.0 ** s_max * 1e-13)
    drel = 0.0
    for E in _directions(S, g, rng):
        if np.any(~small):
            # the stationary reference holds along rate matrices only: off them exp(t(Q + hE)) also gains the
            # factor exp(t h pi^T E 1), which grows with t.  The fit moves Q along rate matrices.
            E = E - np.diag(E.sum(axis=1))
        d_ref = 0.0
        if np.any(small):
            d_ref += _complex_step(Q, times[small], counts[small], E) * counts[small].sum()
        if np.any(~small):
            d_ref += float(_stationary_loss(Q, E, counts[~small])[1])
        d_ref /= sumC
        drel = max(drel, abs(float((g * E).sum()) - d_ref) / abs(d_ref))
    _report("directional derivative rel (dense)", drel, "max(1e-9, 2^s 1e-13)")
    assert drel <= dtol, (drel, dtol)


def _taylor_complex(Qc, times, degrees):
    """sum_{k <= m} (t Qc)^k / k! in complex long double: the polynomial the kernel evaluates at s = 0"""
    S = Qc.shape[0]
    out = []
    for t, m in zip(times, degrees):
        B = LD(t) * Qc
        X = np.eye(S, dtype=CLD)
        term = np.eye(S, dtype=CLD)
        for k in range(1, m + 1):
            term = term @ B / LD(k)
            X = X + term
        out.append(X)
    return np.stack(out)


@pytest.mark.parametrize("S,shape", BANDED_CASES)
def test_top_taylor_term_and_its_adjoint_on_a_banded_matrix(S, shape):
    """At s = 0 the entries m steps above the diagonal of a birth-death Q come from c_m B^m alone; counts sit
    wherever the reference P is far above the truncation bound, so log P and its gradient see the top term."""
    sms = _sms()
    Q, _ = _matrix(S, "tridiagonal", seed=200 + S)
    cn = col_norm(Q)
    norms = [THETA_DOC[m] * (1 - 1e-3) for m in range(1, 10)]
    uniq = np.array(norms) / cn
    idx = np.arange(len(uniq))
    if _shape_of(shape):
        idx = np.resize(idx, sms + 1)
    times = uniq[idx]
    ref = _unif(Q, uniq)
    R = truncation_bound(Q, uniq, [documented_degree(x) for x in norms])
    rng = np.random.default_rng(S)
    counts = rng.integers(1, 20, size=(len(idx), S, S)).astype(np.float64)
    counts *= (ref[idx] > 1e6 * R[idx]).astype(np.float64)  # where truncation moves P by under 1e-6 relative
    eng = FitEngine(times, counts, random_theta(S), num_epochs=0)
    eng.Q.copy_(torch.from_numpy(Q)[None])
    loss, grad = eng.loss_and_grad()
    g = grad[0].cpu().numpy()
    sumC = counts.sum()
    C = counts.astype(LD)
    exp_loss = float(-(C * np.log(np.where(C > 0, ref[idx], 1))).sum() / LD(sumC))
    spad = 8 * ntl(S)
    # |d log P| <= rel + R / P <= (2m + 2)(spad + 2) u + 1e-6 on every counted entry
    lbound = float((C * ((2 * 9 + 2) * (spad + 2) * U64 + R[idx] / np.where(C > 0, ref[idx], 1))).sum() / LD(sumC))
    ldiff = abs(float(loss[0]) - exp_loss)
    _report("banded loss error / bound", ldiff / lbound, 1.0)
    assert ldiff <= lbound, (ldiff, lbound)
    # The gradient is the exact adjoint of the degree-m polynomial the kernel evaluates, so its reference is the
    # complex step of that polynomial (degree from the host's table) in complex long double.  The derivative of the
    # untruncated exp differs from it by paths longer than m that use one step of the direction: near the top
    # term those are not small relative to the entry, so the exact exp is no reference for the adjoint here.
    # The step must stay far below every counted entry: along a dense direction E an entry ~1e-38 reached in d band
    # steps gains t h E_ij in one step, so h = 1e-30 would not be a small perturbation of log P there.
    degrees = [choose_degree(x)[0] for x in norms]
    h = LD(10) ** -1000
    band = (np.abs(np.arange(S)[:, None] - np.arange(S)[None, :]) <= 1).astype(np.float64)
    drel = 0.0
    for E in _directions(S, g, rng, band):
        Pc = _taylor_complex(np.asarray(Q, dtype=CLD) + 1j * h * np.asarray(E, dtype=CLD), uniq, degrees)
        Lc = -(C * np.log(np.where(C > 0, Pc[idx], 1))).sum() / LD(sumC)
        d_ref = float(Lc.imag / h)
        drel = max(drel, abs(float((g * E).sum()) - d_ref) / abs(d_ref))
    _report("banded directional derivative rel", drel, 1e-9)
    assert drel <= 1e-9, drel


# ------------------------------------------------------------------ 4. the fused update against the fp64 oracles
@pytest.mark.parametrize("S,K", FUSED_CASES)
def test_fused_sgd_update_with_mask_matches_the_oracle(S, K):
    sms = _sms()
    K = K or sms + 13
    rng = np.random.default_rng(S * 1000 + K)
    times = np.exp(rng.uniform(np.log(1e-3), np.log(5.0), K))
    half = rng.integers(0, 6, size=(K, S, S)).astype(np.float64)
    counts = half + half.transpose(0, 2, 1)
    mask = (rng.random((S, S)) < 0.8).astype(np.float64)
    mask = np.triu(mask, 1) + np.triu(mask, 1).T + np.eye(S)
    mask[0, 1] = mask[1, 0] = 1.0
    n, lr = 5, 0.05 / counts.sum()
    eng = FitEngine(times, counts, random_theta(S), mask=mask, num_epochs=n, learning_rate=lr, do_adam=False,
                    loss_normalization=False)
    eng.run()
    res = eng.results()
    ref = fit_oracle(times, counts, mask, None, lr, n, do_adam=False, loss_normalization=False, dtype=torch.float64)
    lrel = float(np.max(np.abs(res["loss"] - ref["loss"]) / np.abs(ref["loss"])))
    qrel = max(float(np.max(np.abs(res[k] - ref[k])) / np.max(np.abs(ref[k]))) for k in ("Q_best", "Q_last"))
    _report("fused SGD update: loss rel", lrel, REL_FP64)
    _report("fused SGD update: Q rel", qrel, REL_FP64)
    assert lrel < REL_FP64 and qrel < REL_FP64, (lrel, qrel)


@pytest.mark.parametrize("S", SITE_S)
def test_batched_per_site_fit_matches_the_oracle(S):
    sms = _sms()
    B = 4
    L = sms // B + 3
    rng = np.random.default_rng(S)
    init = np.stack([_matrix(S, "reversible", seed=1000 * S + l)[0] for l in range(L)])
    init /= -np.mean(np.diagonal(init, axis1=1, axis2=2), axis=1)[:, None, None]
    times = np.tile(np.array([0.05, 0.3, 1.0, 3.0]), (L, 1)) * rng.uniform(0.5, 2.0, (L, 1))
    half = rng.integers(0, 8, size=(L, B, S, S)).astype(np.float64)
    counts = half + half.transpose(0, 1, 3, 2)
    n = 8
    got = quantized_transitions_mle_vectorized_over_sites(counts, times, num_epochs=n, initialization=init)
    ref = fit_sites(counts, times, n, init)
    e1 = float(np.max(np.abs(got["loss_per_epoch"] - ref["loss_per_epoch"]) / np.abs(ref["loss_per_epoch"])))
    e2 = float(np.max(np.abs(got["loss_per_epoch_per_site"] - ref["loss_per_epoch_per_site"])
                      / np.abs(ref["loss_per_epoch_per_site"])))
    e3 = float(np.max(np.abs(got["res"] - ref["res"])) / np.max(np.abs(ref["res"])))
    _report("per-site fit: loss, per-site loss, res", max(e1, e2, e3), REL_FP64)
    assert max(e1, e2, e3) < REL_FP64, (e1, e2, e3)


# ------------------------------------------------------------------ 5. range
@pytest.mark.parametrize("S", [4, 20, 32])
def test_exponents_beyond_thirty_squarings_are_reported(S):
    Q, _ = _matrix(S, "reversible", seed=300 + S)
    cn = col_norm(Q)
    with pytest.raises(_lib.CherryError, match=r"4\.0e7"):
        expm_batched(Q, [1.0 / cn, OUT_OF_RANGE * 1.001 / cn])
    P = expm_batched(Q, [OUT_OF_RANGE * 0.999 / cn]).cpu().numpy()
    assert np.all(np.isfinite(P))
    assert choose_degree(OUT_OF_RANGE * 0.999)[1:] == (S_CAP, True)


def test_fit_with_a_bucket_beyond_the_range_raises():
    S, K = 20, 6
    rng = np.random.default_rng(5)
    counts = rng.integers(0, 10, size=(K, S, S)).astype(np.float64)
    eng = FitEngine(np.ones(K), counts, random_theta(S), num_epochs=0)
    cn = col_norm(eng.Q[0].cpu().numpy())
    times = np.linspace(0.1, 2.0, K)
    times[3] = OUT_OF_RANGE * 1.01 / cn
    eng = FitEngine(times, counts, random_theta(S), num_epochs=2)
    eng.run()
    with pytest.raises(_lib.CherryError, match="status 2"):
        eng.results()
