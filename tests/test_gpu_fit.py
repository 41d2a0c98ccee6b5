"""GPU parity tests for the fit (S <= 32 path): the CUDA engine against the fp64 oracle
(tolerance 1e-6 relative, BASELINE.json north_star) and against what the unmodified fp32
reference produced (tolerance 1e-4 relative)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from cherryml_b200 import _lib, caching
from cherryml_b200.estimation import (FitEngine, RateMatrixLearner, quantized_transitions_mle, random_theta,
                                      theta_from_initialization)
from cherryml_b200.io import read_mask_matrix, read_rate_matrix
from oracle.fit_oracle import fit_oracle, loss_and_grad_oracle
from tests.test_oracle_fit import FIT, INP, LG_COUNTS, SMALL_CASES, TOY, load_case

REL_FP64 = 1e-6   # vs the fp64 oracle (north_star: 1e-6 relative in fp64)
REL_FP32 = 1e-4   # vs the reference as shipped (north_star: 1e-4 in fp32)


def random_rate_matrix(S, rng, scale=1.0):
    Q = rng.random((S, S)) * scale
    np.fill_diagonal(Q, 0)
    np.fill_diagonal(Q, -Q.sum(axis=1))
    return Q


@pytest.mark.parametrize("S", [2, 3, 4, 8, 20, 21, 32])
def test_loss_and_gradient_match_the_oracle(S):
    """Times span 9 orders of magnitude: exercises every Taylor degree and up to ~15 squarings."""
    rng = np.random.default_rng(S)
    K = 24
    times = np.exp(rng.uniform(np.log(1e-7), np.log(60.0), K))
    Q = random_rate_matrix(S, rng)
    counts = rng.integers(0, 200, size=(K, S, S)).astype(np.float64)
    counts[rng.random(counts.shape) < 0.3] = 0.0
    eng = FitEngine(times, counts, random_theta(S), num_epochs=0)
    eng.Q.copy_(torch.from_numpy(Q)[None])
    loss, grad = eng.loss_and_grad()
    exp_loss, exp_grad = loss_and_grad_oracle(Q, times, counts)
    assert abs(float(loss[0]) - exp_loss) < 1e-10 * abs(exp_loss)
    g = grad[0].cpu().numpy()
    assert np.max(np.abs(g - exp_grad)) < 1e-9 * np.max(np.abs(exp_grad))


def _run_engine(q, counts, init, mask, g, do_adam=True):
    S = counts.shape[-1]
    m = np.ones((S, S)) if mask is None else mask
    theta0 = theta_from_initialization(init, m) if init is not None else random_theta(S)
    eng = FitEngine(q, counts, theta0, mask=mask, num_epochs=int(g["num_epochs"]), learning_rate=float(g["lr"]),
                    do_adam=do_adam)
    eng.run()
    return eng.results()


@pytest.mark.parametrize("name", sorted(SMALL_CASES))
def test_fit_matches_fp64_oracle_and_reference_run(name):
    q, _, counts, init, mask, g = load_case(name)
    do_adam = "sgd" not in name
    res = _run_engine(q, counts, init, mask, g, do_adam)
    ref = fit_oracle(q, counts, mask, init, float(g["lr"]), int(g["num_epochs"]), do_adam=do_adam,
                     dtype=torch.float64)
    assert np.max(np.abs(res["loss"] - ref["loss"]) / np.abs(ref["loss"])) < REL_FP64
    for key in ref:
        if key.startswith("Q_"):
            scale = np.max(np.abs(ref[key]))
            assert np.max(np.abs(res[key] - ref[key])) < REL_FP64 * scale, key
    # the reference as shipped (fp32 expm)
    assert np.max(np.abs(res["loss"] - g["loss"]) / np.abs(g["loss"])) < REL_FP32
    for key in ("Q_1", "Q_last", "Q_best"):
        scale = np.max(np.abs(g[key]))
        assert np.max(np.abs(res[key] - g[key])) < REL_FP32 * scale, key
    assert np.max(np.abs(res["Q_best"] - g["result"])) < REL_FP32 * np.max(np.abs(g["result"]))


def test_quantized_transitions_mle_stage_function(tmp_path):
    out = str(tmp_path / "mle")
    quantized_transitions_mle(
        count_matrices_path=LG_COUNTS, initialization_path=os.path.join(INP, "equ.txt"), mask_path=None,
        output_rate_matrix_dir=out, stationary_distribution_path=None,
        rate_matrix_parameterization="pande_reversible", device="cuda", learning_rate=1e-1, num_epochs=200,
        do_adam=True,
    )
    g = np.load(os.path.join(FIT, "lg20_init_equ", "reference_run.npz"))
    for name in ("result", "Q_1", "Q_2", "Q_4", "Q_128", "Q_best", "Q_last"):
        Q = read_rate_matrix(os.path.join(out, name + ".txt"))
        assert list(Q.index) == list(Q.columns) and len(Q) == 20
        assert np.max(np.abs(Q.to_numpy() - g[name])) < REL_FP32 * np.max(np.abs(g[name])), name
    import pandas as pd

    df = pd.read_csv(os.path.join(out, "df_res.txt"))
    assert list(df.columns[1:]) == ["nuc_norm", "frob_norm", "loss", "time", "epoch", "frob_norm_diag",
                                    "frob_norm_offdiag"]
    assert np.max(np.abs(df["loss"].to_numpy() - g["loss"]) / g["loss"]) < REL_FP32
    assert float(open(os.path.join(out, "profiling.txt")).read().split()[2]) > 0


def test_mask_pattern_and_incompatible_initialisation(tmp_path):
    """The reference's own fit tests (quantized_transitions_mle_test.py:39-67, 94-104, 130-139)."""
    with pytest.raises(ValueError):
        quantized_transitions_mle(
            count_matrices_path=TOY, initialization_path=os.path.join(INP, "3x3_pande_reversible_initialization.txt"),
            mask_path=os.path.join(INP, "3x3_mask.txt"), output_rate_matrix_dir=str(tmp_path / "a"), num_epochs=3)
    out = str(tmp_path / "b")
    quantized_transitions_mle(
        count_matrices_path=TOY, initialization_path=os.path.join(INP, "3x3_pande_reversible_initialization_mask.txt"),
        mask_path=os.path.join(INP, "3x3_mask.txt"), output_rate_matrix_dir=out, num_epochs=3)
    mask = read_mask_matrix(os.path.join(INP, "3x3_mask.txt")).to_numpy()
    Q = read_rate_matrix(os.path.join(out, "result.txt")).to_numpy()
    assert np.all((np.abs(Q) > 1e-8) == (mask == 1))
    out = str(tmp_path / "c")
    quantized_transitions_mle(
        count_matrices_path=LG_COUNTS, initialization_path=None, mask_path=os.path.join(INP, "20x20_random_mask.txt"),
        output_rate_matrix_dir=out, num_epochs=3)
    mask = read_mask_matrix(os.path.join(INP, "20x20_random_mask.txt")).to_numpy()
    Q = read_rate_matrix(os.path.join(out, "result.txt")).to_numpy()
    assert np.all((np.abs(Q) > 1e-8) == (mask == 1))


def test_batched_independent_problems_match_single_problem_runs():
    """The per-site batch (n_problems > 1): every problem evolves exactly as if run alone."""
    rng = np.random.default_rng(5)
    P, K, S = 7, 9, 20
    times = np.exp(rng.uniform(np.log(0.01), np.log(3.0), (P, K)))
    counts = rng.integers(0, 30, size=(P, K, S, S)).astype(np.float64)
    theta0 = np.stack([random_theta(S, seed=s) for s in range(P)])
    eng = FitEngine(times, counts, theta0, num_epochs=25, best_mode=1, lr_upper=0.2)
    eng.run()
    res = eng.results()
    for p in (0, 3, 6):
        single = FitEngine(times[p], counts[p], theta0[p], num_epochs=25, best_mode=1, lr_upper=0.2)
        single.run()
        r1 = single.results()
        assert np.array_equal(r1["loss"], res["loss_per_problem"][:, p])
        assert np.array_equal(r1["Q_best"], res["Q_best"][p])


def test_loss_decreases_and_graph_replay_equals_eager():
    q, _, counts, init, mask, g = load_case("lg20_init_lg")
    theta0 = theta_from_initialization(init, np.ones((20, 20)))
    a = FitEngine(q, counts, theta0, num_epochs=100)
    a.run()  # >= 64 epochs: replayed from a CUDA graph in chunks of 32
    b = FitEngine(q, counts, theta0, num_epochs=100)
    for _ in range(100):
        b.run(1)  # one epoch per call: plain launches
    ra, rb = a.results(), b.results()
    assert np.array_equal(ra["loss"], rb["loss"]) and np.array_equal(ra["Q_best"], rb["Q_best"])
    assert ra["loss"][-1] < ra["loss"][0]


# ----------------------------------------------------------------- large state spaces (S > 32)
CO_COUNTS = os.path.join(os.path.dirname(FIT), "counting/medium3/refcpp_count_co_matrices_dir_cherries_plus_plus/result.npz")


@pytest.mark.parametrize("S,K", [(36, 6), (64, 5), (100, 7), (400, 4), (36, 160)])
@pytest.mark.parametrize("tmin,grad_tol", [(1e-3, 1e-10), (1e-6, 1e-7)])
def test_large_loss_and_gradient_match_the_oracle(S, K, tmin, grad_tol):
    """With t down to 1e-6 the oracle's own gradient (autograd through torch.matrix_exp's
    block-triangular backward with |dL/dP| ~ 1e9) is only good to ~1e-8 relative, hence the
    looser gradient tolerance there; the loss is tight in both settings."""
    rng = np.random.default_rng(S)
    times = np.exp(rng.uniform(np.log(tmin), np.log(40.0), K))
    times[0], times[-1] = tmin, 55.0  # no squaring / many squarings
    Q = random_rate_matrix(S, rng, scale=2.0 / S)
    counts = rng.integers(0, 50, size=(K, S, S)).astype(np.float64)
    counts[rng.random(counts.shape) < 0.5] = 0.0
    eng = FitEngine(times, counts, random_theta(S), num_epochs=0)
    eng.Q.copy_(torch.from_numpy(Q)[None])
    loss, grad = eng.loss_and_grad()
    exp_loss, exp_grad = loss_and_grad_oracle(Q, times, counts)
    assert abs(float(loss[0]) - exp_loss) < 1e-10 * abs(exp_loss)
    g = grad[0].cpu().numpy()
    assert np.max(np.abs(g - exp_grad)) < grad_tol * np.max(np.abs(exp_grad))


def _co_inputs():
    z = np.load(CO_COUNTS)
    return z["q"], z["counts"]


@pytest.mark.parametrize("name,init,mask", [
    ("co400_init", "coevolution", None),
    ("co400_noinit_mask", None, "aa_coevolution_mask"),
])
def test_large_fit_matches_fp64_oracle_and_reference_run(name, init, mask):
    q, counts = _co_inputs()
    g = np.load(os.path.join(FIT, name, "reference_run.npz"))
    big = np.load(os.path.join(FIT, "inputs", "co400_inputs.npz"))
    init_a = big["coevolution"] if init else None
    mask_a = big["aa_coevolution_mask"].astype(np.float64) if mask else None
    n = int(g["num_epochs"])
    res = _run_engine(q, counts, init_a, mask_a, g)
    ref = fit_oracle(q, counts, mask_a, init_a, float(g["lr"]), n, dtype=torch.float64)
    assert np.max(np.abs(res["loss"] - ref["loss"]) / np.abs(ref["loss"])) < REL_FP64
    for key in ("Q_1", "Q_2", "Q_4", "Q_best", "Q_last"):
        scale = np.max(np.abs(ref[key]))
        assert np.max(np.abs(res[key] - ref[key])) < REL_FP64 * scale, key
    assert np.max(np.abs(res["loss"] - g["loss"]) / np.abs(g["loss"])) < REL_FP32
    for key in ("Q_1", "Q_last", "result"):
        mine = res["Q_best"] if key == "result" else res[key]
        assert np.max(np.abs(mine - g[key])) < REL_FP32 * np.max(np.abs(g[key])), key


def test_large_fit_small_padded_case_vs_oracle():
    """S = 36 (six-letter alphabet pairs): padded to 80 internally; 12 epochs of Adam."""
    rng = np.random.default_rng(9)
    S, K = 36, 8
    times = np.exp(rng.uniform(np.log(0.01), np.log(5.0), K))
    counts = rng.integers(0, 40, size=(K, S, S)).astype(np.float64)
    theta0 = random_theta(S)
    eng = FitEngine(times, counts, theta0, num_epochs=12)
    eng.run()
    res = eng.results()
    ref = fit_oracle(times, counts, None, None, 0.1, 12, dtype=torch.float64)
    assert np.max(np.abs(res["loss"] - ref["loss"]) / np.abs(ref["loss"])) < REL_FP64
    assert np.max(np.abs(res["Q_best"] - ref["Q_best"])) < REL_FP64 * np.max(np.abs(ref["Q_best"]))


@pytest.mark.parametrize("S,K,masked", [(36, 8, False), (100, 6, True), (400, 5, True)])
def test_symmetric_form_equals_the_general_evaluation(S, K, masked, monkeypatch):
    """Symmetric counts + symmetric mask: the epochs run on R Q R^-1 (symmetric) and compute the upper
    tiles only.  Same losses and the same iterates as the general evaluation (CHERRY_FIT_SYMMETRIC=0) to
    rounding -- 12 epochs of Adam amplify a 1e-16 difference to ~1e-12 -- and as the fp64 oracle; the
    times span no squaring ... many squarings.  Unsymmetric counts must fall back to the general form."""
    rng = np.random.default_rng(S + 1)
    tmax = 120.0 / S  # row sums of Q grow with S: up to ~6 squarings
    times = np.exp(rng.uniform(np.log(1e-3 * tmax), np.log(tmax), K))
    times[0], times[-1] = 1e-3 * tmax, tmax
    half = rng.integers(0, 40, size=(K, S, S)).astype(np.float64)
    half[rng.random(half.shape) < 0.4] = 0.0
    counts = half + half.transpose(0, 2, 1)
    mask = None
    if masked:
        m = (rng.random((S, S)) < 0.6).astype(np.float64)
        mask = np.maximum(m, m.T)
        np.fill_diagonal(mask, 1.0)
        counts = counts * mask[None]  # no transitions where the model allows none in one step... and beyond
        counts += (rng.random((S, S)) < 0.05)[None] * 1.0
        counts = 0.5 * (counts + counts.transpose(0, 2, 1))
    theta0 = random_theta(S)
    n = 12

    def run(sym):
        if sym:
            monkeypatch.delenv("CHERRY_FIT_SYMMETRIC", raising=False)
        else:
            monkeypatch.setenv("CHERRY_FIT_SYMMETRIC", "0")
        eng = FitEngine(times, counts, theta0.copy(), num_epochs=n, mask=mask)
        assert eng.symmetric_form == sym
        eng.run()
        return eng.results()

    a, b = run(True), run(False)
    assert np.max(np.abs(a["loss"] - b["loss"]) / np.abs(b["loss"])) < 1e-11
    for key in ("Q_best", "Q_last"):
        assert np.max(np.abs(a[key] - b[key])) < 1e-9 * np.max(np.abs(b[key])), key
    ref = fit_oracle(times, counts, mask, None, 0.1, n, dtype=torch.float64)
    assert np.max(np.abs(a["loss"] - ref["loss"]) / np.abs(ref["loss"])) < REL_FP64
    assert np.max(np.abs(a["Q_last"] - ref["Q_last"])) < REL_FP64 * np.max(np.abs(ref["Q_last"]))
    # unsymmetric counts: general form
    monkeypatch.delenv("CHERRY_FIT_SYMMETRIC", raising=False)
    eng = FitEngine(times, half, theta0.copy(), num_epochs=1, mask=mask)
    assert not eng.symmetric_form


@pytest.mark.parametrize("ta,tb", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("n,batch,ksplit", [(80, 3, 1), (160, 2, 2), (400, 2, 1), (400, 1, 5)])
def test_dmma_gemm_matches_cublas(ta, tb, n, batch, ksplit):
    from cherryml_b200.estimation._gemm import gemm_f64_batched

    gen = torch.Generator(device="cuda").manual_seed(n + batch)
    A = torch.randn(batch, n, n, dtype=torch.float64, device="cuda", generator=gen)
    B = torch.randn(batch, n, n, dtype=torch.float64, device="cuda", generator=gen)
    C0 = torch.randn(batch, n, n, dtype=torch.float64, device="cuda", generator=gen)
    ref = torch.matmul(A.transpose(1, 2) if ta else A, B.transpose(1, 2) if tb else B)
    got = gemm_f64_batched(A, B, ta, tb, ksplit=ksplit)
    assert torch.allclose(got, ref, rtol=1e-12, atol=1e-11)
    acc = gemm_f64_batched(A, B, ta, tb, C=C0.clone(), ksplit=ksplit)
    assert torch.allclose(acc, ref + C0, rtol=1e-12, atol=1e-11)


@pytest.mark.parametrize("S,K", [(20, 24), (48, 6)])
def test_bucket_sharded_epochs_equal_the_single_gpu_run(S, K):
    """The sharded epoch (local loss/gradient -> ONE all-reduce of [dL/dQ | loss] -> update) on a
    1-rank NCCL group must reproduce the graph-replayed single-GPU run: same kernels, same
    reduction order.  (World size 2 is covered on CPU by tests/test_dist_gloo.py and on the GPU
    by ``bench.py --gpus 2``.)"""
    import socket

    import torch.distributed as dist

    created = False
    if not dist.is_initialized():
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
        created = True
    try:
        rng = np.random.default_rng(S)
        times = np.exp(rng.uniform(np.log(1e-3), np.log(8.0), K))
        counts = rng.integers(0, 200, size=(K, S, S)).astype(np.float64)
        counts = counts + counts.transpose(0, 2, 1)
        theta0 = random_theta(S)
        a = FitEngine(times, counts, theta0, num_epochs=70)
        a.run()
        ra = a.results()
        b = FitEngine(times, counts, theta0, num_epochs=70, process_group=dist.group.WORLD)
        b.run()
        rb = b.results()
        assert np.allclose(ra["loss"], rb["loss"], rtol=1e-12, atol=0)
        assert np.allclose(ra["Q_best"], rb["Q_best"], rtol=1e-9, atol=1e-12)
        assert np.allclose(ra["Q_last"], rb["Q_last"], rtol=1e-9, atol=1e-12)
    finally:
        if created:
            dist.destroy_process_group()


@pytest.mark.parametrize("S,K", [(20, 24), (48, 6)])
def test_cherry_loss_autograd_node_in_a_reference_style_loop(S, K):
    """SURVEY 8(b): RateMatrix + torch.optim.Adam + CherryLoss (the CUDA loss/gradient as ONE autograd
    node) reproduce the fp64 oracle's training trajectory (rate.py + trainer.py restated on the CPU),
    for both the small (S <= 32) and the large kernel path."""
    import torch

    from cherryml_b200.estimation import CherryLoss, RateMatrix
    from oracle.fit_oracle import fit_oracle

    rng = np.random.default_rng(S)
    times = np.sort(np.exp(rng.uniform(np.log(0.01), np.log(3.0), K)))
    counts = rng.integers(0, 20, (K, S, S)).astype(np.float64)
    counts = counts + counts.transpose(0, 2, 1) + 30.0 * np.eye(S)[None]
    epochs = 12
    ref = fit_oracle(list(times), counts, num_epochs=epochs, dtype=torch.float64)
    model = RateMatrix(num_states=S, mode="pande_reversible", mask=None, pi_requires_grad=True, device="cuda:0")
    opt = torch.optim.Adam(model.parameters(), lr=0.1)
    t = torch.tensor(times, dtype=torch.float64, device="cuda:0")
    C = torch.tensor(counts, dtype=torch.float64, device="cuda:0")
    total = C.sum()
    losses = []
    for _ in range(epochs):
        opt.zero_grad()
        loss = CherryLoss.apply(model(), t, C) / total
        losses.append(float(loss.detach()))
        loss.backward()
        opt.step()
    assert np.max(np.abs(np.array(losses) - ref["loss"]) / np.abs(ref["loss"])) < 1e-6
    # the node's gradient against torch's own autograd through matrix_exp (fp64, on the GPU)
    Q = model().detach().clone().requires_grad_(True)
    CherryLoss.apply(Q, t, C).backward()
    Q2 = Q.detach().clone().requires_grad_(True)
    (-(C * torch.log(torch.matrix_exp(t[:, None, None] * Q2[None]))).sum()).backward()
    assert float((Q.grad - Q2.grad).abs().max() / Q2.grad.abs().max()) < 1e-9
