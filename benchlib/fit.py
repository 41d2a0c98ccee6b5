"""Fit timings reported by bench.py under the "fit" key (BASELINE.json: "end-to-end fit
seconds (LG 20x20, coevo 400x400)")."""
import ctypes
import time
from typing import Dict, Optional

import numpy as np
import torch

from cherryml_b200 import _lib
from cherryml_b200.estimation._engine import FitEngine, theta_from_initialization
from cherryml_b200.estimation._jtt_ipw import jtt_ipw_from_counts
from benchlib.hostcores import usable_cores


def measure_fp64_gemm_peak(device, n: int = 4096, reps: int = 5) -> float:
    """cuBLAS DGEMM throughput (TFLOP/s) on this GPU: the denominator for the 400x400 fit's
    roofline, measured here because MEASURED_PEAKS.json has no FP64 figure."""
    a = torch.randn(n, n, dtype=torch.float64, device=device)
    b = torch.randn(n, n, dtype=torch.float64, device=device)
    for _ in range(2):
        torch.matmul(a, b)
    torch.cuda.synchronize(device)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize(device)
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * n**3 / (best * 1e-3) / 1e12


def _sync(device, process_group):
    if process_group is not None:
        import torch.distributed as dist

        dist.barrier(group=process_group)
    torch.cuda.synchronize(device)


def timed_fit(times, counts: torch.Tensor, num_epochs: int, mask=None, process_group=None) -> Dict:
    """JTT-IPW initialisation + `num_epochs` Adam epochs + results back on the host.  With a
    process group the buckets are sharded over its ranks (one all-reduce per epoch) and the
    times are the maximum over the ranks."""
    device = counts.device
    _sync(device, process_group)
    t0 = time.perf_counter()
    init = jtt_ipw_from_counts(times, counts, mask=mask)
    S = counts.shape[-1]
    theta0 = theta_from_initialization(init, np.ones((S, S)) if mask is None else mask)
    eng = FitEngine(np.asarray(times), counts, theta0, mask=mask, num_epochs=num_epochs, device=device,
                    process_group=process_group, rate_scale=float(np.max(-np.diag(init))))
    torch.cuda.synchronize(device)
    t_setup = time.perf_counter()
    _lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.run()
    e1.record()
    res = eng.results()
    t1 = time.perf_counter()
    secs = [t1 - t0, t_setup - t0, e0.elapsed_time(e1) * 1e-3]
    n_ranks = 1
    if process_group is not None:
        import torch.distributed as dist

        tt = torch.tensor(secs, dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX, group=process_group)
        secs = [float(x) for x in tt]
        n_ranks = dist.get_world_size(process_group)
    out = {
        "S": int(S), "K": int(len(times)), "num_epochs": int(num_epochs), "n_gpus": n_ranks,
        "sharding": "replica" if n_ranks == 1 else f"buckets over {n_ranks} ranks, one all-reduce of [dL/dQ | loss] per epoch",
        "buckets_this_rank": int(eng.K),
        "seconds_end_to_end": secs[0], "seconds_setup_init": secs[1],
        "seconds_device_epochs": secs[2],
        "ms_per_epoch": secs[2] * 1e3 / max(1, num_epochs),
        "loss_first": float(res["loss"][0]), "loss_last": float(res["loss"][-1]),
        "gpu_launches": _lib.launch_count(),
    }
    if S > 32:
        s = (ctypes.c_int * len(times))()
        mu, deg = ctypes.c_double(0), ctypes.c_int(0)
        _lib.check(_lib.load().cherry_fit_schedule(ctypes.byref(eng.args), s, ctypes.byref(mu), ctypes.byref(deg)),
                   "cherry_fit_schedule")
        sq = int(sum(s[: eng.K]))
        products_fwd = (deg.value - 1) + sq
        sym = bool(eng.symmetric_form)
        if sym:
            # symmetric form: the forward chain and all squaring products compute the tiles on and above the
            # diagonal only (15 of 25 for 400 x 400); the backward chain runs in full
            tn = -(-S // 80)
            upper = (tn * (tn + 1) / 2) / (tn * tn)
            executed = upper * (deg.value - 1) + upper * 3 * sq + 2 * (deg.value - 1)
        else:
            executed = 3.0 * products_fwd
        flops_epoch = executed * 2.0 * S**3
        out.update({
            "symmetric_form": sym,
            "taylor_degree": deg.value, "squarings_total": sq, "squarings_max": int(max(s[: eng.K])),
            "matrix_products_per_epoch": executed, "flop_per_epoch": flops_epoch,
            "tflops_executed": flops_epoch * num_epochs / out["seconds_device_epochs"] / 1e12,
            "mu": mu.value,
        })
    return out


def cpu_fit_baseline(times, counts: torch.Tensor, num_epochs_full: int, epochs_timed: int) -> Dict:
    """The reference's CPU fit on this box's host cores, same counts: the torch-CPU port of
    rate.py + trainer.py (oracle/fit_oracle.py; in fp32 -- the reference's arithmetic -- it
    reproduces the unmodified reference run bit for bit), all host threads, JTT-IPW init.
    A bounded number of epochs is timed and scaled linearly to the full run (epochs are
    identical work)."""
    import os

    from oracle.fit_oracle import fit_oracle

    cores = usable_cores()
    old = torch.get_num_threads()
    torch.set_num_threads(cores)
    try:
        init = jtt_ipw_from_counts(times, counts)
        c = counts.cpu().numpy()
        fit_oracle(times, c, None, init, 0.1, 1, dtype=torch.float32)  # warm-up (thread pools)
        t0 = time.perf_counter()
        fit_oracle(times, c, None, init, 0.1, epochs_timed, dtype=torch.float32)
        dt = time.perf_counter() - t0
    finally:
        torch.set_num_threads(old)
    return {"kind": "port", "cores": cores, "seconds_per_epoch": dt / epochs_timed,
            "seconds_extrapolated": dt / epochs_timed * num_epochs_full,
            "sample": f"{epochs_timed} of {num_epochs_full} epochs timed (torch CPU, fp32 expm as the reference, "
                      f"{cores} threads), scaled linearly"}


def _states_for(S: int):
    from cherryml_b200.utils import amino_acids

    if S == len(amino_acids):
        return list(amino_acids)
    if S == len(amino_acids) ** 2:
        return [a + b for a in amino_acids for b in amino_acids]
    return [f"s{i}" for i in range(S)]


def reference_fit_arms(times, counts: torch.Tensor, num_epochs_full: int, cpu_epochs: int, cuda_epochs: int,
                       workdir: str, timeout_s: int = 180) -> Dict:
    """The UNMODIFIED reference ``quantized_transitions_mle`` (reference
    estimation/_quantized_transitions_mle.py:40-122 -> ratelearner.py:66-152 -> trainer.py:118-243) on
    the SAME count matrices and JTT-IPW initialisation as our arm, as two arms (SURVEY.md 8d item 2):
      * ``cpu``  -- device="cpu", OMP/OPENBLAS threads = all host cores of this box;
      * ``cuda`` -- the reference's own stock device="cuda" path on this B200 (torch.matrix_exp +
        autograd, count tensor re-uploaded every epoch as trainer.py:160-166 does).
    Each arm runs oracle/run_reference_fit.py in its own process on files written here (count matrices
    in the Python writer's layout: exact reprs).  When fewer than ``num_epochs_full`` epochs are timed
    the end-to-end seconds are extrapolated as  (wall - training) + first epoch + (E - 1) * mean later
    epoch  -- epochs are identical work -- and the sample says so."""
    import json
    import os
    import subprocess
    import sys

    from cherryml_b200.io import write_count_matrices_array, write_rate_matrix

    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runner = os.path.join(repo, "oracle", "run_reference_fit.py")
    S = int(counts.shape[-1])
    states = _states_for(S)
    os.makedirs(workdir, exist_ok=True)
    counts_path = os.path.join(workdir, f"counts_{S}.txt")
    init_path = os.path.join(workdir, f"init_{S}.txt")
    write_count_matrices_array(list(times), states, counts.cpu().numpy(), counts_path, "python")
    write_rate_matrix(jtt_ipw_from_counts(times, counts), states, init_path)
    cores = usable_cores()
    out: Dict = {}
    for arm, epochs in (("cpu", cpu_epochs), ("cuda", cuda_epochs)):
        if epochs <= 0:
            continue
        epochs = min(epochs, num_epochs_full)
        odir = os.path.join(workdir, f"ref_{S}_{arm}")
        cmd = [sys.executable, runner, "--counts", counts_path, "--init", init_path, "--device", arm,
               "--epochs", str(epochs), "--threads", str(cores), "--out", odir]
        _log(f"reference arm {S}x{S} {arm}: {epochs} epochs ...")
        # a clean environment: torchrun pins its workers to OMP_NUM_THREADS=1 and exports its rendezvous
        # variables; the reference arm is a plain single process with all host threads
        env = {k: v for k, v in os.environ.items()
               if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "RANK", "LOCAL_RANK",
                            "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK", "MASTER_ADDR", "MASTER_PORT")
               and not k.startswith("TORCHELASTIC")}
        try:
            res = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
            line = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
            if res.returncode != 0 or not line:
                out[arm] = {"error": (res.stderr or res.stdout)[-300:]}
                continue
            r = json.loads(line[-1])
        except Exception as e:  # the extra measurement must not cost the bench line
            out[arm] = {"error": str(e)[:300]}
            continue
        setup = r["wall_seconds"] - r["train_seconds"]
        full = setup + r["first_epoch_seconds"] + (num_epochs_full - 1) * r["seconds_per_epoch"]
        out[arm] = {
            "kind": "reference", "device": arm, "cores": cores if arm == "cpu" else 1,
            "epochs_timed": r["epochs"], "seconds_measured": r["wall_seconds"],
            "seconds_setup_parse_write": setup, "seconds_per_epoch": r["seconds_per_epoch"],
            "seconds_end_to_end": r["wall_seconds"] if epochs == num_epochs_full else full,
            "extrapolated": epochs != num_epochs_full,
            "loss_first": r["loss_first"], "loss_last": r["loss_last"], "torch": r["torch"],
            "sample": (f"unmodified reference quantized_transitions_mle(device='{arm}'), same result.txt and "
                       f"JTT-IPW init as our arm, {r['epochs']} of {num_epochs_full} epochs timed"
                       + ("" if epochs == num_epochs_full else ", later epochs scaled linearly")
                       + (f", {cores} OMP/BLAS threads" if arm == "cpu" else ", torch.matrix_exp + autograd on this GPU")),
        }
    return out


def attach_reference_arms(out: Dict, inputs: Dict) -> None:
    """Reference arms (SURVEY 8d item 2): the UNMODIFIED reference stage on the box's host cores and its
    own device="cuda" path on this GPU, same count matrices and initialisation; the oracle port only
    when the reference package did not travel (oracle/_ref/reference_package.tar.gz absent).

    Run it when nothing else is using the host: the reference's cpu arm is one OpenMP team over all
    cores and its cuda arm is launch-bound on one host thread, so both slow down many times over when
    other ranks of the bench are still working on the same box (measured at N=2: 75 s instead of 1.8 s
    for the 20x20 cpu arm while rank 1 ran its next section).  bench.py therefore defers this call to
    the end, after the other ranks have exited."""
    import shutil
    import tempfile

    from oracle.ref_package import reference_available

    lg_times, lg_counts, grid, co_counts = (inputs[k] for k in ("lg_times", "lg_counts", "grid", "co_counts"))
    num_epochs, ref_epochs = inputs["num_epochs"], inputs["ref_epochs"]
    try:
        if reference_available():
            work = tempfile.mkdtemp(prefix="cherry_ref_fit_")
            lg = reference_fit_arms(lg_times, lg_counts, num_epochs, ref_epochs["lg_cpu"], ref_epochs["lg_cuda"], work)
            co_ref = reference_fit_arms(grid, co_counts, num_epochs, ref_epochs["co_cpu"], ref_epochs["co_cuda"], work)
            shutil.rmtree(work, ignore_errors=True)
            for key, arms in (("lg_20x20", lg), ("coevo_400x400", co_ref)):
                if "cpu" in arms:
                    out[key]["cpu_baseline"] = arms["cpu"]
                if "cuda" in arms:
                    out[key]["reference_cuda"] = arms["cuda"]
                ours = out[key]["seconds_end_to_end"]
                for arm, name in (("cpu", "speedup_vs_reference_cpu"), ("cuda", "speedup_vs_reference_cuda")):
                    if arm in arms and "seconds_end_to_end" in arms[arm]:
                        out[key][name] = arms[arm]["seconds_end_to_end"] / ours
        else:
            out["lg_20x20"]["cpu_baseline"] = cpu_fit_baseline(lg_times, lg_counts, num_epochs, 100)
            out["coevo_400x400"]["cpu_baseline"] = cpu_fit_baseline(grid, co_counts, num_epochs, 2)
    except Exception as e:  # the extra measurement must not cost the bench line
        out["cpu_baseline_error"] = str(e)[:200]


def _log(msg):
    import sys

    sys.stderr.write(f"[bench fit {time.strftime('%H:%M:%S')}] {msg}\n")
    sys.stderr.flush()


def bench_fit(device, lg_times=None, lg_counts: Optional[torch.Tensor] = None, num_epochs: int = 500,
              co_families: int = 16384, process_group=None, cpu_baseline: bool = False,
              ref_epochs: Optional[Dict] = None, defer_reference: bool = False) -> Dict:
    from cherryml_b200.counting._device import count_raw, sorted_grid, symmetrize
    from cherryml_b200.synthetic import as_device_batch, quantization_grid, synthetic_co, synthetic_lg

    grid = quantization_grid()
    K = len(grid)
    ref_epochs = dict({"lg_cpu": 100, "lg_cuda": 100, "co_cpu": 2, "co_cuda": 10}, **(ref_epochs or {}))
    out: Dict = {"metric": "end-to-end fit seconds", "init": "jtt-ipw", "optimizer": "Adam lr=0.1",
                 "dtype": "f64"}
    if lg_counts is None:
        dev = as_device_batch(synthetic_lg(512, 1024, 300, 4, seed=7, device=device), device)
        gd = torch.from_numpy(sorted_grid(grid)).to(device)
        lg_counts = symmetrize(count_raw(dev, gd, K, 20), "lg", K, 20, False)
        lg_times = grid
    # 20 x 20: one wave of CTAs, an epoch is latency -- it stays on one GPU (replicas when N > 1)
    timed_fit(lg_times, lg_counts, 64)  # warm-up (module load, graph instantiation paths)
    out["lg_20x20"] = timed_fit(lg_times, lg_counts, num_epochs)
    _log(f"lg fit done: {out['lg_20x20']['seconds_end_to_end']:.3f} s")
    rank = 0
    if process_group is not None:
        import torch.distributed as dist

        rank = dist.get_rank(process_group)
    # co-evolution counts from synthetic contact-map families (BASELINE config 4 shape)
    from cherryml_b200 import _lib
    from cherryml_b200.counting._device import build_bucket_table_tiles

    lib = _lib.load()
    dev = as_device_batch(synthetic_co(co_families, 1024, 300, seed=11 + rank, device=device), device)
    gd = torch.from_numpy(sorted_grid(grid)).to(device)
    raw = count_raw(dev, gd, K, 20)  # warm-up (and the counts the fit below uses)
    if process_group is not None:  # every rank counted its own families: one all-reduce of the raw histogram
        dist.all_reduce(raw, op=dist.ReduceOp.SUM, group=process_group)
    co_counts = symmetrize(raw, "co", K, 20, False)
    order = torch.empty(dev.n_pairs, dtype=torch.int32, device=device)
    recs = torch.empty(dev.n_pairs * 16, dtype=torch.uint8, device=device)
    ws = torch.empty(2 * (K + 2), dtype=torch.int32, device=device)
    st = _lib.current_stream_ptr()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    reps = 5
    ms_total = ms_kernel = 0.0
    for _ in range(reps):
        raw.zero_()
        torch.cuda.synchronize(device)
        ev[0].record()
        tab = build_bucket_table_tiles(dev, gd, K)
        _lib.check(lib.cherry_sort_pairs_by_bucket(
            _lib.ptr(tab), dev.r_pad, dev.n_pairs, K, _lib.ptr(dev.fams), _lib.ptr(dev.pair_a),
            _lib.ptr(dev.pair_b), _lib.ptr(dev.pair_fam), _lib.ptr(order), _lib.ptr(recs), _lib.ptr(ws), st),
            "cherry_sort_pairs_by_bucket")
        ev[1].record()
        _lib.check(lib.cherry_count_co(_lib.ptr(dev.msa), _lib.ptr(recs), _lib.ptr(ws), dev.n_pairs,
                                       dev.max_row_stride, K, 20, _lib.ptr(raw), st), "cherry_count_co")
        ev[2].record()
        symmetrize(raw, "co", K, 20, False)
        ev[3].record()
        torch.cuda.synchronize(device)
        ms_total += ev[0].elapsed_time(ev[3]) / reps
        ms_kernel += ev[1].elapsed_time(ev[2]) / reps
    # algorithmic bytes of the counting kernel: every residue byte of the contact-paired rows
    # once (4 B per (pair, contact)) + one 16-byte record per pair; the 64 MB histogram stays in L2
    alg_bytes = dev.msa.numel() + 16 * dev.n_pairs
    try:
        import json
        import os

        peak = float(json.load(open(os.path.join(os.path.dirname(os.path.dirname(
            os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        peak, peak_src = 6650.0, "fallback 6650 GB/s"
    achieved = alg_bytes / (ms_kernel * 1e-3) / 1e9
    out["co_counting"] = {
        "workload": f"synthetic co-evolution: {co_families} families x 1024 seqs x 300 sites, perfect "
                    "matching (150 contacts), 100 time buckets",
        "items_examined": dev.n_sites_examined, "ms_per_pass": ms_total,
        "items_per_s": dev.n_sites_examined / (ms_total * 1e-3),
        "roofline": {"bound": "hbm", "kernel": "count_co_sorted_kernel", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "algorithmic_bytes_per_launch": alg_bytes,
                     "kernel_ms": ms_kernel, "peak_source": peak_src},
    }
    del order, recs
    _log(f"co counting done: {ms_total:.3f} ms per pass")
    peak = measure_fp64_gemm_peak(device)
    timed_fit(grid, co_counts, 4, process_group=process_group)
    # The north-star deliverable as ONE timed region (reference estimation_end_to_end/_cherry.py:449-584 from
    # the encoded families on): co-transition counting of this rank's families -> all-reduce of the raw
    # histogram -> symmetrise -> JTT-IPW -> num_epochs Adam epochs (bucket-sharded, one all-reduce per epoch)
    # -> rate matrix on the host.  Wall clock, maximum over the ranks.
    _sync(device, process_group)
    t0 = time.perf_counter()
    raw.zero_()
    count_raw(dev, gd, K, 20, out=raw)
    if process_group is not None:
        dist.all_reduce(raw, op=dist.ReduceOp.SUM, group=process_group)
    co_counts = symmetrize(raw, "co", K, 20, False)
    co = timed_fit(grid, co_counts, num_epochs, process_group=process_group)
    e2e_s = time.perf_counter() - t0
    if process_group is not None:
        tt = torch.tensor([e2e_s], dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX, group=process_group)
        e2e_s = float(tt[0])
    n_ranks = 1 if process_group is None else dist.get_world_size(process_group)
    out["coevo_end_to_end_seconds"] = e2e_s
    _log(f"coevo end to end done: {e2e_s:.3f} s ({co['ms_per_epoch']:.4f} ms per epoch)")
    out["coevo_end_to_end"] = {
        "seconds": e2e_s, "n_gpus": n_ranks, "families_total": co_families * n_ranks,
        "stages": "count_co (families resident in HBM) -> all-reduce -> symmetrise -> JTT-IPW -> "
                  f"{num_epochs} Adam epochs -> rate matrix on host",
        "seconds_fit": co["seconds_end_to_end"], "seconds_counting": e2e_s - co["seconds_end_to_end"]}
    del raw, dev
    co["roofline"] = {"bound": "tensor", "unit": "TFLOP/s", "achieved": co["tflops_executed"], "peak": peak,
                      "frac": co["tflops_executed"] / peak,
                      "peak_source": "cuBLAS DGEMM 4096^3 measured in this run (no FP64 figure in MEASURED_PEAKS.json)"}
    out["coevo_400x400"] = co
    if cpu_baseline and rank == 0:
        inputs = {"lg_times": lg_times, "lg_counts": lg_counts.detach().cpu(), "grid": grid,
                  "co_counts": co_counts.detach().cpu(), "num_epochs": num_epochs, "ref_epochs": ref_epochs}
        if defer_reference:  # the caller runs attach_reference_arms once this rank has the box to itself
            out["_deferred_reference"] = inputs
        else:
            attach_reference_arms(out, inputs)
    return out
