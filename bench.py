#!/usr/bin/env python
"""bench.py -- the hot path on synthetic Pfam-shaped data (BASELINE.json config 3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one counting pass over one batch: bucket table + LG transition histogram of
F families x 1024 sequences x 300 sites into K=100 time buckets (+ the all-reduce of the raw
integer histogram when N > 1, + symmetrisation).  Per-GPU work is fixed (weak scaling: every
rank counts its own F families).  ``value`` = transitions examined per second with the batch
resident in HBM; ``e2e`` = the same through the host-buffer C-ABI entry point
(pinned host arrays -> H2D -> kernels -> D2H).  One JSON line is printed by rank 0.

``--dump-outputs DIR`` writes what the last timed step returned, the symmetrised fp64 count
tensor [K, 20, 20] (320 KB), as ``DIR/counts.npy``.  The batch is generated from a fixed seed, so
two builds run with the same arguments can be compared output for output.

``--impl reference`` times the reference's own CPU implementation (the unmodified C++
program compiled into oracle/_ref, one process per host core on the reference's own family
striping; the C port of the oracle if the binary is absent) on a bounded sample of the same
workload.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from benchlib.hostcores import describe as host_cores, usable_cores

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "cherry transitions counted/s"
UNIT = "transitions/s"
N_SEQS, N_SITES, N_CATS, K_BUCKETS, N_STATES = 1024, 300, 4, 100, 20


_T0 = time.time()


def _log(msg):
    """Progress on stderr (stdout carries the one JSON line)."""
    sys.stderr.write(f"[bench {time.time() - _T0:7.1f}s] {msg}\n")
    sys.stderr.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--families", type=int, default=16384, help="families per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-families", type=int, default=0, help="families in the CPU sample (0 = 16 per core, >= 128)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--text-families", type=int, default=2048,
                    help="families of the larger from-text run (e2e_text_large; 0 = skip)")
    ap.add_argument("--no-fit", action="store_true")
    ap.add_argument("--no-fast-cherries", action="store_true")
    ap.add_argument("--fc-families", type=int, default=2048, help="FastCherries families per GPU")
    ap.add_argument("--no-likelihood", action="store_true")
    ap.add_argument("--no-siterm", action="store_true")
    ap.add_argument("--no-public-api", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step to DIR/counts.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def workload_name(families):
    return (f"synthetic Pfam-scale LG: {families} families x {N_SEQS} seqs x {N_SITES} sites per GPU, "
            f"{K_BUCKETS} time buckets, {N_CATS} site-rate categories")


# ------------------------------------------------------------------ clocks sampling
class ClockSampler:
    """Samples nvidia-smi during the timed region (B200_PROFILING.md clocks line)."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu_index), "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons),
            "samples": len(sm),
        }


# ------------------------------------------------------------ CPU reference / baseline
_RENDERED = {}


def rendered_sample(n_families, seed=0):
    """Text rendering of `n_families` of the workload, written once per process (untimed: both
    the reference programs and our text path start from these files)."""
    import atexit

    from cherryml_b200.synthetic import synthetic_lg, write_text_rendering

    key = (n_families, seed)
    if key not in _RENDERED:
        syn = synthetic_lg(n_families, N_SEQS, N_SITES, N_CATS, seed=seed, device="cpu")
        tmp = tempfile.mkdtemp(prefix="cherry_txt_")
        atexit.register(shutil.rmtree, tmp, True)
        names = write_text_rendering(syn, tmp)
        _RENDERED[key] = (syn, tmp, names)
    return _RENDERED[key]


def default_cpu_families():
    """Sample size of the CPU legs: ~1-2 s of reference time per step on the box's cores."""
    return max(128, 16 * usable_cores())


def cpu_reference_run(n_families, seed=0, workdir=None):
    """Time the reference's CPU counting on a bounded sample of the workload.

    Returns dict(value, unit, cores, kind, sample, seconds).  Text rendering of the sample is
    written before the timer starts (the reference consumes text); the timed region is the
    reference programs themselves, text parsing included, as the reference does it."""
    import numpy as np

    from cherryml_b200.synthetic import (as_count_batch, quantization_grid, synthetic_lg,
                                         write_text_rendering)
    from cherryml_b200.utils import amino_acids

    cores = usable_cores()
    grid = quantization_grid()
    syn, tmp, names = rendered_sample(n_families, seed)
    examined = syn["n_sites_examined"]
    ref_bin = os.path.join(REPO, "oracle", "_ref", "count_transitions")
    if os.path.exists(ref_bin) and os.access(ref_bin, os.X_OK):
        try:
            procs_n = min(cores, n_families)
            cmds = []
            for r in range(procs_n):
                fam_r = names[r::procs_n]  # the reference's MPI striping (.cpp:624-629)
                fpath = os.path.join(tmp, f"families_{r}.txt")
                with open(fpath, "w") as f:
                    f.write(" ".join(fam_r))
                out = os.path.join(tmp, f"out_{r}")
                shutil.rmtree(out, ignore_errors=True)
                os.makedirs(out, exist_ok=True)
                cmds.append([ref_bin, os.path.join(tmp, "tree_dir"), os.path.join(tmp, "msa_dir"),
                             os.path.join(tmp, "site_rates_dir"), str(len(fam_r)), str(N_STATES),
                             str(len(grid)), fpath, *amino_acids, *[str(q) for q in grid], "cherry++", out])
            t0 = time.perf_counter()
            procs = [subprocess.Popen(c, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for c in cmds]
            rcs = [p.wait() for p in procs]
            seconds = time.perf_counter() - t0
            if any(rcs):
                raise RuntimeError(f"reference binary failed: {rcs}")
            # sanity: the reference's summed output equals the oracle on the same sample
            from oracle.counting_oracle import read_count_matrices_text
            from oracle.native import count_batch_oracle

            total = sum(read_count_matrices_text(os.path.join(tmp, f"out_{r}", "result.txt"))[2]
                        for r in range(procs_n))
            # the C++ program reads branch lengths as float32: compare totals only loosely
            if "oracle_total" not in syn:
                syn["oracle_total"] = float(count_batch_oracle(as_count_batch(syn), grid, N_STATES, False).sum())
            if abs(total.sum() - syn["oracle_total"]) > 1e-3 * syn["oracle_total"]:
                raise RuntimeError("reference output disagrees with the oracle on the sample")
        finally:
            pass
        kind, used = "reference", procs_n
        sample = (f"{n_families} of the workload's families ({examined} transitions), unmodified reference "
                  f"C++ program, {procs_n} processes on the reference's family striping, text parsing included")
    else:
        from oracle.native import count_batch_oracle

        batch = as_count_batch(syn)
        t0 = time.perf_counter()
        count_batch_oracle(batch, grid, N_STATES, False)
        seconds = time.perf_counter() - t0
        kind, used = "port", 1
        sample = (f"{n_families} of the workload's families ({examined} transitions), scalar C port of the "
                  "reference loop on pre-encoded arrays (no text parsing), 1 thread")
    return {"value": examined / seconds, "unit": UNIT, "cores": used, "kind": kind, "sample": sample,
            "seconds": seconds}


def text_e2e_run(n_families, seed=0, reps=3):
    """Our path from the SAME text files the reference arm consumes: native multithreaded ingest
    (parse + encode, all host cores) -> pinned host batch -> cherry_count_lg_host (H2D, kernels,
    D2H).  The text rendering is written before the timer starts, as for the reference."""
    from cherryml_b200.counting._device import count_lg_host
    from cherryml_b200.counting._ingest import build_lg_batch_native
    from cherryml_b200.synthetic import quantization_grid, synthetic_lg, write_text_rendering
    from cherryml_b200.utils import amino_acids

    cores = usable_cores()
    grid = quantization_grid()
    syn, tmp, names = rendered_sample(n_families, seed)
    best, ingest_s = float("inf"), 0.0
    for _ in range(reps + 1):  # first pass warms the page cache and the CUDA context
        t0 = time.perf_counter()
        batch = build_lg_batch_native(os.path.join(tmp, "tree_dir"), os.path.join(tmp, "msa_dir"),
                                      os.path.join(tmp, "site_rates_dir"), names, amino_acids, "cherry++",
                                      True, n_threads=cores, pinned=True)
        t1 = time.perf_counter()
        count_lg_host(batch, grid, N_STATES, False)
        t2 = time.perf_counter()
        if t2 - t0 < best:
            best, ingest_s = t2 - t0, t1 - t0
        del batch
    examined = syn["n_sites_examined"]
    return {"value": examined / best, "unit": UNIT, "seconds": best, "seconds_ingest": ingest_s,
            "host_threads": cores,
            "sample": f"{n_families} of the workload's families as text files ({examined} transitions): "
                      "cherry_ingest_lg (parse + encode) -> cherry_count_lg_host; same input as cpu_baseline; "
                      "best of the passes after the first (the page-locked staging buffer is pooled: the first "
                      "batch of a process also pays for pinning it, ~0.2 ms per MB)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    n_fam = args.cpu_families or default_cpu_families()
    for _ in range(args.warmup):
        cpu_reference_run(n_fam)
    times, values, last = [], [], None
    for _ in range(args.steps):
        last = cpu_reference_run(n_fam)
        times.append(last["seconds"])
        values.append(last["value"])
    value = sum(values) / len(values)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_name(args.families), "sample_families_per_step": n_fam},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": last["kind"],
                         "sample": last["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------- our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from cherryml_b200 import _lib
    from cherryml_b200.counting._device import (build_bucket_table_tiles, count_lg_host, count_raw, sorted_grid,
                                                 symmetrize)
    from cherryml_b200.synthetic import as_count_batch, as_device_batch, quantization_grid, synthetic_lg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    lib = _lib.load()

    F = args.families
    grid = quantization_grid()
    K, S = len(grid), N_STATES
    syn = synthetic_lg(F, N_SEQS, N_SITES, N_CATS, seed=1000 + rank, device=device)
    dev = as_device_batch(syn, device)
    grid_dev = torch.from_numpy(sorted_grid(grid)).to(device)
    examined = syn["n_sites_examined"]
    stride = syn["shape"]["stride"]
    n_pairs = dev.n_pairs
    # algorithmic bytes of one counting launch (DESIGN.md): residues read once, site->category
    # groups once per family, pair descriptors + bucket-table row per pair, one histogram flush
    alg_bytes = (dev.msa.numel() + F * (stride // 4) * 2 + n_pairs * (8 + dev.r_pad) + K * S * S * 8)

    raw = torch.zeros((K, S, S), dtype=torch.int64, device=device)
    stream = torch.cuda.current_stream()

    def step(ev=None):
        raw.zero_()
        tab = build_bucket_table_tiles(dev, grid_dev, K)  # per tile, against precomputed decision boundaries
        if ev is not None:
            ev[0].record(stream)
        count_raw(dev, grid_dev, K, S, tab=tab, out=raw)
        if ev is not None:
            ev[1].record(stream)
        if world > 1:
            dist.all_reduce(raw, op=dist.ReduceOp.SUM)
        return symmetrize(raw, "lg", K, S, directed=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        counts = step()
    barrier()
    _log("warm-up steps done")
    # parity gate inside the bench: a 32-family slice of EVERY rank's batch against the oracle
    parity = None
    if True:
        import copy

        from oracle.native import count_batch_oracle

        d3 = copy.copy(dev)
        d3.n_tiles = 32 * (dev.n_tiles // F)
        got = symmetrize(count_raw(d3, grid_dev, K, S), "lg", K, S, False).cpu().numpy()
        host_slice = as_count_batch(dict(syn, msa=syn["msa"][: 32 * N_SEQS * stride]))
        exp = count_batch_oracle(host_slice, grid, S, False, pair_slice=slice(0, 32 * (N_SEQS // 2)))
        parity = bool(np.array_equal(got, exp))
        if world > 1:
            flag = torch.tensor([1 if parity else 0], dtype=torch.int32, device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            parity = bool(int(flag[0]))
        if not parity:
            raise SystemExit("bench.py: GPU counts differ from the oracle on the sample slice")

    sampler = ClockSampler(local_rank)
    _lib.reset_launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if rank == 0:
        sampler.start()
    t_start.record(stream)
    for i in range(args.steps):
        counts = step(evs[i])
    t_end.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count()
    elapsed_ms = t_start.elapsed_time(t_end)
    kernel_ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    if world > 1:
        t = torch.tensor([elapsed_ms, kernel_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, kernel_ms = float(t[0]), float(t[1])
    ms_per_step = elapsed_ms / args.steps
    value = examined * world / (ms_per_step * 1e-3)
    _log(f"timed steps done: {ms_per_step:.3f} ms per step")
    counted = float(counts.sum().item())
    if args.dump_outputs is not None and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "counts.npy"), counts.cpu().numpy())
        _log(f"outputs of the last timed step written to {args.dump_outputs}")

    # ---- strong scaling (BASELINE config 3 as stated: 16k families in total on 1/2/4/8 GPUs): the SAME
    # step, all-reduce inside, on F/N families per rank (the first 1/N of this rank's resident tiles)
    strong = None
    if world > 1:
        import copy

        ds = copy.copy(dev)
        ds.n_tiles = dev.n_tiles // world
        fam_s = F // world
        examined_s = examined // world

        def step_strong():
            raw.zero_()
            count_raw(ds, grid_dev, K, S, tab=build_bucket_table_tiles(ds, grid_dev, K), out=raw)
            dist.all_reduce(raw, op=dist.ReduceOp.SUM)
            return symmetrize(raw, "lg", K, S, directed=False)

        for _ in range(3):
            step_strong()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(args.steps):
            step_strong()
        s1.record(stream)
        barrier()
        t = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_s = float(t[0]) / args.steps
        strong = {"families_total": fam_s * world, "families_per_gpu": fam_s, "ms_per_step": ms_s,
                  "value": examined_s * world / (ms_s * 1e-3), "unit": UNIT,
                  "note": "same step (bucket table, count, NCCL all-reduce of the 320 KB raw histogram, symmetrise) "
                          "on 1/N of the families per rank; efficiency = value / (N * value at N=1 of the weak line)"}
        del ds

    # ---- e2e: host buffers through the C-ABI host entry point
    e2e = None
    host = as_count_batch(syn)
    pinned = {}
    for name in ("msa", "pair_a", "pair_b", "pair_t", "pair_fam"):
        t = torch.from_numpy(getattr(host, name)).pin_memory()
        pinned[name] = t
        setattr(host, name, t.numpy())
    for _ in range(2):
        out, h2d, d2h = count_lg_host(host, grid, S, False)
    if rank == 0 and world == 1:
        assert np.array_equal(out, counts.cpu().numpy()), "host path and device path disagree"
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        out, h2d, d2h = count_lg_host(host, grid, S, False)
    e2e_s = (time.perf_counter() - t0) / args.e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    # the ceiling of any host-buffer path: the bare pinned H2D copy of the same residue buffer (all ranks at once)
    dst = torch.empty(pinned["msa"].numel(), dtype=torch.uint8, device=device)
    dst.copy_(pinned["msa"], non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    dst.copy_(pinned["msa"], non_blocking=True)
    torch.cuda.synchronize()
    copy_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([copy_s], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        copy_s = float(t[0])
    del dst
    e2e = {"value": examined * world / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s * 1e3,
           "h2d_copy_only_ms": copy_s * 1e3, "h2d_copy_only_gbs_per_gpu": pinned["msa"].numel() / copy_s / 1e9,
           "frac_of_h2d_copy_ceiling": copy_s / e2e_s,
           "note": "cherry_count_lg_host: pinned host arrays -> segmented H2D overlapped with counting -> D2H; "
                   "h2d_copy_only = one bare cudaMemcpyAsync of the same pinned residue buffer on every rank at once"}
    del pinned
    _log("e2e (host buffers) done")

    # ---- the fit (every rank takes part when N > 1: bucket-sharded co-evolution fit)
    fit = None
    if not args.no_fit:
        from benchlib.fit import bench_fit

        del dev, syn, host
        torch.cuda.empty_cache()
        fit = bench_fit(device, lg_times=grid, lg_counts=counts,
                        process_group=dist.group.WORLD if world > 1 else None,
                        cpu_baseline=(rank == 0 and not args.no_cpu_baseline), defer_reference=True)
    _log("fit section done")
    # ---- FastCherries (tree estimation, the step before counting): every rank its own families
    fcb = None
    if not args.no_fast_cherries:
        from benchlib.fast_cherries import bench_fast_cherries

        torch.cuda.empty_cache()
        fcb = bench_fast_cherries(device, families=args.fc_families, seed=rank,
                                  cpu_baseline=(world == 1 and rank == 0 and not args.no_cpu_baseline))
        if world > 1:
            t = torch.tensor([fcb["pair_kernel_ms"], fcb["ble_kernel_ms"], fcb["e2e_seconds"]], dtype=torch.float64,
                             device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            fcb["pair_kernel_ms"], fcb["ble_kernel_ms"], fcb["e2e_seconds"] = (float(v) for v in t)
            fam_all = args.fc_families * world
            fcb["families_per_s_kernels"] = fam_all / ((fcb["pair_kernel_ms"] + fcb["ble_kernel_ms"]) * 1e-3)
            fcb["families_per_s_e2e"] = fam_all / fcb["e2e_seconds"]
            fcb["residues_per_s_e2e"] = fam_all * 1024 * 300 / fcb["e2e_seconds"]
            fcb["n_gpus"] = world
    _log("fast_cherries section done")
    llb = None
    if rank == 0 and not args.no_likelihood:
        from benchlib.likelihood import bench_likelihood

        try:
            llb = bench_likelihood(device, cpu_baseline=(world == 1 and not args.no_cpu_baseline))
        except Exception as e:  # never lose the bench line over an extra section
            llb = {"error": str(e)[:300]}
    _log("likelihood section done")
    srb = None
    if rank == 0 and not args.no_siterm:
        from benchlib.siterm import bench_siterm

        try:
            srb = bench_siterm(device, cpu_baseline=(world == 1 and not args.no_cpu_baseline))
        except Exception as e:
            srb = {"error": str(e)[:300]}
    srs = None
    if not args.no_siterm:  # every rank: the per-site fit with a fixed total of sites sharded over the ranks
        from benchlib.siterm import bench_siterm_sharded

        try:
            srs = bench_siterm_sharded(device, dist.group.WORLD if world > 1 else None)
        except Exception as e:
            srs = {"error": str(e)[:300]}
    _log("siterm section done")
    apib = None
    if rank == 0 and world == 1 and not args.no_public_api:
        from benchlib.public_api_demo import bench_public_api_demo

        try:
            apib = bench_public_api_demo()
        except Exception as e:
            apib = {"error": str(e)[:300]}
    _log("public api section done")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if fit is not None and "_deferred_reference" in fit:
        # the reference's own fit arms, timed now that the other ranks are gone and this rank has the
        # box's host cores and its GPU to itself (benchlib/fit.py attach_reference_arms says why)
        from benchlib.fit import attach_reference_arms

        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        if world > 1:
            time.sleep(2.0)  # the other ranks are tearing down
        attach_reference_arms(fit, fit.pop("_deferred_reference"))
        _log("reference fit arms done")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "count_lg_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None,
                "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kernel_ms}
    traffic_file = os.path.join(REPO, "profiles", "count_lg_traffic.json")
    if os.path.exists(traffic_file):
        try:
            roofline["traffic"] = json.load(open(traffic_file)).get("dram_bytes_per_launch")
        except Exception:
            pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_name(F), "l2": "inputs (>5 GB per GPU) larger than L2, no flush needed",
                   "transitions_examined_per_step": examined * world,
                   "transitions_counted_per_step_rank0": counted, "parity_slice_vs_oracle_all_ranks": parity},
        "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "host_cores": host_cores(),
    }
    line["config"]["transitions_counted_per_s"] = counted * world / (ms_per_step * 1e-3)
    if strong is not None:
        line["config"]["strong_scaling"] = strong
    if fit is not None:
        line["fit"] = fit
        # the first clause of BASELINE's metric, inside `config` (the driver keeps config verbatim)
        cfg = line["config"]
        lgf, cof, coc = fit.get("lg_20x20", {}), fit.get("coevo_400x400", {}), fit.get("co_counting", {})
        cfg["fit_lg_seconds"] = lgf.get("seconds_end_to_end")
        cfg["fit_lg_ms_per_epoch"] = lgf.get("ms_per_epoch")
        cfg["fit_coevo_seconds"] = cof.get("seconds_end_to_end")
        cfg["fit_coevo_ms_per_epoch"] = cof.get("ms_per_epoch")
        cfg["fit_coevo_n_gpus"] = cof.get("n_gpus")
        cfg["fit_roofline_frac"] = cof.get("roofline", {}).get("frac")
        cfg["fit_coevo_tflops"] = cof.get("tflops_executed")
        cfg["fit_coevo_symmetric_form"] = cof.get("symmetric_form")
        cfg["co_count_frac"] = coc.get("roofline", {}).get("frac")
        cfg["co_count_items_per_s"] = coc.get("items_per_s")
        cfg["coevo_end_to_end_seconds"] = fit.get("coevo_end_to_end_seconds")
        for key, name in (("lg_20x20", "lg"), ("coevo_400x400", "coevo")):
            f = fit.get(key, {})
            for arm, short in (("cpu_baseline", "cpu"), ("reference_cuda", "cuda")):
                if arm in f and "seconds_end_to_end" in f[arm]:
                    cfg[f"fit_{name}_reference_{short}_seconds"] = f[arm]["seconds_end_to_end"]
                    cfg[f"fit_{name}_speedup_vs_reference_{short}"] = f[arm]["seconds_end_to_end"] / f["seconds_end_to_end"]
    if fcb is not None:
        line["fast_cherries"] = fcb
    if llb is not None:
        line["tree_likelihood"] = llb
    if srb is not None:
        line["siterm"] = srb
    if srs is not None:
        line["siterm_sharded"] = srs
        line["config"]["siterm_sharded_sites_per_s"] = srs.get("sites_per_s")
    if apib is not None:
        line["public_api_demo"] = apib
    if not args.no_cpu_baseline:  # rank 0 (the other ranks have returned above)
        cores = usable_cores()
        n_cpu_fam = args.cpu_families or default_cpu_families()
        cb = cpu_reference_run(n_cpu_fam)
        cb.pop("seconds", None)
        line["cpu_baseline"] = cb
        try:
            line["e2e_text"] = text_e2e_run(n_cpu_fam)
        except Exception as e:  # never lose the bench line over the extra measurement
            line["e2e_text"] = {"error": str(e)[:200]}
        _log("e2e_text done")
        if args.text_families > n_cpu_fam and world == 1:
            # the same from-text path on a batch large enough that the per-call costs (thread start-up, the
            # 320 KB read-back, kernel launches) no longer matter: what the ingest sustains
            try:
                line["e2e_text_large"] = text_e2e_run(args.text_families, seed=1, reps=2)
            except Exception as e:
                line["e2e_text_large"] = {"error": str(e)[:200]}
            _log("e2e_text_large done")
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    # stdout carries exactly ONE line (the JSON): libraries that print banners to file descriptor 1
    # (NCCL's version line at N > 1) are pointed at stderr, the JSON goes to the original stdout
    import builtins

    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    plain_print = builtins.print

    def json_print(*a, **k):
        if len(a) == 1 and isinstance(a[0], str) and a[0].startswith("{") and "file" not in k:
            real_stdout.write(a[0] + "\n")
            real_stdout.flush()
        else:
            plain_print(*a, **k)

    builtins.print = json_print
    try:
        if args.impl == "reference":
            run_reference_arm(args)
        else:
            run_ours(args)
    finally:
        builtins.print = plain_print


if __name__ == "__main__":
    main()
