"""Timing of the exact pair log-likelihood gradient on one GPU (card name and power limit read in the same run).

On the 32 demo families, contact maps reduced by maximal_matching_pairs(., 7) as the public API does, and
Q_2 = LG x LG (get_lg_x_lg_path), per family, CUDA events after a warm-up family:
  expm       one 400 x 400 matrix per distinct branch length (cherry_expm_batched, chunks of 128);
  posterior  cherry_tree_ll_pair_posterior (host tables, inside, outside, edge posteriors);
  gradient   cherry_fit_loss_grad with C = W (chunks of 811 exponents);
  forward    the existing forward-only cherry_tree_log_likelihood (c = 2) on the same matrices, transposed as
             it reads them (the transpose is not timed);
and the posterior's tensor-core FLOPs counted from shapes: per non-root internal node an inside and an
outside product 2 Su^2 n_pairs, per edge the posterior product 2 Su^2 n_pairs ("useful"), and the same with
the tile padding the kernels issue (pairs to 16, states to 128 in the node products and to 64 in the edge
products).  Then one whole PairTreeLikelihoodData.evaluate over all families (host clock, device-synchronised).

    python profiles/pair_ll_grad_driver.py [--reps 2] [--out profiles/pair_ll_grad_b200.txt]
"""
import argparse
import os
import subprocess
import sys
import tarfile
import tempfile
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from cherryml_b200 import _lib  # noqa: E402
from cherryml_b200._public_api import maximal_matching_pairs  # noqa: E402
from cherryml_b200.estimation import PairTreeLikelihoodData  # noqa: E402
from cherryml_b200.evaluation._likelihood import _expm_chunked, _PairFamily, _q_gradient  # noqa: E402
from cherryml_b200.io import read_contact_map, read_msa, read_rate_matrix, read_tree, write_contact_map  # noqa: E402
from cherryml_b200.markov_chain import compute_stationary_distribution, get_lg_x_lg_path  # noqa: E402
from cherryml_b200.utils import amino_acids as AA  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def posterior_flops(fam):
    """(useful, issued) FLOPs of the three products of one posterior pass."""
    nodes = fam.nodes_host
    Su, N = fam.S * fam.S, fam.n_pairs
    n_int = int(np.sum((nodes["flags"][:-1] & 1) == 0))  # internal nodes other than the root (the last node)
    n_edges = fam.n_nodes - 1
    useful = 2.0 * Su * Su * N * (2 * n_int + n_edges)
    Np = -(-N // 16) * 16
    node = 2.0 * Np * (-(-Su // 128) * 128) * (-(-Su // 16) * 16)
    Sp = -(-Su // 64) * 64
    return useful, node * 2 * n_int + 2.0 * Sp * Sp * Np * n_edges


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [f"card: {card()}"]
    lib = _lib.load()
    dev = torch.device("cuda")
    tmp = tempfile.mkdtemp()
    with tarfile.open(os.path.join(REPO, "tests", "golden", "demo_data.tar.xz")) as tf:
        fams = sorted(n.split("/")[1][:-4] for n in tf.getnames() if n.startswith("trees/") and n.endswith(".txt"))
        tf.extractall(tmp, members=[tf.getmember(f"{d}/{f}.txt") for d in ("msas", "trees", "contact_maps")
                                    for f in fams])
    os.makedirs(os.path.join(tmp, "matched"))
    for f in fams:
        cm = read_contact_map(os.path.join(tmp, "contact_maps", f + ".txt"))
        matched = np.zeros_like(cm)
        for i, j in maximal_matching_pairs(cm, 7):
            matched[i, j] = matched[j, i] = 1
        write_contact_map(matched, os.path.join(tmp, "matched", f + ".txt"))
    Q = read_rate_matrix(get_lg_x_lg_path()).to_numpy()
    pi = torch.from_numpy(compute_stationary_distribution(Q)).to(dev)
    Qd = torch.from_numpy(np.array(Q)).to(dev)
    lines.append(f"Q_2 = LG x LG, {len(fams)} demo families, maximal-matching contact maps (minimum distance 7); "
                 f"CUDA events, mean of {args.reps} calls per family after a warm-up family")
    lines.append("family: leaves, pairs, distinct lengths | expm ms | posterior ms (useful / issued TFLOP/s) | "
                 "gradient ms | forward-only ms | posterior speed-up over forward")
    tot = dict(expm=0.0, post=0.0, grad=0.0, fwd=0.0)
    order = [fams[0]] + fams  # the first family twice: its first pass is the warm-up and is not reported
    for k, f in enumerate(order):
        fam = _PairFamily(read_tree(os.path.join(tmp, "trees", f + ".txt")), read_msa(os.path.join(tmp, "msas", f + ".txt")),
                          read_contact_map(os.path.join(tmp, "matched", f + ".txt")), AA, dev)
        n_m = len(fam.exponents)
        t = torch.from_numpy(fam.exponents).to(dev)
        box = {}

        def run_expm():
            box["P"] = _expm_chunked(Q, fam.exponents, dev, transpose=False)

        def run_post():
            box["post"] = fam.posterior(box["P"], pi)

        def run_grad():
            box["g"] = _q_gradient(Qd, t, box["post"][1])

        t_expm = events_ms(run_expm, args.reps)
        t_post = events_ms(run_post, args.reps)
        t_grad = events_ms(run_grad, args.reps)
        # forward only, on the transposed matrices it reads
        Pt = torch.empty_like(box["P"])
        _lib.check(lib.cherry_tree_ll_transpose(_lib.ptr(box["P"]), n_m, 400, _lib.ptr(Pt), _lib.current_stream_ptr()),
                   "cherry_tree_ll_transpose")
        d_nodes = torch.from_numpy(fam.nodes_host.view(np.uint8).reshape(-1)).to(dev)
        d_pidx = torch.from_numpy(fam.p_index).to(dev)
        d_cat = torch.zeros(max(1, fam.n_pairs), dtype=torch.int32, device=dev)
        nbytes = int(lib.cherry_tree_ll_scratch_bytes(20, 2, fam.n_pairs, fam.max_depth))
        scratch = torch.empty(max(8, nbytes), dtype=torch.uint8, device=dev)
        ll_fwd = torch.empty(max(1, fam.n_pairs), dtype=torch.float64, device=dev)

        def run_fwd():
            _lib.check(lib.cherry_tree_log_likelihood(_lib.ptr(d_nodes), fam.n_nodes, _lib.ptr(d_pidx), 1, _lib.ptr(Pt),
                                                      _lib.ptr(fam.obs), _lib.ptr(d_cat), _lib.ptr(pi), 20, 2,
                                                      fam.n_pairs, fam.max_depth, _lib.ptr(scratch), nbytes,
                                                      _lib.ptr(ll_fwd), _lib.current_stream_ptr()),
                       "cherry_tree_log_likelihood")

        t_fwd = events_ms(run_fwd, args.reps)
        ll_post = box["post"][0].double()
        dev_rel = float(((ll_post - ll_fwd[: fam.n_pairs]).abs() / ll_fwd[: fam.n_pairs].abs().clamp(min=1.0)).max())
        del Pt, box, scratch
        torch.cuda.empty_cache()
        if k == 0:
            continue
        useful, issued = posterior_flops(fam)
        tot["expm"] += t_expm
        tot["post"] += t_post
        tot["grad"] += t_grad
        tot["fwd"] += t_fwd
        lines.append(f"{f}: {len(fam.nodes_host[fam.nodes_host['flags'] & 1 == 1])} leaves, {fam.n_pairs} pairs, "
                     f"{n_m} lengths | {t_expm:.2f} | {t_post:.2f} ({useful / t_post / 1e9:.1f} / "
                     f"{issued / t_post / 1e9:.1f}) | {t_grad:.2f} | {t_fwd:.2f} | {t_fwd / t_post:.2f}x "
                     f"(max pair ll difference {dev_rel:.1e})")
    lines.append(f"sum over families: expm {tot['expm']:.1f} ms, posterior {tot['post']:.1f} ms, gradient "
                 f"{tot['grad']:.1f} ms, forward-only {tot['fwd']:.1f} ms")
    data = PairTreeLikelihoodData(os.path.join(tmp, "trees"), os.path.join(tmp, "msas"),
                                  os.path.join(tmp, "matched"), fams, AA, dev)
    data.evaluate(Qd, pi)  # warm-up
    for key in data.timing:
        data.timing[key] = 0.0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    total, gQ, gpi = data.evaluate(Qd, pi)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    tm = data.timing
    lines.append(f"one PairTreeLikelihoodData.evaluate over all {len(fams)} families ({data.n_pairs} pairs, "
                 f"{data.n_exponents} distinct lengths): {wall * 1e3:.0f} ms wall; expm {tm['expm'] * 1e3:.0f} ms, "
                 f"posterior {tm['posterior'] * 1e3:.0f} ms, gradient {tm['loss_grad'] * 1e3:.0f} ms; "
                 f"log-likelihood {float(total)!r}")
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
