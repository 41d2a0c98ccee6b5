"""Timing of the exact branch-length gradient on one GPU (card name and power limit read in the same run).

1. 13gs_1_A (1024 leaves x 210 sites, LG): cherry_tree_ll_posterior against cherry_tree_ll_edge_derivatives
   on the same prepared inputs (host tables, forward, backward, reductions), CUDA events over repeated
   launches after a warm-up, the two alternated over three rounds.
2. branch_length_mle on all demo families: per-epoch time split into expm, posterior (the edge-derivative
   launches and their copies back) and host (parameters, exponent tables, Adam), from the stage's
   profiling file.

    python profiles/branch_length_driver.py [--epochs 100] [--out profiles/branch_length_b200.txt]
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
from cherryml_b200.evaluation._likelihood import _expm_transposed, _SiteFamily  # noqa: E402
from cherryml_b200.io import read_msa, read_rate_matrix, read_site_rates, read_tree  # noqa: E402
from cherryml_b200.markov_chain import _rate_matrix_path, compute_stationary_distribution  # noqa: E402
from cherryml_b200.utils import amino_acids as AA  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=100)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [f"card: {card()}"]
    tmp = tempfile.mkdtemp()
    with tarfile.open(os.path.join(REPO, "tests", "golden", "demo_data.tar.xz")) as tf:
        members = [m for m in tf.getmembers() if m.name.split("/")[0] in ("msas", "trees", "site_rates")]
        tf.extractall(tmp, members=members)
    fams = sorted(f[:-4] for f in os.listdir(os.path.join(tmp, "trees")) if f.endswith(".txt"))
    Q = read_rate_matrix(_rate_matrix_path("lg")).to_numpy()
    pi = compute_stationary_distribution(Q)

    # 1. posterior pass vs the same pass with edge derivatives, 13gs_1_A
    fam_name = "13gs_1_A"
    tree = read_tree(os.path.join(tmp, "trees", fam_name + ".txt"))
    fam = _SiteFamily(tree, read_msa(os.path.join(tmp, "msas", fam_name + ".txt")),
                      read_site_rates(os.path.join(tmp, "site_rates", fam_name + ".txt")), AA, "cuda")
    P = _expm_transposed(Q, fam.exponents, "cuda")
    d_pi = torch.from_numpy(pi).cuda()
    d_Q = torch.from_numpy(np.ascontiguousarray(Q)).cuda()
    lib = _lib.load()
    n_m = len(fam.exponents)
    sizes = (20, fam.n_nodes, fam.max_depth, fam.n_cats, n_m, fam.n_units, _lib.ptr(fam.unit_cat))
    post_bytes = int(lib.cherry_tree_ll_posterior_scratch_bytes(*sizes))
    der_bytes = int(lib.cherry_tree_ll_edge_derivatives_scratch_bytes(*sizes))
    scratch = torch.empty(der_bytes, dtype=torch.uint8, device="cuda")
    ll = torch.empty(fam.n_units, dtype=torch.float64, device="cuda")
    W = torch.empty((n_m, 20, 20), dtype=torch.float64, device="cuda")
    root = torch.empty(20, dtype=torch.float64, device="cuda")
    dtau = torch.empty((fam.n_nodes, fam.n_cats), dtype=torch.float64, device="cuda")
    head = (_lib.ptr(fam.nodes), fam.n_nodes, fam.max_depth, _lib.ptr(fam.p_index), fam.n_cats, _lib.ptr(P), n_m,
            _lib.ptr(fam.obs), _lib.ptr(fam.unit_cat), _lib.ptr(d_pi))

    def posterior():
        _lib.check(lib.cherry_tree_ll_posterior(*head, 20, fam.n_units, _lib.ptr(scratch), post_bytes, _lib.ptr(ll),
                                                _lib.ptr(W), _lib.ptr(root), _lib.current_stream_ptr()), "posterior")

    def derivatives():
        _lib.check(lib.cherry_tree_ll_edge_derivatives(*head, _lib.ptr(d_Q), 20, fam.n_units, _lib.ptr(scratch),
                                                       der_bytes, _lib.ptr(ll), _lib.ptr(W), _lib.ptr(root),
                                                       _lib.ptr(dtau), _lib.current_stream_ptr()), "derivatives")

    t_p, t_d = [], []
    for _ in range(3):
        t_p.append(events_ms(posterior, args.reps))
        t_d.append(events_ms(derivatives, args.reps))
    lines.append(f"{fam_name}: {len(tree.leaves())} leaves x {fam.n_units} sites, {fam.n_cats} rate categories, "
                 f"{n_m} distinct exponents; CUDA events, 1 warm-up + {args.reps} calls, 3 alternated rounds")
    lines.append(f"  cherry_tree_ll_posterior:        " + ", ".join(f"{x:.3f}" for x in t_p) +
                 f" ms per call; scratch {post_bytes / 1e6:.1f} MB")
    lines.append(f"  cherry_tree_ll_edge_derivatives: " + ", ".join(f"{x:.3f}" for x in t_d) +
                 f" ms per call; scratch {der_bytes / 1e6:.1f} MB")
    lines.append(f"  extra cost of the derivatives (median of rounds): "
                 f"{np.median(t_d) - np.median(t_p):.3f} ms ({100 * (np.median(t_d) / np.median(t_p) - 1):.1f}%)")

    # 2. branch_length_mle, all demo families
    from cherryml_b200.phylogeny_estimation import branch_length_mle

    out = {k: os.path.join(tmp, "blmle", k) for k in ("output_tree_dir", "output_site_rates_dir",
                                                      "output_likelihood_dir")}
    t0 = time.time()
    branch_length_mle(tree_dir=os.path.join(tmp, "trees"), site_rates_dir=os.path.join(tmp, "site_rates"),
                      msa_dir=os.path.join(tmp, "msas"), families=fams, rate_matrix_path=_rate_matrix_path("lg"),
                      amino_acids=AA, num_epochs=args.epochs, **out)
    wall = time.time() - t0
    prof = open(os.path.join(out["output_tree_dir"], fams[0] + ".profiling")).read().splitlines()[1]
    # "(stage over N families, E epochs: expm X s, posterior Y s, host Z s)"
    parts = dict(p.strip().split()[:2] for p in prof.split(":", 1)[1].rstrip(")").split(","))
    n_eval = args.epochs + 1
    n_sites = sum(len(read_site_rates(os.path.join(tmp, "site_rates", f + ".txt"))) for f in fams)
    lines.append(f"branch_length_mle, {len(fams)} demo families ({n_sites} sites), {args.epochs} epochs "
                 f"({n_eval} evaluations), wall {wall:.2f} s (reading and encoding included)")
    lines.append("  per evaluation: " + ", ".join(f"{k} {1e3 * float(v) / n_eval:.1f} ms" for k, v in parts.items()))
    from cherryml_b200.evaluation import dp_likelihood_computation

    start = sum(dp_likelihood_computation(
        tree=read_tree(os.path.join(tmp, "trees", f + ".txt")), msa=read_msa(os.path.join(tmp, "msas", f + ".txt")),
        contact_map=None, site_rates=read_site_rates(os.path.join(tmp, "site_rates", f + ".txt")), amino_acids=AA,
        pi_1=pi, Q_1=Q)[0] for f in fams)
    best = sum(float(open(os.path.join(out["output_likelihood_dir"], f + ".txt")).readline()) for f in fams)
    lines.append(f"  summed log-likelihood under LG: given (FastTree) lengths {start!r} -> kept iterates {best!r}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
