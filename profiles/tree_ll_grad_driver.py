"""Timing of the exact likelihood gradient on one GPU (card name and power limit read in the same run).

1. 13gs_1_A (1024 leaves x 210 sites, LG): cherry_tree_log_likelihood alone against
   cherry_tree_ll_posterior (forward with stores, backward, reduction, plus its host index tables),
   CUDA events over repeated launches on prepared inputs.
2. tree_likelihood_mle on all demo families: per-epoch time split into expm, posterior, loss_grad and
   host (profiling.txt of the stage).
3. The numpy oracle's gradient of 13gs_1_A on the host, for scale.

    python profiles/tree_ll_grad_driver.py [--epochs 10] [--out profiles/tree_ll_grad_b200.txt]
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
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [f"card: {card()}"]
    lib = _lib.load()
    tmp = tempfile.mkdtemp()
    with tarfile.open(os.path.join(REPO, "tests", "golden", "demo_data.tar.xz")) as tf:
        members = [m for m in tf.getmembers() if m.name.split("/")[0] in ("msas", "trees", "site_rates")]
        tf.extractall(tmp, members=members)
    fams = sorted(f[:-4] for f in os.listdir(os.path.join(tmp, "trees")) if f.endswith(".txt"))
    Q = read_rate_matrix(_rate_matrix_path("lg")).to_numpy()
    pi = compute_stationary_distribution(Q)

    # 1. forward alone vs the posterior pass, 13gs_1_A
    fam_name = "13gs_1_A"
    tree = read_tree(os.path.join(tmp, "trees", fam_name + ".txt"))
    msa = read_msa(os.path.join(tmp, "msas", fam_name + ".txt"))
    rates = read_site_rates(os.path.join(tmp, "site_rates", fam_name + ".txt"))
    fam = _SiteFamily(tree, msa, rates, AA, "cuda")
    P = _expm_transposed(Q, fam.exponents, "cuda")
    d_pi = torch.from_numpy(pi).cuda()
    d_pidx = torch.from_numpy(fam.p_index).cuda()
    d_cat = torch.from_numpy(fam.unit_cat).cuda()
    fwd_bytes = int(lib.cherry_tree_ll_scratch_bytes(20, 1, fam.n_units, fam.max_depth))
    fwd_scratch = torch.empty(fwd_bytes, dtype=torch.uint8, device="cuda")
    ll = torch.empty(fam.n_units, dtype=torch.float64, device="cuda")

    def forward():
        _lib.check(lib.cherry_tree_log_likelihood(_lib.ptr(fam.nodes), fam.n_nodes, _lib.ptr(d_pidx), fam.n_cats,
                                                  _lib.ptr(P), _lib.ptr(fam.obs), _lib.ptr(d_cat), _lib.ptr(d_pi), 20,
                                                  1, fam.n_units, fam.max_depth, _lib.ptr(fwd_scratch), fwd_bytes,
                                                  _lib.ptr(ll), _lib.current_stream_ptr()), "forward")

    n_m = len(fam.exponents)
    post_bytes = int(lib.cherry_tree_ll_posterior_scratch_bytes(20, fam.n_nodes, fam.max_depth, fam.n_cats, n_m,
                                                                fam.n_units, _lib.ptr(fam.unit_cat)))
    post_scratch = torch.empty(post_bytes, dtype=torch.uint8, device="cuda")
    W = torch.empty((n_m, 20, 20), dtype=torch.float64, device="cuda")
    root = torch.empty(20, dtype=torch.float64, device="cuda")

    def posterior():
        _lib.check(lib.cherry_tree_ll_posterior(_lib.ptr(fam.nodes), fam.n_nodes, fam.max_depth,
                                                _lib.ptr(fam.p_index), fam.n_cats, _lib.ptr(P), n_m, _lib.ptr(fam.obs),
                                                _lib.ptr(fam.unit_cat), _lib.ptr(d_pi), 20, fam.n_units,
                                                _lib.ptr(post_scratch), post_bytes, _lib.ptr(ll), _lib.ptr(W),
                                                _lib.ptr(root), _lib.current_stream_ptr()), "posterior")

    t_f = events_ms(forward, args.reps)
    t_p = events_ms(posterior, args.reps)
    lines.append(f"{fam_name}: {len(tree.leaves())} leaves x {fam.n_units} sites, {fam.n_cats} rate categories, "
                 f"{n_m} distinct exponents")
    lines.append(f"  cherry_tree_log_likelihood (forward only): {t_f:.3f} ms per call (CUDA events, {args.reps} calls)")
    lines.append(f"  cherry_tree_ll_posterior (host tables + forward with stores + backward + reduce): {t_p:.3f} ms "
                 f"per call; scratch {post_bytes / 1e6:.1f} MB")

    # 2. tree_likelihood_mle, all demo families
    from cherryml_b200.estimation import tree_likelihood_mle

    out = os.path.join(tmp, "mle")
    t0 = time.time()
    tree_likelihood_mle(tree_dir=os.path.join(tmp, "trees"), msa_dir=os.path.join(tmp, "msas"),
                        site_rates_dir=os.path.join(tmp, "site_rates"), families=fams, amino_acids=AA,
                        initialization_path=_rate_matrix_path("lg"), num_epochs=args.epochs,
                        output_rate_matrix_dir=out)
    wall = time.time() - t0
    prof = open(os.path.join(out, "profiling.txt")).read().splitlines()
    vals = {ln.split(":")[0]: float(ln.split(":")[1].split()[0]) for ln in prof[1:]}
    n_eval = args.epochs + 1
    lines.append(f"tree_likelihood_mle, {len(fams)} demo families, {args.epochs} epochs ({n_eval} evaluations), "
                 f"wall {wall:.2f} s: {prof[0]}")
    lines.append("  per evaluation: " + ", ".join(
        f"{k} {1e3 * vals[k] / n_eval:.1f} ms" for k in ("expm", "posterior", "loss_grad", "host and rest")) +
        f"; set-up (read and encode, once) {vals['Set-up (read and encode)']:.2f} s")
    lines.append(f"  log-likelihood: LG start -> best {open(os.path.join(out, 'log_likelihood.txt')).read().strip()}")

    # 3. numpy oracle, 13gs_1_A
    from oracle.likelihood_grad_oracle import log_likelihood_gradient

    t0 = time.time()
    log_likelihood_gradient(tree, msa, rates, AA, pi, Q)
    lines.append(f"numpy oracle gradient of {fam_name} on the host: {time.time() - t0:.2f} s")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
