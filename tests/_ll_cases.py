"""Shared fixtures of the likelihood tests: the FastTree-verified known answers of the reference's
tests/evaluation_tests/likelihood_test.py (restated here with its 1a92_1_A data fixture under
tests/golden/likelihood/1a92), the goldens made by tests/golden/make_golden_likelihood.py, and the seeded
models, trees, MSAs, simulations and demo families of the likelihood-gradient tests."""
import json
import os
import tarfile

import numpy as np

from cherryml_b200.io import Tree, read_msa, read_rate_matrix, read_site_rates, read_tree
from cherryml_b200.markov_chain import chain_product, compute_stationary_distribution
from tests.conftest import GOLDEN

AA = list("ARNDCQEGHILKMFPSTWYV")
DNA = list("ACGT")
LL_DIR = os.path.join(GOLDEN, "likelihood")


def rate_matrix(name):
    from cherryml_b200.markov_chain import _rate_matrix_path

    return read_rate_matrix(_rate_matrix_path(name)).to_numpy()


def _tree(nodes, edges):
    t = Tree()
    t.add_nodes(nodes)
    t.add_edges(edges)
    return t


def fasttree_kats():
    """(name, tree, msa, contact_map, site_rates, pi_1, Q_1, pi_2, Q_2, ll, lls, decimals).
    likelihood_test.py:242-284 (3 seqs), :291-331 (4 seqs), :338-378 (gaps), :385-429 (equ x equ),
    :918-953 (1a92_1_A, 1/2/4/20 rate categories)."""
    wag, equ = rate_matrix("wag"), rate_matrix("equ")
    pi_wag = compute_stationary_distribution(wag)
    equ2 = chain_product(equ, equ)
    pi_equ2 = compute_stationary_distribution(equ2)
    out = []
    t3 = _tree(["r", "l1", "l2", "l3"], [("r", "l1", 0.0), ("r", "l2", 1.120547166), ("r", "l3", 3.402392896)])
    out.append(("wag_3_seqs", t3, {"l1": "S", "l2": "T", "l3": "G"}, np.eye(1), [1.0], pi_wag, wag, None, None,
                -7.343870, [-7.343870], 4))
    t4 = _tree(["r", "i1", "l1", "l2", "l3", "l4"],
               [("r", "l1", 0.0), ("r", "l2", 1.121562482), ("r", "i1", 1.719057732), ("i1", "l3", 1.843908633),
                ("i1", "l4", 2.740236263)])
    out.append(("wag_4_seqs_gaps", t4, {"l1": "SS", "l2": "TT", "l3": "GG", "l4": "D-"}, np.eye(2), [1.0, 1.0],
                pi_wag, wag, pi_equ2, equ2, -17.436349, [-10.092142, -7.344207], 4))
    out.append(("equ_x_equ_3_seqs", t3, {"l1": "SK", "l2": "TI", "l3": "GL"}, np.ones((2, 2)), [1.0, 1.0],
                compute_stationary_distribution(equ), equ, pi_equ2, equ2, -9.382765 * 2, [-9.382765, -9.382765], 4))
    d = os.path.join(LL_DIR, "1a92")
    msa = read_msa(os.path.join(d, "msa.txt"))
    for cats, ll in ((1, -4649.6146), (2, -4397.8184), (4, -4337.8688), (20, -4307.0638)):
        rates = read_site_rates(os.path.join(d, f"site_rates_{cats}_cat.txt"))
        out.append((f"1a92_{cats}_cat", read_tree(os.path.join(d, f"tree_{cats}_cat.txt")), msa, np.eye(len(rates)),
                    rates, pi_wag, wag, None, None, ll, None, 4))
    return out


def pair_matrix(case):
    Q1 = rate_matrix(case["Q1"])
    if case["pair_model"] is None:
        return None
    base = chain_product(Q1, Q1)
    if case["pair_model"] == "product":
        return base
    rng = np.random.default_rng(case["pair_seed"])
    pi = compute_stationary_distribution(base)
    n = base.shape[0]
    sym = rng.uniform(0.5, 1.5, (n, n))
    sym = (sym + sym.T) / 2
    Q = (base / pi[None, :]) * sym * pi[None, :]
    Q[np.arange(n), np.arange(n)] = 0
    Q[np.arange(n), np.arange(n)] = -Q.sum(axis=1)
    return Q


def golden_cases():
    with open(os.path.join(LL_DIR, "cases.json")) as f:
        cases = json.load(f)
    out = []
    for c in cases:
        t = Tree()
        t.add_nodes(c["names"])
        for i in range(1, len(c["names"])):
            t.add_edge(c["names"][c["parent"][i]], c["names"][i], c["length"][i])
        L = len(c["site_rates"])
        cmap = None
        if c["contact_map_given"]:
            cmap = np.eye(L) if not c["pairs"] else np.zeros((L, L))
            for a, b in c["pairs"]:
                cmap[a, b] = cmap[b, a] = 1
        Q1 = rate_matrix(c["Q1"])
        Q2 = pair_matrix(c)
        out.append(dict(tree=t, msa=c["msa"], contact_map=cmap, site_rates=c["site_rates"], Q1=Q1,
                        pi1=compute_stationary_distribution(Q1), Q2=Q2,
                        pi2=None if Q2 is None else compute_stationary_distribution(Q2), ll=c["ll"], lls=c["lls"]))
    return out


# ------------------------------------------------------------------ seeded cases of the gradient tests

def _random_reversible(S, seed, mask=None):
    rng = np.random.default_rng(seed)
    pi = rng.dirichlet(np.full(S, 5.0))
    sym = rng.uniform(0.2, 2.0, (S, S))
    sym = (sym + sym.T) / 2
    if mask is not None:
        sym = sym * mask
    Q = sym * pi[None, :]
    np.fill_diagonal(Q, 0.0)
    np.fill_diagonal(Q, -Q.sum(axis=1))
    return Q / -np.sum(pi * np.diag(Q)), pi


def _model(name, S):
    if name in ("lg", "wag"):
        Q = rate_matrix(name)
        return Q, compute_stationary_distribution(Q)
    return _random_reversible(S, seed=S)


def _random_tree(n_leaves, rng, root_children=2, zero_branch=False):
    """Random rooted tree: random joins down to `root_children` subtrees under the root."""
    t = Tree()
    names = [f"L{i}" for i in range(n_leaves)]
    t.add_nodes(names)
    edges = []
    pool = list(names)
    k = 0
    while len(pool) > root_children:
        a, b = rng.choice(len(pool), 2, replace=False)
        p = f"n{k}"
        k += 1
        t.add_node(p)
        edges += [(p, pool[a], float(rng.lognormal(-2, 0.8))), (p, pool[b], float(rng.lognormal(-2, 0.8)))]
        pool = [x for i, x in enumerate(pool) if i not in (a, b)] + [p]
    t.add_node("root")
    edges += [("root", x, float(rng.lognormal(-2, 0.8))) for x in pool]
    if zero_branch:
        edges[0] = (edges[0][0], edges[0][1], 0.0)
    t.add_edges(edges)
    return t


def _random_msa(tree, alphabet, L, rng, gap_frac=0.1, all_gap_column=False):
    msa = {}
    for v in tree.leaves():
        s = rng.choice(alphabet, L)
        s[rng.random(L) < gap_frac] = "-" if "-" not in alphabet else "X"
        if all_gap_column:
            s[0] = "-" if "-" not in alphabet else "X"
        msa[v] = "".join(s)
    return msa


def _rates(L, n_cats, rng):
    cats = [0.1, 3.0] + [float(x) for x in rng.uniform(0.2, 2.5, max(0, n_cats - 2))]
    cats = cats[:n_cats] if n_cats > 1 else [1.0]
    r = [cats[i % n_cats] for i in range(L)]
    rng.shuffle(r)
    return r


def _star_of_cherries(n_cherries, rng):
    t = Tree()
    t.add_node("root")
    for c in range(n_cherries):
        p, a, b = f"c{c}", f"c{c}a", f"c{c}b"
        t.add_nodes([p, a, b])
        t.add_edges([("root", p, float(rng.lognormal(-3, 1))), (p, a, float(rng.lognormal(-2, 1))),
                     (p, b, float(rng.lognormal(-2, 1)))])
    return t


def _caterpillar(n_leaves, rng):
    """Maximally deep tree (depth n_leaves - 1)."""
    t = Tree()
    t.add_node("n0")
    prev = "n0"
    for i in range(n_leaves - 1):
        leaf, nxt = f"L{i}", f"n{i + 1}"
        t.add_node(leaf)
        t.add_edge(prev, leaf, float(rng.lognormal(-2, 1)))
        if i == n_leaves - 2:
            t.add_node(f"L{i + 1}")
            t.add_edge(prev, f"L{i + 1}", float(rng.lognormal(-2, 1)))
        else:
            t.add_node(nxt)
            t.add_edge(prev, nxt, float(rng.lognormal(-2, 1)))
            prev = nxt
    return t


def _demo_family(tmp_dir, fam="13gs_1_A"):
    """(tree, msa, site rates) of a demo family, extracted under `tmp_dir`."""
    with tarfile.open(os.path.join(GOLDEN, "demo_data.tar.xz")) as tf:
        tf.extractall(tmp_dir, members=[tf.getmember(f"{d}/{fam}.txt") for d in ("msas", "trees", "site_rates")])
    return (read_tree(os.path.join(tmp_dir, "trees", f"{fam}.txt")), read_msa(os.path.join(tmp_dir, "msas", f"{fam}.txt")),
            read_site_rates(os.path.join(tmp_dir, "site_rates", f"{fam}.txt")))


def _write_families(root, fams, alphabet=AA):
    """fams: {name: (tree, msa, site_rates)} -> (tree_dir, msa_dir, site_rates_dir)."""
    from cherryml_b200.io import write_msa, write_site_rates, write_tree

    dirs = [os.path.join(root, d) for d in ("trees", "msas", "site_rates")]
    for d in dirs:
        os.makedirs(d, exist_ok=True)
    for name, (tree, msa, rates) in fams.items():
        write_tree(tree, os.path.join(dirs[0], name + ".txt"))
        write_msa(msa, os.path.join(dirs[1], name + ".txt"))
        write_site_rates(rates, os.path.join(dirs[2], name + ".txt"))
    return dirs


def _simulate_family(Q, pi, n_leaves, L, rng):
    """Sites evolved down a random tree under (Q, pi); site rates from three categories."""
    from scipy.linalg import expm

    tree = _random_tree(n_leaves, rng)
    rates = [float(r) for r in rng.choice([0.5, 1.0, 2.0], L)]
    cats = sorted(set(rates))
    cat = np.array([cats.index(r) for r in rates])
    states = {tree.root(): rng.choice(len(pi), L, p=pi)}
    for v in reversed(tree.postorder_traversal()):
        if v == tree.root():
            continue
        p, length = tree.parent(v)
        cdf = np.cumsum(np.stack([expm(length * r * Q) for r in cats]), axis=2)  # [cats, S, S]
        rows = cdf[cat, states[p]]  # [L, S]
        states[v] = np.minimum((rng.random(L)[:, None] > rows).sum(axis=1), len(pi) - 1)
    msa = {v: "".join(AA[s] for s in states[v]) for v in tree.leaves()}
    return tree, msa, rates


def _synthetic_cases():
    """(id, tree, msa, site_rates, alphabet, model name)."""
    aa21 = AA + ["-"]
    out = []
    rng = np.random.default_rng(11)
    t = _random_tree(12, rng)
    out.append(("lg_1cat", t, _random_msa(t, AA, 30, rng), _rates(30, 1, rng), AA, "lg"))
    t = _random_tree(10, rng, root_children=3, zero_branch=True)
    out.append(("wag_4cat_gapcol_zero_branch", t, _random_msa(t, AA, 40, rng, all_gap_column=True),
                _rates(40, 4, rng), AA, "wag"))
    t = _random_tree(9, rng)
    out.append(("random_20cat", t, _random_msa(t, AA, 60, rng), _rates(60, 20, rng), AA, "random"))
    t = _random_tree(8, rng, root_children=4)
    out.append(("dna_4cat_multifurcating", t, _random_msa(t, DNA, 50, rng), _rates(50, 4, rng), DNA, "random"))
    t = _random_tree(11, rng, zero_branch=True)
    out.append(("s21_gaps_as_state", t, _random_msa(t, aa21, 45, rng, all_gap_column=True), _rates(45, 4, rng), aa21,
                "random"))
    single = Tree()
    single.add_node("only")
    out.append(("single_leaf", single, {"only": "ARND-"}, [1.0, 1.0, 2.0, 0.5, 1.0], AA, "lg"))
    t = _caterpillar(60, rng)
    out.append(("caterpillar_60", t, _random_msa(t, AA, 77, rng, gap_frac=0.2), _rates(77, 4, rng), AA, "lg"))
    t = _star_of_cherries(512, rng)
    out.append(("star_512_cherries", t, _random_msa(t, AA, 24, rng), _rates(24, 4, rng), AA, "wag"))
    for i, c in enumerate(golden_cases()):
        cm = c["contact_map"]
        if cm is None or not np.any(cm - np.diag(np.diag(cm))):
            out.append((f"golden_{i}", c["tree"], c["msa"], c["site_rates"], AA, "lg"))
    return out


def _scratch_formula(S, n_nodes, max_depth, n_cats, n_matrices, unit_cat):
    """Bytes of cherry_tree_ll_posterior's scratch."""
    G = max(1, 256 // S)
    counts = np.bincount(unit_cat, minlength=n_cats)
    ctas = int(sum((c + G - 1) // G for c in counts))
    doubles = ctas * (3 * n_nodes * G * S + 2 * (max_depth + 1) * G * S + n_nodes * S * S + S)
    ints = ctas * G + ctas + (n_cats + 1) + (n_matrices + 1) + (n_nodes - 1) * n_cats + n_nodes * n_cats
    return 8 * doubles + 4 * ints
