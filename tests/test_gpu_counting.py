"""GPU parity tests for counting: the CUDA path (through the C ABI and the public stage
functions) against the reference goldens and the oracle.  Bit-exact: integer/byte work."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from cherryml_b200 import _lib, caching
from cherryml_b200.counting import count_co_transitions, count_transitions, device_result
from cherryml_b200.counting._device import (count_batch, count_lg_host, count_raw, sorted_grid,
                                             symmetrize, to_device)
from cherryml_b200.io import read_count_matrices_array
from cherryml_b200.synthetic import (as_count_batch, as_device_batch, quantization_grid, synthetic_co,
                                     synthetic_lg)
from cherryml_b200.utils import amino_acids
from oracle.counting_oracle import read_count_matrices_text
from oracle.native import count_batch_oracle
from tests.test_oracle_counting import CO_CASES, GRID_CO, GRID_LG, LG_CASES, MEDIUM3, MODES


@pytest.mark.parametrize("case", LG_CASES, ids=lambda c: f"{c[0]}-{c[4]}")
@pytest.mark.parametrize("use_cpp", [True, False])
def test_count_transitions_reference_tiny_goldens(golden_counting, tmp_path, case, use_cpp):
    ds, fams, aa, grid, mode, gdir = case
    root = os.path.join(golden_counting, ds)
    out = str(tmp_path / "out")
    count_transitions(
        tree_dir=f"{root}/tree_dir", msa_dir=f"{root}/msa_dir", site_rates_dir=f"{root}/site_rates_dir",
        families=fams, amino_acids=aa, quantization_points=grid, edge_or_cherry=mode,
        output_count_matrices_dir=out, num_processes=3, use_cpp_implementation=use_cpp,
    )
    q, states, counts = read_count_matrices_array(os.path.join(out, "result.txt"))
    gq, gstates, gcounts = read_count_matrices_text(os.path.join(golden_counting, ds, gdir, "result.txt"))
    assert np.allclose(q, gq) and states == gstates
    assert np.array_equal(counts, gcounts)
    assert open(os.path.join(out, "profiling.txt")).read().split()[2].replace(".", "").replace("e-", "").isdigit()


@pytest.mark.parametrize("case", CO_CASES, ids=lambda c: f"{c[0]}-{c[4]}")
def test_count_co_transitions_reference_tiny_goldens(golden_counting, tmp_path, case):
    ds, fams, aa, grid, mode, gdir = case
    root = os.path.join(golden_counting, ds)
    out = str(tmp_path / "out")
    count_co_transitions(
        tree_dir=f"{root}/tree_dir", msa_dir=f"{root}/msa_dir", contact_map_dir=f"{root}/contact_map_dir",
        families=fams, amino_acids=aa, quantization_points=grid, edge_or_cherry=mode,
        minimum_distance_for_nontrivial_contact=2, output_count_matrices_dir=out, num_processes=2,
    )
    q, states, counts = read_count_matrices_array(os.path.join(out, "result.txt"))
    gq, gstates, gcounts = read_count_matrices_text(os.path.join(golden_counting, ds, gdir, "result.txt"))
    assert np.allclose(q, gq) and states == gstates
    assert np.array_equal(counts, gcounts)


@pytest.mark.parametrize("mode,tag,msa_sub", MODES)
@pytest.mark.parametrize("personality", ["cpp", "py"])
def test_count_transitions_medium3_vs_reference_run(golden_counting, tmp_path, mode, tag, msa_sub, personality):
    m3 = os.path.join(golden_counting, "medium3")
    out = str(tmp_path / "out")
    count_transitions(
        tree_dir=f"{m3}/tree_dir", msa_dir=f"{m3}/{msa_sub}", site_rates_dir=f"{m3}/site_rates_dir",
        families=MEDIUM3, amino_acids=amino_acids, quantization_points=GRID_LG, edge_or_cherry=mode,
        output_count_matrices_dir=out, use_cpp_implementation=(personality == "cpp"),
    )
    golden_path = f"{m3}/ref{personality}_count_matrices_dir_{tag}/result.txt"
    _, _, gcounts = read_count_matrices_text(golden_path)
    _, _, counts = read_count_matrices_array(os.path.join(out, "result.txt"))
    assert np.array_equal(counts, gcounts)
    # the written file is byte-identical to what the reference program wrote
    assert open(os.path.join(out, "result.txt")).read() == open(golden_path).read()
    grid, states, dev = device_result(out)
    assert np.array_equal(dev.cpu().numpy(), gcounts)


@pytest.mark.parametrize("mode,tag,msa_sub", MODES)
def test_count_co_transitions_medium3_vs_reference_run(golden_counting, tmp_path, mode, tag, msa_sub):
    m3 = os.path.join(golden_counting, "medium3")
    out = str(tmp_path / "out")
    count_co_transitions(
        tree_dir=f"{m3}/tree_dir", msa_dir=f"{m3}/{msa_sub}", contact_map_dir=f"{m3}/contact_map_dir",
        families=MEDIUM3, amino_acids=amino_acids, quantization_points=GRID_CO, edge_or_cherry=mode,
        minimum_distance_for_nontrivial_contact=7, output_count_matrices_dir=out,
    )
    gcounts = np.load(f"{m3}/refcpp_count_co_matrices_dir_{tag}/result.npz")["counts"]
    _, _, dev = device_result(out)
    assert np.array_equal(dev.cpu().numpy(), gcounts)
    _, _, counts = read_count_matrices_array(os.path.join(out, "result.txt"))
    assert np.array_equal(counts, gcounts)  # every cell < 1e6, so 6 significant digits are exact


def test_cache_dir_semantics(golden_counting, tmp_path):
    root = os.path.join(golden_counting, "tiny")
    kw = dict(tree_dir=f"{root}/tree_dir", msa_dir=f"{root}/msa_dir", site_rates_dir=f"{root}/site_rates_dir",
              families=["fam1", "fam2", "fam3"], amino_acids=["I", "L", "S", "T"],
              quantization_points=[1.99, 10.01], edge_or_cherry="cherry")
    with pytest.raises(caching.CacheUsageError):
        count_transitions(kw["tree_dir"], **{k: v for k, v in kw.items() if k != "tree_dir"})
    caching.set_cache_dir(str(tmp_path / "cache"))
    try:
        res = count_transitions(**kw)
        out = res["output_count_matrices_dir"]
        assert os.path.exists(os.path.join(out, "result.success"))
        mtime = os.path.getmtime(os.path.join(out, "result.txt"))
        res2 = count_transitions(**kw, num_processes=7)  # excluded arg: same key, cached
        assert res2 == res and os.path.getmtime(os.path.join(out, "result.txt")) == mtime
    finally:
        caching.set_cache_dir(None)


@pytest.mark.parametrize("n_cats,K", [(4, 100), (20, 129), (1, 7)])
def test_lg_synthetic_vs_oracle(n_cats, K):
    grid = quantization_grid(lo=-(K // 2), hi=K - K // 2 - 1)
    assert len(grid) == K
    syn = synthetic_lg(48, 256, 300, n_cats, seed=11)
    batch = as_count_batch(syn)
    exp = count_batch_oracle(batch, grid, 20, False)
    got = count_batch(batch, grid, 20, directed=False).cpu().numpy()
    assert np.array_equal(got, exp)
    got_dir = count_batch(batch, grid, 20, directed=True).cpu().numpy()
    assert np.array_equal(got_dir, count_batch_oracle(batch, grid, 20, True))
    host, h2d, d2h = count_lg_host(batch, grid, 20, False)
    assert np.array_equal(host, exp) and h2d > batch.msa.size and d2h == exp.nbytes


def test_lg_histogram_too_large_for_shared_memory_falls_back_to_global_atomics():
    grid = [float("%.8f" % (0.001 * 1.05**i)) for i in range(200)]  # 200*400*4 B = 320 KB > 227 KB
    syn = synthetic_lg(8, 128, 150, 4, seed=5)
    batch = as_count_batch(syn)
    got = count_batch(batch, grid, 20, directed=False).cpu().numpy()
    assert np.array_equal(got, count_batch_oracle(batch, grid, 20, False))


def test_lg_ragged_shapes_and_small_alphabet():
    """Families of different sizes in one batch, 4-letter alphabet (others become skips)."""
    from cherryml_b200.counting._ingest import _BatchBuilder, lg_column_layout

    rng = np.random.default_rng(2)
    builder = _BatchBuilder("lg")
    for f, (n_rows, L) in enumerate([(2, 1), (6, 17), (40, 333), (10, 64), (2, 1500)]):
        rates = rng.choice([0.25, 1.0, 3.0], size=L)
        vals, dest, group_cat, stride = lg_column_layout(rates)
        rows = np.full((n_rows, stride), 4, dtype=np.uint8)
        rows[:, dest] = rng.integers(0, 5, size=(n_rows, L)).astype(np.uint8)  # 4 == S is the skip code
        a = np.arange(0, n_rows, 2, dtype=np.int32)
        builder.add_family(f"f{f}", rows, a, a + 1, rng.lognormal(-0.5, 1.0, len(a)), vals, group_cat, stride // 4, L)
    batch = builder.finish()
    grid = [0.05 * 1.3**i for i in range(20)]
    got = count_batch(batch, grid, 4, directed=False).cpu().numpy()
    assert np.array_equal(got, count_batch_oracle(batch, grid, 4, False))
    assert got.sum() > 0


def test_out_of_range_residue_is_rejected():
    syn = synthetic_lg(2, 8, 32, 4, seed=1)
    batch = as_count_batch(syn)
    batch.msa = batch.msa.copy()
    batch.msa[37] = 21  # > S
    with pytest.raises(_lib.CherryError, match="bytes > 20"):
        count_batch(batch, quantization_grid(), 20, directed=False)


def test_empty_batch():
    from cherryml_b200.counting._ingest import _BatchBuilder

    for kind, shape in (("lg", (3, 20, 20)), ("co", (3, 400, 400))):
        got = count_batch(_BatchBuilder(kind).finish(), [0.1, 1.0, 2.0], 20, directed=False)
        assert tuple(got.shape) == shape and float(got.sum()) == 0.0


def test_co_synthetic_vs_oracle():
    grid = quantization_grid()
    syn = synthetic_co(24, 128, 200, seed=13)
    batch = as_count_batch(syn)
    for directed in (False, True):
        got = count_batch(batch, grid, 20, directed=directed).cpu().numpy()
        assert np.array_equal(got, count_batch_oracle(batch, grid, 20, directed))


def test_sort_pairs_by_bucket():
    """The device counting sort groups the pairs by bucket; pairs outside the grid go last."""
    rng = np.random.default_rng(4)
    for n_pairs, K, r_pad in ((1, 3, 4), (777, 7, 4), (100_003, 129, 8), (5000, 254, 4)):
        tab = np.full((n_pairs, r_pad), 255, dtype=np.uint8)
        tab[:, 0] = rng.integers(0, K + 3, n_pairs)  # K..K+2 never occur in a real table, 255 does
        tab[tab[:, 0] >= K, 0] = 255
        tab_d = torch.from_numpy(tab).cuda()
        order = torch.empty(n_pairs, dtype=torch.int32, device="cuda")
        ws = torch.empty(2 * (K + 2), dtype=torch.int32, device="cuda")
        rc = _lib.load().cherry_sort_pairs_by_bucket(_lib.ptr(tab_d), r_pad, n_pairs, K, 0, 0, 0, 0,
                                                     _lib.ptr(order), 0, _lib.ptr(ws),
                                                     _lib.current_stream_ptr())
        _lib.check(rc, "sort")
        order, ws = order.cpu().numpy(), ws.cpu().numpy()
        b = np.minimum(tab[:, 0].astype(np.int64), K)
        assert np.array_equal(np.sort(order), np.arange(n_pairs))
        assert np.array_equal(ws[: K + 2], np.concatenate([[0], np.cumsum(np.bincount(b, minlength=K + 1))]))
        assert np.all(np.diff(b[order]) >= 0)


def test_co_ragged_families_and_small_alphabets():
    """Families with 0 .. 3000 contacts, odd row counts, pairs outside the grid, S = 3 and
    S = 20 (shared-memory histogram) and S = 24 (global reductions only)."""
    from cherryml_b200.counting._ingest import _BatchBuilder, contact_paired_rows

    for S in (3, 20, 24):
        rng = np.random.default_rng(S)
        builder = _BatchBuilder("co")
        for f, (n_rows, L, P) in enumerate([(2, 9, 0), (6, 17, 3), (40, 333, 160), (11, 64, 31), (2, 7000, 3000),
                                            (300, 40, 20)]):
            enc = rng.integers(0, S + 1, size=(n_rows, L)).astype(np.uint8)  # S is the skip code
            enc[1::2] = np.where(rng.random((len(enc[1::2]), L)) < 0.6, enc[0 : 2 * len(enc[1::2]) : 2], enc[1::2])
            contacts = np.stack([rng.integers(0, L, P), rng.integers(0, L, P)], axis=1).astype(np.int32)
            rows = contact_paired_rows(enc, contacts, S)
            a = np.arange(0, n_rows - 1, 2, dtype=np.int32)
            t = rng.lognormal(-0.5, 1.5, len(a))
            builder.add_family(f"f{f}", rows, a, a + 1, t, np.ones(1), contacts, P, P)
        batch = builder.finish()
        grid = [0.05 * 1.3**i for i in range(15)]
        for directed in (False, True):
            got = count_batch(batch, grid, S, directed=directed).cpu().numpy()
            assert np.array_equal(got, count_batch_oracle(batch, grid, S, directed))
        assert got.sum() > 0


def test_co_row_longer_than_a_stage_is_an_error():
    from cherryml_b200.counting._ingest import _BatchBuilder, contact_paired_rows

    builder = _BatchBuilder("co")
    P = 9000  # 18000 bytes per row > 16384
    contacts = np.zeros((P, 2), dtype=np.int32)
    rows = contact_paired_rows(np.zeros((2, 4), dtype=np.uint8), contacts, 20)
    builder.add_family("f", rows, np.array([0]), np.array([1]), np.array([0.5]), np.ones(1), contacts, P, P)
    with pytest.raises(_lib.CherryError, match="exceeds"):
        count_batch(builder.finish(), [0.1, 1.0], 20, directed=False)


def test_full_size_properties_co():
    """BASELINE config-4 shape on a slice (1024 families x 1024 x 300, perfect matching):
    conservation, the symmetries of the symmetrised tensor, and a 16-family slice vs the oracle."""
    grid = quantization_grid()
    K = len(grid)
    n_fams, n_pairs = 1024, 512
    syn = synthetic_co(n_fams, 1024, 300, seed=5, device="cuda")
    dev = as_device_batch(syn, "cuda")
    grid_dev = torch.from_numpy(sorted_grid(grid)).cuda()
    raw = count_raw(dev, grid_dev, K, 20)
    total = int(raw.sum(dtype=torch.int64).item())
    stride = syn["shape"]["stride"]
    rows = syn["msa"].view(n_fams, n_pairs, 2, stride // 2, 2)
    valid = (rows < 20).all(dim=4).all(dim=2)  # [fam, pair, contact]
    in_grid = ((syn["pair_t"] >= grid[0]) & (syn["pair_t"] <= grid[-1])).view(n_fams, n_pairs, 1)
    assert total == int((valid & in_grid).sum().item())
    sym = symmetrize(raw, "co", K, 20, directed=False)
    assert torch.equal(sym, sym.transpose(1, 2)) and float(sym.sum().item()) == float(total)
    perm = (torch.arange(400, device="cuda") % 20) * 20 + torch.arange(400, device="cuda") // 20
    assert torch.equal(sym, sym[:, perm][:, :, perm])
    # counting twice into the same buffer doubles every cell (accumulate semantics)
    raw2 = count_raw(dev, grid_dev, K, 20, out=raw.clone())
    assert torch.equal(raw2, 2 * raw)
    import copy
    batch = as_count_batch(syn)
    sl = slice(0, 16 * n_pairs)
    exp = count_batch_oracle(batch, grid, 20, False, pair_slice=sl)
    d3 = copy.copy(dev)
    d3.n_pairs = 16 * n_pairs
    d3.n_tiles = 16 * (dev.n_tiles // n_fams)
    got = symmetrize(count_raw(d3, grid_dev, K, 20), "co", K, 20, False).cpu().numpy()
    assert np.array_equal(got, exp)


@pytest.mark.parametrize("kind", ["lg", "co"])
def test_more_quantization_points_than_one_pass_addresses(kind):
    """The reference has no bound on the number of quantization points (_count_transitions.cpp:295-307,
    quantization_grid_num_steps >= 127 gives K > 254); the kernels address 254 buckets per pass, longer grids
    are counted in passes over overlapping sub-grids.  K = 300 and K = 600, bit-exact against the oracle,
    including values exactly at and one ulp around the sub-grid seams."""
    for K in (300, 600):
        grid = [0.0005 * 1.02**i for i in range(K)]
        if kind == "lg":
            syn = synthetic_lg(6, 64, 96, 4, seed=K)
        else:
            syn = synthetic_co(3, 32, 60, seed=K)
        # pair lengths on and around the grid points next to the seams (rate 1 exists in neither batch's
        # categories exactly, so also plain multiples are exercised through the random lengths)
        t = syn["pair_t"].clone()
        g = np.array(grid)
        seam = np.concatenate([g[250:256], np.nextafter(g[250:256], 0), np.nextafter(g[250:256], np.inf),
                               np.sqrt(g[250:255] * g[251:256])])
        n = min(len(seam), t.numel())
        t[:n] = torch.from_numpy(seam[:n])
        syn["pair_t"] = t
        batch = as_count_batch(syn)
        got = count_batch(batch, grid, 20, directed=False).cpu().numpy()
        assert np.array_equal(got, count_batch_oracle(batch, grid, 20, False))
        assert got[252:].sum() > 0 and got[:252].sum() > 0


def test_full_size_properties_lg():
    """BASELINE config-3 shape on one GPU slice (2048 families x 1024 x 300): size-independent
    properties -- conservation (every valid, in-grid site counted once), symmetry, linearity
    over a split of the families, and agreement of a 64-family slice with the oracle."""
    grid = quantization_grid()
    K = len(grid)
    syn = synthetic_lg(2048, 1024, 300, 4, seed=3, device="cuda")
    dev = as_device_batch(syn, "cuda")
    grid_dev = torch.from_numpy(sorted_grid(grid)).cuda()
    raw = count_raw(dev, grid_dev, K, 20)
    total = int(raw.sum().item())
    # conservation, computed independently with torch ops on the device
    n_pairs, stride = 512, syn["shape"]["stride"]
    rows = syn["msa"].view(2048, n_pairs, 2, stride)
    valid = (rows[:, :, 0, :] < 20) & (rows[:, :, 1, :] < 20)
    rates = torch.from_numpy(syn["rate_vals"][:4]).cuda()
    cat = torch.from_numpy(syn["aux"][: stride // 4].astype(np.int64)).cuda().repeat_interleave(4)
    tt = syn["pair_t"].view(2048, n_pairs, 1) * rates[cat].view(1, 1, stride)
    in_grid = (tt >= grid[0]) & (tt <= grid[-1])
    assert total == int((valid & in_grid).sum().item())
    sym = symmetrize(raw, "lg", K, 20, directed=False)
    assert torch.equal(sym, sym.transpose(1, 2)) and float(sym.sum().item()) == float(total)
    # linearity: counts(first half of the tiles) + counts(second half) == counts(all)
    import copy
    half = dev.n_tiles // 2
    d1, d2 = copy.copy(dev), copy.copy(dev)
    d1.n_tiles = half
    d2.tiles, d2.n_tiles = dev.tiles[half * 16:], dev.n_tiles - half
    assert torch.equal(count_raw(d1, grid_dev, K, 20) + count_raw(d2, grid_dev, K, 20), raw)
    # a 64-family slice against the oracle
    batch = as_count_batch(syn)
    sl = slice(0, 64 * n_pairs)
    exp = count_batch_oracle(batch, grid, 20, False, pair_slice=sl)
    d3 = copy.copy(dev)
    d3.n_tiles = 64 * (dev.n_tiles // 2048)
    got = symmetrize(count_raw(d3, grid_dev, K, 20), "lg", K, 20, False).cpu().numpy()
    assert np.array_equal(got, exp)


@pytest.mark.parametrize("grid_kind", ["geometric", "repeated_point", "zero_point"])
def test_bucket_table_tiles_at_bucket_boundaries(grid_kind):
    """t*rate exactly at / a few ulps around the geometric midpoints and the grid points: the table's
    precomputed decision boundaries must be the reference's switch points exactly; a grid with a repeated
    or a zero point takes the binary search, whose product-based fast comparison must fall back to the
    reference expression where needed (at zero the products tie and the quotients are infinite)."""
    from cherryml_b200 import _lib
    from oracle.native import quantization_idx_c

    lg = np.array(sorted(GRID_LG))
    grid = lg
    if grid_kind == "repeated_point":
        grid = np.array(sorted(list(lg) + [lg[7], lg[40]]))
    elif grid_kind == "zero_point":
        grid = np.concatenate([[0.0], lg])
    mids = np.sqrt(grid[:-1] * grid[1:])
    near = [mids, grid]
    for base in (mids, grid):
        lo, hi = base, base
        for _ in range(4):
            lo, hi = np.nextafter(lo, 0), np.nextafter(hi, np.inf)
            near += [lo, hi]
    ts = np.concatenate(near + [0.5 * (grid[:-1] + grid[1:]),
                                np.exp(np.random.default_rng(0).uniform(np.log(lg[0] / 2), np.log(lg[-1] * 2), 5000))])
    syn = synthetic_lg(1, 2 * len(ts), 16, 4, seed=0)
    syn["pair_t"] = torch.from_numpy(ts.copy())
    rates = np.array([1.0, 0.5, 3.0, 1.0 / 3.0])
    syn["rate_vals"] = rates.copy()
    dev = as_device_batch(syn, "cuda")
    grid_dev = torch.from_numpy(grid).cuda()
    tab = torch.full((dev.n_pairs * dev.r_pad,), 77, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().cherry_build_bucket_table_tiles(
        _lib.ptr(dev.pair_t), _lib.ptr(dev.tiles), dev.n_tiles, _lib.ptr(dev.fams), _lib.ptr(dev.rate_vals),
        _lib.ptr(grid_dev), len(grid), dev.r_pad, _lib.ptr(tab), _lib.current_stream_ptr()),
        "cherry_build_bucket_table_tiles")
    tab = tab.cpu().numpy().reshape(len(ts), 4)
    for i, t in enumerate(ts):
        for r in range(4):
            exp = quantization_idx_c(t * rates[r], grid)
            assert tab[i, r] == (255 if exp < 0 else exp), (t, rates[r])


@pytest.mark.parametrize("families_per_batch", [1, 2])
def test_streamed_batches_equal_the_single_batch(golden_counting, tmp_path, families_per_batch):
    """More families than `families_per_batch`: chunks are ingested by host threads while the
    previous chunk is counted; the raw integer histograms add up exactly, so the files are the
    reference program's byte for byte as in the single-batch tests above."""
    m3 = os.path.join(golden_counting, "medium3")
    out = str(tmp_path / "lg")
    count_transitions(
        tree_dir=f"{m3}/tree_dir", msa_dir=f"{m3}/msa_dir", site_rates_dir=f"{m3}/site_rates_dir",
        families=MEDIUM3, amino_acids=amino_acids, quantization_points=GRID_LG, edge_or_cherry="cherry++",
        output_count_matrices_dir=out, use_cpp_implementation=True, num_processes=4,
        families_per_batch=families_per_batch,
    )
    golden = f"{m3}/refcpp_count_matrices_dir_cherries_plus_plus/result.txt"
    assert open(os.path.join(out, "result.txt")).read() == open(golden).read()
    out = str(tmp_path / "co")
    count_co_transitions(
        tree_dir=f"{m3}/tree_dir", msa_dir=f"{m3}/msa_dir", contact_map_dir=f"{m3}/contact_map_dir",
        families=MEDIUM3, amino_acids=amino_acids, quantization_points=GRID_CO, edge_or_cherry="cherry++",
        minimum_distance_for_nontrivial_contact=7, output_count_matrices_dir=out, num_processes=4,
        families_per_batch=families_per_batch,
    )
    gcounts = np.load(f"{m3}/refcpp_count_co_matrices_dir_cherries_plus_plus/result.npz")["counts"]
    _, _, dev = device_result(out)
    assert np.array_equal(dev.cpu().numpy(), gcounts)
