"""Run the counting kernels on an encoded batch (device side of the counting stage).

PyTorch owns the device buffers and the stream; all compute is the CUDA library behind
the C ABI (``include/cherryml_b200.h``).  No CPU fallback.
"""
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from .. import _lib
from ._ingest import CountBatch

# (pairs x contacts) per co-transition launch is kept below this so no uint32 cell can wrap
_CO_MAX_ITEMS_PER_LAUNCH = (1 << 32) - 1


@dataclass
class DeviceBatch:
    kind: str
    msa: torch.Tensor
    fams: torch.Tensor
    pair_a: torch.Tensor
    pair_b: torch.Tensor
    pair_t: torch.Tensor
    pair_fam: torch.Tensor
    rate_vals: torch.Tensor
    aux: torch.Tensor
    tiles: torch.Tensor
    r_pad: int
    n_pairs: int
    n_tiles: int
    n_sites_examined: int
    tile_items: Optional[np.ndarray] = None  # host copy, co only: items per tile
    max_row_stride: int = 0  # co only

    def nbytes(self) -> int:
        return sum(
            t.numel() * t.element_size()
            for t in (self.msa, self.fams, self.pair_a, self.pair_b, self.pair_t,
                      self.pair_fam, self.rate_vals, self.aux, self.tiles)
        )


def _as_device(arr: np.ndarray, device, pin: bool = False) -> torch.Tensor:
    raw = np.ascontiguousarray(arr).view(np.uint8).reshape(-1)
    t = torch.from_numpy(raw)
    if pin:
        t = t.pin_memory()
    return t.to(device, non_blocking=pin)


def to_device(batch: CountBatch, device="cuda") -> DeviceBatch:
    """Upload a host batch.  Tensors are raw byte tensors; the kernels see typed pointers."""
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.CherryError("cherryml_b200 counting runs on CUDA devices only")
    _lib.load()
    tile_items = None
    if batch.kind == "co" and batch.tiles.shape[0]:
        tile_items = batch.tiles["n_pairs"].astype(np.int64) * batch.fams["aux_cnt"][
            batch.tiles["fam"]
        ].astype(np.int64)
    return DeviceBatch(
        kind=batch.kind,
        msa=_as_device(batch.msa, device),
        fams=_as_device(batch.fams, device),
        pair_a=_as_device(batch.pair_a, device),
        pair_b=_as_device(batch.pair_b, device),
        pair_t=_as_device(batch.pair_t, device),
        pair_fam=_as_device(batch.pair_fam, device),
        rate_vals=_as_device(batch.rate_vals, device),
        # the co-transition kernels read contact-paired rows, not the contact list
        aux=_as_device(batch.aux if batch.kind == "lg" else np.zeros(0, np.int32), device),
        tiles=_as_device(batch.tiles, device),
        r_pad=batch.r_pad,
        n_pairs=batch.n_pairs,
        n_tiles=int(batch.tiles.shape[0]),
        n_sites_examined=batch.n_sites_examined,
        tile_items=tile_items,
        max_row_stride=int(batch.fams["row_stride"].max()) if batch.fams.shape[0] else 16,
    )


def sorted_grid(quantization_points: Sequence[float]) -> np.ndarray:
    grid = np.array(sorted(float(q) for q in quantization_points), dtype=np.float64)
    if grid.size == 0:
        raise ValueError("quantization_points is empty")
    return grid  # more than _lib.MAX_BUCKETS points: count_raw makes several passes over sub-grids


def validate_residues(msa: torch.Tensor, num_states: int) -> None:
    """Raise unless every residue byte is <= num_states (the skip code)."""
    lib = _lib.load()
    n = msa.numel() // 16 * 16
    flag = torch.zeros(1, dtype=torch.int32, device=msa.device)
    rc = lib.cherry_validate_residues(_lib.ptr(msa), n, int(num_states), _lib.ptr(flag),
                                      _lib.current_stream_ptr())
    _lib.check(rc, "cherry_validate_residues")
    bad_tail = bool((msa[n:] > num_states).any().item()) if n < msa.numel() else False
    if int(flag.item()) != 0 or bad_tail:
        raise _lib.CherryError(
            f"residue buffer holds bytes > {num_states}: encode with the same alphabet that is "
            "passed to the counting call (skip code == number of states)"
        )


def build_bucket_table_tiles(dev: DeviceBatch, grid_dev: torch.Tensor, K: int) -> torch.Tensor:
    """The bucket table of the pairs covered by the batch's tiles, built one warp per tile."""
    lib = _lib.load()
    tab = torch.empty(max(1, dev.n_pairs * dev.r_pad), dtype=torch.uint8, device=dev.msa.device)
    if dev.n_tiles:
        rc = lib.cherry_build_bucket_table_tiles(
            _lib.ptr(dev.pair_t), _lib.ptr(dev.tiles), dev.n_tiles, _lib.ptr(dev.fams), _lib.ptr(dev.rate_vals),
            _lib.ptr(grid_dev), K, dev.r_pad, _lib.ptr(tab), _lib.current_stream_ptr(),
        )
        _lib.check(rc, "cherry_build_bucket_table_tiles")
    return tab


def count_raw(
    dev: DeviceBatch,
    grid_dev: torch.Tensor,
    K: int,
    S: int,
    tab: Optional[torch.Tensor] = None,
    out: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """Raw directed integer histogram on the device (``_count_raw_one``).  The kernels address at most
    ``_lib.MAX_BUCKETS`` (254) buckets through a one-byte table; the reference has no bound
    (``_count_transitions.cpp:295-307``), so a longer grid is counted in passes over sub-grids of 252 points
    extended by one neighbour on each side: a value's nearest grid point and both of that point's neighbours
    are then in the same sub-grid, so the decision is the full grid's, and the values that fall to the two
    extra points are masked out of the pass (they belong to the neighbouring pass)."""
    if K <= _lib.MAX_BUCKETS:
        return _count_raw_one(dev, grid_dev, K, S, tab, out)
    if tab is not None:
        raise _lib.CherryError(f"a precomputed bucket table addresses at most {_lib.MAX_BUCKETS} buckets")
    device = dev.msa.device
    if out is None:
        shape = (K, S, S) if dev.kind == "lg" else (K, S * S, S * S)
        out = torch.zeros(shape, dtype=torch.int64 if dev.kind == "lg" else torch.int32, device=device)
    step = _lib.MAX_BUCKETS - 2
    for lo in range(0, K, step):
        hi = min(K, lo + step)
        elo, ehi = max(0, lo - 1), min(K, hi + 1)
        sub = grid_dev[elo:ehi].contiguous()
        ks = ehi - elo
        sub_tab = build_bucket_table_tiles(dev, sub, ks)
        if dev.n_pairs:
            if elo < lo:
                sub_tab[sub_tab == 0] = _lib.NO_BUCKET
            if ehi > hi:
                sub_tab[sub_tab == ks - 1] = _lib.NO_BUCKET
        part = _count_raw_one(dev, sub, ks, S, sub_tab, None)
        out[lo:hi] += part[lo - elo: lo - elo + (hi - lo)]
    return out


def _count_raw_one(
    dev: DeviceBatch,
    grid_dev: torch.Tensor,
    K: int,
    S: int,
    tab: Optional[torch.Tensor] = None,
    out: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """Raw directed integer histogram on the device, K <= _lib.MAX_BUCKETS.

    LG: uint64 ``[K,S,S]`` (returned as an int64 tensor); co: uint32 ``[K,S*S,S*S]``
    (returned as an int32 tensor).  ``out`` is accumulated into when given.
    """
    lib = _lib.load()
    device = dev.msa.device
    stream = _lib.current_stream_ptr()
    if tab is None:
        tab = build_bucket_table_tiles(dev, grid_dev, K)
    if dev.kind == "lg":
        if out is None:
            out = torch.zeros((K, S, S), dtype=torch.int64, device=device)
        if dev.n_tiles:
            rc = lib.cherry_count_lg(
                _lib.ptr(dev.msa), _lib.ptr(dev.fams), _lib.ptr(dev.pair_a), _lib.ptr(dev.pair_b),
                _lib.ptr(tab), dev.r_pad, _lib.ptr(dev.aux), _lib.ptr(dev.tiles), dev.n_tiles,
                K, S, _lib.ptr(out), stream,
            )
            _lib.check(rc, "cherry_count_lg")
        return out
    n = S * S
    if out is None:
        out = torch.zeros((K, n, n), dtype=torch.int32, device=device)
    if dev.n_tiles:
        total_items = int(dev.tile_items.sum()) if dev.tile_items is not None else 0
        if total_items > _CO_MAX_ITEMS_PER_LAUNCH:
            raise _lib.CherryError(
                f"{total_items} (pair, contact) items in one batch could wrap a uint32 cell; "
                "split the families into several batches"
            )
        order = torch.empty(dev.n_pairs, dtype=torch.int32, device=device)
        recs = torch.empty(dev.n_pairs * 16, dtype=torch.uint8, device=device)
        ws = torch.empty(2 * (K + 2), dtype=torch.int32, device=device)
        rc = lib.cherry_sort_pairs_by_bucket(
            _lib.ptr(tab), dev.r_pad, dev.n_pairs, K, _lib.ptr(dev.fams), _lib.ptr(dev.pair_a),
            _lib.ptr(dev.pair_b), _lib.ptr(dev.pair_fam), _lib.ptr(order), _lib.ptr(recs), _lib.ptr(ws),
            stream,
        )
        _lib.check(rc, "cherry_sort_pairs_by_bucket")
        rc = lib.cherry_count_co(
            _lib.ptr(dev.msa), _lib.ptr(recs), _lib.ptr(ws), dev.n_pairs, dev.max_row_stride, K, S,
            _lib.ptr(out), stream,
        )
        _lib.check(rc, "cherry_count_co")
    return out


def symmetrize(raw: torch.Tensor, kind: str, K: int, S: int, directed: bool) -> torch.Tensor:
    """fp64 count tensor with the reference's 0.5 / 0.25 weights applied (exact)."""
    lib = _lib.load()
    stream = _lib.current_stream_ptr()
    if kind == "lg":
        out = torch.empty((K, S, S), dtype=torch.float64, device=raw.device)
        rc = lib.cherry_symmetrize_lg(_lib.ptr(raw), K, S, int(directed), _lib.ptr(out), stream)
        _lib.check(rc, "cherry_symmetrize_lg")
    else:
        n = S * S
        out = torch.empty((K, n, n), dtype=torch.float64, device=raw.device)
        rc = lib.cherry_symmetrize_co(_lib.ptr(raw), K, S, int(directed), _lib.ptr(out), stream)
        _lib.check(rc, "cherry_symmetrize_co")
    return out


def count_batch(
    batch: CountBatch,
    quantization_points: Sequence[float],
    num_states: int,
    directed: bool,
    device="cuda",
    process_group=None,
) -> torch.Tensor:
    """Encoded host batch -> symmetrised fp64 count tensor on the device.

    With ``process_group`` (torch.distributed, one process per GPU) each rank passes the
    batch of ITS families; the raw integer histograms are summed with one all-reduce, so
    the result is bit-identical for any number of ranks.
    """
    grid = sorted_grid(quantization_points)
    K = int(grid.size)
    dev = to_device(batch, device)
    validate_residues(dev.msa, num_states)
    grid_dev = torch.from_numpy(grid).to(dev.msa.device)
    raw = count_raw(dev, grid_dev, K, num_states)
    if process_group is not None:
        import torch.distributed as dist

        dist.all_reduce(raw, op=dist.ReduceOp.SUM, group=process_group)
    return symmetrize(raw, batch.kind, K, num_states, directed)


def count_batches_streamed(
    build_batch,
    family_chunks: Sequence[Sequence[str]],
    kind: str,
    quantization_points: Sequence[float],
    num_states: int,
    directed: bool,
    device="cuda",
    process_group=None,
) -> torch.Tensor:
    """Chunks of families through ingest -> H2D -> counting with the ingest of chunk i+1 (host
    threads of the library, the GIL is released during the call) running while chunk i is uploaded
    and counted; ``build_batch(families) -> CountBatch``.  The raw integer histograms of the chunks
    add up exactly, so the result does not depend on the chunking."""
    from concurrent.futures import ThreadPoolExecutor

    grid = sorted_grid(quantization_points)
    K = int(grid.size)
    dev = torch.device(device)
    raw = None
    co_items = 0  # the co histogram has uint32 cells and is accumulated over ALL chunks
    chunks = [c for c in family_chunks if len(c)]
    with ThreadPoolExecutor(max_workers=1) as pool:
        pending = pool.submit(build_batch, chunks[0]) if chunks else None
        for i in range(len(chunks)):
            batch = pending.result()
            pending = pool.submit(build_batch, chunks[i + 1]) if i + 1 < len(chunks) else None
            d = to_device(batch, dev)
            validate_residues(d.msa, num_states)
            if kind == "co" and d.tile_items is not None:
                co_items += int(d.tile_items.sum())
                if co_items > _CO_MAX_ITEMS_PER_LAUNCH:
                    raise _lib.CherryError(
                        f"more than {_CO_MAX_ITEMS_PER_LAUNCH} (pair, contact) items in one call could wrap a "
                        "uint32 cell of the co-transition histogram; count the families in several calls")
            grid_dev = torch.from_numpy(grid).to(d.msa.device)
            raw = count_raw(d, grid_dev, K, num_states, out=raw)
            torch.cuda.synchronize(d.msa.device)  # the host batch (pooled pinned buffer) may be reused now
            del batch, d
    if raw is None:
        n = num_states if kind == "lg" else num_states * num_states
        raw = torch.zeros((K, n, n), dtype=torch.int64 if kind == "lg" else torch.int32, device=dev)
    if process_group is not None:
        import torch.distributed as dist

        dist.all_reduce(raw, op=dist.ReduceOp.SUM, group=process_group)
    return symmetrize(raw, kind, K, num_states, directed)


def count_lg_host(batch: CountBatch, quantization_points: Sequence[float], num_states: int,
                  directed: bool):
    """End-to-end LG counting from HOST buffers through ``cherry_count_lg_host``.

    ``batch`` arrays may be numpy arrays or (pinned) CPU torch tensors viewed as numpy.
    Returns ``(counts fp64 [K,S,S] numpy, h2d_bytes, d2h_bytes)``.  The copies, the kernels
    and the read-back all happen inside the call.
    """
    import ctypes

    if batch.kind != "lg":
        raise ValueError("count_lg_host takes an LG batch")
    lib = _lib.load()
    grid = sorted_grid(quantization_points)
    K, S = int(grid.size), int(num_states)
    out = np.empty((K, S, S), dtype=np.float64)
    h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
    rc = lib.cherry_count_lg_host(
        _lib.ptr(batch.msa), int(batch.msa.size), _lib.ptr(batch.fams), int(batch.fams.shape[0]),
        _lib.ptr(batch.pair_a), _lib.ptr(batch.pair_b), _lib.ptr(batch.pair_t), int(batch.pair_a.shape[0]),
        _lib.ptr(batch.rate_vals), int(batch.rate_vals.shape[0]),
        _lib.ptr(batch.aux), int(batch.aux.shape[0]), _lib.ptr(batch.tiles), int(batch.tiles.shape[0]),
        _lib.ptr(grid), K, S, int(batch.r_pad), int(directed), _lib.ptr(out),
        ctypes.addressof(h2d), ctypes.addressof(d2h),
    )
    _lib.check(rc, "cherry_count_lg_host")
    return out, int(h2d.value), int(d2h.value)
