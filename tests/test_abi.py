"""The C-ABI library loads and exports exactly what include/cherryml_b200.h declares
(no compute calls: runs without a GPU)."""
import os
import re

import pytest

from cherryml_b200 import _lib

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    text = open(os.path.join(REPO, "include", "cherryml_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cherry_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_and_loads():
    from cherryml_b200.csrc.build import build

    build()
    lib = _lib.load()
    assert b"sm_100a" in lib.cherry_version()
    assert lib.cherry_last_error() is not None
    lib.cherry_reset_launch_count()
    assert lib.cherry_launch_count() == 0


def test_every_declared_symbol_is_exported_and_bound():
    lib = _lib.load()
    declared = _declared_functions()
    assert declared, "no declarations parsed from the header"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == _lib.exported_symbols(), "ctypes signatures out of sync with the header"


def test_struct_layouts_match_header():
    assert _lib.FAM_DESC_DTYPE.itemsize == 32
    assert [_lib.FAM_DESC_DTYPE.fields[n][1] for n in
            ("msa_off", "row_stride", "n_chunks", "aux_off", "aux_cnt", "rate_off", "n_rates")] == [
        0, 8, 12, 16, 20, 24, 28]
    assert _lib.TILE_DTYPE.itemsize == 16


def test_argument_validation_without_gpu():
    """Null pointers / bad sizes are rejected before anything touches CUDA."""
    lib = _lib.load()
    assert lib.cherry_count_lg(0, 0, 0, 0, 0, 4, 0, 0, 1, 10, 20, 0, 0) == -1
    assert b"null pointer" in lib.cherry_last_error()
    assert lib.cherry_build_bucket_table_tiles(0, 0, 1, 0, 0, 0, 10, 4, 0, 0) == -1
    assert b"null pointer" in lib.cherry_last_error()
    assert lib.cherry_count_lg_host(0, 16, 0, 1, 0, 0, 0, 1, 0, 4, 0, 1, 0, 1, 0, 10, 20, 4, 0, 0, 0, 0) == -1
    assert b"null pointer" in lib.cherry_last_error()
    with pytest.raises(_lib.CherryError):
        _lib.check(lib.cherry_symmetrize_lg(0, 1, 1, 0, 0, 0), "cherry_symmetrize_lg")


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libcherryml_b200.so")
    with pytest.raises(_lib.CherryError, match="no CPU fallback"):
        _lib.load()


def test_product_package_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under cherryml_b200/ may import it (or read /root/reference)."""
    pkg = os.path.join(REPO, "cherryml_b200")
    offenders = []
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if not fn.endswith(".py"):
                continue
            text = open(os.path.join(dirpath, fn)).read()
            if re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M) or "/root/reference" in text:
                offenders.append(os.path.relpath(os.path.join(dirpath, fn), REPO))
    assert offenders == []


def test_large_fit_sizes_without_gpu():
    """S > 32: the K limit of the header is enforced by the sizing call, and the power-chain work lists of every
    padded size up to 800 fit the workspace carved for them (the sizing call fails otherwise)."""
    import ctypes

    from cherryml_b200.markov_chain import LARGE_MAX_K

    text = open(os.path.join(REPO, "include", "cherryml_b200.h")).read()
    assert int(re.search(r"#define CHERRY_LARGE_FIT_MAX_K (\d+)", text).group(1)) == LARGE_MAX_K
    lib = _lib.load()
    n = ctypes.c_size_t(0)
    for S in list(range(33, 801, 80)) + list(range(80, 801, 80)):
        assert lib.cherry_fit_workspace_bytes(S, 4, 1, ctypes.byref(n)) == 0, (S, lib.cherry_last_error())
        assert n.value > 0
    assert lib.cherry_fit_workspace_bytes(36, LARGE_MAX_K, 1, ctypes.byref(n)) == 0
    assert lib.cherry_fit_workspace_bytes(36, LARGE_MAX_K + 1, 1, ctypes.byref(n)) == -3
    assert b"limit of %d" % LARGE_MAX_K in lib.cherry_last_error()


def test_small_fit_sizes_without_gpu():
    """S <= 32: the sizing call answers for every S, for one and for 400 buckets, one and 331 problems, and the
    answer covers the matrix slots that do not stay in shared memory for every CTA, plus the arrival counters."""
    import ctypes

    lib = _lib.load()
    n = ctypes.c_size_t(0)
    for S in range(1, 33):
        spad = (S + 7) // 8 * 8
        slot_bytes = spad * (spad + 4) * 8
        resident = min(220 * 1024 // slot_bytes, 43, 20 if S <= 24 else 43)  # 9 Taylor + 30 squaring + 4 slots
        for K in (1, 400):
            for P in (1, 331):
                assert lib.cherry_fit_workspace_bytes(S, K, P, ctypes.byref(n)) == 0, (S, K, P, lib.cherry_last_error())
                spill = (43 - resident) * slot_bytes * P * K
                assert n.value >= spill + 4 * P, (S, K, P, n.value)
                assert n.value <= spill + 4 * P + 512, (S, K, P, n.value)
