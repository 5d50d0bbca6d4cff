"""Device-resident sparse graphs: the handle that replaces the reference's torch sparse COO tensor.

``DeviceCSR`` is what ``TorchGraphInterface.convert_sparse_mat_to_tensor`` (reference
``base/torch_interface.py:8-12``) returns in this package: CSR arrays in HBM (int64 row offsets,
int32 columns, fp32 values) plus the split plan for power-law rows that ``hgr_spmm_f32`` consumes,
and (lazily) the CSR of the transpose for the backward pass.  It still quacks like the tensor the
encoders held: ``.shape``, ``._nnz()``, ``.t()``.

Layout in HBM (per matrix): ``indptr`` 8 B x (rows + 1), ``indices`` 4 B x nnz, ``values`` 4 B x nnz,
plan arrays 4 B x (heavy rows + chunks) + 8 B x (heavy rows + 1).  The normalised bipartite adjacency
is bit-exactly symmetric (SURVEY.md section 9.5), so its transpose is the same object and the backward
pass re-reads the same arrays.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

_N_SM_DEFAULT = 148


def _n_sm(device) -> int:
    if torch.cuda.is_available() and torch.device(device).type == "cuda":
        return torch.cuda.get_device_properties(device).multi_processor_count
    return _N_SM_DEFAULT


def default_chunk_nnz(nnz: int, n_sm: int = _N_SM_DEFAULT, n_cols: int = 0) -> int:
    """Chunk length for splitting long rows: a power of two in [64, 1024] that leaves every SM about
    128 chunks' worth of nonzeros, so small L2-resident graphs keep a short critical path and the
    1 B-interaction graph keeps the partial-row traffic below 0.1 % of the gather traffic.  The wider the gathered table, the
    more of it a chunk of a long row spans (columns ascend inside a row): above 2 M / 6 M table rows the cap drops to 512 / 256
    so that a chunk stays near one L2 window (measured on the blocks of the 2- and 8-GPU graphs, profiles/spmm_r2.md section 5)."""
    t = max(1, nnz // (n_sm * 128))
    t = 1 << (t.bit_length() - 1)
    cap = 1024 if n_cols <= 2_000_000 else (512 if n_cols <= 6_000_000 else 256)
    return int(min(cap, max(64, t)))


def split_plan(indptr: np.ndarray, chunk_nnz: int):
    """Host-side plan: rows longer than ``chunk_nnz`` and their chunk ranges (see hgr_csr_t)."""
    deg = np.diff(indptr)
    heavy = np.nonzero(deg > chunk_nnz)[0].astype(np.int32)
    per = (deg[heavy] + chunk_nnz - 1) // chunk_nnz
    ptr = np.zeros(heavy.size + 1, dtype=np.int64)
    np.cumsum(per, out=ptr[1:])
    owner = np.repeat(np.arange(heavy.size, dtype=np.int32), per)
    return heavy, ptr, owner


def window_split_plan_host(indptr: np.ndarray, indices: np.ndarray, window_shift: int, min_seg: int, max_seg: int, min_span: int = 0):
    """The rule of ``hgr_window_split_count / _fill`` (csrc/split_plan.cu) restated with python loops: the checker of the
    device plan in the tests.  Returns ``(heavy_rows int32, heavy_chunk_ptr int64, chunk_owner int32, chunk_start int64)``."""
    heavy, ptr, owner, start = [], [0], [], []
    for r in range(indptr.size - 1):
        s, e = int(indptr[r]), int(indptr[r + 1])
        cuts = [s]
        windows = e > s and (int(indices[e - 1]) >> window_shift) - (int(indices[s]) >> window_shift) >= min_span
        for j in range(s + 1, e):
            ln = j - cuts[-1]
            if ln >= max_seg or (windows and (int(indices[j]) >> window_shift) != (int(indices[j - 1]) >> window_shift) and ln >= min_seg):
                cuts.append(j)
        if len(cuts) > 1:
            owner += [len(heavy)] * len(cuts)
            heavy.append(r)
            start += cuts
            ptr.append(ptr[-1] + len(cuts))
    return (np.asarray(heavy, dtype=np.int32), np.asarray(ptr, dtype=np.int64), np.asarray(owner, dtype=np.int32),
            np.asarray(start, dtype=np.int64))


def window_split_plan(indptr: torch.Tensor, indices: torch.Tensor, window_shift: int, min_seg: int, max_seg: int, min_span: int = 0):
    """Window-aligned split plan on the device (include/hgr.h: hgr_window_split_count / _fill): a row is cut where it leaves a
    window of ``2 ** window_shift`` rows of the gathered table once the chunk holds ``min_seg`` nonzeros, and every ``max_seg``
    nonzeros at the latest; rows whose columns span fewer than ``min_span`` windows are only cut by the cap.  Returns device tensors ``(heavy_rows, heavy_chunk_ptr, chunk_owner, chunk_start)``."""
    if indptr.dtype != torch.int64 or indices.dtype != torch.int32 or not (indptr.is_cuda and indices.is_cuda):
        raise TypeError("window_split_plan wants CUDA tensors: int64 indptr, int32 indices")
    indptr, indices = indptr.contiguous(), indices.contiguous()
    lib = _lib.lib()
    dev = indptr.device
    n_rows = int(indptr.numel()) - 1
    with torch.cuda.device(dev):
        st = _lib.stream_ptr()
        n_seg = torch.ones(max(n_rows, 1), dtype=torch.int32, device=dev)
        _lib.check(lib.hgr_window_split_count(indptr.data_ptr(), indices.data_ptr(), n_rows, int(window_shift), int(min_seg), int(max_seg),
                                              int(min_span), n_seg.data_ptr(), st))
        n_seg = n_seg[:n_rows]
        heavy = torch.nonzero(n_seg > 1).flatten().to(torch.int32)
        per = n_seg[heavy.long()].to(torch.int64)
        ptr = torch.zeros(heavy.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(per, 0, out=ptr[1:])
        owner = torch.repeat_interleave(torch.arange(heavy.numel(), dtype=torch.int32, device=dev), per)
        start = torch.empty(int(owner.numel()), dtype=torch.int64, device=dev)
        _lib.check(lib.hgr_window_split_fill(indptr.data_ptr(), indices.data_ptr(), heavy.data_ptr(), ptr.data_ptr(), int(heavy.numel()),
                                             int(window_shift), int(min_seg), int(max_seg), int(min_span), start.data_ptr(), st))
    return heavy, ptr, owner, start


_SPLIT_WINDOW_SHIFT = 17  # 2^17 rows = 32 MB of a D = 64 table
_SPLIT_MIN_SEG = 128
_SPLIT_MIN_SPAN = 3  # windows between a row's first and last column before window crossings cut it (> 64 MB of table)


_RUN = 32  # work-list entries that stay together: a whole thread block for every supported width (8 / 16 / 32 row groups)


_WINDOW_ROWS = 1 << 17  # 32 MB of a D = 64 table


def _work_items(indptr, heavy_rows, n_chunks, chunk_nnz, heavy_chunk_ptr, chunk_owner, chunk_start):
    """What every schedule orders: the chunk entries (``~c``) with the first nonzero and length of each chunk, the non-empty whole
    rows (ascending) with their lengths, and the empty rows (ascending)."""
    dev = indptr.device
    n_rows = indptr.numel() - 1
    deg = indptr[1:] - indptr[:-1]
    light = torch.ones(n_rows, dtype=torch.bool, device=dev)
    if heavy_rows.numel():
        light[heavy_rows.long()] = False
    rows = torch.nonzero(light & (deg > 0)).flatten()
    empty = torch.nonzero(light & (deg == 0)).flatten()
    c_ids = ~torch.arange(n_chunks, dtype=torch.int32, device=dev)
    if n_chunks:
        own = chunk_owner.long()
        row_end = indptr[heavy_rows.long()[own] + 1]
        if chunk_start is not None:
            c_start = chunk_start
            last = torch.arange(1, n_chunks + 1, device=dev) == heavy_chunk_ptr[own + 1]
            c_len = torch.where(last, row_end, torch.cat([chunk_start[1:], chunk_start[:1]])) - c_start
        else:
            c_start = indptr[heavy_rows.long()[own]] + (torch.arange(n_chunks, device=dev) - heavy_chunk_ptr[own]) * chunk_nnz
            c_len = torch.clamp(row_end - c_start, max=chunk_nnz)
    else:
        c_start = c_len = torch.empty(0, dtype=torch.long, device=dev)
    return c_ids, c_start, c_len, rows, deg[rows], empty


def _windowed_schedule(indptr, indices, items, window_rows):
    """Work items ordered by the table window their FIRST column falls in; inside a window chunks before rows, rows by
    descending length.  Columns ascend inside a row, so the chunks of all long rows walk the gathered table front to back
    together: a window of embedding rows is fetched from DRAM once and then served from L2 to every long row that
    references it (popular users sit in most popular items' rows), instead of once per row."""
    c_ids, c_start, c_len, rows, r_len, empty = items
    c_first = indices[c_start].long() // window_rows
    r_first = indices[indptr[rows]].long() // window_rows
    big = int(indptr[-1]) + 2  # longer than any row or chunk
    # sort key: window, then descending length (a full chunk is never shorter than a whole row of the same plan, so chunks
    # lead; the groups of a block and the two half-warps of a warp get work of nearly the same length)
    key_c = c_first * (2 * big) + (big - c_len)
    key_r = r_first * (2 * big) + 1 + (big - r_len)
    ids = torch.cat([c_ids, rows.to(torch.int32)])
    order = torch.sort(torch.cat([key_c, key_r]), stable=True).indices
    return torch.cat([ids[order], empty.to(torch.int32)]).contiguous()


def _spread_schedule(indptr, indices, items, window_rows):
    """The windowed order for the chunks, with the whole rows SPREAD evenly through it instead of sitting in the window of their
    first column.  For a row-partitioned block whose propagation publishes every finished row to all ranks (fused all-gather):
    the whole rows are most of the output rows, and in the windowed order they all run in the first windows (every user row starts
    in rank 0's item range), so the exchange is squeezed into the first half of the kernel and stalls it.  Here runs of ``_RUN``
    rows of equal length (a whole thread block) are shuffled with a fixed seed and merged with the chunk runs in proportion to
    their nonzeros: finished rows -- and the NVLink traffic they cause -- leave at a steady rate from the first block to the last."""
    c_ids, c_start, c_len, rows, r_len, empty = items
    if c_ids.numel() == 0 or rows.numel() == 0:
        return _windowed_schedule(indptr, indices, items, window_rows)
    dev = indptr.device
    # chunks: window of the first column, then descending length
    big = int(indptr[-1]) + 2  # longer than any chunk
    c_order = torch.sort((indices[c_start].long() // window_rows) * big + (big - c_len), stable=True).indices
    c_ids, c_len = c_ids[c_order], c_len[c_order]
    # rows: runs of equal length, shuffled
    r_order = torch.sort(r_len, descending=True, stable=True).indices
    n_runs = -(-int(rows.numel()) // _RUN)
    gen = torch.Generator()
    gen.manual_seed(0x5eed)
    run_pos = torch.empty(n_runs, dtype=torch.long)
    run_pos[torch.randperm(n_runs, generator=gen)] = torch.arange(n_runs)
    slot = run_pos.to(dev)[torch.arange(rows.numel(), device=dev) // _RUN] * _RUN + torch.arange(rows.numel(), device=dev) % _RUN
    r_order = r_order[torch.sort(slot).indices]
    rows, r_len = rows[r_order], r_len[r_order]

    def run_keys(lengths):  # fraction of the list's nonzeros that precede the run an entry belongs to
        n = lengths.numel()
        before = torch.cumsum(lengths, 0) - lengths
        first = before[torch.arange(0, n, _RUN, device=dev)]
        return first.to(torch.float64)[torch.arange(n, device=dev) // _RUN] / max(float(lengths.sum()), 1.0)

    merged = torch.sort(torch.cat([run_keys(c_len), run_keys(r_len)]), stable=True).indices  # ties: the chunk run first
    return torch.cat([torch.cat([c_ids, rows.to(torch.int32)])[merged], empty.to(torch.int32)]).contiguous()


def work_schedule(indptr: torch.Tensor, heavy_rows: torch.Tensor, n_chunks: int, chunk_nnz: int, mode: str,
                  indices: torch.Tensor | None = None, heavy_chunk_ptr: torch.Tensor | None = None,
                  chunk_owner: torch.Tensor | None = None, n_cols: int = 0, chunk_start: torch.Tensor | None = None) -> torch.Tensor:
    """The ``hgr_csr_t::work_order`` list (int32, device): which row or chunk every row group of the propagation kernel takes.

    ``binned``       chunk entries first, then the unsplit rows by descending length (stable): the two half-warps of a
                     warp and the groups of a block get rows of (nearly) the same length and retire together, and the
                     longest rows start first, so the grid has no long-row tail.
    ``windowed[:W]`` items ordered by the W-row window of the gathered table their first column falls in (``_windowed_schedule``).
    ``spread[:W]``   the windowed order for the chunks, whole rows spread evenly through it (``_spread_schedule``): the schedule of a
                     row-partitioned block whose kernel publishes its rows to many ranks.
    ``auto``         ``windowed`` when the gathered table is larger than 64 MB, else ``binned`` (the default).

    Measured on B200 (profiles/spmm_r2.md), 1.25 M x 0.25 M x 125 M graph, one launch: rows in stored order without a list
    6.27 ms, binned 4.71 - 5.01, windowed 4.13 - 4.20.
    Only the schedule changes: each row is accumulated by one row group in stored order, so results are bit-identical."""
    if mode == "auto":
        # a table that fits L2 (<= 64 MB of 256-byte rows) needs no windows: pure length binning measured 10 % faster there
        mode = "windowed" if n_cols * 256 > (64 << 20) else "binned"
    name, _, window = mode.partition(":")
    if name not in ("binned", "windowed", "spread") or (name == "binned" and window):
        raise ValueError("unknown propagation schedule %r (auto | binned | windowed[:W] | spread[:W])" % (mode,))
    items = _work_items(indptr, heavy_rows, n_chunks, chunk_nnz, heavy_chunk_ptr, chunk_owner, chunk_start)
    if name == "binned":
        c_ids, _, _, rows, r_len, empty = items
        order = torch.sort(r_len, descending=True, stable=True).indices
        return torch.cat([c_ids, rows[order].to(torch.int32), empty.to(torch.int32)]).contiguous()
    schedule = _spread_schedule if name == "spread" else _windowed_schedule
    return schedule(indptr, indices, items, int(window) if window else _WINDOW_ROWS)


class DeviceCSR:
    """CSR matrix in device memory + split plan + work schedule + ctypes descriptor (``hgr_csr_t``)."""

    def __init__(self, indptr: torch.Tensor, indices: torch.Tensor, values: torch.Tensor, shape, symmetric: bool = False,
                 chunk_nnz: int | None = None, transpose: "DeviceCSR | None" = None, split: str = "auto"):
        if indptr.dtype != torch.int64 or indices.dtype != torch.int32 or values.dtype != torch.float32:
            raise TypeError("DeviceCSR wants int64 indptr, int32 indices, float32 values")
        if not (indptr.is_cuda and indices.is_cuda and values.is_cuda):
            raise _lib.HgrError("DeviceCSR arrays must live on a CUDA device (there is no CPU path)")
        self.indptr, self.indices, self.values = indptr.contiguous(), indices.contiguous(), values.contiguous()
        self.shape = (int(shape[0]), int(shape[1]))
        self.device = indptr.device
        self.symmetric = bool(symmetric) and self.shape[0] == self.shape[1]
        self._t = transpose
        self._ws = {}
        nnz = int(self.indices.numel())
        self.chunk_nnz = int(chunk_nnz) if chunk_nnz else default_chunk_nnz(nnz, _n_sm(self.device), self.shape[1])
        # How long rows are cut.  "fixed": every chunk_nnz nonzeros.  "window[:shift[:min_seg[:min_span]]]": where the row leaves a window of
        # 2^shift rows of the gathered table (window_split_plan), at most chunk_nnz nonzeros per chunk.  "auto": windows when the
        # gathered table cannot stay in L2 (> 64 MB of 256-byte rows) and the caller did not fix chunk_nnz, else fixed.
        if split == "auto":
            split = "window" if (self.shape[1] * 256 > (64 << 20) and not chunk_nnz and nnz > 0) else "fixed"
        self.split = split
        dev = self.device
        self.chunk_start = None
        if split.startswith("window"):
            f = split.split(":")
            shift = int(f[1]) if len(f) > 1 else _SPLIT_WINDOW_SHIFT
            min_seg = int(f[2]) if len(f) > 2 else _SPLIT_MIN_SEG
            min_span = int(f[3]) if len(f) > 3 else _SPLIT_MIN_SPAN
            self.heavy_rows, self.heavy_chunk_ptr, self.chunk_owner, self.chunk_start = window_split_plan(
                self.indptr, self.indices, shift, min_seg, max(self.chunk_nnz, min_seg), min_span)
        elif split == "fixed":
            heavy, ptr, owner = split_plan(self.indptr.cpu().numpy(), self.chunk_nnz)
            self.heavy_rows = torch.from_numpy(heavy).to(dev)
            self.heavy_chunk_ptr = torch.from_numpy(ptr).to(dev)
            self.chunk_owner = torch.from_numpy(owner).to(dev)
        else:
            raise ValueError("unknown split plan %r (fixed | window[:shift[:min_seg]] | auto)" % (split,))
        d = _lib.CsrDesc()
        d.n_rows, d.n_cols, d.nnz = self.shape[0], self.shape[1], nnz
        d.indptr, d.indices, d.values = self.indptr.data_ptr(), self.indices.data_ptr(), self.values.data_ptr()
        d.chunk_nnz, d.n_heavy_rows, d.n_chunks = self.chunk_nnz, int(self.heavy_rows.numel()), int(self.chunk_owner.numel())
        d.heavy_rows, d.heavy_chunk_ptr, d.chunk_owner = (self.heavy_rows.data_ptr(), self.heavy_chunk_ptr.data_ptr(),
                                                          self.chunk_owner.data_ptr())
        d.chunk_start = None if self.chunk_start is None or d.n_chunks == 0 else self.chunk_start.data_ptr()
        self.desc = d
        self.set_schedule("auto")

    def set_schedule(self, mode: str) -> "DeviceCSR":
        """Choose how the propagation kernel's row groups are handed rows and chunks (``work_schedule``); results do not change."""
        self.schedule = mode
        self.work_order = work_schedule(self.indptr, self.heavy_rows, int(self.desc.n_chunks), self.chunk_nnz, mode, self.indices,
                                        self.heavy_chunk_ptr, self.chunk_owner, self.shape[1],
                                        self.chunk_start if self.desc.chunk_start else None)
        self.desc.work_order = self.work_order.data_ptr()
        self.desc.n_work = int(self.work_order.numel())
        return self

    # ---- what the reference's encoders touch on the sparse tensor -------------------------------
    def _nnz(self) -> int:
        return int(self.indices.numel())

    is_sparse = True  # what `adj.is_sparse` answered for the COO tensor this handle replaces

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        """The reference's encoders call ``torch.sparse.mm(self.sparse_norm_adj, x)`` themselves (model/graph/LightGCN.py:133,
        HCCF.py:199, SGL.py:156-160 ...).  With a ``DeviceCSR`` as the first operand torch hands the call over to this hook, and
        the product runs on ``hgr_spmm_f32`` with its hand-written backward (``ops.spmm``) -- the unmodified encoder source keeps
        working.  Anything else torch might do with the handle is refused loudly."""
        import torch as _t

        name = getattr(func, "__name__", "")
        if name in ("_sparse_mm", "mm", "matmul", "spmm") and len(args) == 2 and isinstance(args[0], DeviceCSR) and isinstance(args[1], _t.Tensor):
            from . import ops

            return ops.spmm(args[0], args[1])
        raise _lib.HgrError("torch.%s is not supported on a DeviceCSR (only adj @ dense: torch.sparse.mm / torch.mm / torch.matmul)" % name)

    def _indices(self) -> torch.Tensor:
        """COO coordinates ``[2, nnz]`` int64, row-major -- what ``sparse_tensor._indices()`` gave the reference (LightGCN.py:118
        builds an unused all-ones copy from it).  Returned on the HOST: the legacy ``torch.sparse.FloatTensor(i, v, shape)``
        constructor those lines use only takes CPU tensors."""
        rows = torch.repeat_interleave(torch.arange(self.shape[0], device=self.device, dtype=torch.int64), self.indptr[1:] - self.indptr[:-1])
        return torch.stack([rows, self.indices.to(torch.int64)]).cpu()

    def _values(self) -> torch.Tensor:
        return self.values.cpu()

    def t(self) -> "DeviceCSR":
        if self.symmetric:
            return self
        if self._t is None:
            self._t = transpose_csr(self)
            self._t._t = self
        return self._t

    # ---- same sparsity pattern, other values (edge dropout) ---------------------------------------
    def transpose_permutation(self) -> torch.Tensor:
        """For a structurally symmetric matrix: ``tperm[p]`` = position of entry (c, r) for the p-th entry (r, c).
        Computed once (one sort-free ``searchsorted`` over the canonical keys) and cached."""
        tp = getattr(self, "_tperm", None)
        if tp is None:
            n = self.shape[1]
            rows = torch.repeat_interleave(torch.arange(self.shape[0], device=self.device, dtype=torch.int64),
                                           self.indptr[1:] - self.indptr[:-1])
            cols = self.indices.to(torch.int64)
            tp = torch.searchsorted(rows * n + cols, cols * n + rows)
            if self.shape[0] != self.shape[1] or not bool((self.indices[tp.clamp(max=max(cols.numel() - 1, 0))] == rows.to(torch.int32)).all()):
                raise ValueError("transpose_permutation needs a structurally symmetric matrix with sorted columns")
            self._tperm = tp
        return tp

    def with_values(self, values: torch.Tensor, t_values: torch.Tensor | None = None) -> "DeviceCSR":
        """A matrix with THIS sparsity pattern (and split plan) and other values; ``t_values`` are the values of its
        transpose in this same pattern (structurally symmetric matrices: ``values[transpose_permutation()]``).
        No host work, no synchronisation: explicit zeros stand in for dropped entries, which leaves every sum
        bit-identical to the compacted matrix (fma(0, x, acc) == acc)."""
        import copy

        out = copy.copy(self)
        out.values = values.contiguous()
        out.symmetric = False
        d = _lib.CsrDesc.from_buffer_copy(self.desc)
        d.values = out.values.data_ptr()
        out.desc = d
        out._tperm = getattr(self, "_tperm", None)
        out._t = None
        if t_values is not None:
            t = copy.copy(self)
            t.values = t_values.contiguous()
            t.symmetric = False
            td = _lib.CsrDesc.from_buffer_copy(self.desc)
            td.values = t.values.data_ptr()
            t.desc = td
            t._t, out._t = out, t
        return out

    def to(self, *a, **k):  # `.to(device)` / `.cuda()` on an already-resident handle are no-ops
        return self

    cuda = to

    # ---- construction --------------------------------------------------------------------------
    @classmethod
    def from_host(cls, indptr, indices, values, shape, device="cuda", **kw) -> "DeviceCSR":
        dev = torch.device(device)
        return cls(torch.as_tensor(np.ascontiguousarray(indptr, dtype=np.int64)).to(dev),
                   torch.as_tensor(np.ascontiguousarray(indices, dtype=np.int32)).to(dev),
                   torch.as_tensor(np.ascontiguousarray(values, dtype=np.float32)).to(dev), shape, **kw)

    @classmethod
    def from_scipy(cls, mat, device="cuda", symmetric: bool | None = None, **kw) -> "DeviceCSR":
        m = mat.tocsr()
        if not m.has_sorted_indices:
            m = m.copy()
            m.sort_indices()
        if symmetric is None:
            symmetric = m.shape[0] == m.shape[1] and (m != m.T).nnz == 0
        return cls.from_host(m.indptr, m.indices, m.data, m.shape, device=device, symmetric=symmetric, **kw)

    def workspace(self, d: int) -> torch.Tensor | None:
        """Partial-row buffer for the split plan ([n_chunks, D] fp32), cached per D."""
        need = int(self.desc.n_chunks) * d if self.desc.n_heavy_rows > 0 else 0
        if need == 0:
            return None
        ws = self._ws.get(d)
        if ws is None:
            ws = torch.empty(need, dtype=torch.float32, device=self.device)
            self._ws[d] = ws
        return ws

    def to_host(self, drop_zeros: bool = False):
        """``(indptr, indices, values)`` as numpy arrays; ``drop_zeros`` removes the explicit zeros an edge-dropped
        matrix carries (``with_values``), giving the compacted CSR the reference builds."""
        ip, ix, dv = self.indptr.cpu().numpy(), self.indices.cpu().numpy(), self.values.cpu().numpy()
        if drop_zeros:
            keep = dv != 0
            rows = np.repeat(np.arange(ip.size - 1), np.diff(ip))[keep]
            ip = np.zeros_like(ip)
            np.cumsum(np.bincount(rows, minlength=ip.size - 1), out=ip[1:])
            ix, dv = ix[keep], dv[keep]
        return ip, ix, dv


def transpose_csr(a: DeviceCSR) -> DeviceCSR:
    """CSR of A^T (needed when A is not symmetric: edge-dropped or rectangular matrices).  A stable
    sort by column keeps rows ascending inside every transposed row."""
    n_rows, n_cols = a.shape
    rows = torch.repeat_interleave(torch.arange(n_rows, device=a.device, dtype=torch.int32), a.indptr[1:] - a.indptr[:-1])
    order = torch.sort(a.indices, stable=True).indices
    counts = torch.bincount(a.indices, minlength=n_cols)
    indptr = torch.zeros(n_cols + 1, dtype=torch.int64, device=a.device)
    torch.cumsum(counts, 0, out=indptr[1:])
    return DeviceCSR(indptr, rows[order].contiguous(), a.values[order].contiguous(), (n_cols, n_rows),
                     chunk_nnz=a.chunk_nnz, split=a.split)


# ------------------------------------------------------------------------------------------------
# Device builders (csrc/graph_build.cu) -- replace the scipy / python-list path of the reference's
# data layer: data/ui_graph.py:70-84,95-112 and data/graph.py:11-25.
# ------------------------------------------------------------------------------------------------
def host_pow_lut(n: int, exponent: float) -> np.ndarray:
    """``np.power(arange(n, float32), exponent)`` with inf -> 0, computed on THIS host: the reference's
    normalisation values are whatever numpy's (not correctly rounded) float32 pow returns here
    (data/graph.py:15-16,21-22; SURVEY.md F10)."""
    with np.errstate(divide="ignore"):
        lut = np.power(np.arange(n, dtype=np.float32), np.float32(exponent))
    lut[np.isinf(lut)] = 0.0
    return lut.astype(np.float32)


def _as_i32(x, device) -> torch.Tensor:
    t = torch.as_tensor(x)
    return t.to(device=device, dtype=torch.int32).contiguous()


def _build(kind: str, a: torch.Tensor, b: torch.Tensor, n_rows: int, n_cols: int, n_users: int = 0, n_items: int = 0):
    dev = a.device
    if dev.type != "cuda":
        raise _lib.HgrError("graph construction runs on the GPU (no CPU path)")
    n_in = int(a.numel())
    n_sorted = 2 * n_in if kind == "bipartite" else n_in
    lib = _lib.lib()
    ws_bytes = int(lib.hgr_build_csr_workspace_bytes(n_sorted))
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
    off = (-ws.data_ptr()) % 256
    indptr = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
    indices = torch.empty(max(n_sorted, 1), dtype=torch.int32, device=dev)
    values = torch.empty(max(n_sorted, 1), dtype=torch.float32, device=dev)
    row_entries = torch.empty(max(n_rows, 1), dtype=torch.int32, device=dev)
    nnz = torch.zeros(1, dtype=torch.int64, device=dev)
    st = _lib.stream_ptr()
    if kind == "bipartite":
        rc = lib.hgr_bipartite_to_csr(a.data_ptr(), b.data_ptr(), n_in, n_users, n_items, indptr.data_ptr(), indices.data_ptr(),
                                      values.data_ptr(), row_entries.data_ptr(), nnz.data_ptr(), ws.data_ptr() + off, ws_bytes, st)
    else:
        rc = lib.hgr_coo_to_csr(a.data_ptr(), b.data_ptr(), n_in, n_rows, n_cols, indptr.data_ptr(), indices.data_ptr(),
                                values.data_ptr(), row_entries.data_ptr(), nnz.data_ptr(), ws.data_ptr() + off, ws_bytes, st)
    _lib.check(rc)
    n = int(nnz.item())  # the one synchronisation of the build: the output size
    del ws
    return indptr, indices[:n].clone(), values[:n].clone(), row_entries[:n_rows]


def _scale(indptr, indices, values, n_rows, row_scale, col_scale):
    _lib.check(_lib.lib().hgr_csr_scale(indptr.data_ptr(), indices.data_ptr(), values.data_ptr(), n_rows, _lib.ptr(row_scale),
                                        _lib.ptr(col_scale), _lib.stream_ptr()))


def _degree_scale(deg: torch.Tensor, exponent: float) -> torch.Tensor:
    max_deg = int(deg.max().item()) if deg.numel() else 0
    lut = torch.from_numpy(host_pow_lut(max_deg + 1, exponent)).to(deg.device)
    out = torch.empty(deg.numel(), dtype=torch.float32, device=deg.device)
    over = torch.zeros(1, dtype=torch.int32, device=deg.device)
    _lib.check(_lib.lib().hgr_degree_scale(deg.data_ptr(), deg.numel(), lut.data_ptr(), lut.numel(), out.data_ptr(), over.data_ptr(),
                                           _lib.stream_ptr()))
    if int(over.item()) != 0:
        raise _lib.HgrError("degree outside the normalisation table")
    return out


def build_norm_adj(user_idx, item_idx, n_users: int, n_items: int, device="cuda", chunk_nnz=None, normalize: bool = True) -> DeviceCSR:
    """``Interaction.norm_adj`` built on the device: the (U+I)^2 bipartite adjacency of the dense
    interaction list (duplicates summed) with ``(D^-1/2 A) D^-1/2`` values, bit-identical to
    ``Graph.normalize_graph_mat(Interaction.ui_adj)`` (data/graph.py:11-19).  ``normalize=False`` returns
    ``ui_adj`` itself (data/ui_graph.py:70-84)."""
    dev = torch.device(device)
    u, i = _as_i32(user_idx, dev), _as_i32(item_idx, dev)
    n = n_users + n_items
    indptr, indices, values, deg = _build("bipartite", u, i, n, n, n_users, n_items)
    if normalize:
        d = _degree_scale(deg, -0.5)
        _scale(indptr, indices, values, n, d, d)
    out = DeviceCSR(indptr, indices, values, (n, n), symmetric=True, chunk_nnz=chunk_nnz)
    out.degree = deg
    return out


def build_interaction_csr(user_idx, item_idx, n_users: int, n_items: int, device="cuda", transpose: bool = False,
                          row_normalize: bool = False, chunk_nnz=None) -> DeviceCSR:
    """``Interaction.interaction_mat`` (``transpose``: ``inv_interaction_mat``), data/ui_graph.py:95-112;
    ``row_normalize`` applies the rectangular branch ``D^-1 R`` of ``normalize_graph_mat`` (data/graph.py:20-24).
    Also the training-item mask of full-ranking evaluation (user -> sorted train items)."""
    dev = torch.device(device)
    u, i = _as_i32(user_idx, dev), _as_i32(item_idx, dev)
    (r, c, nr, nc) = (i, u, n_items, n_users) if transpose else (u, i, n_users, n_items)
    indptr, indices, values, deg = _build("coo", r, c, nr, nc)
    if row_normalize:
        _scale(indptr, indices, values, nr, _degree_scale(deg, -1.0), None)
    out = DeviceCSR(indptr, indices, values, (nr, nc), chunk_nnz=chunk_nnz)
    out.degree = deg
    return out


# ------------------------------------------------------------------------------------------------
# Hypergraph incidence for the scatter form of ED-HNN message passing
# (model/layers/layers2/EquivSetConv2.py:85-100, EquivSetGNN2.py:105-133, HCCF_diffusion.py:291-308,382-402)
# ------------------------------------------------------------------------------------------------
class Incidence:
    """Row-normalised incidence pair of a hypergraph given as (vertex, hyperedge) pairs:
    ``to_edges = De^-1 H^T`` ([n_edges, n_nodes]) and ``to_nodes = Dv^-1 H`` ([n_nodes, n_edges]).
    ``to_edges @ X`` is ``torch_scatter.scatter(X[V], E, reduce='mean')`` and ``to_nodes @ Xe`` is
    ``scatter(Xe[E], V, reduce='mean', dim_size=n_nodes)``: an empty segment gives a zero row, exactly
    pytorch-scatter's ``sum / clamp(count, 1)``.  Built once; the reference re-derives (V, E) with
    ``torch.nonzero(H > 0)`` on a dense matrix every forward."""

    def __init__(self, to_edges: DeviceCSR, to_nodes: DeviceCSR):
        self.to_edges, self.to_nodes = to_edges, to_nodes
        self.n_edges, self.n_nodes = to_edges.shape


def _csr_keys(m: DeviceCSR) -> torch.Tensor:
    rows = torch.repeat_interleave(torch.arange(m.shape[0], device=m.device, dtype=torch.int64), m.indptr[1:] - m.indptr[:-1])
    return rows * m.shape[1] + m.indices.to(torch.int64)


def pair_positions(inc: Incidence, vertex, edges):
    """Where each (vertex, hyperedge) pair sits in ``inc.to_edges`` and in ``inc.to_nodes`` (both canonical CSR): the maps that
    let a per-pair weight vector (HD2's attention, model/graph/HD2.py:630-632) become CSR values.  Pairs must be unique."""
    dev = inc.to_edges.device
    v = torch.as_tensor(vertex).to(dev, torch.int64)
    e = torch.as_tensor(edges).to(dev, torch.int64)
    pos_e = torch.searchsorted(_csr_keys(inc.to_edges), e * inc.n_nodes + v)
    pos_n = torch.searchsorted(_csr_keys(inc.to_nodes), v * inc.n_edges + e)
    return pos_e, pos_n


def incidence_from_csr(h: DeviceCSR) -> Incidence:
    """The star expansion HGNN_HD4 feeds to EquivSetGNN2 (model/graph/HGNN_HD4.py:389,397; EquivSetGNN2.py:105-133):
    ``(V, E) = nonzero(dense(H) > 0)`` of a matrix that is already sparse on the device -- every stored entry once, whatever
    its multiplicity.  No dense (U+I)^2 copy, no ``nonzero`` per forward."""
    rows = torch.repeat_interleave(torch.arange(h.shape[0], device=h.device, dtype=torch.int32), h.indptr[1:] - h.indptr[:-1])
    keep = h.values > 0
    return build_incidence(rows[keep], h.indices[keep], h.shape[0], h.shape[1], device=h.device)


class HyperNormAdj:
    """``Graph.normalize_graph_mat_hyper`` (data/graph.py:28-42): ``Dv^-1/2 H De^-1 H^T Dv^-1/2`` kept FACTORED,
    ``left = (Dv^-1/2 H) De^-1`` ([n_v, n_e]) and ``right = H^T Dv^-1/2`` ([n_e, n_v]), both ``DeviceCSR`` with scipy's
    roundings.  The reference multiplies the factors out with scipy (a two-hop matrix: nearly dense for a power-law graph);
    here the operator is applied as two propagations, which is also how every encoder uses it."""

    def __init__(self, left: DeviceCSR, right: DeviceCSR):
        self.left, self.right = left, right
        self.shape = (left.shape[0], right.shape[1])
        self.device = left.device

    def matmul(self, x: torch.Tensor) -> torch.Tensor:
        from . import ops

        return ops.spmm(self.left, ops.spmm(self.right, x))

    __matmul__ = matmul

    def t(self):
        return self  # symmetric operator


def normalize_graph_mat_hyper(h: DeviceCSR) -> HyperNormAdj:
    dev = h.device
    n_v, n_e = h.shape
    rows = torch.repeat_interleave(torch.arange(n_v, device=dev), h.indptr[1:] - h.indptr[:-1])
    rowsum = torch.zeros(n_v, dtype=torch.float32, device=dev).index_add_(0, rows, h.values)
    colsum = torch.zeros(n_e, dtype=torch.float32, device=dev).index_add_(0, h.indices.long(), h.values)
    rs, cs = rowsum.to(torch.int32), colsum.to(torch.int32)
    if not (torch.equal(rs.float(), rowsum) and torch.equal(cs.float(), colsum)):
        raise _lib.HgrError("normalize_graph_mat_hyper on the device needs integer row / column sums (unit-weight incidences)")
    dv, de = _degree_scale(rs, -0.5), _degree_scale(cs, -1.0)
    lv = h.values.clone()
    _scale(h.indptr, h.indices, lv, n_v, dv, de)  # (dv[r] * h) * de[c]: scipy's d_v.dot(adj).dot(d_e)
    left = DeviceCSR(h.indptr, h.indices, lv, h.shape, chunk_nnz=h.chunk_nnz, split=h.split)
    ht = h.t()
    rv = ht.values.clone()
    _scale(ht.indptr, ht.indices, rv, n_e, None, dv)  # h * dv[c]: adj.T.dot(d_v)
    right = DeviceCSR(ht.indptr, ht.indices, rv, ht.shape, chunk_nnz=ht.chunk_nnz, split=ht.split)
    return HyperNormAdj(left, right)


def build_incidence(vertex, edges, n_nodes: int, n_edges: int | None = None, device="cuda") -> Incidence:
    dev = torch.device(device)
    v, e = _as_i32(vertex, dev), _as_i32(edges, dev)
    if n_edges is None:
        n_edges = int(e.max().item()) + 1 if e.numel() else 0
    # duplicated (v, e) pairs are summed into a multiplicity, like scatter() visiting the pair twice
    to_nodes = build_interaction_csr(v, e, n_nodes, n_edges, device=dev, row_normalize=True)
    to_edges = build_interaction_csr(v, e, n_nodes, n_edges, device=dev, transpose=True, row_normalize=True)
    return Incidence(to_edges, to_nodes)


def incidence_from_dense(h: torch.Tensor) -> Incidence:
    """``generate_V_E`` (model/layers/layers2/EquivSetGNN2.py:105-133): pairs = ``nonzero(H > 0)``."""
    nz = torch.nonzero(h > 0)
    return build_incidence(nz[:, 0], nz[:, 1], h.shape[0], h.shape[1], device=h.device)
