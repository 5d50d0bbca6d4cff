"""Argument validation of the five producers that publish finished rows into gathered tables (the fused all-gather of
sharded training): the propagation epilogue, the LayerNorm backward, publish_rows, add_rows and the rows x small-matrix
product.  A bad destination list is refused with an error message before anything is launched.  No GPU is needed: every
call below is refused by the host-side checks, and every call also carries a second defect (no work list, an unsupported
width or a NULL operand) that a later check refuses, so no kernel could run even if the gather check were missing."""
import ctypes as C

import pytest

FAKE = 1 << 20  # a 16-byte aligned address that is never dereferenced: every call is refused on the host


@pytest.fixture(scope="module")
def lib():
    from hypergraph_diffusion_for_recommendation_b200 import _lib, build

    build.build()  # nvcc cross-compiles for sm_100a without a GPU
    return _lib


def _bad_gathers(lib):
    """(name, hgr_gather_t) pairs that every producer must refuse.  Built by hand: make_gather cannot hold 9 tables."""
    cases = []

    def g(n_gather, out=(), row_offset=0, mc=None):
        gt = lib.Gather()
        gt.n_gather = n_gather
        for j, p in enumerate(out):
            gt.out[j] = p
        gt.row_offset = row_offset
        gt.mc = mc
        cases.append(gt)
        return gt

    g(9, [FAKE] * lib.HGR_MAX_GATHER)
    g(-1)
    g(1, [None])
    g(1, [FAKE + 4])
    g(3, [FAKE, FAKE + 16, FAKE + 8])  # a misaligned table after two good ones
    g(1, [FAKE], row_offset=-1)
    g(0, mc=FAKE + 8)
    return list(zip(["n_gather=9", "n_gather=-1", "null_table", "misaligned_table", "misaligned_third_table", "negative_row_offset",
                     "misaligned_mc"], cases))


def _no_work_list_desc(lib):
    """A 4 x 4 matrix without nonzeros and without a work list: hgr_spmm_f32 refuses it after all other checks."""
    d = lib.CsrDesc()
    d.n_rows, d.n_cols, d.nnz = 4, 4, 0
    d.indptr = FAKE
    return d


def _spmm_with(lib, gt):
    ep = lib.Epilogue()
    ep.scale = 1.0
    ep.n_gather = gt.n_gather
    for j in range(lib.HGR_MAX_GATHER):
        ep.gather_out[j] = gt.out[j]
    ep.gather_row_offset = gt.row_offset
    ep.gather_mc = gt.mc
    d = _no_work_list_desc(lib)
    return lib.lib().hgr_spmm_f32(C.byref(d), FAKE, FAKE, 64, C.byref(ep), None, 0, None)


def _leaky_ln_bwd_with(lib, gt):  # D = 48 is unsupported
    return lib.lib().hgr_leaky_ln_bwd_gather_f32(FAKE, FAKE, None, 1e-5, 1, 0.3, 4, 48, FAKE, None, None, None, C.byref(gt), None)


def _publish_with(lib, gt):  # x is NULL
    return lib.lib().hgr_publish_rows_f32(None, 4, 64, C.byref(gt), None)


def _add_rows_with(lib, gt):  # a, b and out are NULL
    return lib.lib().hgr_add_rows_f32(None, None, 4, 64, None, C.byref(gt), None)


def _rows_times_small_with(lib, gt):  # A1, B and Y are NULL
    return lib.lib().hgr_rows_times_small_gather_f32(None, 64, None, 0, None, 64, 4, None, None, 0, C.byref(gt), None)


PRODUCERS = {"spmm": _spmm_with, "leaky_ln_bwd": _leaky_ln_bwd_with, "publish_rows": _publish_with, "add_rows": _add_rows_with,
             "rows_times_small": _rows_times_small_with}


@pytest.mark.parametrize("producer", sorted(PRODUCERS))
def test_every_producer_refuses_a_bad_gather_before_launching(lib, producer):
    handle = lib.lib()
    call = PRODUCERS[producer]
    for what, gt in _bad_gathers(lib):
        before = handle.hgr_launch_count()
        rc = call(lib, gt)
        msg = handle.hgr_last_error()
        assert rc == -1, (producer, what, rc, msg)
        assert b"gather" in msg, (producer, what, msg)  # refused by the gather check, not by the second defect
        assert handle.hgr_launch_count() == before, (producer, what)


def test_spmm_refuses_a_null_output_without_a_gather_destination(lib):
    """Y may be NULL only when the epilogue publishes the rows somewhere else."""
    handle = lib.lib()
    d = _no_work_list_desc(lib)
    ep = lib.Epilogue()
    ep.scale = 1.0
    before = handle.hgr_launch_count()
    for epi in (None, C.byref(ep)):
        rc = handle.hgr_spmm_f32(C.byref(d), FAKE, None, 64, epi, None, 0, None)
        assert rc == -1 and b"NULL" in handle.hgr_last_error()
    assert handle.hgr_launch_count() == before
