"""Long lists (64 < K <= 256) in full-rank evaluation, the checks that need no GPU: the workspace of hgr_fullrank_topk_f32
(unchanged for K <= 64, never larger for a long list than for K = 64 at the same shape), the argument validation of the
widened range, and the find_k_largest merge rule the refquirk replay relies on, at K beyond the golden cases (K <= 20)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from oracle import hgr_oracle as O

REF = os.environ.get("HGR_REFERENCE", "")

# hgr_fullrank_topk_workspace_bytes(n_test, n_items, 64, K, 0) for K = 20, 40, 64
WORKSPACE_K_LE_64 = {
    (52_000, 92_000): {20: 1_006_567_424, 40: 1_808_728_064, 64: 2_771_320_832},
    (262_144, 250_000): {20: 1_834_176_256, 40: 2_840_809_216, 64: 4_048_768_768},
    (30_000, 41_000): {20: 922_060_544, 40: 1_734_051_584, 64: 2_708_440_832},
}
HGR_ERR_INVALID, HGR_ERR_WORKSPACE = -1, -4


@pytest.fixture(scope="module")
def lib():
    from hypergraph_diffusion_for_recommendation_b200 import _lib, build

    build.build()  # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


@pytest.mark.parametrize("shape", sorted(WORKSPACE_K_LE_64))
def test_workspace_of_short_lists_is_unchanged_and_bounds_long_lists(lib, shape):
    n_test, n_items = shape
    for k, want in WORKSPACE_K_LE_64[shape].items():
        assert lib.hgr_fullrank_topk_workspace_bytes(n_test, n_items, 64, k, 0) == want, k
    k64 = WORKSPACE_K_LE_64[shape][64]
    for k in (65, 100, 256):
        for engine in (0, 2):
            assert lib.hgr_fullrank_topk_workspace_bytes(n_test, n_items, 64, k, engine) <= k64, (k, engine)


def _topk(lib, n_items, K, mode, engine, n_test=1, workspace=None):
    """One hgr_fullrank_topk_f32 call with 16-byte-aligned dummy arrays: only the validation before any launch may run."""
    buf = np.zeros(max(n_items, 8) * 64 + 64, np.float32)
    base = buf.ctypes.data + (-buf.ctypes.data) % 16
    keep = (buf, np.zeros(16, np.int64))
    p = base
    rc = lib.hgr_fullrank_topk_f32(p, 4, p, n_items, 64, p, n_test, keep[1].ctypes.data, p, K, mode, engine, p, p, None,
                                   workspace, 0, None)
    return rc, lib.hgr_last_error()


def test_refquirk_mode_accepts_lists_of_up_to_256_items(lib):
    rc, _ = _topk(lib, 300, 256, 1, 0, n_test=0)
    assert rc == 0
    rc, msg = _topk(lib, 300, 257, 1, 0, n_test=0)
    assert rc == HGR_ERR_INVALID and b"K <= 256" in msg


def test_tensor_engine_accepts_lists_of_up_to_256_items(lib):
    rc, msg = _topk(lib, 300, 256, 0, 2)
    assert rc == HGR_ERR_WORKSPACE, msg  # past the engine check: only the (missing) workspace stops it
    rc, msg = _topk(lib, 300, 257, 0, 2)
    assert rc == HGR_ERR_INVALID and b"K <= 256" in msg
    rc, msg = _topk(lib, 300, 256, 1, 2)
    assert rc == HGR_ERR_WORKSPACE, msg


def merge_rule(k, c):
    """find_k_largest's result restated: the first k entries of the merge of A = candidates 0..k-1 sorted (score desc, id asc)
    and B = the exact top-k, A's entries first on equal scores."""
    a = sorted(range(k), key=lambda i: (-c[i], i))
    b = sorted(range(c.size), key=lambda i: (-c[i], i))[:k]
    out, ia, ib = [], 0, 0
    while len(out) < k:
        if ia < k and (ib >= k or c[a[ia]] >= c[b[ib]]):
            out.append(a[ia])
            ia += 1
        else:
            out.append(b[ib])
            ib += 1
    return np.array(out, np.int64), c[out]


def long_cases(ties):
    rng = np.random.default_rng(256 + ties)
    for k in (65, 100, 256):
        for n in (k + 40, 3 * k, 2000):
            c = rng.permutation(n).astype(np.float32) / n - 0.5  # distinct scores
            if ties:
                c = np.round(c * 8) / 8
            c[rng.random(n) < 0.2] = -10e8
            yield k, c.astype(np.float32)


def test_oracle_find_k_largest_follows_the_merge_rule_at_long_k():
    for k, c in long_cases(ties=False):
        ids, sc = O.find_k_largest(k, c)
        want_ids, want_sc = merge_rule(k, c)
        # masked entries of A (-10e8) tie among themselves: compare them as a set, everything else position by position
        live = want_sc > -10e8
        assert np.array_equal(ids[live], want_ids[live]), (k, c.size)
        assert np.array_equal(sc.view(np.uint32), want_sc.view(np.uint32)), (k, c.size)
        assert set(ids[~live].tolist()) == set(want_ids[~live].tolist())


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs HGR_REFERENCE: a checkout of the unmodified reference project")
def test_oracle_find_k_largest_matches_the_reference_at_long_k():
    sys.path.insert(0, REF)
    try:
        from util.algorithm import find_k_largest
    finally:
        sys.path.remove(REF)
    for ties in (False, True):
        for k, c in long_cases(ties):
            ids, sc = find_k_largest(k, c)
            o_ids, o_sc = O.find_k_largest(k, c)
            assert np.array_equal(np.asarray(ids, np.int64), o_ids), (k, c.size, ties)
            assert np.array_equal(np.asarray(sc, np.float32).view(np.uint32), o_sc.view(np.uint32)), (k, c.size, ties)
