"""The fused all-gather stores on one GPU.  Five producers can store their finished rows, besides their local output, at
``row_offset`` of up to HGR_MAX_GATHER destination tables: the propagation epilogue, the LayerNorm backward, publish_rows,
add_rows and the rows x small-matrix product.  In sharded training those tables are peer-mapped on other GPUs; a kernel
cannot tell them from local buffers, so the unicast path is checked here with local tables: the rows land at the offset in
every table, bit for bit, and nothing else in any table is touched.  (The multicast path needs an NVLS object and is not
covered here.)"""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from oracle import hgr_oracle as O

from conftest import rowwise_rel_err as rel_err

pytestmark = pytest.mark.gpu
SENTINEL = 0x7FC0BEEF  # a NaN bit pattern no kernel produces
WIDTHS = [32, 64, 128]
LAYOUTS = [(1, 1), (1, 2), (3, 1), (3, 2), (8, 1), (8, 2)]  # (tables, row_offset in units of the producer's rows)


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def tables(k, rows, d):
    return [torch.full((3 * rows, d), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32) for _ in range(k)]


def assert_published(outs, off, want):
    """Rows [off, off + n) of every table are ``want``; every other row still holds the sentinel."""
    n = want.shape[0]
    w = bits(want)
    for j, t in enumerate(outs):
        tb = bits(t)
        assert torch.equal(tb[off:off + n], w), j
        assert bool((tb[:off] == SENTINEL).all()) and bool((tb[off + n:] == SENTINEL).all()), j


@pytest.fixture(scope="module")
def hgr():
    from hypergraph_diffusion_for_recommendation_b200 import _lib, graph, ops

    assert torch.cuda.is_available()
    _lib.lib()
    return types.SimpleNamespace(lib=_lib, graph=graph, ops=ops)


@pytest.fixture(scope="module")
def plans(hgr):
    """The 8 000-node power-law adjacency without split rows, cut every 64 nonzeros (group reduce) and every 8 (group and
    block reduce)."""
    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions

    g = powerlaw_interactions(3000, 5000, 120_000, seed=3)
    csr = O.build_norm_adj(g.train_u, g.train_i, 3000, 5000)
    out = {c: hgr.graph.DeviceCSR.from_host(*csr, (8000, 8000), symmetric=True, chunk_nnz=c) for c in (1 << 30, 64, 8)}
    chunks = (out[8].heavy_chunk_ptr[1:] - out[8].heavy_chunk_ptr[:-1]).cpu()
    assert out[1 << 30].desc.n_heavy_rows == 0 and out[64].desc.n_heavy_rows > 0
    assert bool((chunks <= 64).any()) and bool((chunks > 64).any())
    return out


@pytest.mark.parametrize("ln", [False, True])
@pytest.mark.parametrize("chunk", [1 << 30, 64, 8])
@pytest.mark.parametrize("d", WIDTHS)
def test_spmm_epilogue_publishes_every_row(hgr, plans, d, chunk, ln):
    a = plans[chunk]
    n = a.shape[0]
    gen = torch.Generator(device="cuda").manual_seed(d + chunk)
    x = torch.randn(n, d, generator=gen, device="cuda")
    kw = dict(slope=0.3)
    if ln:
        kw.update(gamma=torch.randn(d, generator=gen, device="cuda"), beta=torch.randn(d, generator=gen, device="cuda"))
    y_plain = hgr.ops.spmm_raw(a, x, hgr.ops._epilogue(**kw))
    for k, m in LAYOUTS:
        off = m * n
        outs = tables(k, n, d)
        y = hgr.ops.spmm_raw(a, x, hgr.ops._epilogue(gather_ptrs=[t.data_ptr() for t in outs], gather_row_offset=off, **kw))
        assert torch.equal(bits(y), bits(y_plain))
        assert_published(outs, off, y)
        outs = tables(k, n, d)  # Y NULL: the tables are the only destination
        assert hgr.ops.spmm_raw(a, x, hgr.ops._epilogue(gather_ptrs=[t.data_ptr() for t in outs], gather_row_offset=off, **kw),
                                no_local_out=True) is None
        assert_published(outs, off, y)


@pytest.mark.parametrize("with_gamma", [False, True])
@pytest.mark.parametrize("d", WIDTHS)
def test_leaky_ln_bwd_publishes_dpre(hgr, d, with_gamma):
    n = 1237
    gen = torch.Generator(device="cuda").manual_seed(d)
    pre, dy = torch.randn(n, d, generator=gen, device="cuda"), torch.randn(n, d, generator=gen, device="cuda")
    gamma = 1 + 0.1 * torch.randn(d, generator=gen, device="cuda") if with_gamma else None
    want = hgr.ops.leaky_ln_bwd(pre, dy, gamma, 1e-5, 0.3)
    for k, m in LAYOUTS:
        outs = tables(k, n, d)
        got = hgr.ops.leaky_ln_bwd(pre, dy, gamma, 1e-5, 0.3, [t.data_ptr() for t in outs], m * n)
        for g, w in zip(got, want):
            assert (g is None) == (w is None) and (g is None or torch.equal(bits(g), bits(w)))
        assert_published(outs, m * n, want[0])


@pytest.mark.parametrize("d", WIDTHS)
def test_publish_rows(hgr, d):
    n = 1237
    x = torch.randn(n, d, generator=torch.Generator(device="cuda").manual_seed(d), device="cuda")
    for k, m in LAYOUTS:
        outs = tables(k, n, d)
        hgr.ops.publish_rows(x, [t.data_ptr() for t in outs], m * n)
        assert_published(outs, m * n, x)
    lib = hgr.lib.lib()
    torch.cuda.synchronize()
    before = lib.hgr_launch_count()
    hgr.ops.publish_rows(x, [], n)  # nothing to publish: nothing launched
    assert lib.hgr_launch_count() == before


@pytest.mark.parametrize("d", WIDTHS)
def test_add_rows_publishes_the_sum(hgr, d):
    """hgr_add_rows_f32 called directly: ops.add_rows publishes only through a sharded graph."""
    n = 1237
    gen = torch.Generator(device="cuda").manual_seed(d)
    a, b = torch.randn(n, d, generator=gen, device="cuda"), torch.randn(n, d, generator=gen, device="cuda")
    lib = hgr.lib.lib()
    for k, m in LAYOUTS:
        outs = tables(k, n, d)
        out = torch.full((n, d), float("nan"), device="cuda")
        g = hgr.lib.make_gather([t.data_ptr() for t in outs], m * n)
        hgr.lib.check(lib.hgr_add_rows_f32(a.data_ptr(), b.data_ptr(), n, d, out.data_ptr(), C.byref(g), hgr.lib.stream_ptr()))
        assert torch.equal(bits(out), bits(a + b))
        assert_published(outs, m * n, out)


@pytest.mark.parametrize("N", [32, 64, 128, 256])
def test_rows_times_small_publishes_its_rows(hgr, N):
    n, K = 1237, 64  # not a multiple of the 64-row tile
    gen = torch.Generator(device="cuda").manual_seed(N)
    a = torch.randn(n, K, generator=gen, device="cuda")
    b = 0.2 * torch.randn(K, N, generator=gen, device="cuda")
    bias = torch.randn(N, generator=gen, device="cuda")
    y_plain = hgr.ops.rows_times_small(a, None, b, bias, relu=True)
    want = torch.relu(a.double() @ b.double() + bias.double())
    assert rel_err(y_plain, want) < 1e-5
    for k, m in LAYOUTS:
        outs = tables(k, n, N)
        y = hgr.ops.rows_times_small(a, None, b, bias, relu=True, gather=([t.data_ptr() for t in outs], m * n, 0))
        assert torch.equal(bits(y), bits(y_plain))
        assert_published(outs, m * n, y)
