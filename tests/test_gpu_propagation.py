"""GPU parity of the propagation path (libhgr.so through the C ABI) against the oracle and the
reference-generated golden vectors.  Bit-exact where a row is accumulated sequentially; 1e-5
relative (north_star) everywhere else, tolerance written at each assert."""
import types

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import hgr_oracle as O

pytestmark = pytest.mark.gpu
RTOL = 1e-5


from conftest import rowwise_rel_err as rel_err  # noqa: E402  row-wise: each embedding row against its own magnitude


def bits(a):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def params(golden, prefix):
    return {k[len(prefix):]: torch.from_numpy(golden[k]) for k in golden.files if k.startswith(prefix)}


@pytest.fixture(scope="module")
def hgr():
    import hypergraph_diffusion_for_recommendation_b200 as pkg
    from hypergraph_diffusion_for_recommendation_b200 import _lib, encoders, graph, ops

    assert torch.cuda.is_available()
    _lib.lib()  # raises if libhgr.so is missing: there is no fallback
    return types.SimpleNamespace(pkg=pkg, lib=_lib, enc=encoders, graph=graph, ops=ops)


@pytest.fixture(scope="module")
def adj(hgr, pl_graph):
    n = pl_graph["n_users"] + pl_graph["n_items"]
    return hgr.graph.DeviceCSR.from_host(*pl_graph["csr"], (n, n), symmetric=True, chunk_nnz=1 << 20)


@pytest.fixture(scope="module")
def data(pl_graph):
    n = pl_graph["n_users"] + pl_graph["n_items"]
    ip, ix, dv = pl_graph["csr"]
    return types.SimpleNamespace(n_users=pl_graph["n_users"], n_items=pl_graph["n_items"],
                                 norm_adj=sp.csr_matrix((dv, ix, ip), shape=(n, n)))


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------------------ SpMM
def test_spmm_bit_exact_vs_oracle_and_reference(hgr, golden, pl_graph, adj):
    y = hgr.ops.spmm_raw(adj, cuda(golden["spmm_X"]))
    assert np.array_equal(bits(y), bits(O.spmm(*pl_graph["csr"], golden["spmm_X"])))
    assert np.array_equal(bits(y), bits(golden["spmm_Y"]))  # torch.sparse.mm on CPU, same bits


@pytest.mark.parametrize("d", [32, 64, 128])
def test_spmm_widths_and_split_rows(hgr, pl_graph, d):
    n = pl_graph["n_users"] + pl_graph["n_items"]
    rng = np.random.default_rng(d)
    x = rng.standard_normal((n, d)).astype(np.float32)
    ref = O.spmm(*pl_graph["csr"], x)
    whole = hgr.graph.DeviceCSR.from_host(*pl_graph["csr"], (n, n), symmetric=True, chunk_nnz=1 << 20)
    assert whole.desc.n_heavy_rows == 0
    assert np.array_equal(bits(hgr.ops.spmm_raw(whole, cuda(x))), bits(ref))
    split = hgr.graph.DeviceCSR.from_host(*pl_graph["csr"], (n, n), symmetric=True, chunk_nnz=8)
    assert split.desc.n_heavy_rows > 0
    y1, y2 = hgr.ops.spmm_raw(split, cuda(x)), hgr.ops.spmm_raw(split, cuda(x))
    assert np.array_equal(bits(y1), bits(y2))  # deterministic: no atomics
    assert rel_err(y1, ref) < RTOL
    light = np.diff(pl_graph["csr"][0]) <= 8
    assert np.array_equal(bits(y1)[light], bits(ref)[light])  # unsplit rows stay bit-exact


def test_spmm_empty_rows_and_empty_matrix(hgr):
    indptr = np.array([0, 0, 2, 2, 3, 3], dtype=np.int64)
    indices = np.array([4, 0, 1], dtype=np.int32)
    vals = np.array([0.5, -2.0, 3.0], dtype=np.float32)
    a = hgr.graph.DeviceCSR.from_host(indptr, indices, vals, (5, 5))
    x = np.arange(5 * 32, dtype=np.float32).reshape(5, 32)
    y = hgr.ops.spmm_raw(a, cuda(x)).cpu().numpy()
    assert np.array_equal(y, O.spmm(indptr, indices, vals, x))
    assert not y[[0, 2, 4]].any()
    e = hgr.graph.DeviceCSR.from_host(np.zeros(4, dtype=np.int64), np.zeros(0, np.int32), np.zeros(0, np.float32), (3, 7))
    assert not hgr.ops.spmm_raw(e, torch.ones(7, 64, device="cuda")).any()
    with pytest.raises(ValueError):
        hgr.ops.spmm_raw(a, torch.ones(5, 48, device="cuda"))  # unsupported width fails loudly
    with pytest.raises(hgr.lib.HgrError):
        hgr.ops.spmm_raw(a, torch.ones(5, 64))  # CPU tensor: no fallback


def test_spmm_refuses_a_matrix_without_work_list(hgr, pl_graph):
    """Row groups take their rows and chunks from hgr_csr_t::work_order only: the descriptor of a non-empty matrix without a
    list is refused before anything is launched.  Every pointer is valid device memory, so a library that accepted the
    descriptor would run the product instead of failing."""
    import ctypes as C

    n = pl_graph["n_users"] + pl_graph["n_items"]
    a = hgr.graph.DeviceCSR.from_host(*pl_graph["csr"], (n, n), symmetric=True, split="fixed")
    d = hgr.lib.CsrDesc.from_buffer_copy(a.desc)
    d.work_order, d.n_work = None, 0
    x, y = torch.ones(n, 64, device="cuda"), torch.zeros(n, 64, device="cuda")
    ws = a.workspace(64)
    lib = hgr.lib.lib()
    before = lib.hgr_launch_count()
    rc = lib.hgr_spmm_f32(C.byref(d), x.data_ptr(), y.data_ptr(), 64, None, hgr.lib.ptr(ws), 0 if ws is None else ws.numel() * 4,
                          hgr.lib.stream_ptr())
    assert rc == -1 and b"work list" in lib.hgr_last_error()
    assert lib.hgr_launch_count() == before


def test_spmm_epilogue_stages(hgr, pl_graph, adj):
    n = pl_graph["n_users"] + pl_graph["n_items"]
    rng = np.random.default_rng(3)
    x, res, a0, a1 = (rng.standard_normal((n, 64)).astype(np.float32) for _ in range(4))
    gamma, beta = rng.standard_normal(64).astype(np.float32), rng.standard_normal(64).astype(np.float32)
    z = O.spmm(*pl_graph["csr"], x)
    pre = torch.empty(n, 64, device="cuda")
    keep = [cuda(gamma), cuda(beta), cuda(res), cuda(a0), cuda(a1)]  # the descriptor only borrows the tensors
    ep = hgr.ops._epilogue(slope=0.3, gamma=keep[0], beta=keep[1], residual=keep[2], addends=(keep[3], keep[4]), scale=0.25, pre=pre)
    y = hgr.ops.spmm_raw(adj, cuda(x), ep)
    want = (O.layer_norm(O.leaky_relu(z, 0.3), gamma, beta) + res + (a0 + a1)) * np.float32(0.25)
    assert np.array_equal(bits(pre), bits(z))
    assert rel_err(y, want) < RTOL
    del keep


def test_spmm_properties_on_a_larger_graph(hgr):
    """Size-independent checks at a size the oracle still finishes quickly: A 1 = rowsum,
    linearity, and <y, A x> = <A y, x> for the symmetric adjacency."""
    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions

    g = powerlaw_interactions(3000, 5000, 120_000, seed=3)
    csr = O.build_norm_adj(g.train_u, g.train_i, 3000, 5000)
    a = hgr.graph.DeviceCSR.from_host(*csr, (8000, 8000), symmetric=True)
    assert a.desc.n_heavy_rows > 0  # the default plan splits the popular items
    rng = np.random.default_rng(0)
    x = rng.standard_normal((8000, 64)).astype(np.float32)
    z = rng.standard_normal((8000, 64)).astype(np.float32)
    y = hgr.ops.spmm_raw(a, cuda(x))
    assert rel_err(y, O.spmm(*csr, x)) < RTOL
    ones = hgr.ops.spmm_raw(a, torch.ones(8000, 64, device="cuda"))
    rowsum = np.bincount(np.repeat(np.arange(8000), np.diff(csr[0])), weights=csr[2].astype(np.float64), minlength=8000)
    assert rel_err(ones[:, 0], rowsum) < RTOL
    lin = hgr.ops.spmm_raw(a, cuda(2 * x - 3 * z))
    assert rel_err(lin, 2 * y.cpu().numpy() - 3 * hgr.ops.spmm_raw(a, cuda(z)).cpu().numpy()) < 1e-4
    yz = hgr.ops.spmm_raw(a, cuda(z))
    lhs = float((cuda(z).double() * y.double()).sum())
    rhs = float((yz.double() * cuda(x).double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1.0)


# ------------------------------------------------------------------------------------------ autograd ops
def test_spmm_backward_matches_reference_autograd(hgr, golden, adj):
    x = cuda(golden["spmm_X"]).requires_grad_(True)
    y = hgr.ops.spmm(adj, x)
    (y * cuda(golden["spmm_G"])).sum().backward()
    assert rel_err(x.grad, golden["spmm_dX"]) < RTOL


def test_hgconv_forward_backward(hgr, golden, adj):
    x = cuda(golden["hgconv_X"]).requires_grad_(True)
    y = hgr.ops.hgconv(adj, x, slope=0.5)
    assert rel_err(y, golden["hgconv_Y_act"]) < RTOL
    (y * cuda(golden["spmm_G"])).sum().backward()
    assert rel_err(x.grad, golden["hgconv_dX_act"]) < RTOL
    with torch.no_grad():
        y0 = hgr.ops.hgconv(adj, x, slope=None)
    assert np.array_equal(bits(y0), bits(golden["hgconv_Y_noact"]))  # symmetric A, sequential rows: same bits as torch CPU


def test_hgconv_asymmetric_after_edge_drop(hgr, golden, adj):
    dropped = hgr.enc.SpAdjDropEdge()(adj, float(golden["drop_keep"]), rand=torch.from_numpy(golden["drop_rand"]))
    # the dropped matrix keeps the pattern of the adjacency with zeroed values; compacted, it is the reference's matrix
    ip, ix, dv = dropped.to_host(drop_zeros=True)
    rows = np.repeat(np.arange(ip.size - 1), np.diff(ip))
    assert np.array_equal(np.stack([rows, ix]), golden["drop_indices"])
    assert np.array_equal(bits(dv), bits(golden["drop_values"]))
    x = cuda(golden["drop_X"])
    assert np.array_equal(bits(hgr.ops.spmm_raw(dropped, x)), bits(golden["drop_Y"]))
    y = hgr.enc.HGCNConv(0.3)(dropped, x, act=True)
    assert rel_err(y, golden["drop_hgconv_Y"]) < RTOL
    # transpose handle: (A^T)^T round trip and A^T x against the oracle
    tip, tix, tdv = O.csr_transpose(ip.astype(np.int64), ix.astype(np.int64), dv, dropped.shape[1])
    t = dropped.t()
    th = t.to_host(drop_zeros=True)
    assert np.array_equal(th[0], tip) and np.array_equal(th[1], tix) and np.array_equal(bits(th[2]), bits(tdv))
    assert t.t() is dropped
    # a matrix that is not structurally symmetric still takes the compacting path
    rect = hgr.graph.DeviceCSR.from_host(ip, ix, dv, dropped.shape)
    d2 = hgr.enc.SpAdjDropEdge()(rect, 0.5, rand=torch.from_numpy(np.random.default_rng(0).random(ix.size).astype(np.float32)))
    assert d2._nnz() < rect._nnz() and np.array_equal(bits(hgr.ops.spmm_raw(d2.t().t(), x)), bits(hgr.ops.spmm_raw(d2, x)))


def test_lightgcn_propagate_and_backward(hgr, golden, adj, pl_graph):
    e0 = cuda(np.concatenate([golden["lgcn_user_emb0"], golden["lgcn_item_emb0"]], 0)).requires_grad_(True)
    out = hgr.ops.lightgcn_propagate(adj, e0, 3)
    u = pl_graph["n_users"]
    assert rel_err(out[:u], golden["lgcn_user_out"]) < RTOL and rel_err(out[u:], golden["lgcn_item_out"]) < RTOL
    g = cuda(golden["spmm_G"])
    (out * g).sum().backward()
    # d/dE0 of mean_k A^k E0 contracted with G is mean_k A^k G (A symmetric)
    want = O.lgcn_forward(pl_graph["csr"], golden["spmm_G"][:u], golden["spmm_G"][u:], 3)
    assert rel_err(e0.grad, np.concatenate(want, 0)) < RTOL
    s = hgr.ops.lightgcn_propagate(adj, e0.detach(), 2, sum_readout=True)
    e = e0.detach().cpu().numpy()
    e1 = O.spmm(*pl_graph["csr"], e)
    assert rel_err(s, e + e1 + O.spmm(*pl_graph["csr"], e1)) < RTOL


# ------------------------------------------------------------------------------------------ encoders
def test_lgcn_encoder_matches_reference(hgr, golden, data):
    enc = hgr.enc.LGCN_Encoder(data, 64, 3)
    enc.load_state_dict({"embedding_dict.user_emb": torch.from_numpy(golden["lgcn_user_emb0"]),
                         "embedding_dict.item_emb": torch.from_numpy(golden["lgcn_item_emb0"])}, strict=True)
    enc = enc.cuda()
    with torch.no_grad():
        ue, ie = enc()
    assert rel_err(ue, golden["lgcn_user_out"]) < RTOL and rel_err(ie, golden["lgcn_item_out"]) < RTOL


def test_equiv_set_conv_matches_reference(hgr, golden, data, adj):
    esc = hgr.enc.EquivSetConv(64, 64, data.n_users, data.n_items, mlp1_layers=0, mlp2_layers=0, mlp3_layers=1, alpha=0.0,
                               aggr="mean", dropout=0.5, normalization="ln", input_norm=True, data=data)
    esc.load_state_dict(params(golden, "esc_param/"), strict=True)  # same state_dict keys as the reference module
    esc = esc.cuda().eval()
    x = cuda(golden["esc_X"]).requires_grad_(True)
    y = esc(x, adj, x, None)
    assert rel_err(y, golden["esc_Y"]) < RTOL
    (y * cuda(golden["spmm_G"])).sum().backward()
    assert rel_err(x.grad, golden["esc_dX"]) < 2e-5
    for k, p in esc.named_parameters():
        assert rel_err(p.grad, golden["esc_grad/" + k]) < 2e-5, k


def test_local_aware_encoder_matches_reference(hgr, golden, data, adj):
    lae = hgr.enc.LocalAwareEncoder(data, 64, 64, 2, 0.3, 0.2)
    lae.load_state_dict(params(golden, "lae_param/"), strict=True)
    lae = lae.cuda().eval()
    e0 = cuda(golden["lae_E0"]).requires_grad_(True)
    lu, li = lae(e0, lae.sparse_norm_adj)
    assert rel_err(lu, golden["lae_user_out"]) < RTOL and rel_err(li, golden["lae_item_out"]) < RTOL
    (torch.cat([lu, li], 0) * cuda(golden["spmm_G"])).sum().backward()
    assert rel_err(e0.grad, golden["lae_dE0"]) < 2e-5
    checked = 0
    for k, p in lae.named_parameters():
        if "lae_grad/" + k in golden.files:
            assert rel_err(p.grad, golden["lae_grad/" + k]) < 5e-5, k
            checked += 1
    assert checked >= 10


def test_hccf_encoder_matches_reference(hgr, golden, data):
    conf = dict(lrate=0.001, lr_decay=0.9, max_epoch=1, batch_size=64, reg=0.1, embedding_size=64, hyper_dim=32, drop_rate=0.5,
                p=0.1, n_layers=2)
    hc = hgr.enc.HCCFEncoder(conf, data)
    hc.load_state_dict(params(golden, "hccf_param/"), strict=True)
    hc = hc.cuda().eval()
    with torch.no_grad():
        hu, hi, gcn_h, hyp_h = hc(keep_rate=1.0)
    assert rel_err(hu, golden["hccf_user_out"]) < RTOL and rel_err(hi, golden["hccf_item_out"]) < RTOL
    for l in range(2):
        assert rel_err(gcn_h[l], golden["hccf_gcn_%d" % l]) < RTOL
        assert rel_err(hyp_h[l], golden["hccf_hyp_%d" % l]) < RTOL  # tall-and-skinny fp32 products in a different order


# ------------------------------------------------------------------------------------ scatter-mean form (SURVEY.md a-6)
@pytest.mark.parametrize("n,k,d", [(1, 32, 32), (63, 64, 64), (3001, 128, 64), (30011, 128, 64), (4097, 256, 128), (2500, 32, 128)])
def test_hyperedge_products_forward_backward(hgr, n, k, d):
    """HGNNLayer.forward on the tall-and-skinny kernels (csrc/hyperedge.cu) against the float64 oracle: forward, both
    gradients, ragged row counts (not a multiple of the 32-row staging tile or the 64-row output tile)."""
    rng = np.random.default_rng(n + k + d)
    h = (rng.standard_normal((n, k)) * 0.3).astype(np.float32)
    e = rng.standard_normal((n, d)).astype(np.float32)
    g = rng.standard_normal((n, d)).astype(np.float32)
    ht, et = cuda(h).requires_grad_(True), cuda(e).requires_grad_(True)
    assert hgr.ops.hyperedge_supported(ht, et)
    y = hgr.ops.hyperedge(ht, et)
    assert rel_err(y, O.hyperedge(h, e)) < RTOL  # 1e-5 relative (north_star), fp32 sums in a different order
    (y * cuda(g)).sum().backward()
    dh, de = O.hyperedge_grads(h, e, g)
    assert rel_err(ht.grad, dh) < RTOL and rel_err(et.grad, de) < RTOL
    y2 = hgr.ops.hyperedge(ht.detach(), et.detach())
    assert np.array_equal(bits(y2), bits(y))  # partials are added in block order: reproducible
    t = hgr.ops.tall_skinny_tn(cuda(h), cuda(e))
    assert rel_err(t, h.astype(np.float64).T @ e.astype(np.float64)) < RTOL
    with pytest.raises(ValueError):
        hgr.ops.hyperedge(torch.ones(8, 48, device="cuda"), torch.ones(8, 64, device="cuda"))  # unsupported width fails loudly
    with pytest.raises(hgr.lib.HgrError):
        hgr.ops.tall_skinny_tn(torch.ones(8, 48, device="cuda"), torch.ones(8, 64, device="cuda"))


@pytest.mark.parametrize("n,k,w", [(5, 64, 128), (3001, 64, 128), (20000, 32, 64), (777, 128, 32)])
def test_tall_times_small_forward_backward(hgr, n, k, w):
    """HCCF's ``hyper = E0 @ W`` (HCCF.py:178-179) on the libhgr kernels against float64: output, dE0 and the tall-skinny dW."""
    rng = np.random.default_rng(n + w)
    x = rng.standard_normal((n, k)).astype(np.float32)
    m = (rng.standard_normal((k, w)) * 0.2).astype(np.float32)
    g = rng.standard_normal((n, w)).astype(np.float32)
    xt, mt = cuda(x).requires_grad_(True), cuda(m).requires_grad_(True)
    y = hgr.ops.tall_times_small(xt, mt)
    (y * cuda(g)).sum().backward()
    x64, m64, g64 = x.astype(np.float64), m.astype(np.float64), g.astype(np.float64)
    assert rel_err(y, x64 @ m64) < RTOL
    assert rel_err(xt.grad, g64 @ m64.T) < RTOL and rel_err(mt.grad, x64.T @ g64) < RTOL
    with pytest.raises(ValueError):
        hgr.ops.tall_times_small(torch.ones(8, 48, device="cuda"), torch.ones(48, 64, device="cuda"))


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("n,k,w", [(4096, 64, 64), (10001, 32, 128), (5000, 128, 64)])
def test_linear_layer_kernel_matches_torch(hgr, n, k, w, relu):
    """``ops.linear`` (nn.Linear.forward [+ ReLU] of the MLP / LocalAwareEncoder input layers on the rows x small-matrix kernel,
    weight gradient on the tall-skinny reduce) against float64: output and all three gradients."""
    import torch.nn.functional as F

    rng = np.random.default_rng(n + w + relu)
    x = rng.standard_normal((n, k)).astype(np.float32)
    wt = (rng.standard_normal((w, k)) * 0.2).astype(np.float32)
    b = rng.standard_normal(w).astype(np.float32)
    g = rng.standard_normal((n, w)).astype(np.float32)
    xs, ws, bs = cuda(x).requires_grad_(True), cuda(wt).requires_grad_(True), cuda(b).requires_grad_(True)
    y = hgr.ops.linear(xs, ws, bs, relu=relu)
    (y * cuda(g)).sum().backward()
    xr, wr, br = (torch.from_numpy(v).double().requires_grad_(True) for v in (x, wt, b))
    yr = F.linear(xr, wr, br)
    yr = torch.relu(yr) if relu else yr
    (yr * torch.from_numpy(g).double()).sum().backward()
    assert rel_err(y, yr.detach().numpy()) < RTOL
    assert rel_err(xs.grad, xr.grad.numpy()) < RTOL and rel_err(ws.grad, wr.grad.numpy()) < RTOL and rel_err(bs.grad, br.grad.numpy()) < RTOL
    small = hgr.ops.linear(torch.ones(8, k, device="cuda"), ws.detach(), bs.detach(), relu=relu)  # short inputs stay on F.linear
    assert small.shape == (8, w)


def test_scatter_mean_form_matches_reference_golden_and_oracle(hgr, golden):
    from hypergraph_diffusion_for_recommendation_b200 import graph

    v, e, x = golden["scat_V"], golden["scat_E"], golden["scat_X"]
    inc = graph.build_incidence(v, e, x.shape[0])
    xt = cuda(x).requires_grad_(True)
    y = hgr.ops.scatter_mean_conv(inc, xt)
    assert rel_err(y, golden["scat_Y"]) < RTOL  # the reference's torch_scatter path
    assert rel_err(y, O.scatter_mean_conv(v, e, x, x.shape[0])) < RTOL
    # backward against torch autograd of the same index_add / clamp(count, 1) arithmetic
    g = cuda(np.random.default_rng(2).standard_normal(x.shape).astype(np.float32))
    (y * g).sum().backward()
    import torch

    xr = torch.from_numpy(x).requires_grad_(True)
    vt, et = torch.from_numpy(v).long(), torch.from_numpy(e).long()
    n_e = int(et.max()) + 1
    xe = torch.zeros(n_e, x.shape[1]).index_add_(0, et, xr[vt]) / torch.bincount(et, minlength=n_e).clamp(min=1)[:, None]
    xv = torch.zeros(x.shape[0], x.shape[1]).index_add_(0, vt, xe[et]) / torch.bincount(vt, minlength=x.shape[0]).clamp(min=1)[:, None]
    (xv * g.cpu()).sum().backward()
    assert rel_err(xt.grad, xr.grad) < RTOL


def test_scatter_mean_ragged_incidence_with_empty_segments(hgr):
    from hypergraph_diffusion_for_recommendation_b200 import encoders, graph

    rng = np.random.default_rng(8)
    n, n_e, d = 500, 64, 64
    v = rng.integers(0, n - 50, 4000)          # the last 50 vertices belong to no hyperedge
    e = rng.integers(0, n_e, 4000)
    e[e == 13] = 12                            # hyperedge 13 is empty
    pairs = np.unique(np.stack([v, e], 1), axis=0)
    v, e = pairs[:, 0], pairs[:, 1]
    x = rng.standard_normal((n, d)).astype(np.float32)
    inc = graph.build_incidence(v, e, n, n_e)
    y = hgr.ops.scatter_mean_conv(inc, cuda(x))
    assert rel_err(y, O.scatter_mean_conv(v, e, x, n)) < RTOL
    assert float(y[-50:].abs().max()) == 0.0   # empty segments give zero rows
    # the dense-incidence entry point of the reference (generate_V_E: nonzero(H > 0))
    import torch

    h = torch.zeros(n, n_e)
    h[torch.from_numpy(v), torch.from_numpy(e)] = 0.7
    inc2 = graph.incidence_from_dense(h.cuda())
    assert rel_err(hgr.ops.scatter_mean_conv(inc2, cuda(x)), y) < 1e-6
    conv = encoders.EquivSetConvScatter(d, d, mlp1_layers=0, mlp2_layers=0, mlp3_layers=0, aggr='mean', alpha=0.0)
    out = conv(cuda(x), torch.from_numpy(v).cuda(), torch.from_numpy(e).cuda(), cuda(x))
    assert rel_err(out, y) < 1e-6


# ------------------------------------------------------------------------------------ SGL (augmentation + InfoNCE views)
def test_sgl_encoder_views_and_device_augmentor(hgr, pl_graph):
    from hypergraph_diffusion_for_recommendation_b200 import augmentor

    n_users, n_items = pl_graph["n_users"], pl_graph["n_items"]
    u, i = cuda(pl_graph["u"]), cuda(pl_graph["i"])
    ku, ki = augmentor.GraphAugmentor.edge_dropout(u, i, 0.3)
    assert ku.numel() == int(u.numel() * 0.7)
    pairs = set(zip(pl_graph["u"].tolist(), pl_graph["i"].tolist()))
    assert set(zip(ku.tolist(), ki.tolist())) <= pairs and len(set(zip(ku.tolist(), ki.tolist()))) == ku.numel()
    nu, ni = augmentor.GraphAugmentor.node_dropout(u, i, n_users, n_items, 0.2)
    assert n_users - len(set(nu.tolist())) >= int(n_users * 0.2) - 0 and nu.numel() < u.numel()
    # the perturbed Laplacian is exactly the oracle's normalised adjacency of the kept interactions
    adj = augmentor.convert_to_laplacian_mat(ku, ki, n_users, n_items)
    want = O.build_norm_adj(ku.cpu().numpy(), ki.cpu().numpy(), n_users, n_items)
    got = adj.to_host()
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and np.array_equal(bits(got[2]), bits(want[2]))
    # encoder: clean forward == LightGCN; perturbed views differ; the contrastive loss is differentiable
    n = n_users + n_items
    data = types.SimpleNamespace(n_users=n_users, n_items=n_items, train_u=u, train_i=i, norm_adj=None,
                                 norm_adj_device=hgr.graph.DeviceCSR.from_host(*pl_graph["csr"], (n, n), symmetric=True))
    torch.manual_seed(0)
    enc = hgr.enc.SGL_Encoder(data, 64, 0.2, 3, 0.2, 1).cuda()
    ue, ie = enc()
    ego = torch.cat([enc.embedding_dict['user_emb'], enc.embedding_dict['item_emb']], 0)
    ref_u, ref_i = O.lgcn_forward(pl_graph["csr"], ego[:n_users].detach().cpu().numpy(), ego[n_users:].detach().cpu().numpy(), 3)
    assert rel_err(ue, ref_u) < 1e-6 and rel_err(ie, ref_i) < 1e-6
    p1, p2 = enc.graph_reconstruction(), enc.graph_reconstruction()
    v1, _ = enc(p1)
    assert not torch.equal(v1, ue)
    loss = enc.cal_cl_loss([torch.arange(0, n_users, 2), torch.arange(0, n_items, 3)], p1, p2)
    loss.backward()
    assert torch.isfinite(loss) and float(enc.embedding_dict['user_emb'].grad.abs().sum()) > 0
    # per-layer list of perturbed graphs (aug_type 2 in the paper) gives the same result as one graph used for every layer
    a, b = enc([p1, p1, p1]), enc(p1)
    assert rel_err(a[0], b[0]) < 1e-6


# ------------------------------------------------------------------------------------------ more callers of the path
@pytest.fixture(scope="module")
def more_golden():
    import os

    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "more_encoders.npz"))


def _facade(more_golden):
    from hypergraph_diffusion_for_recommendation_b200 import data as D

    return D.Interaction(None, more_golden["train"].tolist(), more_golden["test"].tolist())


def test_sht_encoder_matches_reference(hgr, more_golden):
    """SHTEncoder (LightGCN-sum + low-rank hypergraph transform) on the façade's device adjacency against the reference's
    CPU outputs and parameter gradients (tests/golden/make_golden_more_encoders.py)."""
    g = more_golden
    n_layers, hyper_dim, n_hyper = (int(v) for v in g["sht_args"])
    args = {"max_epoch": 1, "batch_size": 64, "lrate": 0.01, "lr_decay": 0.9, "reg": 0.0, "embedding_size": 64, "hyper_dim": hyper_dim,
            "drop_rate": 0.2, "p": 0.1, "n_layers": n_layers, "cl_rate": 1e-4, "temp": 0.2, "seed": 20, "early_stopping_steps": 20,
            "hyperedge_num": n_hyper}
    m = hgr.enc.SHTEncoder(_facade(g), args).cuda()
    m.load_state_dict(params(g, "sht_param/"), strict=True)
    emb, hu, hi = m()
    assert rel_err(emb, g["sht_embeds"]) < RTOL and rel_err(hu, g["sht_hyper_u"]) < RTOL and rel_err(hi, g["sht_hyper_i"]) < RTOL
    ((emb * cuda(g["sht_w0"])).sum() + (hu * cuda(g["sht_w1"])).sum() + (hi * cuda(g["sht_w2"])).sum()).backward()
    for k, p in m.named_parameters():
        assert rel_err(p.grad, g["sht_grad/" + k]) < 2e-5, k


def test_dhcf_encoder_rectangular_hgconv_matches_reference(hgr, more_golden):
    """DHCF_Encoder: HGCNConv on the rectangular [users, items] interaction matrix and on its transpose (the reference densifies
    the matrix); outputs and embedding gradients against the reference."""
    g = more_golden
    layers, hyper_dim, p = int(g["dhcf_args"][0]), int(g["dhcf_args"][1]), float(g["dhcf_args"][2])
    m = hgr.enc.DHCF_Encoder(None, _facade(g), {"input_dim": 64, "hyper_dim": hyper_dim, "p": p, "drop_rate": 0.2, "n_layers": layers}).cuda()
    m.load_state_dict(params(g, "dhcf_param/"), strict=True)
    assert m.adj.shape == (m.data.n_users, m.data.n_items) and m.adj.t().shape == (m.data.n_items, m.data.n_users)
    ue, ie = m()
    assert ue.shape[1] == (layers + 1) * hyper_dim
    assert rel_err(ue, g["dhcf_user_out"]) < RTOL and rel_err(ie, g["dhcf_item_out"]) < RTOL
    ((ue * cuda(g["dhcf_wu"])).sum() + (ie * cuda(g["dhcf_wi"])).sum()).backward()
    assert rel_err(m.embedding_dict["user_emb"].grad, g["dhcf_grad_user"]) < 2e-5
    assert rel_err(m.embedding_dict["item_emb"].grad, g["dhcf_grad_item"]) < 2e-5


def test_sgl_encoder_on_the_data_facade_with_repeated_training_pairs(hgr):
    """ADVICE r1: ``SGL_Encoder.graph_reconstruction`` on ``data.Interaction`` (no ``train_u`` attribute there), with a training file
    that lists some pairs twice: the reference perturbs ``interaction_mat.nonzero()`` -- distinct pairs, unit weights
    (data/augmentor.py:32-42) -- so the perturbed Laplacian has no weight-2 edge and the edge count is of the distinct pairs."""
    from hypergraph_diffusion_for_recommendation_b200 import data as D

    rng = np.random.default_rng(4)
    pairs = np.unique(np.stack([rng.integers(0, 40, 600), 1000 + rng.integers(0, 70, 600)], 1), axis=0)
    listed = np.concatenate([pairs, pairs[::5]])  # every fifth pair twice
    train = [[int(u), int(i), 1.0] for u, i in listed]
    test = [[int(u), int(i), 1.0] for u, i in pairs[::7]]
    data = D.Interaction(None, train, test)
    enc = hgr.enc.SGL_Encoder(data, 64, 0.25, 2, 0.2, 1).cuda()
    adj = enc.graph_reconstruction()
    ip, ix, dv = adj.to_host(drop_zeros=True)
    kept = int(pairs.shape[0] * 0.75)
    assert ix.size == 2 * kept                                   # int(E_distinct * (1 - drop_rate)) edges, both directions
    deg = np.diff(ip).astype(np.float64)
    rows = np.repeat(np.arange(ip.size - 1), np.diff(ip))
    want = 1.0 / np.sqrt(deg[rows] * deg[ix])                     # unit weights: every value is d[r] d[c]
    assert np.abs(dv - want).max() < 1e-6
    ue, ie = enc(adj)
    assert ue.shape == (data.n_users, 64) and torch.isfinite(ue).all() and torch.isfinite(ie).all()


def test_drop_edges_philox_mask_is_a_consistent_transpose_pair_and_changes_with_the_step(hgr, adj):
    """``hgr_drop_edges_f32`` without host random numbers (SURVEY 8b seam 6): keep rate, rescaling, the mirrored launch really is
    the transpose of the dropped matrix, same seed -> same mask, and the device-side step counter gives a new mask."""
    keep = 0.7
    d1 = hgr.enc.drop_edges(adj, keep, seed=11)
    ip, ix, dv = d1.to_host()
    full = adj.to_host()[2]
    kept = dv != 0
    assert abs(kept.mean() - keep) < 0.05
    assert np.array_equal(bits(dv[kept]), bits((full[kept] / np.float32(keep)).astype(np.float32)))  # true division of the kept values
    n = adj.shape[0]
    import scipy.sparse as sp

    a = sp.csr_matrix((dv, ix, ip), shape=(n, n))
    tp, ti, tv = d1.t().to_host()
    at = sp.csr_matrix((tv, ti, tp), shape=(n, n))
    assert (a.T != at).nnz == 0                                            # mirror launch == transpose of the dropped matrix
    assert (a != a.T).nnz > 0                                              # the two directions of an edge are dropped independently
    d2 = hgr.enc.drop_edges(adj, keep, seed=11)
    assert np.array_equal(bits(d2.to_host()[2]), bits(dv))                 # counter-based: reproducible
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    s0 = hgr.enc.drop_edges(adj, keep, seed=11, step=step).to_host()[2]
    step += 1
    s1 = hgr.enc.drop_edges(adj, keep, seed=11, step=step).to_host()[2]
    assert np.array_equal(bits(s0), bits(dv)) and not np.array_equal(bits(s0), bits(s1))
    x = cuda(np.random.default_rng(0).standard_normal((n, 64)).astype(np.float32)).requires_grad_(True)
    y = hgr.ops.spmm(d1, x)
    y.sum().backward()
    want = np.asarray(at @ np.ones((n, 64), np.float32))                   # d/dx sum(A x) = A^T 1
    assert rel_err(x.grad, want) < RTOL


def test_window_split_plan_matches_rule_and_oracle_under_every_schedule(hgr, pl_graph):
    """The window-aligned split plan (csrc/split_plan.cu): the device walk gives the plan of the python restatement; the
    propagation with it is reproducible, independent of the schedule, within 1e-5 of the oracle and bit-exact on whole rows."""
    from hypergraph_diffusion_for_recommendation_b200 import graph

    n = pl_graph["n_users"] + pl_graph["n_items"]
    indptr, indices, vals = pl_graph["csr"]
    shift, min_seg, max_seg = 4, 3, 12  # 16-row windows of the 150-row table
    for span in (3, 0):
        want = graph.window_split_plan_host(indptr, indices, shift, min_seg, max_seg, span)
        got = graph.window_split_plan(cuda(indptr.astype(np.int64)), cuda(indices.astype(np.int32)), shift, min_seg, max_seg, span)
        for w, g in zip(want, got):
            assert np.array_equal(w, g.cpu().numpy())
    assert want[0].size > 10 and want[3].size > 2 * want[0].size
    a = hgr.graph.DeviceCSR.from_host(indptr, indices, vals, (n, n), symmetric=True, chunk_nnz=max_seg, split="window:%d:%d:0" % (shift, min_seg))
    assert a.split.startswith("window") and a.desc.chunk_start
    assert (int(a.desc.n_heavy_rows), int(a.desc.n_chunks)) == (want[0].size, want[3].size)
    x = np.random.default_rng(3).standard_normal((n, 64)).astype(np.float32)
    ref = O.spmm(indptr, indices, vals, x)
    outs = []
    for sched in ("binned", "windowed:16", "spread:16"):
        a.set_schedule(sched)
        outs.append(hgr.ops.spmm_raw(a, cuda(x)))
    for y in outs[1:]:
        assert torch.equal(y, outs[0])
    assert rel_err(outs[0], ref) < RTOL
    whole = np.ones(n, dtype=bool)
    whole[want[0]] = False
    assert np.array_equal(bits(outs[0])[whole], bits(ref)[whole])
    # backward goes through the same plan (symmetric matrix): gradient of sum(Y * G) is A^T G
    g = np.random.default_rng(4).standard_normal((n, 64)).astype(np.float32)
    xt = cuda(x).requires_grad_(True)
    (hgr.ops.spmm(a, xt) * cuda(g)).sum().backward()
    assert rel_err(xt.grad, O.spmm(indptr, indices, vals, g)) < RTOL
