"""CPU oracle for the embedding-propagation / loss / full-rank-eval hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this module; the product path (``hypergraph_diffusion_for_recommendation_b200``)
never does and fails loudly when ``libhgr.so`` is missing.

Every function restates one call site of the reference (paths relative to
``/root/reference/HD_SELFRec``) in numpy, with the bit-sensitive inner loops in ``hgr_oracle.c``.
Parity is PINNED: ``tests/test_oracle_golden.py`` checks every function here against
``tests/golden/reference_vectors_*.npz``, produced by running the reference itself
(``tests/golden/make_golden.py``).  The reference has no tests or golden vectors of its
own (SURVEY.md F3).

Third-party arithmetic the reference calls on this path and that is restated here
(SURVEY.md section 8c): torch (pinned 1.10.1 in the reference's requirements.txt; 2.11.0 in the
build container) ``torch.sparse.mm`` = per-row sequential FMA; pytorch-scatter 2.1.0
``scatter(reduce='mean')`` = sum / clamp(count, 1); numpy ``np.power`` float32 (not correctly
rounded: consumed through a lookup table built on the same host); scipy CSR construction
(duplicates summed, columns sorted); numba 0.53.1 ``find_k_largest``.
"""
from __future__ import annotations

import ctypes
import math
import os

import numpy as np

from . import build as _build

_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        path = _build.build()
        lib = ctypes.CDLL(path)
        i64p, f32p = ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_float)
        lib.hgr_oracle_spmm_f32.argtypes = [i64p, i64p, f32p, ctypes.c_int64, ctypes.c_int64, f32p, f32p]
        lib.hgr_oracle_scores_f32.argtypes = [f32p, f32p, ctypes.c_int64, ctypes.c_int64, f32p]
        lib.hgr_oracle_find_k_largest.argtypes = [ctypes.c_int64, f32p, ctypes.c_int64, i64p, f32p]
        lib.hgr_oracle_topk_exact.argtypes = [ctypes.c_int64, f32p, ctypes.c_int64, i64p, f32p]
        for f in (lib.hgr_oracle_spmm_f32, lib.hgr_oracle_scores_f32, lib.hgr_oracle_find_k_largest,
                  lib.hgr_oracle_topk_exact):
            f.restype = None
        _LIB = lib
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


MASK_SCORE = np.float32(-10e8)  # base/graph_recommender.py:80


# --------------------------------------------------------------------------------------------
# (a-1) adjacency construction                       data/ui_graph.py:70-84, data/graph.py:11-42
# --------------------------------------------------------------------------------------------
def pow_lut(n: int, exponent: float) -> np.ndarray:
    """``np.power(float32 degree, exponent)`` with inf -> 0 (data/graph.py:15-16,21-22) for every
    integer degree below ``n``.  numpy's float32 pow is not correctly rounded (SURVEY.md F10), so
    the product takes this table, built on the same host, instead of recomputing the power."""
    with np.errstate(divide="ignore"):
        lut = np.power(np.arange(n, dtype=np.float32), np.float32(exponent))
    lut[np.isinf(lut)] = 0.0
    return lut.astype(np.float32)


def coo_to_csr_sum(rows, cols, vals, n_rows, n_cols):
    """scipy ``csr_matrix((v, (r, c)))`` semantics: duplicates summed, columns sorted."""
    rows = np.asarray(rows, dtype=np.int64)
    cols = np.asarray(cols, dtype=np.int64)
    key = rows * n_cols + cols
    order = np.argsort(key, kind="stable")
    key, vals = key[order], np.asarray(vals, dtype=np.float32)[order]
    uniq, start = np.unique(key, return_index=True)
    data = np.add.reduceat(vals.astype(np.float64), start).astype(np.float32) if key.size else vals
    r, c = uniq // n_cols, uniq % n_cols
    indptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.add.at(indptr, r + 1, 1)
    return np.cumsum(indptr), c.astype(np.int64), data


def csr_transpose(indptr, indices, data, n_cols):
    n_rows = indptr.size - 1
    rows = np.repeat(np.arange(n_rows, dtype=np.int64), np.diff(indptr))
    order = np.argsort(indices, kind="stable")
    t_indptr = np.zeros(n_cols + 1, dtype=np.int64)
    np.add.at(t_indptr, indices + 1, 1)
    return np.cumsum(t_indptr), rows[order], data[order]


def bipartite_adjacency(u, i, n_users, n_items):
    """``Interaction.__create_sparse_bipartite_adjacency`` (data/ui_graph.py:70-84):
    ``A = [[0, R], [R^T, 0]]`` with unit weights, duplicate interactions summed."""
    u = np.asarray(u, dtype=np.int64)
    i = np.asarray(i, dtype=np.int64)
    n = n_users + n_items
    rows = np.concatenate([u, i + n_users])
    cols = np.concatenate([i + n_users, u])
    return coo_to_csr_sum(rows, cols, np.ones(rows.size, dtype=np.float32), n, n)


def normalize_graph_mat(indptr, indices, data, n_cols):
    """``Graph.normalize_graph_mat`` (data/graph.py:11-25): square -> (D^-1/2 A) D^-1/2 with two
    float32 multiplies per entry; rectangular -> D^-1 A."""
    n_rows = indptr.size - 1
    rows = np.repeat(np.arange(n_rows), np.diff(indptr))
    rowsum = np.zeros(n_rows, dtype=np.float64)
    np.add.at(rowsum, rows, data.astype(np.float64))
    rowsum = rowsum.astype(np.float32)
    deg = rowsum.astype(np.int64)
    assert np.all(deg == rowsum), "integer weights only"
    if n_rows == n_cols:
        d = pow_lut(int(deg.max()) + 1 if deg.size else 1, -0.5)[deg]
        out = ((d[rows] * data).astype(np.float32) * d[indices]).astype(np.float32)
    else:
        d = pow_lut(int(deg.max()) + 1 if deg.size else 1, -1.0)[deg]
        out = (d[rows] * data).astype(np.float32)
    return indptr, indices, out


def build_norm_adj(u, i, n_users, n_items):
    """``Interaction.norm_adj`` (data/ui_graph.py:37-38): canonical CSR of D^-1/2 A D^-1/2."""
    n = n_users + n_items
    ip, ix, dv = bipartite_adjacency(u, i, n_users, n_items)
    return normalize_graph_mat(ip, ix, dv, n)


def interaction_matrix(u, i, n_users, n_items):
    """``Interaction.__create_sparse_interaction_matrix`` (data/ui_graph.py:95-112): R as CSR."""
    return coo_to_csr_sum(u, i, np.ones(len(u), dtype=np.float32), n_users, n_items)


def laplacian_of_interaction(indptr, indices, data, n_users, n_items):
    """``Interaction.convert_to_laplacian_mat`` (data/ui_graph.py:86-93), used by SGL views."""
    rows = np.repeat(np.arange(n_users, dtype=np.int64), np.diff(indptr))
    n = n_users + n_items
    r = np.concatenate([rows, indices + n_users])
    c = np.concatenate([indices + n_users, rows])
    ip, ix, dv = coo_to_csr_sum(r, c, np.concatenate([data, data]), n, n)
    return normalize_graph_mat(ip, ix, dv, n)


def drop_edges(indptr, indices, data, rand, keep):
    """``SpAdjDropEdge.forward`` (model/graph/HCCF.py:213-226): keep nonzero k iff
    ``floor(rand[k] + keep)`` is 1, rescale by ``1 / keep``; order preserved."""
    rows = np.repeat(np.arange(indptr.size - 1, dtype=np.int64), np.diff(indptr))
    mask = np.floor(rand.astype(np.float32) + np.float32(keep)).astype(bool)
    new_ip = np.zeros(indptr.size, dtype=np.int64)
    np.add.at(new_ip, rows[mask] + 1, 1)
    return np.cumsum(new_ip), indices[mask], (data[mask] / np.float32(keep)).astype(np.float32)


# --------------------------------------------------------------------------------------------
# (a-3 .. a-7) propagation
# --------------------------------------------------------------------------------------------
def spmm(indptr, indices, data, x):
    """``torch.sparse.mm(A, X)`` (model/graph/LightGCN.py:133): sequential FMA per row."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    indices = np.ascontiguousarray(indices, dtype=np.int64)
    data = np.ascontiguousarray(data, dtype=np.float32)
    y = np.empty((indptr.size - 1, x.shape[1]), dtype=np.float32)
    _lib().hgr_oracle_spmm_f32(_p(indptr, ctypes.c_int64), _p(indices, ctypes.c_int64), _p(data, ctypes.c_float),
                               indptr.size - 1, x.shape[1], _p(x, ctypes.c_float), _p(y, ctypes.c_float))
    return y


def spmm_f64(indptr, indices, data, x):
    """The same product accumulated in float64 (numpy), rounded once: the value both the reference's sequential fp32 chain
    and any other fp32 summation order approximate.  Used by the parity tests for rows with 10^5 .. 10^6 nonzeros, where the
    sequential fp32 chain of ``torch.sparse.mm`` is itself further than 1e-5 from the exact sum."""
    indptr = np.asarray(indptr, dtype=np.int64)
    out = np.zeros((indptr.size - 1, x.shape[1]), dtype=np.float64)
    for r in range(indptr.size - 1):
        s, e = int(indptr[r]), int(indptr[r + 1])
        for b in range(s, e, 1 << 18):  # blocks bound the gathered temporary (2^18 x D doubles)
            t = min(e, b + (1 << 18))
            out[r] += np.asarray(data[b:t], dtype=np.float64) @ np.asarray(x[np.asarray(indices[b:t])], dtype=np.float64)
    return out


def lgcn_forward(csr, user_emb, item_emb, n_layers):
    """``LGCN_Encoder.forward`` (model/graph/LightGCN.py:129-140): L propagations, then the mean of
    the L+1 layer outputs (torch.mean over a stacked [N, L+1, D] tensor)."""
    ego = np.concatenate([user_emb, item_emb], 0).astype(np.float32)
    layers = [ego]
    for _ in range(n_layers):
        ego = spmm(*csr, ego)
        layers.append(ego)
    mean = np.mean(np.stack(layers, 1).astype(np.float64), 1).astype(np.float32)
    return mean[: user_emb.shape[0]], mean[user_emb.shape[0]:]


def sht_forward(csr, u_emb, i_emb, u_hyper, i_hyper, n_layers):
    """``SHTEncoder.forward`` (model/graph/SHT.py:192-203): ``embeds = sum_k A^k E`` (k = 0..L), then the low-rank hypergraph
    transform ``embeds @ (hyper.T @ hyper)`` on the user and item halves (float64 accumulation, rounded once)."""
    ego = np.concatenate([u_emb, i_emb], 0).astype(np.float32)
    lats = [ego]
    for _ in range(n_layers):
        lats.append(spmm(*csr, lats[-1]))
    emb = lats[0].copy()
    for t in lats[1:]:
        emb = emb + t
    n_u = u_emb.shape[0]

    def hg(e, h):
        h64 = h.astype(np.float64)
        return (e.astype(np.float64) @ (h64.T @ h64)).astype(np.float32)

    return emb, hg(emb[:n_u], u_hyper), hg(emb[n_u:], i_hyper)


def dhcf_forward(r_csr, u_emb, i_emb, n_layers, slope):
    """``DHCF_Encoder.forward`` (model/graph/DHCF.py:170-186): per layer ``leaky(R (R^T U))`` and ``leaky(R^T (R I))`` of the INPUT
    tables (the reference does not chain the layers), concatenated after the inputs along the feature axis.  ``r_csr`` is the
    ``[users, items]`` interaction matrix (the reference densifies it; the products are the same sums)."""
    rt = csr_transpose(*r_csr, i_emb.shape[0])
    us, its = [u_emb], [i_emb]
    for _ in range(n_layers):
        us.append(hgconv(r_csr, u_emb, slope, csr_t=rt))
        its.append(hgconv(rt, i_emb, slope, csr_t=r_csr))
    return np.concatenate(us, 1), np.concatenate(its, 1)


def leaky_relu(x, slope):
    return np.where(x >= 0, x, x * np.float32(slope)).astype(np.float32)


def hgconv(csr, x, slope=None, csr_t=None):
    """``HGCNConv.forward`` (model/graph/HGNN_HD3.py:540-553): ``act(A (A^T X))``; ``slope=None``
    is the ``act=False`` branch.  ``csr_t`` (the CSR of A^T) defaults to a fresh transpose."""
    if csr_t is None:
        csr_t = csr_transpose(*csr, x.shape[0])
    y = spmm(*csr, spmm(*csr_t, x))
    return y if slope is None else leaky_relu(y, slope)


def layer_norm(x, gamma, beta, eps=1e-5):
    x64 = x.astype(np.float64)
    mu = x64.mean(-1, keepdims=True)
    var = ((x64 - mu) ** 2).mean(-1, keepdims=True)
    return ((x64 - mu) / np.sqrt(var + eps) * gamma.astype(np.float64) + beta.astype(np.float64)).astype(np.float32)


def equiv_set_conv(csr, x, params, prefix="", csr_t=None):
    """``EquivSetConv.forward`` (model/graph/HGNN_HD3.py:705-720) with the reference's fixed
    hyper-parameters (W1 = identity, W2 = slice of the concat, AdaptiveAvgPool1d(D) = identity,
    alpha = 0, W = Linear(LayerNorm(.)), HGCNConv slope 0.5)."""
    g = lambda k: params[prefix + k]
    xe = layer_norm(hgconv(csr, x, 0.5, csr_t), g("lns.0.weight"), g("lns.0.bias")) + x
    xv = layer_norm(hgconv(csr, xe, 0.5, csr_t), g("lns.1.weight"), g("lns.1.bias")) + xe
    h = layer_norm(xv, g("W.normalizations.0.weight"), g("W.normalizations.0.bias"))
    return (h.astype(np.float64) @ g("W.lins.0.weight").astype(np.float64).T + g("W.lins.0.bias")).astype(np.float32)


def equiv_set_gnn(csr, x, params, prefix="", csr_t=None):
    """``EquivSetGNN.forward`` (model/graph/HGNN_HD3.py:596-610) in eval mode (dropout = identity)."""
    g = lambda k: params[prefix + k]
    h = np.maximum((x.astype(np.float64) @ g("lin_in.weight").astype(np.float64).T + g("lin_in.bias")).astype(np.float32), 0)
    h = equiv_set_conv(csr, h, params, prefix + "conv.", csr_t)
    return np.maximum(h, 0)


def local_aware_encoder(csr, ego, params, n_layers, n_users, csr_t=None):
    """``LocalAwareEncoder.forward`` (model/graph/HGNN_HD3.py:410-427), eval mode."""
    res = ego
    for k in range(n_layers):
        if k != n_layers - 1:
            ego = equiv_set_gnn(csr, ego, params, "edhnn_layers.%d." % k, csr_t) + res
        else:
            ego = layer_norm(hgconv(csr, ego, None, csr_t), params["lns.%d.weight" % k], params["lns.%d.bias" % k]) + res
    return ego[:n_users], ego[n_users:]


def hyperedge(adj, emb):
    """``HGNNLayer.forward`` (model/graph/HCCF.py:206-211): ``adj @ (adj.T @ emb)`` for the dense learned incidence
    ``adj [n, hyper_dim]``, accumulated in float64 and rounded once (the reference's fp32 BLAS order is unspecified)."""
    a = np.asarray(adj, dtype=np.float64)
    return (a @ (a.T @ np.asarray(emb, dtype=np.float64))).astype(np.float32)


def hyperedge_grads(adj, emb, dy):
    """Gradients of ``sum(hyperedge(adj, emb) * dy)`` w.r.t. ``adj`` and ``emb`` (float64)."""
    a, e, g = (np.asarray(v, dtype=np.float64) for v in (adj, emb, dy))
    t, dt = a.T @ e, a.T @ g
    return (g @ t.T + e @ dt.T).astype(np.float32), (a @ dt).astype(np.float32)


def hccf_forward(csr, params, n_layers, n_users):
    """``HCCFEncoder.forward`` (model/graph/HCCF.py:173-191) with keep_rate = 1 and dropout off."""
    ue, ie = params["embedding_dict.user_emb"], params["embedding_dict.item_emb"]
    hidden = [np.concatenate([ue, ie], 0)]
    hu = (ue.astype(np.float64) @ params["embedding_dict.user_w"].astype(np.float64)).astype(np.float32)
    hi = (ie.astype(np.float64) @ params["embedding_dict.item_w"].astype(np.float64)).astype(np.float32)
    gcn_h, hyp_h = [], []

    hgnn = hyperedge

    for _ in range(n_layers):
        gcn = spmm(*csr, hidden[-1])
        hyp = np.concatenate([hgnn(hu, hidden[-1][:n_users]), hgnn(hi, hidden[-1][n_users:])], 0)
        gcn_h.append(gcn)
        hyp_h.append(hyp)
        hidden.append(gcn + hyp)
    emb = hidden[0].copy()
    for h in hidden[1:]:
        emb = emb + h
    return emb[:n_users], emb[n_users:], gcn_h, hyp_h


def scatter_mean_conv(v, e, x, n_nodes):
    """Scatter form of ED-HNN message passing (model/layers/layers2/EquivSetConv2.py:85-100) with
    identity MLPs and alpha = 0: ``Xe = segment_mean_E(X[V])``, ``Xv = segment_mean_V(Xe[E])``;
    an empty segment yields 0 (pytorch-scatter 2.1.0 ``scatter(reduce='mean')``)."""
    d = x.shape[1]
    n_e = int(e.max()) + 1
    xe = np.zeros((n_e, d), dtype=np.float64)
    np.add.at(xe, e, x[v].astype(np.float64))
    xe /= np.maximum(np.bincount(e, minlength=n_e), 1)[:, None]
    xe = xe.astype(np.float32)
    xv = np.zeros((n_nodes, d), dtype=np.float64)
    np.add.at(xv, v, xe[e].astype(np.float64))
    xv /= np.maximum(np.bincount(v, minlength=n_nodes), 1)[:, None]
    return xv.astype(np.float32)


# --------------------------------------------------------------------------------------------
# (a-8, a-9) losses with analytic gradients            util/loss_torch.py:5-9,17-21,32-40,103-110
def scatter_mean_conv_weighted(v, e, x, att, n_nodes):
    """The attention-weighted scatter convolution (model/graph/HD2.py:624-643 with W1 = identity, W2 = slice, alpha = 0,
    before W): ``Xe = segment_mean_E(X[V] * att)``, ``Xv = segment_mean_V(Xe[E])``; ``att`` is one weight per (v, e) pair."""
    d = x.shape[1]
    n_e = int(e.max()) + 1
    xe = np.zeros((n_e, d), dtype=np.float64)
    np.add.at(xe, e, (x[v] * np.asarray(att, dtype=np.float32).reshape(-1, 1)).astype(np.float64))
    xe = (xe / np.maximum(np.bincount(e, minlength=n_e), 1)[:, None]).astype(np.float32)
    xv = np.zeros((n_nodes, d), dtype=np.float64)
    np.add.at(xv, v, xe[e].astype(np.float64))
    return (xv / np.maximum(np.bincount(v, minlength=n_nodes), 1)[:, None]).astype(np.float32)


def _mlp_w(x, params, prefix):
    """``MLP`` with one layer and InputNorm (model/layers/MLP.py:109-117): ``Linear(LayerNorm(x))``."""
    h = layer_norm(x, params[prefix + "normalizations.0.weight"], params[prefix + "normalizations.0.bias"])
    return (h.astype(np.float64) @ params[prefix + "lins.0.weight"].astype(np.float64).T + params[prefix + "lins.0.bias"]).astype(np.float32)


def equiv_set_gnn_scatter(v, e, x, params, prefix, n_nodes):
    """``EquivSetGNN.forward`` of the scatter form in eval mode (model/layers/layers2/EquivSetGNN2.py:83-103 =
    model/graph/HCCF_diffusion.py:358-380): ``relu(lin_in(x))`` -> scatter convolution -> ``W`` -> ``relu``."""
    h = np.maximum((x.astype(np.float64) @ params[prefix + "lin_in.weight"].astype(np.float64).T + params[prefix + "lin_in.bias"]).astype(np.float32), 0)
    return np.maximum(_mlp_w(scatter_mean_conv(v, e, h, n_nodes), params, prefix + "conv.W."), 0)


def hd4_local_aware_encoder(csr, ui_pattern, ego, params, n_layers, n_users):
    """``LocalAwareEncoder.forward`` of HGNN_HD4 (model/graph/HGNN_HD4.py:391-405), eval mode: every layer but the last is the
    scatter-form ``EquivSetGNN2`` over ``(V, E) = nonzero(ui_adj > 0)`` (EquivSetGNN2.py:105-133) plus the residual; the last is
    ``lns[0](HGCNConv(norm_adj, act=False)) + res``.  ``ui_pattern`` = (indptr, indices) of the bipartite adjacency."""
    ip, ix = ui_pattern
    v = np.repeat(np.arange(ip.size - 1), np.diff(ip))
    e = np.asarray(ix)
    res = ego
    for k in range(n_layers):
        if k != n_layers - 1:
            ego = equiv_set_gnn_scatter(v, e, ego, params, "edhnn_layers.%d." % k, ego.shape[0]) + res
        else:
            ego = layer_norm(hgconv(csr, ego, None), params["lns.0.weight"], params["lns.0.bias"]) + res
    return ego[:n_users], ego[n_users:]


def hccf_diffusion_forward(csr, params, n_layers, n_users):
    """``HCCFEncoder.forward`` of HCCF_diffusion (model/graph/HCCF_diffusion.py:197-217) with keep_rate = 1 and dropout off:
    per layer ``gcn = A h``; the hypergraph branch is the scatter-form EquivSetGNN over the SIGN pattern of the learned incidence
    ``H = E0 W`` (``generate_V_E``: ``nonzero(H > 0)``, :382-402), users and items separately, one shared ``edhnnlayer``."""
    ue, ie = params["embedding_dict.user_emb"], params["embedding_dict.item_emb"]
    hidden = [np.concatenate([ue, ie], 0)]
    pats = []
    for emb, w in ((ue, params["embedding_dict.user_w"]), (ie, params["embedding_dict.item_w"])):
        h = (emb.astype(np.float64) @ w.astype(np.float64)).astype(np.float32)
        nz = np.argwhere(h > 0)
        pats.append((nz[:, 0], nz[:, 1]))
    gcn_h, hyp_h = [], []
    for _ in range(n_layers):
        cur = hidden[-1]
        gcn = spmm(*csr, cur)
        hu = equiv_set_gnn_scatter(pats[0][0], pats[0][1], cur[:n_users], params, "edhnnlayer.", n_users)
        hi = equiv_set_gnn_scatter(pats[1][0], pats[1][1], cur[n_users:], params, "edhnnlayer.", cur.shape[0] - n_users)
        gcn_h.append(gcn)
        hyp_h.append(np.concatenate([hu, hi], 0))
        hidden.append(gcn + hyp_h[-1])
    emb = hidden[0].copy()
    for h in hidden[1:]:
        emb = emb + h
    return emb[:n_users], emb[n_users:], gcn_h, hyp_h


def normalize_graph_mat_hyper(indptr, indices, data, n_cols):
    """``Graph.normalize_graph_mat_hyper`` (data/graph.py:28-42) in FACTORED form: ``left = (Dv^-1/2 H) De^-1`` and
    ``right = H^T Dv^-1/2`` as CSR triples, each value with scipy's roundings; the reference's matrix is
    ``(left @ H^T) @ Dv^-1/2 = left @ right``."""
    indptr = np.asarray(indptr, dtype=np.int64)
    indices = np.asarray(indices, dtype=np.int64)
    data = np.asarray(data, dtype=np.float32)
    n_rows = indptr.size - 1
    rows = np.repeat(np.arange(n_rows), np.diff(indptr))
    rowsum = np.zeros(n_rows, dtype=np.float32)
    np.add.at(rowsum, rows, data)
    colsum = np.zeros(n_cols, dtype=np.float32)
    np.add.at(colsum, indices, data)
    with np.errstate(divide="ignore"):
        de = np.power(colsum, np.float32(-1))
        dv = np.power(rowsum, np.float32(-0.5))
    de[np.isinf(de)] = 0
    dv[np.isinf(dv)] = 0
    left = ((dv[rows] * data).astype(np.float32) * de[indices]).astype(np.float32)
    t_ptr, t_idx, t_val = csr_transpose(indptr, indices, data, n_cols)
    right = (t_val * dv[t_idx]).astype(np.float32)
    return (indptr, indices, left), (t_ptr, t_idx, right)


# --------------------------------------------------------------------------------------------
def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def bpr_l2_from_tables(user_tab, item_tab, u, p, n, reg, batch_size):
    """``bpr_loss`` + ``l2_reg_loss / batch_size`` on rows gathered from the tables
    (model/graph/LightGCN.py:52-55).  Returns (rec_loss, reg_loss, dUserTab, dItemTab)."""
    ut, it = user_tab.astype(np.float64), item_tab.astype(np.float64)
    ue, pe, ne = ut[u], it[p], it[n]
    x = (ue * pe).sum(1) - (ue * ne).sum(1)
    s = _sigmoid(x)
    rec = np.mean(-np.log(10e-6 + s))
    nu, np_, nn = np.sqrt((ue ** 2).sum()), np.sqrt((pe ** 2).sum()), np.sqrt((ne ** 2).sum())
    regl = reg * (nu + np_ + nn) / batch_size
    gx = -(s * (1 - s)) / (10e-6 + s) / len(u)
    c = reg / batch_size
    d_ue = gx[:, None] * (pe - ne) + c * ue / nu
    d_pe = gx[:, None] * ue + c * pe / np_
    d_ne = -gx[:, None] * ue + c * ne / nn
    du, di = np.zeros_like(ut), np.zeros_like(it)
    np.add.at(du, u, d_ue)
    np.add.at(di, p, d_pe)
    np.add.at(di, n, d_ne)
    return np.float32(rec), np.float32(regl), du.astype(np.float32), di.astype(np.float32)


def _normalize_rows(x, eps=1e-12):
    nrm = np.maximum(np.sqrt((x ** 2).sum(1, keepdims=True)), eps)
    return x / nrm, nrm


def _normalize_bwd(g, y, nrm):
    """Gradient of y = x / ||x|| w.r.t. x given upstream g."""
    return (g - y * (g * y).sum(1, keepdims=True)) / nrm


def contrast_loss(e1, e2, nodes, temp):
    """``contrastLoss`` (util/loss_torch.py:103-110).  Returns (loss, dE1, dE2); the row
    normalisation runs over the whole tables but only the picked rows receive gradient."""
    a, na = _normalize_rows(e1.astype(np.float64)[nodes] + 1e-8)
    b, nb = _normalize_rows(e2.astype(np.float64)[nodes] + 1e-8)
    logits = a @ b.T / temp
    ex = np.exp(logits)
    deno = ex.sum(1) + 1e-8
    pos = (a * b).sum(1) / temp
    loss = -np.mean(pos - np.log(deno))
    m = len(nodes)
    w = ex / deno[:, None]  # d log(deno) / d logits
    g_logits = w / m
    ga = (-(b / temp) / m) + g_logits @ b / temp
    gb = (-(a / temp) / m) + g_logits.T @ a / temp
    d1, d2 = np.zeros(e1.shape, np.float64), np.zeros(e2.shape, np.float64)
    d1[nodes] = _normalize_bwd(ga, a, na)
    d2[nodes] = _normalize_bwd(gb, b, nb)
    return np.float32(loss), d1.astype(np.float32), d2.astype(np.float32)


def info_nce(v1, v2, temp):
    """``InfoNCE`` (util/loss_torch.py:32-40) with b_cos=True.  Returns (loss, dV1, dV2)."""
    a, na = _normalize_rows(v1.astype(np.float64))
    b, nb = _normalize_rows(v2.astype(np.float64))
    ex = np.exp(a @ b.T / temp)
    ttl = ex.sum(1)
    pos = np.exp((a * b).sum(1) / temp)
    ratio = pos / ttl
    loss = np.mean(-np.log(ratio + 10e-6))
    m = a.shape[0]
    g_ratio = -1.0 / (ratio + 10e-6) / m
    g_pos = g_ratio / ttl
    g_ttl = -g_ratio * pos / ttl ** 2
    g_logits = g_ttl[:, None] * ex / temp
    g_dot = g_pos * pos / temp
    ga = g_dot[:, None] * b + g_logits @ b
    gb = g_dot[:, None] * a + g_logits.T @ a
    return np.float32(loss), _normalize_bwd(ga, a, na).astype(np.float32), _normalize_bwd(gb, b, nb).astype(np.float32)


# --------------------------------------------------------------------------------------------
# (a-10) full-ranking evaluation     base/graph_recommender.py:61-92, util/algorithm.py:143-173
# --------------------------------------------------------------------------------------------
def scores(user_vec, item_emb):
    user_vec = np.ascontiguousarray(user_vec, dtype=np.float32)
    item_emb = np.ascontiguousarray(item_emb, dtype=np.float32)
    out = np.empty(item_emb.shape[0], dtype=np.float32)
    _lib().hgr_oracle_scores_f32(_p(user_vec, ctypes.c_float), _p(item_emb, ctypes.c_float), item_emb.shape[0],
                                 item_emb.shape[1], _p(out, ctypes.c_float))
    return out


def find_k_largest(k, cand):
    """Literal ``find_k_largest`` including the duplicate quirk (SURVEY.md F9)."""
    cand = np.ascontiguousarray(cand, dtype=np.float32)
    ids, sc = np.zeros(k, dtype=np.int64), np.zeros(k, dtype=np.float32)
    _lib().hgr_oracle_find_k_largest(k, _p(cand, ctypes.c_float), cand.size, _p(ids, ctypes.c_int64), _p(sc, ctypes.c_float))
    return ids, sc


def topk_exact(k, cand):
    cand = np.ascontiguousarray(cand, dtype=np.float32)
    ids, sc = np.zeros(k, dtype=np.int64), np.zeros(k, dtype=np.float32)
    _lib().hgr_oracle_topk_exact(k, _p(cand, ctypes.c_float), cand.size, _p(ids, ctypes.c_int64), _p(sc, ctypes.c_float))
    return ids, sc


def fullrank_topk(user_emb, item_emb, test_users, train_indptr, train_indices, k, mode="exact"):
    """``GraphRecommender.test`` (base/graph_recommender.py:61-92) for dense user ids: score every
    item, overwrite the user's training items with -10e8, take the top ``k``.  ``mode='exact'`` is
    the true top-k (ties by ascending id); ``mode='refquirk'`` replays ``find_k_largest``."""
    ids = np.zeros((len(test_users), k), dtype=np.int64)
    sc = np.zeros((len(test_users), k), dtype=np.float32)
    pick = topk_exact if mode == "exact" else find_k_largest
    for r, u in enumerate(test_users):
        c = scores(user_emb[u], item_emb)
        c[train_indices[train_indptr[u]:train_indptr[u + 1]]] = MASK_SCORE
        ids[r], sc[r] = pick(k, c)
    return ids, sc


def ranking_evaluation(test_items, rec_ids, top_n):
    """``ranking_evaluation`` + ``Metric`` (util/evaluation.py:9-15,18-30,45-53,85-97,158-185).
    ``test_items[r]`` is the list of ground-truth item ids of the r-th test user in test-file
    order, ``rec_ids[r]`` the recommended ids.  Returns the reference's list of strings."""
    out = []
    for n in top_n:
        hits, total, recall_sum, ndcg_sum = [], 0, 0, 0
        for truth, rec in zip(test_items, rec_ids):
            pred = list(rec[:n])
            tset = set(truth)  # dict keys in the reference: unique, insertion-ordered
            uniq_truth = list(dict.fromkeys(truth))
            h = len(tset.intersection(set(pred)))
            hits.append(h)
            total += len(uniq_truth)
            dcg = 0
            for pos, it in enumerate(pred):
                if it in tset:
                    dcg += 1.0 / math.log(pos + 2, 2)
            idcg = 0
            for pos in range(len(uniq_truth[:n])):
                idcg += 1.0 / math.log(pos + 2, 2)
            ndcg_sum += dcg / idcg
        recall_list = [h / len(dict.fromkeys(t)) for h, t in zip(hits, test_items)]
        out.append("Top " + str(n) + "\n")
        out.append("Hit Ratio:" + str(round(sum(hits) / total, 5)) + "\n")
        out.append("Precision:" + str(round(sum(hits) / (len(hits) * n), 5)) + "\n")
        out.append("Recall:" + str(round(sum(recall_list) / len(recall_list), 5)) + "\n")
        out.append("NDCG:" + str(round(ndcg_sum / len(hits), 5)) + "\n")
    return out


# ------------------------------------------------------------------------------------------------ data layer
def load_data_set(path):
    """``FileIO.load_data_set`` (data/loader.py:24-38): header skipped, tab-or-comma split per line, weight 1."""
    from re import split

    data = []
    with open(path) as f:
        next(f)
        for line in f:
            items = split(',', line.strip()) if '\t' not in line else split('\t', line.strip())
            data.append([int(items[0]), int(items[1]), 1.0])
    return data


def generate_set(training_data, test_data):
    """``Interaction.__generate_set`` (data/ui_graph.py:43-68), the python loop itself: dense ids by first appearance,
    dict-of-dict training / test sets (a rewritten pair keeps its slot and takes the new rating), ``user_history_dict``
    lists for rating-1 entries, test entries of unknown users skipped.  Returns plain dicts / a set."""
    user, item, id2user, id2item = {}, {}, {}, {}
    training_set_u, training_set_i, test_set, history = {}, {}, {}, {}
    test_set_item = set()
    for u, i, r in training_data:
        u, i = int(u), int(i)
        if u not in user:
            user[u] = len(user)
            id2user[user[u]] = u
        if i not in item:
            item[i] = len(item)
            id2item[item[i]] = i
        if r == 1.0:
            history.setdefault(u, []).append(i)
        training_set_u.setdefault(u, {})[i] = r
        training_set_i.setdefault(i, {})[u] = r
    for u, i, r in test_data:
        if u not in user:
            continue
        test_set.setdefault(u, {})[i] = r
        test_set_item.add(i)
    return dict(user=user, item=item, id2user=id2user, id2item=id2item, training_set_u=training_set_u,
                training_set_i=training_set_i, test_set=test_set, user_history_dict=history, test_set_item=test_set_item)
