"""Full-ranking evaluation on libhgr.so: the drop-in for ``GraphRecommender.test`` and ``util.evaluation``.

Reference call sites replaced (paths relative to HD_SELFRec/):

==============================  ==================================================================
``fullrank_topk``                the body of ``GraphRecommender.test`` -- base/graph_recommender.py:61-92
                                 (= base/main_recommender.py:64-100): ``predict`` (model/graph/LightGCN.py:99-102),
                                 the ``candidates[train item] = -10e8`` loop (:78-80) and ``find_k_largest``
                                 (util/algorithm.py:143-173), for ALL test users in one call
``EvalData``                     the parts of ``Interaction`` the loop touches (data/ui_graph.py:18-68,149-150):
                                 ``test_set`` order, ``user``/``item``/``id2item`` maps, ``user_rated``
``test``                         returns the same ``rec_list`` dict ``{raw_user: [(raw_item, score), ...]}``
``ranking_evaluation``           util/evaluation.py:158-185 with ``Metric.hits/hit_ratio/precision/recall/NDCG``
                                 (:9-15,18-30,45-53,85-97): same list of strings, same 5-decimal rounding
``ranking_evaluation_ids``       the same strings straight from the ``[n_test, K]`` id matrix (no dicts)
==============================  ==================================================================

Top-K semantics (include/hgr.h): ``mode='exact'`` is the true top-K (score descending, ties by ascending
item id); ``mode='refquirk'`` replays ``find_k_largest`` as shipped, duplicates included (SURVEY.md F9).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib

MODES = {"exact": 0, "refquirk": 1}
ENGINES = {"auto": 0, "simt": 1, "tensor": 2}


def fullrank_topk(user_emb: torch.Tensor, item_emb: torch.Tensor, test_users: torch.Tensor, train_indptr: torch.Tensor,
                  train_indices: torch.Tensor, k: int, mode: str = "exact", engine: str = "auto", return_stats: bool = False):
    """Top-``k`` items for every test user.  Returns device tensors ``(ids int32 [n_test, k], scores float32
    [n_test, k])`` (+ a uint64[4] stats tensor).  ``train_indptr`` (int64 [n_users + 1]) / ``train_indices``
    (int32, ascending inside a row) are the training interaction matrix used as the mask.  ``k`` goes to the C ABI unchanged:
    both modes take ``k <= 256`` (the tensor-core path when the width is 64), ``mode='exact'`` also any larger ``k`` (SIMT path)."""
    if not (user_emb.is_cuda and item_emb.is_cuda):
        raise _lib.HgrError("embedding tables must be CUDA tensors (no CPU path)")
    if user_emb.dtype != torch.float32 or item_emb.dtype != torch.float32 or user_emb.dim() != 2 or item_emb.dim() != 2:
        raise TypeError("embedding tables must be 2-D float32")
    if user_emb.shape[1] != item_emb.shape[1]:
        raise ValueError("user and item embeddings differ in width")
    dev = user_emb.device
    user_emb, item_emb = user_emb.detach().contiguous(), item_emb.detach().contiguous()
    test_users = test_users.to(device=dev, dtype=torch.int32).contiguous()
    train_indptr = train_indptr.to(device=dev, dtype=torch.int64).contiguous()
    train_indices = train_indices.to(device=dev, dtype=torch.int32).contiguous()
    if train_indptr.numel() != user_emb.shape[0] + 1:
        raise ValueError("train_indptr must have n_users + 1 entries")
    n_test, n_items, d = int(test_users.numel()), int(item_emb.shape[0]), int(user_emb.shape[1])
    lib = _lib.lib()
    ids = torch.empty((n_test, k), dtype=torch.int32, device=dev)
    scores = torch.empty((n_test, k), dtype=torch.float32, device=dev)
    stats = torch.zeros(4, dtype=torch.int64, device=dev)
    ws_bytes = int(lib.hgr_fullrank_topk_workspace_bytes(n_test, n_items, d, k, ENGINES[engine]))
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
    off = (-ws.data_ptr()) % 256
    _lib.check(lib.hgr_fullrank_topk_f32(user_emb.data_ptr(), user_emb.shape[0], item_emb.data_ptr(), n_items, d,
                                         test_users.data_ptr(), n_test, train_indptr.data_ptr(), _lib.ptr(train_indices), k,
                                         MODES[mode], ENGINES[engine], ids.data_ptr(), scores.data_ptr(), stats.data_ptr(),
                                         ws.data_ptr() + off, ws_bytes, _lib.stream_ptr()))
    ws.record_stream(torch.cuda.current_stream())
    return (ids, scores, stats) if return_stats else (ids, scores)


class EvalData:
    """Device-side view of what ``GraphRecommender.test`` reads from ``Interaction``: the test users in
    ``test_set`` order, the training matrix as the mask, raw-id maps for building ``rec_list``."""

    def __init__(self, data, device="cuda"):
        dev = torch.device(device)
        self.data = data
        if hasattr(data, "eval_arrays"):  # the array-backed façade (data.Interaction): no python loop over interactions
            users, self.raw_users, self.truth_indptr, self.truth_items, self.id2item = data.eval_arrays()
            self.test_users = torch.from_numpy(users.astype(np.int32)).to(dev)
            mask = data.interaction_mat  # DeviceCSR, user -> sorted training items
            self.train_indptr, self.train_indices = mask.indptr, mask.indices
            return
        self.raw_users = list(data.test_set.keys())
        self.test_users = torch.tensor([data.user[u] for u in self.raw_users], dtype=torch.int32, device=dev)
        mat = data.interaction_mat.tocsr()
        if not mat.has_sorted_indices:
            mat = mat.copy()
            mat.sort_indices()
        self.train_indptr = torch.from_numpy(mat.indptr.astype(np.int64)).to(dev)
        self.train_indices = torch.from_numpy(mat.indices.astype(np.int32)).to(dev)
        self.id2item = np.array([data.id2item[i] for i in range(data.n_items)])
        # ground truth as CSR over test users: dense item id, or -1 for items never seen in training
        truth, ptr = [], [0]
        for u in self.raw_users:
            truth.extend(data.item.get(it, -1) for it in data.test_set[u])
            ptr.append(len(truth))
        self.truth_indptr = np.asarray(ptr, dtype=np.int64)
        self.truth_items = np.asarray(truth, dtype=np.int64)

    @classmethod
    def from_arrays(cls, n_users, n_items, train_u, train_i, test_u, test_i, device="cuda"):
        """Build from dense id arrays (synthetic graphs): test users in order of first appearance."""
        self = cls.__new__(cls)
        dev = torch.device(device)
        order = np.lexsort((train_i, train_u))
        tu, ti = np.asarray(train_u)[order], np.asarray(train_i)[order]
        keep = np.ones(tu.size, dtype=bool)
        keep[1:] = (tu[1:] != tu[:-1]) | (ti[1:] != ti[:-1])
        tu, ti = tu[keep], ti[keep]
        indptr = np.zeros(n_users + 1, dtype=np.int64)
        np.cumsum(np.bincount(tu, minlength=n_users), out=indptr[1:])
        self.train_indptr = torch.from_numpy(indptr).to(dev)
        self.train_indices = torch.from_numpy(ti.astype(np.int32)).to(dev)
        test_u, test_i = np.asarray(test_u), np.asarray(test_i)
        uniq, first = np.unique(test_u, return_index=True)
        users = uniq[np.argsort(first, kind="stable")]
        self.raw_users = users.tolist()
        self.test_users = torch.from_numpy(users.astype(np.int32)).to(dev)
        o = np.argsort(test_u, kind="stable")
        su, si = test_u[o], test_i[o]
        starts = np.searchsorted(su, users, side="left")
        ends = np.searchsorted(su, users, side="right")
        self.truth_indptr = np.zeros(users.size + 1, dtype=np.int64)
        np.cumsum(ends - starts, out=self.truth_indptr[1:])
        self.truth_items = np.concatenate([si[a:b] for a, b in zip(starts, ends)]).astype(np.int64) if users.size else np.zeros(0, np.int64)
        self.id2item = np.arange(n_items)
        self.data = None
        return self


def test(recommender, user_emb: torch.Tensor, item_emb: torch.Tensor, mode: str = "refquirk", engine: str = "auto"):
    """Drop-in body for ``GraphRecommender.test``: ``rec_list[raw_user] = [(raw_item, score), ...]`` of length
    ``recommender.max_N`` for every user of ``recommender.data.test_set``.  ``mode='refquirk'`` (default here)
    reproduces the reference's lists exactly; ``'exact'`` gives the duplicate-free top-K.  ``max_N`` up to 256 works in both
    modes (``fullrank_topk``)."""
    ev = getattr(recommender, "_hgr_eval_data", None)
    if ev is None:
        ev = EvalData(recommender.data, device=user_emb.device)
        recommender._hgr_eval_data = ev
    ids, scores = fullrank_topk(user_emb, item_emb, ev.test_users, ev.train_indptr, ev.train_indices, int(recommender.max_N),
                                mode=mode, engine=engine)
    ids_h, scores_h = ids.cpu().numpy(), scores.cpu().numpy()  # one D2H of [n_test, K] instead of n_items floats per user
    names = ev.id2item[ids_h]
    return {u: list(zip(names[r].tolist(), scores_h[r])) for r, u in enumerate(ev.raw_users)}


# ------------------------------------------------------------------------------------------------
# metrics (host logic; util/evaluation.py)
# ------------------------------------------------------------------------------------------------
def ranking_evaluation(origin, res, N):
    """Reference signature: ``origin[user] = {item: rating}``, ``res[user] = [(item, score), ...]``."""
    if len(origin) != len(res):
        print('The Lengths of test set and predicted set do not match!')
        raise SystemExit(-1)
    users = list(res.keys())
    item_index = {}
    truth, tptr, pred = [], [0], []
    max_n = max(N)

    def idx(it):
        return item_index.setdefault(it, len(item_index))

    for u in users:
        truth.extend(idx(it) for it in origin[u])
        tptr.append(len(truth))
        row = [idx(p[0]) for p in res[u][:max_n]]
        pred.append(row + [-2] * (max_n - len(row)))
    # metric sums follow the iteration order of `origin` for hit ratio and of `res` for the rest; all are
    # plain sums over users, accumulated below in `res` order exactly as the reference's loops do
    return ranking_evaluation_ids(np.asarray(tptr, dtype=np.int64), np.asarray(truth, dtype=np.int64),
                                  np.asarray(pred, dtype=np.int64).reshape(len(users), max_n), N)


def ranking_evaluation_ids(truth_indptr, truth_items, rec_ids, N):
    """The reference's metric strings from id matrices.  ``truth_items[truth_indptr[r]:truth_indptr[r+1]]`` are the
    ground-truth item ids of test user ``r`` (unique; -1 = unknown item, never hit), ``rec_ids[r]`` the
    recommended ids, best first.  Every float is produced by the same sequence of double operations as
    ``Metric.*`` so the rounded strings are identical."""
    rec_ids = np.asarray(rec_ids)
    n_users, k = rec_ids.shape
    n_truth = np.diff(truth_indptr)
    # hit matrix: rec_ids[r, j] in truth(r)
    key_t = np.repeat(np.arange(n_users, dtype=np.int64), n_truth) * (1 << 32) + (truth_items.astype(np.int64) & 0xffffffff)
    key_t = np.sort(key_t[truth_items >= 0])
    key_r = (np.arange(n_users, dtype=np.int64)[:, None] * (1 << 32) + (rec_ids.astype(np.int64) & 0xffffffff)).ravel()
    pos = np.searchsorted(key_t, key_r)
    pos[pos >= key_t.size] = max(key_t.size - 1, 0)
    hit = ((key_t[pos] == key_r) if key_t.size else np.zeros(key_r.size, bool)).reshape(n_users, k) & (rec_ids >= 0)
    disc = np.array([1.0 / math.log(n + 2, 2) for n in range(k)], dtype=np.float64)
    measure = []
    for n in N:
        m = min(n, k)  # a list shorter than N is used whole (res[user][:n])
        h = hit[:, :m]
        # Metric.hits counts a SET intersection: a duplicated recommendation (refquirk) counts once
        first = np.ones_like(h)
        for j in range(1, m):
            first[:, j] = ~(rec_ids[:, :j] == rec_ids[:, j:j + 1]).any(axis=1)
        hits = (h & first).sum(axis=1)
        hits_l = hits.tolist()
        total_num = int(n_truth.sum())
        hit_num = 0
        for x in hits_l:
            hit_num += x
        hr = round(hit_num / total_num, 5)
        prec = round(sum(hits_l) / (n_users * n), 5)
        recall_list = [a / b for a, b in zip(hits_l, n_truth.tolist())]
        recall = round(sum(recall_list) / len(recall_list), 5)
        # NDCG sums 1/log2(pos + 2) over EVERY hit position (duplicates included), in position order
        dcg = np.zeros(n_users, dtype=np.float64)
        for j in range(m):
            dcg = np.where(h[:, j], dcg + disc[j], dcg)
        idcg_tab = np.zeros(max(k, n) + 1, dtype=np.float64)
        acc = 0
        for j in range(max(k, n)):
            acc += 1.0 / math.log(j + 2, 2)
            idcg_tab[j + 1] = acc
        idcg = idcg_tab[np.minimum(n_truth, n)]
        sum_ndcg = 0
        for x in (dcg / idcg).tolist():
            sum_ndcg += x
        ndcg = round(sum_ndcg / n_users, 5)
        measure.append('Top ' + str(n) + '\n')
        measure += ['Hit Ratio:' + str(hr) + '\n', 'Precision:' + str(prec) + '\n', 'Recall:' + str(recall) + '\n',
                    'NDCG:' + str(ndcg) + '\n']
    return measure


def ranking_evaluation_device(truth_indptr, truth_items, rec_ids: torch.Tensor, N, host_sums: bool = False):
    """``ranking_evaluation_ids`` on the device: the per-user work (set intersections, DCG: ``hgr_rank_metrics``) AND the sums
    over users (``hgr_rank_metric_sums``: one thread per sum adds the users' terms in the reference's order, python's
    ``sum()`` arithmetic included), so only ``3 x len(N)`` numbers come back and the strings are identical to
    ``ranking_evaluation``.  ``host_sums=True`` keeps the sums in python loops (the cross-check of the device reducer)."""
    import sys

    dev = rec_ids.device
    rec_ids = rec_ids.to(torch.int32).contiguous()
    n_users, k = rec_ids.shape
    tp_dev = torch.as_tensor(np.asarray(truth_indptr, dtype=np.int64)).to(dev)
    ti = torch.as_tensor(np.asarray(truth_items, dtype=np.int64)).to(dev)
    n_truth = (tp_dev[1:] - tp_dev[:-1])
    # sort every truth row ascending (row id is the major key), on the device
    rows = torch.repeat_interleave(torch.arange(n_users, dtype=torch.int64, device=dev), n_truth)
    ti_sorted = (torch.sort(rows * (1 << 32) + (ti + 1)).values & 0xffffffff).sub_(1).to(torch.int32)
    top = sorted(int(n) for n in N)
    top_dev = torch.tensor(top, dtype=torch.int32, device=dev)
    disc = torch.tensor([1.0 / math.log(p + 2, 2) for p in range(k)], dtype=torch.float64, device=dev)
    hits = torch.empty((n_users, len(top)), dtype=torch.int32, device=dev)
    dcg = torch.empty((n_users, len(top)), dtype=torch.float64, device=dev)
    lib = _lib.lib()
    _lib.check(lib.hgr_rank_metrics(rec_ids.data_ptr(), n_users, k, tp_dev.data_ptr(), ti_sorted.data_ptr(), top_dev.data_ptr(),
                                    len(top), disc.data_ptr(), hits.data_ptr(), dcg.data_ptr(), _lib.stream_ptr()))
    total_num = int(n_truth.sum())
    idcg_tab = [0.0]
    for j in range(max(max(top), k)):
        idcg_tab.append(idcg_tab[-1] + 1.0 / math.log(j + 2, 2))
    if host_sums:
        hits_h, dcg_h = hits.cpu().numpy(), dcg.cpu().numpy()
        n_truth_l = n_truth.tolist()
    else:
        idcg_dev = torch.tensor(idcg_tab, dtype=torch.float64, device=dev)
        hit_sum = torch.empty(len(top), dtype=torch.int64, device=dev)
        rec_sum = torch.empty(len(top), dtype=torch.float64, device=dev)
        ndcg_sum = torch.empty(len(top), dtype=torch.float64, device=dev)
        _lib.check(lib.hgr_rank_metric_sums(hits.data_ptr(), dcg.data_ptr(), tp_dev.data_ptr(), n_users, len(top), top_dev.data_ptr(),
                                            idcg_dev.data_ptr(), len(idcg_tab), 1 if sys.version_info >= (3, 12) else 0,
                                            hit_sum.data_ptr(), rec_sum.data_ptr(), ndcg_sum.data_ptr(), _lib.stream_ptr()))
        hit_sum, rec_sum, ndcg_sum = hit_sum.tolist(), rec_sum.tolist(), ndcg_sum.tolist()
    measure = []
    for n in N:
        q = top.index(int(n))
        if host_sums:
            hits_l = hits_h[:, q].tolist()
            hit_num = 0
            for x in hits_l:
                hit_num += x
            recall_list = [a / b for a, b in zip(hits_l, n_truth_l)]
            sum_recall = sum(recall_list)
            sum_ndcg = 0
            for d, m in zip(dcg_h[:, q].tolist(), n_truth_l):
                sum_ndcg += d / idcg_tab[min(m, n)]
        else:
            hit_num, sum_recall, sum_ndcg = hit_sum[q], rec_sum[q], ndcg_sum[q]
        hr = round(hit_num / total_num, 5)
        prec = round(hit_num / (n_users * n), 5)
        recall = round(sum_recall / n_users, 5)
        ndcg = round(sum_ndcg / n_users, 5)
        measure.append('Top ' + str(n) + '\n')
        measure += ['Hit Ratio:' + str(hr) + '\n', 'Precision:' + str(prec) + '\n', 'Recall:' + str(recall) + '\n',
                    'NDCG:' + str(ndcg) + '\n']
    return measure
