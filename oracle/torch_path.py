"""The reference's CPU torch path for the hot path, restated call for call.  TEST INFRASTRUCTURE ONLY.

Used (a) by tests to cross-check gradients of the CUDA path against torch autograd on the same
arithmetic the reference runs, and (b) by ``bench.py`` as the ``cpu_baseline`` / ``--impl reference``
arm: the reference is pure Python over ``torch.sparse.mm`` / ``torch.mm`` / LayerNorm / Adam, and
``/root/reference`` does not exist on the GPU box, so the same sequence of torch calls is restated
here (kind = "port").  Pinned against ``tests/golden/reference_vectors_*.npz`` by
``tests/test_oracle_golden.py::test_torch_path_*``.  Never imported by the product package.

Call sites restated (paths relative to /root/reference/HD_SELFRec):
  base/torch_interface.py:8-12      COO tensor from the scipy CSR (int64 indices, uncoalesced)
  model/graph/LightGCN.py:129-140   LGCN_Encoder.forward
  model/graph/HGNN_HD3.py:540-553   HGCNConv.forward
  model/graph/HGNN_HD3.py:705-720   EquivSetConv.forward (W1 = id, W2 = slice, W = Linear(LN(.)))
  model/graph/HGNN_HD3.py:596-610   EquivSetGNN.forward
  model/graph/HGNN_HD3.py:410-427   LocalAwareEncoder.forward
  util/loss_torch.py:5-9,17-21      bpr_loss, l2_reg_loss
  model/graph/LightGCN.py:49-66     one training step (forward, losses, .item() x3, backward, Adam)
  base/graph_recommender.py:61-92   test(): per-user GEMV, train-item mask, find_k_largest
  util/sampler.py:237-264           next_batch_pairwise: per-sample python rejection loop over random.choice
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import hgr_oracle as O


def coo_from_csr(indptr, indices, data, shape) -> torch.Tensor:
    rows = np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr))
    i = torch.from_numpy(np.stack([rows, np.asarray(indices, dtype=np.int64)]))
    return torch.sparse_coo_tensor(i, torch.from_numpy(np.asarray(data, dtype=np.float32)), tuple(shape))


def bpr_loss(user_emb, pos_item_emb, neg_item_emb):
    pos_score = torch.mul(user_emb, pos_item_emb).sum(dim=1)
    neg_score = torch.mul(user_emb, neg_item_emb).sum(dim=1)
    return torch.mean(-torch.log(10e-6 + torch.sigmoid(pos_score - neg_score)))


def l2_reg_loss(reg, *args):
    emb_loss = 0
    for emb in args:
        emb_loss = emb_loss + torch.norm(emb, p=2)
    return emb_loss * reg


class LGCN(nn.Module):
    def __init__(self, adj, n_users, n_items, emb_size, n_layers):
        super().__init__()
        self.adj, self.n_users, self.layers = adj, n_users, n_layers
        init = nn.init.xavier_uniform_
        self.embedding_dict = nn.ParameterDict({'user_emb': nn.Parameter(init(torch.empty(n_users, emb_size))),
                                                'item_emb': nn.Parameter(init(torch.empty(n_items, emb_size)))})

    def forward(self):
        ego = torch.cat([self.embedding_dict['user_emb'], self.embedding_dict['item_emb']], 0)
        all_emb = [ego]
        for _ in range(self.layers):
            ego = torch.sparse.mm(self.adj, ego)
            all_emb += [ego]
        out = torch.mean(torch.stack(all_emb, dim=1), dim=1)
        return out[:self.n_users], out[self.n_users:]


def hgcnconv(adj, embs, slope=None):
    y = torch.sparse.mm(adj, torch.sparse.mm(adj.t(), embs))
    return y if slope is None else F.leaky_relu(y, slope)


class EquivSetConv(nn.Module):
    def __init__(self, width):
        super().__init__()
        self.lns = nn.ModuleList([nn.LayerNorm(width) for _ in range(2)])
        self.W = nn.ModuleDict({'normalizations': nn.ModuleList([nn.LayerNorm(width)]), 'lins': nn.ModuleList([nn.Linear(width, width)])})

    def forward(self, X, adj):
        Xe = self.lns[0](hgcnconv(adj, X, 0.5)) + X
        Xev = torch.cat([X, Xe], -1)[..., X.shape[-1]:]
        Xv = self.lns[1](hgcnconv(adj, Xev, 0.5)) + Xev
        return self.W['lins'][0](self.W['normalizations'][0](Xv))


class EquivSetGNN(nn.Module):
    def __init__(self, width, dropout=0.5):
        super().__init__()
        self.lin_in = nn.Linear(width, width)
        self.conv = EquivSetConv(width)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x, adj):
        x = self.dropout(x)
        x = F.relu(self.lin_in(x))
        x = self.dropout(x)
        x = F.relu(self.conv(x, adj))
        return self.dropout(x)


class LocalAwareEncoder(nn.Module):
    def __init__(self, adj, n_users, width, n_layers):
        super().__init__()
        self.adj, self.n_users, self.layers = adj, n_users, n_layers
        self.edhnn_layers = nn.ModuleList([EquivSetGNN(width) for _ in range(n_layers)])
        self.lns = nn.ModuleList([nn.LayerNorm(width) for _ in range(n_layers)])

    def forward(self, ego, adj=None):
        adj = self.adj if adj is None else adj
        res = ego
        for k in range(self.layers):
            if k != self.layers - 1:
                ego = self.edhnn_layers[k](ego, adj) + res
            else:
                ego = self.lns[k](hgcnconv(self.adj, ego, None)) + res
        return ego[:self.n_users], ego[self.n_users:]


class HGNNModel(nn.Module):
    """HGNNModel in ``--mode=local_only`` (model/graph/HGNN_HD3.py:248-330): tables + LocalAwareEncoder."""

    def __init__(self, adj, n_users, n_items, width, n_layers):
        super().__init__()
        init = nn.init.xavier_uniform_
        self.embedding_dict = nn.ParameterDict({'user_emb': nn.Parameter(init(torch.empty(n_users, width))),
                                                'item_emb': nn.Parameter(init(torch.empty(n_items, width)))})
        self.hgnn_layer_local = LocalAwareEncoder(adj, n_users, width, n_layers)

    def forward(self):
        ego = torch.cat([self.embedding_dict['user_emb'], self.embedding_dict['item_emb']], 0)
        return self.hgnn_layer_local(ego)


def contrast_loss(embeds1, embeds2, nodes, temp):
    """util/loss_torch.py:103-110."""
    embeds1 = F.normalize(embeds1 + 1e-8, p=2)
    embeds2 = F.normalize(embeds2 + 1e-8, p=2)
    pck1, pck2 = embeds1[nodes], embeds2[nodes]
    nume = torch.exp(torch.sum(pck1 * pck2, dim=-1) / temp)
    deno = torch.exp(pck1 @ pck2.T / temp).sum(-1) + 1e-8
    return -torch.log(nume / deno).mean()


class HCCF(nn.Module):
    """``HCCFEncoder`` (model/graph/HCCF.py:136-226): per layer an edge-dropped GCN propagation plus the learned dense
    hyperedge two-stage on users and items; sum readout; returns the per-layer GCN / hypergraph tables for the SSL loss."""

    def __init__(self, adj, n_users, n_items, width, n_edges, n_layers, drop_rate=0.2):
        super().__init__()
        self.adj, self.n_users, self.n_layers = adj, n_users, n_layers
        init = nn.init.xavier_uniform_
        self.embedding_dict = nn.ParameterDict({
            'user_emb': nn.Parameter(init(torch.empty(n_users, width))), 'item_emb': nn.Parameter(init(torch.empty(n_items, width))),
            'user_w': nn.Parameter(init(torch.empty(width, n_edges))), 'item_w': nn.Parameter(init(torch.empty(width, n_edges)))})
        self.drop_out = nn.Dropout(drop_rate)

    def drop_edges(self, keep_rate):
        if keep_rate == 1.0:
            return self.adj
        adj = self.adj.coalesce()
        vals, idxs = adj.values(), adj.indices()
        mask = ((torch.rand(vals.size()) + keep_rate).floor()).type(torch.bool)  # HCCF.py:217-226
        return torch.sparse_coo_tensor(idxs[:, mask], vals[mask] / keep_rate, adj.shape)

    def forward(self, keep_rate=0.5):
        n_users = self.n_users
        embeddings = torch.cat([self.embedding_dict['user_emb'], self.embedding_dict['item_emb']], 0)
        hidden, gcn_hidden, hgnn_hidden = [embeddings], [], []
        hyper_uu = self.embedding_dict['user_emb'] @ self.embedding_dict['user_w']
        hyper_ii = self.embedding_dict['item_emb'] @ self.embedding_dict['item_w']
        for _ in range(self.n_layers):
            gcn_emb = torch.sparse.mm(self.drop_edges(keep_rate), hidden[-1])
            hu, hi = self.drop_out(hyper_uu), self.drop_out(hyper_ii)
            hyper_uemb = torch.mm(hu, torch.mm(hu.T, hidden[-1][:n_users]))
            hyper_iemb = torch.mm(hi, torch.mm(hi.T, hidden[-1][n_users:]))
            gcn_hidden += [gcn_emb]
            hgnn_hidden += [torch.cat([hyper_uemb, hyper_iemb], 0)]
            hidden += [gcn_emb + hgnn_hidden[-1]]
        embeddings = sum(hidden)
        return embeddings[:n_users], embeddings[n_users:], gcn_hidden, hgnn_hidden


def train_step_hccf(model, optimizer, u_idx, p_idx, n_idx, temp, ss_rate, keep_rate):
    """model/graph/HCCF.py:79-95 with calcLosses (:59-68).  The SSL nodes are the batch's unique user / positive-item ids
    (the shipped code passes the gathered EMBEDDINGS to torch.unique(...long()), which collapses the node set to {0};
    bench.py times the intended computation on both arms and says so in its config)."""
    n_users = model.n_users
    user_emb, item_emb, gcn_l, hyp_l = model(keep_rate=keep_rate)
    rec_loss = bpr_loss(user_emb[u_idx], item_emb[p_idx], item_emb[n_idx])
    un, pn = torch.unique(u_idx), torch.unique(p_idx)
    ssl = 0
    for g, h in zip(gcn_l, hyp_l):
        g = g.detach()
        ssl = ssl + contrast_loss(g[:n_users], h[:n_users], un, temp) + contrast_loss(g[n_users:], h[n_users:], pn, temp)
    ssl = ssl * ss_rate
    loss = rec_loss + ssl
    vals = (loss.item(), rec_loss.item(), float(ssl))
    optimizer.zero_grad()
    loss.backward()
    optimizer.step()
    return vals


def train_step(model, optimizer, u_idx, p_idx, n_idx, reg, batch_size):
    """model/graph/LightGCN.py:49-66 (same body in HGNN_HD3.py:138-160)."""
    user_all, item_all = model()
    ue, pe, ne = user_all[u_idx], item_all[p_idx], item_all[n_idx]
    rec_loss = bpr_loss(ue, pe, ne)
    reg_loss = l2_reg_loss(reg, ue, pe, ne) / batch_size
    loss = rec_loss + reg_loss
    vals = (loss.item(), rec_loss.item(), reg_loss.item())
    optimizer.zero_grad()
    loss.backward()
    optimizer.step()
    return vals


def evaluate_users(user_emb, item_emb, test_users, train_indptr, train_indices, max_n):
    """base/graph_recommender.py:61-92 with LightGCN.predict (:99-102): one GEMV per user, python-side
    masking of the training items, find_k_largest (the C restatement of the numba routine)."""
    rec = np.zeros((len(test_users), max_n), dtype=np.int64)
    for r, u in enumerate(test_users):
        cand = torch.matmul(user_emb[u], item_emb.transpose(0, 1)).cpu().numpy()
        for it in train_indices[train_indptr[u]:train_indptr[u + 1]]:
            cand[it] = -10e8
        rec[r], _ = O.find_k_largest(max_n, cand)
    return rec


def sample_batch_pairwise(users, items, training_set_u, item_list, n_negs=1, choice=None):
    """The per-batch body of ``next_batch_pairwise`` (util/sampler.py:248-263): for every positive pair one python-level
    ``random.choice(item_list)`` redrawn while the item is in the user's training set, then three ``torch.LongTensor``s.
    ``training_set_u[user]`` is any container with hash membership (the reference holds dicts); ids are already dense."""
    import random

    choice = choice or random.choice
    u_idx, i_idx, j_idx = [], [], []
    for k, user in enumerate(users):
        i_idx.append(items[k])
        u_idx.append(user)
        seen = training_set_u[user]
        for _ in range(n_negs):
            neg_item = choice(item_list)
            while neg_item in seen:
                neg_item = choice(item_list)
            j_idx.append(neg_item)
    return torch.LongTensor(u_idx), torch.LongTensor(i_idx), torch.LongTensor(j_idx)
