#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

The reference (DanbiAubrey/Hypergraph_diffusion_for_recommendation, mounted read-only at
/root/reference/HD_SELFRec) has no tests and no golden vectors of its own (SURVEY.md F3), so the
fixtures that pin the oracle are produced here by importing the reference's own classes on CPU
and dumping their inputs and outputs.  Nothing is copied from the reference: it is imported,
called, and only arrays are stored.

    python tests/golden/make_golden.py            # needs /root/reference; rewrites tests/golden/*.npz

Shims (SURVEY.md section 9): ``.cuda()`` becomes the identity on this CPU-only host and
``torch_scatter`` / ``torch_sparse`` (absent here; imported by the HGNN_HD3 module chain) are
stubbed.  The stubs are never on a code path whose output is stored, except
``torch_scatter.scatter`` for the scatter-mean form, which follows pytorch-scatter 2.1.0's
documented semantics (sum via index_add, mean = sum / clamp(count, 1)).
"""
import glob
import os
import random
import sys
import tempfile
import types
import warnings

import numpy as np

REF = os.environ.get("HGR_REFERENCE", "/root/reference/HD_SELFRec")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
warnings.filterwarnings("ignore")


def install_shims():
    import torch

    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self

    ts = types.ModuleType("torch_scatter")

    def scatter(src, index, dim=0, out=None, dim_size=None, reduce="sum"):
        if dim < 0:
            dim += src.dim()
        if dim_size is None:
            dim_size = int(index.max()) + 1
        shape = list(src.shape)
        shape[dim] = dim_size
        res = torch.zeros(shape, dtype=src.dtype)
        res.index_add_(dim, index, src)
        if reduce == "mean":
            cnt = torch.bincount(index, minlength=dim_size).clamp(min=1).to(src.dtype)
            view = [1] * src.dim()
            view[dim] = dim_size
            res = res / cnt.view(view)
        return res

    ts.scatter = scatter
    sys.modules["torch_scatter"] = ts
    tsp = types.ModuleType("torch_sparse")
    tsp.spspmm = tsp.spmm = lambda *a, **k: None
    sys.modules["torch_sparse"] = tsp


def seed_all(s):
    import torch

    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


def csr_parts(m):
    m = m.tocsr()
    return m.indptr.astype(np.int64), m.indices.astype(np.int64), m.data.astype(np.float32)


def main():
    if not os.path.isdir(REF):
        raise SystemExit("reference tree not found at %s" % REF)
    install_shims()
    import torch

    torch.set_num_threads(1)  # sequential accumulation order on CPU
    work = tempfile.mkdtemp(prefix="hgr_golden_")
    os.chdir(work)
    os.symlink(os.path.join(REF, "conf"), "conf")
    os.makedirs("log", exist_ok=True)
    sys.path.insert(0, REF)
    sys.dont_write_bytecode = True

    from data.ui_graph import Interaction
    from data.graph import Graph
    from base.torch_interface import TorchGraphInterface
    from base.graph_recommender import GraphRecommender
    from util.loss_torch import bpr_loss, l2_reg_loss, contrastLoss, InfoNCE
    from util.algorithm import find_k_largest
    from util.evaluation import ranking_evaluation
    from util.sampler import next_batch_pairwise
    from model.graph.LightGCN import LGCN_Encoder
    import model.graph.HGNN_HD3 as HD3
    import model.graph.HCCF as HCCF
    from model.layers.layers2.EquivSetConv2 import EquivSetConv as EquivSetConvScatter

    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions

    out = {}

    # ------------------------------------------------------------------ (i) adjacency, hand graph
    # 3 users (raw 10, 11, 12), 4 train items (raw 100..103); interaction (10,100) is duplicated
    # (scipy sums duplicates -> weight 2), item 104 appears only in the test set, user 13 only in test.
    hand_train = [[10, 100, 1.0], [10, 101, 1.0], [11, 101, 1.0], [10, 100, 1.0], [12, 102, 1.0],
                  [12, 103, 1.0], [11, 103, 1.0], [12, 101, 1.0]]
    hand_test = [[10, 102, 1.0], [11, 104, 1.0], [13, 100, 1.0], [12, 100, 1.0]]
    hand = Interaction(None, [list(t) for t in hand_train], [list(t) for t in hand_test])
    ip, ix, dv = csr_parts(hand.norm_adj)
    out["hand_train"] = np.array(hand_train, dtype=np.float64)
    out["hand_test"] = np.array(hand_test, dtype=np.float64)
    out["hand_norm_indptr"], out["hand_norm_indices"], out["hand_norm_data"] = ip, ix, dv
    ip, ix, dv = csr_parts(hand.ui_adj)
    out["hand_ui_indptr"], out["hand_ui_indices"], out["hand_ui_data"] = ip, ix, dv
    ip, ix, dv = csr_parts(hand.norm_interaction_mat)  # rectangular branch: D^-1 R
    out["hand_normR_indptr"], out["hand_normR_indices"], out["hand_normR_data"] = ip, ix, dv
    ip, ix, dv = csr_parts(Graph.normalize_graph_mat_hyper(hand.interaction_mat))
    out["hand_hyper_indptr"], out["hand_hyper_indices"], out["hand_hyper_data"] = ip, ix, dv
    out["hand_id2user"] = np.array([hand.id2user[k] for k in range(hand.n_users)])
    out["hand_id2item"] = np.array([hand.id2item[k] for k in range(hand.n_items)])

    # ------------------------------------------------------------------ small power-law graph
    g = powerlaw_interactions(60, 90, 600, seed=7)
    train = [[int(u), int(i) + g.n_users, 1.0] for u, i in zip(g.train_u, g.train_i)]
    test = [[int(u), int(i) + g.n_users, 1.0] for u, i in zip(g.test_u, g.test_i)]
    data = Interaction(None, [list(t) for t in train], [list(t) for t in test])
    U, I = data.n_users, data.n_items
    N = U + I
    D = 64
    out["pl_train"] = np.array(train, dtype=np.float64)
    out["pl_test"] = np.array(test, dtype=np.float64)
    out["pl_dense_u"] = np.array([data.user[t[0]] for t in train])
    out["pl_dense_i"] = np.array([data.item[t[1]] for t in train])
    out["pl_id2user"] = np.array([data.id2user[k] for k in range(U)])
    out["pl_id2item"] = np.array([data.id2item[k] for k in range(I)])
    ip, ix, dv = csr_parts(data.norm_adj)
    out["pl_norm_indptr"], out["pl_norm_indices"], out["pl_norm_data"] = ip, ix, dv
    # degree -> d^-1/2 table as numpy computes it on this host (SURVEY.md F10)
    deg = np.asarray(data.ui_adj.sum(1)).flatten().astype(np.float32)
    out["pl_deg"] = deg
    out["pow_lut"] = np.power(np.arange(0, 4097, dtype=np.float32), np.float32(-0.5))
    # SGL-style laplacian of the interaction matrix (data/ui_graph.py:86-93)
    ip, ix, dv = csr_parts(data.convert_to_laplacian_mat(data.interaction_mat))
    out["pl_lap_indptr"], out["pl_lap_indices"], out["pl_lap_data"] = ip, ix, dv
    coo = TorchGraphInterface.convert_sparse_mat_to_tensor(data.norm_adj)
    out["pl_coo_indices"] = coo._indices().numpy()
    out["pl_coo_values"] = coo._values().numpy()

    # ------------------------------------------------------------------ (ii) encoders
    seed_all(11)
    enc = LGCN_Encoder(data, D, 3)
    with torch.no_grad():
        ue, ie = enc()
    out["lgcn_user_emb0"] = enc.embedding_dict["user_emb"].detach().numpy()
    out["lgcn_item_emb0"] = enc.embedding_dict["item_emb"].detach().numpy()
    out["lgcn_user_out"], out["lgcn_item_out"] = ue.numpy(), ie.numpy()
    # one raw propagation and its autograd gradient
    X = torch.randn(N, D, requires_grad=True)
    Y = torch.sparse.mm(enc.sparse_norm_adj, X)
    G = torch.randn(N, D)
    (Y * G).sum().backward()
    out["spmm_X"], out["spmm_Y"], out["spmm_G"], out["spmm_dX"] = X.detach().numpy(), Y.detach().numpy(), G.numpy(), X.grad.numpy()

    # HGCNConv: activation on (slope 0.5) and off
    conv = HD3.HGCNConv(leaky=0.5)
    X2 = torch.randn(N, D, requires_grad=True)
    Ya = conv(enc.sparse_norm_adj, X2, act=True)
    (Ya * G).sum().backward()
    out["hgconv_X"], out["hgconv_Y_act"], out["hgconv_dX_act"] = X2.detach().numpy(), Ya.detach().numpy(), X2.grad.numpy()
    with torch.no_grad():
        out["hgconv_Y_noact"] = conv(enc.sparse_norm_adj, X2, act=False).numpy()

    # EquivSetConv (HGNN_HD3.py:655-720) with the reference's own hyper-parameters
    seed_all(12)
    esc = HD3.EquivSetConv(D, D, U, I, mlp1_layers=0, mlp2_layers=0, mlp3_layers=1, alpha=0.0, aggr="mean",
                           dropout=0.5, normalization="ln", input_norm=True, hypergraph=None, data=data)
    esc.eval()
    for p in esc.parameters():  # non-trivial LayerNorm affine parameters
        p.data = p.data + 0.1 * torch.randn_like(p)
    X3 = torch.randn(N, D, requires_grad=True)
    Y3 = esc(X3, enc.sparse_norm_adj, X3, data.ui_adj)
    (Y3 * G).sum().backward()
    out["esc_X"], out["esc_Y"], out["esc_dX"] = X3.detach().numpy(), Y3.detach().numpy(), X3.grad.numpy()
    for k, v in esc.state_dict().items():
        out["esc_param/" + k] = v.numpy()
    for k, p in esc.named_parameters():
        out["esc_grad/" + k] = p.grad.numpy()

    # LocalAwareEncoder (HGNN_HD3.py:352-427), eval mode (dropout off), 2 layers
    seed_all(13)
    lae = HD3.LocalAwareEncoder(data, D, D, 2, 0.3, 0.2, torch.device("cpu"))
    lae.eval()
    for p in lae.parameters():
        p.data = p.data + 0.05 * torch.randn_like(p)
    E0 = torch.nn.init.xavier_uniform_(torch.empty(N, D)).requires_grad_(True)
    lu, li = lae(E0, lae.sparse_norm_adj)
    (torch.cat([lu, li], 0) * G).sum().backward()
    out["lae_E0"], out["lae_user_out"], out["lae_item_out"], out["lae_dE0"] = E0.detach().numpy(), lu.detach().numpy(), li.detach().numpy(), E0.grad.numpy()
    for k, v in lae.state_dict().items():
        out["lae_param/" + k] = v.numpy()
    for k, p in lae.named_parameters():
        if p.grad is not None:
            out["lae_grad/" + k] = p.grad.numpy()

    # HCCFEncoder (HCCF.py:136-191): keep_rate=1, eval mode => deterministic
    seed_all(14)
    hconf = dict(lrate=0.001, lr_decay=0.9, max_epoch=1, batch_size=64, reg=0.1, embedding_size=D, hyper_dim=32,
                 drop_rate=0.5, p=0.1, n_layers=2)
    hc = HCCF.HCCFEncoder(hconf, data)
    hc.eval()
    hu, hi, gcn_h, hyp_h = hc(keep_rate=1.0)
    for k, v in hc.state_dict().items():
        out["hccf_param/" + k] = v.numpy()
    out["hccf_user_out"], out["hccf_item_out"] = hu.detach().numpy(), hi.detach().numpy()
    for l in range(2):
        out["hccf_gcn_%d" % l] = gcn_h[l].detach().numpy()
        out["hccf_hyp_%d" % l] = hyp_h[l].detach().numpy()
    # SpAdjDropEdge with a replayable mask (HCCF.py:213-226): same torch.rand stream re-drawn here
    seed_all(15)
    dropped = HCCF.SpAdjDropEdge()(hc.sparse_norm_adj, 0.7)
    seed_all(15)
    out["drop_rand"] = torch.rand(hc.sparse_norm_adj._values().size()).numpy()
    out["drop_keep"] = np.float32(0.7)
    out["drop_indices"] = dropped._indices().numpy()
    out["drop_values"] = dropped._values().numpy()
    Xd = torch.randn(N, D)
    out["drop_X"] = Xd.numpy()
    out["drop_Y"] = torch.sparse.mm(dropped, Xd).numpy()
    out["drop_hgconv_Y"] = HD3.HGCNConv(leaky=0.3)(dropped, Xd, act=True).numpy()  # asymmetric A: A (A^T X)

    # scatter-mean form (layers2/EquivSetConv2.py:85-100), W1/W2/W = identity / slice, alpha 0
    seed_all(16)
    esc2 = EquivSetConvScatter(D, D, mlp1_layers=0, mlp2_layers=0, mlp3_layers=0, alpha=0.0, aggr="mean")
    Hd = torch.tensor(np.asarray(data.ui_adj.todense()))
    nz = torch.nonzero(Hd > 0)
    V, E = nz[:, 0], nz[:, 1]
    Xs = torch.randn(N, D)
    out["scat_V"], out["scat_E"], out["scat_X"] = V.numpy(), E.numpy(), Xs.numpy()
    with torch.no_grad():
        out["scat_Y"] = esc2(Xs, V, E, Xs).numpy()

    # ------------------------------------------------------------------ (iii) losses + grads
    seed_all(21)
    random.seed(21)
    batch = next(next_batch_pairwise(data, 128))
    u_idx, p_idx, n_idx = batch
    out["tri_u"], out["tri_p"], out["tri_n"] = u_idx.numpy(), p_idx.numpy(), n_idx.numpy()
    ut = torch.randn(U, D, requires_grad=True)
    it = torch.randn(I, D, requires_grad=True)
    ue_, pe_, ne_ = ut[u_idx], it[p_idx], it[n_idx]
    rec = bpr_loss(ue_, pe_, ne_)
    reg = l2_reg_loss(0.1, ue_, pe_, ne_) / 2048
    (rec + reg).backward()
    out["loss_user_tab"], out["loss_item_tab"] = ut.detach().numpy(), it.detach().numpy()
    out["loss_bpr"], out["loss_reg"] = rec.detach().numpy(), reg.detach().numpy()
    out["loss_reg_lambda"], out["loss_reg_batch_size"] = np.float32(0.1), np.int64(2048)
    out["loss_dU"], out["loss_dI"] = ut.grad.numpy(), it.grad.numpy()

    e1 = torch.randn(U, D, requires_grad=True)
    e2 = torch.randn(U, D, requires_grad=True)
    nodes = torch.unique(u_idx)
    cl = contrastLoss(e1, e2, nodes, 0.2)
    cl.backward()
    out["cl_e1"], out["cl_e2"], out["cl_nodes"], out["cl_temp"] = e1.detach().numpy(), e2.detach().numpy(), nodes.numpy(), np.float32(0.2)
    out["cl_loss"], out["cl_d1"], out["cl_d2"] = cl.detach().numpy(), e1.grad.numpy(), e2.grad.numpy()
    v1 = torch.randn(96, D, requires_grad=True)
    v2 = torch.randn(96, D, requires_grad=True)
    nce = InfoNCE(v1, v2, 0.2)
    nce.backward()
    out["nce_v1"], out["nce_v2"], out["nce_temp"] = v1.detach().numpy(), v2.detach().numpy(), np.float32(0.2)
    out["nce_loss"], out["nce_d1"], out["nce_d2"] = nce.detach().numpy(), v1.grad.numpy(), v2.grad.numpy()

    # sampler stream for replay: python `random` state -> triples (util/sampler.py:237-264)
    random.seed(33)
    samp = list(next_batch_pairwise(data, 256))
    out["samp_u"] = np.concatenate([b[0].numpy() for b in samp])
    out["samp_p"] = np.concatenate([b[1].numpy() for b in samp])
    out["samp_n"] = np.concatenate([b[2].numpy() for b in samp])

    # ------------------------------------------------------------------ (iv) find_k_largest
    rng = np.random.default_rng(5)
    cases = [np.array([5, 3, 1, 4, 2, .5], dtype=np.float32),
             np.array([-1e9, 3, -1e9, 4, 2, 3, 3, .5], dtype=np.float32),
             np.array([1, 1, 1, 1, 1, 1, 1, 1, 1, 1], dtype=np.float32)]
    ks = [3, 3, 4]
    for _ in range(40):
        n = int(rng.integers(25, 120))
        c = rng.standard_normal(n).astype(np.float32)
        if rng.random() < 0.5:
            c = np.round(c * 2) / 2  # many exact ties
        c[rng.random(n) < 0.2] = -10e8
        cases.append(c.astype(np.float32))
        ks.append(int(rng.integers(1, 21)))
    for j, (c, k) in enumerate(zip(cases, ks)):
        ids, sc = find_k_largest(k, c)
        out["fkl_in_%d" % j] = c
        out["fkl_k_%d" % j] = np.int64(k)
        out["fkl_ids_%d" % j] = np.array(ids, dtype=np.int64)
        out["fkl_scores_%d" % j] = np.array(sc, dtype=np.float32)
    out["fkl_n"] = np.int64(len(cases))

    # ------------------------------------------------------------------ (v) test() + ranking_evaluation
    seed_all(41)
    ue_t = torch.randn(U, D) * 0.3
    ie_t = torch.randn(I, D) * 0.3
    shell = types.SimpleNamespace(data=data, max_N=20)

    def predict(u):  # LightGCN.predict (LightGCN.py:99-102)
        uid = data.get_user_id(u)
        return torch.matmul(ue_t[uid], ie_t.transpose(0, 1)).cpu().numpy()

    shell.predict = predict
    import io
    import contextlib

    with contextlib.redirect_stdout(io.StringIO()):
        rec_list = GraphRecommender.test(shell)
    users = list(data.test_set.keys())
    out["eval_user_emb"], out["eval_item_emb"] = ue_t.numpy(), ie_t.numpy()
    out["eval_users_raw"] = np.array(users)
    out["eval_rec_items_raw"] = np.array([[p[0] for p in rec_list[u]] for u in users])
    out["eval_rec_scores"] = np.array([[p[1] for p in rec_list[u]] for u in users], dtype=np.float32)
    measures = ranking_evaluation(data.test_set, rec_list, [10, 20])
    out["eval_measures"] = np.array(measures)
    out["eval_topN"] = np.array([10, 20])

    # consecutive runs of arrays of at most 0.9 MB go to reference_vectors_<n>.npz: float data barely compresses and no
    # stored file may exceed 1 MB.  tests/conftest.py reads the parts back in order as one mapping
    parts, size = [{}], 0
    for k, a in out.items():
        a = np.asarray(a)
        if parts[-1] and size + a.nbytes > 900_000:
            parts.append({})
            size = 0
        parts[-1][k] = a
        size += a.nbytes
    for old in glob.glob(os.path.join(HERE, "reference_vectors_*.npz")):
        os.remove(old)
    for n, part in enumerate(parts):
        path = os.path.join(HERE, "reference_vectors_%d.npz" % n)
        np.savez_compressed(path, **part)
        print("wrote", path, "(%d arrays, %.1f KB)" % (len(part), os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
