"""Pin the CPU oracle against vectors produced by the unmodified reference.

The reference has no tests of its own (SURVEY.md F3); ``tests/golden/reference_vectors_*.npz`` hold the
outputs of the reference's classes on seeded inputs (``tests/golden/make_golden.py``).  Integer /
index results must match exactly, floating point within the tolerance written in each test.
"""
import numpy as np
import pytest

from oracle import hgr_oracle as O

RTOL = 1e-5  # north_star: propagated embeddings and losses within 1e-5 relative in fp32


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def canon(indptr, indices, data):
    """Sort every CSR row by column (scipy leaves `csr_matrix((v, (r, c)))` products unsorted)."""
    rows = np.repeat(np.arange(indptr.size - 1), np.diff(indptr))
    order = np.lexsort((indices, rows))
    return indptr, indices[order], data[order]


def params(golden, prefix):
    return {k[len(prefix):]: golden[k] for k in golden.files if k.startswith(prefix)}


# ------------------------------------------------------------------------------------ adjacency
def test_hand_graph_adjacency_bit_exact(golden):
    tr = golden["hand_train"]
    user = {r: k for k, r in enumerate(golden["hand_id2user"])}
    item = {r: k for k, r in enumerate(golden["hand_id2item"])}
    u = np.array([user[int(t[0])] for t in tr])
    i = np.array([item[int(t[1])] for t in tr])
    U, I = len(user), len(item)
    assert (U, I) == (3, 4)  # user 13 and item 104 are test-only and get no id
    ip, ix, dv = O.bipartite_adjacency(u, i, U, I)
    assert np.array_equal(ip, golden["hand_ui_indptr"]) and np.array_equal(ix, golden["hand_ui_indices"])
    assert np.array_equal(dv, golden["hand_ui_data"]) and dv.max() == 2.0  # duplicate (10,100) summed
    ip, ix, dv = O.build_norm_adj(u, i, U, I)
    assert np.array_equal(ip, golden["hand_norm_indptr"]) and np.array_equal(ix, golden["hand_norm_indices"])
    assert np.array_equal(dv.view(np.uint32), golden["hand_norm_data"].view(np.uint32))
    r = O.interaction_matrix(u, i, U, I)
    ip, ix, dv = O.normalize_graph_mat(*r, I)  # rectangular branch
    gip, gix, gdv = canon(golden["hand_normR_indptr"], golden["hand_normR_indices"], golden["hand_normR_data"])
    assert np.array_equal(ip, gip) and np.array_equal(ix, gix)
    assert np.array_equal(dv.view(np.uint32), gdv.view(np.uint32))


def test_powerlaw_adjacency_bit_exact(golden, pl_graph):
    ip, ix, dv = pl_graph["csr"]
    assert np.array_equal(ip, golden["pl_norm_indptr"]) and np.array_equal(ix, golden["pl_norm_indices"])
    assert np.array_equal(dv.view(np.uint32), golden["pl_norm_data"].view(np.uint32))
    # COO handed to torch by TorchGraphInterface (base/torch_interface.py:8-12) is the CSR order
    rows = np.repeat(np.arange(ip.size - 1), np.diff(ip))
    assert np.array_equal(np.stack([rows, ix]), golden["pl_coo_indices"])
    assert np.array_equal(dv, golden["pl_coo_values"])
    lut_ref = np.where(np.isinf(golden["pow_lut"]), np.float32(0), golden["pow_lut"]).astype(np.float32)
    assert np.array_equal(O.pow_lut(4097, -0.5).view(np.uint32), lut_ref.view(np.uint32))


def test_laplacian_and_reference_id_order(golden, pl_graph):
    from hypergraph_diffusion_for_recommendation_b200.synth import reference_dense_ids

    tr = golden["pl_train"]
    du, di, id2u, id2i = reference_dense_ids(tr[:, 0].astype(np.int64), tr[:, 1].astype(np.int64))
    assert np.array_equal(du, golden["pl_dense_u"]) and np.array_equal(di, golden["pl_dense_i"])
    assert np.array_equal(id2u, golden["pl_id2user"]) and np.array_equal(id2i, golden["pl_id2item"])
    r = O.interaction_matrix(pl_graph["u"], pl_graph["i"], pl_graph["n_users"], pl_graph["n_items"])
    ip, ix, dv = O.laplacian_of_interaction(*r, pl_graph["n_users"], pl_graph["n_items"])
    assert np.array_equal(ip, golden["pl_lap_indptr"]) and np.array_equal(ix, golden["pl_lap_indices"])
    assert np.array_equal(dv.view(np.uint32), golden["pl_lap_data"].view(np.uint32))


def test_drop_edges_replays_reference_mask(golden, pl_graph):
    ip, ix, dv = O.drop_edges(*pl_graph["csr"], golden["drop_rand"], float(golden["drop_keep"]))
    rows = np.repeat(np.arange(ip.size - 1), np.diff(ip))
    assert np.array_equal(np.stack([rows, ix]), golden["drop_indices"])
    assert np.array_equal(dv.view(np.uint32), golden["drop_values"].view(np.uint32))
    y = O.spmm(ip, ix, dv, golden["drop_X"])
    assert np.array_equal(y.view(np.uint32), golden["drop_Y"].view(np.uint32))
    y2 = O.hgconv((ip, ix, dv), golden["drop_X"], 0.3)  # asymmetric A: A (A^T X)
    assert rel_err(y2, golden["drop_hgconv_Y"]) < RTOL


# ------------------------------------------------------------------------------------ propagation
def test_spmm_bit_exact_and_symmetric_backward(golden, pl_graph):
    y = O.spmm(*pl_graph["csr"], golden["spmm_X"])
    assert np.array_equal(y.view(np.uint32), golden["spmm_Y"].view(np.uint32))
    # A is bit-exactly symmetric, so autograd's A^T dY equals A dY up to summation order
    dx = O.spmm(*pl_graph["csr"], golden["spmm_G"])
    assert rel_err(dx, golden["spmm_dX"]) < RTOL


def test_lgcn_forward(golden, pl_graph):
    ue, ie = O.lgcn_forward(pl_graph["csr"], golden["lgcn_user_emb0"], golden["lgcn_item_emb0"], 3)
    assert rel_err(ue, golden["lgcn_user_out"]) < RTOL and rel_err(ie, golden["lgcn_item_out"]) < RTOL


def test_hgconv(golden, pl_graph):
    y = O.hgconv(pl_graph["csr"], golden["hgconv_X"], 0.5)
    assert rel_err(y, golden["hgconv_Y_act"]) < RTOL
    y = O.hgconv(pl_graph["csr"], golden["hgconv_X"], None)
    assert rel_err(y, golden["hgconv_Y_noact"]) < RTOL
    # symmetric A: A (A^T X) == A (A X) bit-exactly (SURVEY.md section 9.5)
    y2 = O.spmm(*pl_graph["csr"], O.spmm(*pl_graph["csr"], golden["hgconv_X"]))
    assert np.array_equal(y2.view(np.uint32), golden["hgconv_Y_noact"].view(np.uint32))


def test_equiv_set_conv_and_local_encoder(golden, pl_graph):
    y = O.equiv_set_conv(pl_graph["csr"], golden["esc_X"], params(golden, "esc_param/"))
    assert rel_err(y, golden["esc_Y"]) < RTOL
    lu, li = O.local_aware_encoder(pl_graph["csr"], golden["lae_E0"], params(golden, "lae_param/"), 2, pl_graph["n_users"])
    assert rel_err(lu, golden["lae_user_out"]) < RTOL and rel_err(li, golden["lae_item_out"]) < RTOL


def test_hccf_forward(golden, pl_graph):
    hu, hi, gcn_h, hyp_h = O.hccf_forward(pl_graph["csr"], params(golden, "hccf_param/"), 2, pl_graph["n_users"])
    assert rel_err(hu, golden["hccf_user_out"]) < RTOL and rel_err(hi, golden["hccf_item_out"]) < RTOL
    for l in range(2):
        assert rel_err(gcn_h[l], golden["hccf_gcn_%d" % l]) < RTOL
        assert rel_err(hyp_h[l], golden["hccf_hyp_%d" % l]) < RTOL


def test_scatter_mean_form(golden):
    y = O.scatter_mean_conv(golden["scat_V"], golden["scat_E"], golden["scat_X"], golden["scat_X"].shape[0])
    assert rel_err(y, golden["scat_Y"]) < RTOL


# ------------------------------------------------------------------------------------ losses
def test_bpr_l2(golden):
    rec, reg, du, di = O.bpr_l2_from_tables(golden["loss_user_tab"], golden["loss_item_tab"], golden["tri_u"], golden["tri_p"],
                                            golden["tri_n"], float(golden["loss_reg_lambda"]), int(golden["loss_reg_batch_size"]))
    assert rel_err(rec, golden["loss_bpr"]) < RTOL and rel_err(reg, golden["loss_reg"]) < RTOL
    assert rel_err(du, golden["loss_dU"]) < RTOL and rel_err(di, golden["loss_dI"]) < RTOL


def test_contrast_and_infonce(golden):
    loss, d1, d2 = O.contrast_loss(golden["cl_e1"], golden["cl_e2"], golden["cl_nodes"], float(golden["cl_temp"]))
    assert rel_err(loss, golden["cl_loss"]) < RTOL
    assert rel_err(d1, golden["cl_d1"]) < 5e-5 and rel_err(d2, golden["cl_d2"]) < 5e-5
    loss, d1, d2 = O.info_nce(golden["nce_v1"], golden["nce_v2"], float(golden["nce_temp"]))
    assert rel_err(loss, golden["nce_loss"]) < RTOL
    assert rel_err(d1, golden["nce_d1"]) < 5e-5 and rel_err(d2, golden["nce_d2"]) < 5e-5


# ------------------------------------------------------------------------------------ evaluation
def test_find_k_largest_quirk_bit_exact(golden):
    for j in range(int(golden["fkl_n"])):
        ids, sc = O.find_k_largest(int(golden["fkl_k_%d" % j]), golden["fkl_in_%d" % j])
        assert np.array_equal(ids, golden["fkl_ids_%d" % j]), j
        assert np.array_equal(sc, golden["fkl_scores_%d" % j]), j
    ids, _ = O.find_k_largest(3, np.array([5, 3, 1, 4, 2, .5], dtype=np.float32))
    assert list(ids) == [0, 0, 3]  # SURVEY.md F9: ids < K are re-inserted
    ids, _ = O.topk_exact(3, np.array([5, 3, 1, 4, 2, .5], dtype=np.float32))
    assert list(ids) == [0, 3, 1]
    ids, _ = O.topk_exact(4, np.ones(10, dtype=np.float32))
    assert list(ids) == [0, 1, 2, 3]  # ties by ascending id


def test_fullrank_eval_and_metrics(golden, pl_graph):
    id2item = golden["pl_id2item"]
    user = {r: k for k, r in enumerate(golden["pl_id2user"])}
    item = {r: k for k, r in enumerate(id2item)}
    users_raw = golden["eval_users_raw"]
    test_users = np.array([user[int(r)] for r in users_raw])
    tip, tix, _ = O.interaction_matrix(pl_graph["u"], pl_graph["i"], pl_graph["n_users"], pl_graph["n_items"])
    ids, sc = O.fullrank_topk(golden["eval_user_emb"], golden["eval_item_emb"], test_users, tip, tix, 20, mode="refquirk")
    assert np.array_equal(id2item[ids], golden["eval_rec_items_raw"])  # index parity incl. the quirk
    assert rel_err(sc, golden["eval_rec_scores"]) < RTOL
    # metrics: ground truth per test user in test-file order, raw ids (items unseen in training stay raw)
    truth = {int(r): [] for r in users_raw}
    for uu, ii, _ in golden["pl_test"]:
        if int(uu) in truth:
            truth[int(uu)].append(int(ii))
    test_items = [truth[int(r)] for r in users_raw]
    strings = O.ranking_evaluation(test_items, id2item[ids], [10, 20])
    assert strings == [str(s) for s in golden["eval_measures"]]
    # exact mode differs from the quirk only by the duplicated ids < K
    ids_x, _ = O.fullrank_topk(golden["eval_user_emb"], golden["eval_item_emb"], test_users, tip, tix, 20, mode="exact")
    for a, b in zip(ids, ids_x):
        assert len(set(b)) == 20 and set(a) <= set(b)


# ------------------------------------------------------------------------------------ torch restatement (CPU baseline arm)
def test_torch_path_encoders_match_reference(golden, pl_graph):
    import torch

    from oracle import torch_path as T

    torch.set_num_threads(1)
    n = pl_graph["n_users"] + pl_graph["n_items"]
    adj = T.coo_from_csr(*pl_graph["csr"], (n, n))
    lae = T.LocalAwareEncoder(adj, pl_graph["n_users"], 64, 2)
    lae.load_state_dict({k: torch.from_numpy(v) for k, v in params(golden, "lae_param/").items()}, strict=True)
    lae.eval()
    e0 = torch.from_numpy(golden["lae_E0"]).requires_grad_(True)
    lu, li = lae(e0)
    assert rel_err(lu.detach().numpy(), golden["lae_user_out"]) < RTOL and rel_err(li.detach().numpy(), golden["lae_item_out"]) < RTOL
    (torch.cat([lu, li], 0) * torch.from_numpy(golden["spmm_G"])).sum().backward()
    assert rel_err(e0.grad.numpy(), golden["lae_dE0"]) < RTOL
    lg = T.LGCN(adj, pl_graph["n_users"], pl_graph["n_items"], 64, 3)
    lg.load_state_dict({"embedding_dict.user_emb": torch.from_numpy(golden["lgcn_user_emb0"]),
                        "embedding_dict.item_emb": torch.from_numpy(golden["lgcn_item_emb0"])})
    with torch.no_grad():
        ue, ie = lg()
    assert np.array_equal(ue.numpy(), golden["lgcn_user_out"]) and np.array_equal(ie.numpy(), golden["lgcn_item_out"])


def test_torch_path_losses_and_eval_match_reference(golden, pl_graph):
    import torch

    from oracle import torch_path as T

    ut = torch.from_numpy(golden["loss_user_tab"])
    it = torch.from_numpy(golden["loss_item_tab"])
    u, p, n = (torch.from_numpy(golden[k]) for k in ("tri_u", "tri_p", "tri_n"))
    assert rel_err(T.bpr_loss(ut[u], it[p], it[n]).numpy(), golden["loss_bpr"]) < 1e-6
    assert rel_err((T.l2_reg_loss(0.1, ut[u], it[p], it[n]) / 2048).numpy(), golden["loss_reg"]) < 1e-6
    user = {r: k for k, r in enumerate(golden["pl_id2user"])}
    test_users = np.array([user[int(r)] for r in golden["eval_users_raw"]])
    tip, tix, _ = O.interaction_matrix(pl_graph["u"], pl_graph["i"], pl_graph["n_users"], pl_graph["n_items"])
    rec = T.evaluate_users(torch.from_numpy(golden["eval_user_emb"]), torch.from_numpy(golden["eval_item_emb"]), test_users, tip, tix, 20)
    assert np.array_equal(golden["pl_id2item"][rec], golden["eval_rec_items_raw"])


def test_sht_and_dhcf_encoders_against_the_reference():
    """The oracle's restatements of two more callers of the path (SHTEncoder, DHCF_Encoder) against the reference's own outputs
    (tests/golden/more_encoders.npz, make_golden_more_encoders.py)."""
    import os

    from hypergraph_diffusion_for_recommendation_b200 import data as D

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "more_encoders.npz"))
    d = D.Interaction(None, g["train"].tolist(), g["test"].tolist())
    u, i = d.dense_training_pairs()
    csr = O.build_norm_adj(u, i, d.n_users, d.n_items)
    n_layers = int(g["sht_args"][0])
    emb, hu, hi = O.sht_forward(csr, g["sht_param/uEmbeds"], g["sht_param/iEmbeds"], g["sht_param/uHyper"], g["sht_param/iHyper"], n_layers)

    def rel(a, b):
        return np.abs(a.astype(np.float64) - b.astype(np.float64)).max() / np.abs(b).max()

    assert rel(emb, g["sht_embeds"]) < 1e-6 and rel(hu, g["sht_hyper_u"]) < 1e-5 and rel(hi, g["sht_hyper_i"]) < 1e-5
    r = O.interaction_matrix(u, i, d.n_users, d.n_items)
    ue, ie = O.dhcf_forward(r, g["dhcf_param/embedding_dict.user_emb"], g["dhcf_param/embedding_dict.item_emb"], int(g["dhcf_args"][0]),
                            float(g["dhcf_args"][2]))
    # the reference multiplies a DENSIFIED matrix (dense fp32 GEMM order); same sums, other order
    assert rel(ue, g["dhcf_user_out"]) < 1e-5 and rel(ie, g["dhcf_item_out"]) < 1e-5


# ------------------------------------------------------------------------------------------ scatter-form consumers (SURVEY a-6)
@pytest.fixture(scope="module")
def scat():
    import os

    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scatter_encoders.npz"))


def _scat_graph(scat):
    from hypergraph_diffusion_for_recommendation_b200.synth import reference_dense_ids

    du, di, id2u, id2i = reference_dense_ids(scat["train"][:, 0].astype(np.int64), scat["train"][:, 1].astype(np.int64))
    return du, di, id2u.size, id2i.size


def _params(npz, prefix):
    return {k[len(prefix):]: npz[k] for k in npz.files if k.startswith(prefix)}


def test_oracle_hd4_local_aware_encoder_matches_the_reference(scat):
    """HGNN_HD4.LocalAwareEncoder (model/graph/HGNN_HD4.py:391-405) as run by tests/golden/make_golden_scatter_encoders.py."""
    du, di, nu, ni = _scat_graph(scat)
    csr = O.build_norm_adj(du, di, nu, ni)
    ip, ix, _ = O.bipartite_adjacency(du, di, nu, ni)
    ue, ie = O.hd4_local_aware_encoder(csr, (ip, ix), scat["hd4_E0"], _params(scat, "hd4_param/"), 2, nu)
    assert rel_err(ue, scat["hd4_user_out"]) < RTOL and rel_err(ie, scat["hd4_item_out"]) < RTOL


def test_oracle_hccf_diffusion_encoder_matches_the_reference(scat):
    """HCCF_diffusion.HCCFEncoder (model/graph/HCCF_diffusion.py:197-217) with keep_rate 1, eval mode."""
    du, di, nu, ni = _scat_graph(scat)
    csr = O.build_norm_adj(du, di, nu, ni)
    hu, hi, gcn_h, hyp_h = O.hccf_diffusion_forward(csr, _params(scat, "hdf_param/"), 2, nu)
    assert rel_err(hu, scat["hdf_user_out"]) < RTOL and rel_err(hi, scat["hdf_item_out"]) < RTOL
    for l in range(2):
        assert rel_err(gcn_h[l], scat["hdf_gcn_%d" % l]) < RTOL and rel_err(hyp_h[l], scat["hdf_hyp_%d" % l]) < RTOL


def test_oracle_attention_weighted_scatter_matches_the_reference(scat):
    """HD2.EquivSetConv.forward (model/graph/HD2.py:624-643): per-edge attention on the node -> hyperedge stage."""
    xv = O.scatter_mean_conv_weighted(scat["att_V"], scat["att_E"], scat["att_X"], scat["att_atts"], scat["att_X"].shape[0])
    y = O._mlp_w(xv, _params(scat, "att_param/"), "W.")
    assert rel_err(y, scat["att_Y"]) < RTOL


def test_oracle_normalize_graph_mat_hyper_matches_the_reference(scat):
    """Graph.normalize_graph_mat_hyper (data/graph.py:28-42): the factored form reproduces the reference's matrix -- its values
    after multiplying the two factors out (float64 product of fp32 factors, 1e-6) and its action on a table."""
    import scipy.sparse as sp

    du, di, nu, ni = _scat_graph(scat)
    for name, (ip, ix, dv), shape in (("inter", O.interaction_matrix(du, di, nu, ni), (nu, ni)),
                                      ("adj", O.bipartite_adjacency(du, di, nu, ni), (nu + ni, nu + ni))):
        (lp, li, lv), (rp, ri, rv) = O.normalize_graph_mat_hyper(ip, ix, dv, shape[1])
        left = sp.csr_matrix((lv.astype(np.float64), li, lp), shape=shape)
        right = sp.csr_matrix((rv.astype(np.float64), ri, rp), shape=(shape[1], shape[0]))
        prod = (left @ right).tocsr()
        prod.sort_indices()
        assert np.array_equal(prod.indptr, scat["hyper_%s_indptr" % name]) and np.array_equal(prod.indices, scat["hyper_%s_indices" % name])
        assert np.abs(prod.data - scat["hyper_%s_data" % name]).max() <= 1e-6 * np.abs(scat["hyper_%s_data" % name]).max()
        x = scat["hyper_%s_X" % name]
        y = O.spmm(lp, li, lv, O.spmm(rp, ri, rv, x))
        assert rel_err(y, scat["hyper_%s_Y" % name]) < RTOL
