"""Long lists (64 < K <= 256) in full-rank evaluation on the GPU: the tensor path's candidate pool, its block-wide re-scoring
and the block-per-user refquirk replay against the CPU oracle.  Bar: top-K item ids AND scores bit-exact (ties by ascending
item id), as in test_gpu_eval.py."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from oracle import hgr_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUB = os.path.join(ROOT, "tests", "refstub")
LONG_K = [65, 100, 128, 200, 256]
ENGINES = ("simt", "tensor", "auto")


@pytest.fixture(scope="module")
def E():
    import torch

    from hypergraph_diffusion_for_recommendation_b200 import _lib, evaluation

    assert torch.cuda.is_available()
    _lib.lib()
    return evaluation


def cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def train_csr(u, i, n_users):
    order = np.lexsort((i, u))
    u, i = np.asarray(u)[order], np.asarray(i)[order]
    keep = np.ones(u.size, bool)
    keep[1:] = (u[1:] != u[:-1]) | (i[1:] != i[:-1])
    u, i = u[keep], i[keep]
    ptr = np.zeros(n_users + 1, np.int64)
    np.cumsum(np.bincount(u, minlength=n_users), out=ptr[1:])
    return ptr, i.astype(np.int32)


def run(E, ue, ie, test_users, ptr, idx, k, mode, engine):
    ids, sc, stats = E.fullrank_topk(cuda(ue), cuda(ie), cuda(np.asarray(test_users, np.int32)), cuda(ptr), cuda(idx), k, mode=mode,
                                     engine=engine, return_stats=True)
    return ids.cpu().numpy().astype(np.int64), sc.cpu().numpy(), stats.cpu().numpy()


def check_exact(E, ue, ie, test_users, ptr, idx, k, engines=ENGINES, modes=("exact", "refquirk")):
    out = {}
    for mode in modes:
        want_ids, want_sc = O.fullrank_topk(ue, ie, test_users, ptr, idx, k, mode=mode)
        for engine in engines:
            ids, sc, stats = run(E, ue, ie, test_users, ptr, idx, k, mode, engine)
            bad = np.nonzero((ids != want_ids).any(axis=1))[0]
            assert bad.size == 0, "K=%d %s/%s: %d users differ, first %d: got %s want %s" % (
                k, mode, engine, bad.size, bad[0], ids[bad[0]], want_ids[bad[0]])
            assert np.array_equal(sc.view(np.uint32), want_sc.view(np.uint32)), "K=%d %s/%s scores not bit-exact" % (k, mode, engine)
            assert stats[3] < 1_000_000, "tensor-score error reached %.2f of the proven bound" % (stats[3] / 1e6)
            out[(mode, engine)] = stats
    return out


@pytest.mark.parametrize("k", LONG_K)
def test_random_trained_and_layernorm_like_embeddings(E, k):
    rng = np.random.default_rng(k)
    n_users, n_items, d = 700, 3000, 64
    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions

    g = powerlaw_interactions(n_users, n_items, 40_000, seed=3)
    ptr, idx = train_csr(g.train_u, g.train_i, n_users)
    ue = (rng.standard_normal((n_users, d)) * 0.1).astype(np.float32)
    ie = (rng.standard_normal((n_items, d)) * 0.1).astype(np.float32)
    test_users = rng.permutation(n_users)[:600]
    check_exact(E, ue, ie, test_users, ptr, idx, k)
    # "trained": the user's training items score highest, so the mask decides the list
    ue2 = ue.copy()
    for u in range(n_users):
        its = idx[ptr[u]:ptr[u + 1]]
        if its.size:
            ue2[u] = ie[its].mean(axis=0) * 3
    ie2 = ie * (1 + 4 * rng.random((n_items, 1))).astype(np.float32)  # uneven item norms
    stats = check_exact(E, ue2, ie2, test_users, ptr, idx, k)
    assert stats[("exact", "tensor")][2] == 0, "no user should need the brute-force fallback here (%d did)" % stats[("exact", "tensor")][2]
    assert stats[("exact", "tensor")][0] > 0  # the tensor path ran (candidates were emitted)
    # LayerNorm-like tables: every score of a user within a fraction of a percent of ||u|| ||i||
    ue3 = (1.0 + 0.05 * rng.standard_normal((n_users, d))).astype(np.float32)
    ie3 = (1.0 + 0.05 * rng.standard_normal((n_items, d))).astype(np.float32)
    check_exact(E, ue3, ie3, test_users, ptr, idx, k, modes=("exact",))


def test_popular_items_with_low_ids_do_not_overflow_the_pool(E):
    """The case of test_gpu_eval.py's popular-low-ids test at K = 100: the first 150 items are every user's best."""
    rng = np.random.default_rng(77)
    n_users, n_items, k = 12_000, 40_000, 100
    common = rng.standard_normal(64).astype(np.float32)
    ue = (0.1 * rng.standard_normal((n_users, 64)) + 0.5 * common).astype(np.float32)
    ie = (0.1 * rng.standard_normal((n_items, 64))).astype(np.float32)
    ie[:150] += (0.5 * common * rng.uniform(0.5, 1.5, (150, 1))).astype(np.float32)
    tu = rng.integers(0, n_users, 100_000)
    ti = np.minimum((rng.pareto(1.2, 100_000) * 40).astype(np.int64), n_items - 1)
    ptr, idx = train_csr(tu, ti, n_users)
    users = np.arange(0, n_users, 97)
    want_ids, want_sc = O.fullrank_topk(ue, ie, users, ptr, idx, k, mode="exact")
    ids, sc, stats = run(E, ue, ie, np.arange(n_users, dtype=np.int32), ptr, idx, k, "exact", "tensor")
    assert np.array_equal(ids[users], want_ids) and np.array_equal(sc[users].view(np.uint32), want_sc.view(np.uint32))
    assert stats[2] == 0, "%d users overflowed their candidate pools" % stats[2]
    assert stats[3] < 1_000_000


def test_pool_overflow_falls_back_to_exact_path(E):
    """Scores increasing with the item id: far more items than the pool holds meet the threshold, every user goes to the
    brute-force kernel, and the result does not change."""
    n_users, n_items, d, k = 5, 6000, 64, 100
    ue = np.zeros((n_users, d), np.float32)
    ue[:, 0] = 1.0
    ie = np.zeros((n_items, d), np.float32)
    ie[:, 0] = np.linspace(0.1, 5.0, n_items, dtype=np.float32)
    ptr, idx = train_csr(np.array([0, 0, 1]), np.array([5999, 5998, 17]), n_users)
    stats = check_exact(E, ue, ie, np.arange(n_users), ptr, idx, k)
    assert stats[("exact", "tensor")][2] == n_users


@pytest.mark.parametrize("k", [100, 256])
def test_users_with_fewer_unmasked_items_than_k(E, k):
    rng = np.random.default_rng(k + 6)
    n_users, n_items, d = 9, 300, 64
    unmasked = [5, 0, 100, 300, 299, 1, k - 1, k, k + 1]
    tu, ti = [], []
    for u, n_free in enumerate(unmasked):
        its = rng.permutation(n_items)[:n_items - n_free]
        tu += [u] * its.size
        ti += list(its)
    ptr, idx = train_csr(np.array(tu, np.int64), np.array(ti, np.int64), n_users)
    ue = (rng.standard_normal((n_users, d)) * 0.1).astype(np.float32)
    ie = (rng.standard_normal((n_items, d)) * 0.1).astype(np.float32)
    check_exact(E, ue, ie, np.arange(n_users), ptr, idx, k, modes=("exact",))


@pytest.mark.parametrize("k", [100, 256])
def test_ragged_item_count_and_many_sub_ranges(E, k):
    """Few users x 20 011 items: not a multiple of the 128-item tile, and the catalogue is cut into many sub-ranges."""
    rng = np.random.default_rng(7 + k)
    n_users, n_items, d = 300, 20_011, 64
    ptr, idx = train_csr(rng.integers(0, n_users, 9000), rng.integers(0, n_items, 9000), n_users)
    ue = (rng.standard_normal((n_users, d)) * 0.1).astype(np.float32)
    ie = (rng.standard_normal((n_items, d)) * 0.1).astype(np.float32)
    test_users = rng.permutation(n_users)[:257]
    stats = check_exact(E, ue, ie, test_users, ptr, idx, k)
    s = stats[("exact", "tensor")]
    assert s[2] == 0 and s[0] < 257 * 20 * k and s[1] <= s[0]  # far fewer candidates than scores (5.1 M)


def test_engines_agree_at_gowalla_scale(E):
    """30 k users x 41 k items, K = 100: the tensor path and the fp32 brute force return identical ids and scores."""
    import torch

    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions

    n_users, n_items, d, k = 30_000, 41_000, 64, 100
    g = powerlaw_interactions(n_users, n_items, 1_000_000, seed=1234)
    ev = E.EvalData.from_arrays(n_users, n_items, g.train_u, g.train_i, g.test_u, g.test_i)
    torch.manual_seed(0)
    ue = torch.nn.init.xavier_uniform_(torch.empty(n_users, d)).cuda()
    ie = torch.nn.init.xavier_uniform_(torch.empty(n_items, d)).cuda()
    sub = ev.test_users[:4096]
    a_ids, a_sc, stats = E.fullrank_topk(ue, ie, ev.test_users, ev.train_indptr, ev.train_indices, k, engine="tensor", return_stats=True)
    b_ids, b_sc = E.fullrank_topk(ue, ie, sub, ev.train_indptr, ev.train_indices, k, engine="simt")
    assert torch.equal(a_ids[:4096], b_ids) and torch.equal(a_sc[:4096], b_sc)
    assert int(stats[2]) == 0 and int(stats[3]) < 1_000_000
    sc = a_sc.cpu().numpy()
    assert (np.diff(sc, axis=1) <= 0).all()


@pytest.mark.parametrize("n_test", [11_008, 14_080, 18_432])
def test_every_user_count_gets_the_full_sample_of_bucket_maxima(E, n_test):
    """43 - 73 blocks of 256 users are where a plan of 5 - 7 sample segments would leave 320 - 448 bucket maxima (< 2 K at
    K = 256) and a quarter or more of the users would fill their pools.  Long lists always sample 8 segments x 2 column
    halves = 512 maxima: at 92 000 items nobody falls back, and the tensor path equals the fp32 brute force."""
    import torch

    n_items, d, k = 92_000, 64, 256
    rng = np.random.default_rng(n_test)
    deg = rng.integers(5, 60, n_test)
    tu = np.repeat(np.arange(n_test), deg)
    ti = np.minimum((rng.pareto(1.0, tu.size) * 50).astype(np.int64), n_items - 1)
    ptr, idx = train_csr(tu, ti, n_test)
    torch.manual_seed(n_test)
    ue = torch.nn.init.xavier_uniform_(torch.empty(n_test, d)).cuda()
    ie = torch.nn.init.xavier_uniform_(torch.empty(n_items, d)).cuda()
    users = torch.randperm(n_test, device="cuda").to(torch.int32)
    a_ids, a_sc, stats = E.fullrank_topk(ue, ie, users, cuda(ptr), cuda(idx), k, engine="tensor", return_stats=True)
    assert int(stats[2]) == 0, "%d of %d users overflowed their candidate pools" % (int(stats[2]), n_test)
    assert int(stats[3]) < 1_000_000
    sub = users[:512]
    b_ids, b_sc = E.fullrank_topk(ue, ie, sub, cuda(ptr), cuda(idx), k, engine="simt")
    assert torch.equal(a_ids[:512], b_ids) and torch.equal(a_sc[:512], b_sc)


def test_install_evaluates_top_100_lists_like_the_oracle():
    """A reference-style model with item_ranking = "10,20,50,100" (max_N = 100): fast_evaluation runs through install()'s
    refquirk seam, and its strings equal the oracle's metrics on the oracle's refquirk lists from the same tables."""
    code = """
    import random, sys
    import numpy as np, torch
    sys.path.insert(0, %r)
    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions
    from oracle import hgr_oracle as O
    g = powerlaw_interactions(400, 600, 12000, seed=3)
    train = [[int(u), 10000 + int(i), 1.0] for u, i in zip(g.train_u, g.train_i)]
    test = [[int(u), 10000 + int(i), 1.0] for u, i in zip(g.test_u, g.test_i)]
    import hypergraph_diffusion_for_recommendation_b200 as hgr
    hgr.install(%r)
    import model.graph.LightGCN as M
    kw = dict(item_ranking="10,20,50,100", batch_size=2048, embedding_size=64, n_layers=2, max_epoch=2, lrate=0.01, reg=1e-4)
    torch.manual_seed(5); random.seed(5)
    rec = M.LightGCN(None, train, test, **kw)
    rec.train()
    assert rec.max_N == 100
    meas, lists = rec.fast_evaluation(0)
    assert len(meas) == 20 and meas[15] == "Top 100\\n", meas
    assert all(len(v) == 100 for v in lists.values())
    d = rec.data
    ue, ie = rec.user_emb.detach().cpu().numpy(), rec.item_emb.detach().cpu().numpy()
    tu = np.array([d.user[u] for u, i, _ in train]); ti = np.array([d.item[i] for u, i, _ in train])
    order = np.lexsort((ti, tu)); tu, ti = tu[order], ti[order]
    keep = np.ones(tu.size, bool); keep[1:] = (tu[1:] != tu[:-1]) | (ti[1:] != ti[:-1])
    tu, ti = tu[keep], ti[keep]
    ptr = np.zeros(d.n_users + 1, np.int64); np.cumsum(np.bincount(tu, minlength=d.n_users), out=ptr[1:])
    users = list(d.test_set)
    ids, _ = O.fullrank_topk(ue, ie, np.array([d.user[u] for u in users]), ptr, ti.astype(np.int32), 100, mode="refquirk")
    rec_ids = [[d.id2item[int(i)] for i in row] for row in ids]
    assert rec_ids == [[i for i, _ in lists[u]] for u in users]
    want = O.ranking_evaluation([list(d.test_set[u]) for u in users], rec_ids, [10, 20, 50, 100])
    assert meas == want, (meas, want)
    print("OK", meas[15:])
    """ % (ROOT, STUB)
    env = dict(os.environ, PYTHONPATH=ROOT, PYTHONDONTWRITEBYTECODE="1")
    p = subprocess.run([sys.executable, "-c", textwrap.dedent(code)], capture_output=True, text=True, env=env, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + "\n" + p.stderr[-4000:]
    assert "OK" in p.stdout
