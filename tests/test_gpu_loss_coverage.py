"""The fused loss kernels past their grid caps, at every width and on saturated, repeated and degenerate inputs.

BPR + L2 (csrc/loss_bpr.cu) caps its grid at kLossMaxBlocks blocks and strides over the batch beyond 1 184 x groups-per-block
triples; bench.py's workload takes 56 such passes per step.  contrastLoss / InfoNCE (csrc/loss_ssl.cu) cut the looped
dimension into ssl_splits(M) slices.  Every check is against an independent float64 evaluation of the reference's own
expressions (util/loss_torch.py): the numpy oracle where the case is small, float64 torch autograd on the device where the
batch or the [M, M] logits would not fit a CPU test."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import hgr_oracle as O

from conftest import global_rel_err as grad_err
from conftest import rowwise_rel_err as rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
BPR_GRAD = 2e-5  # the global gradient bars of test_gpu_losses.py
SSL_GRAD = 5e-5
WIDTHS = [32, 64, 128]
LOSS_MAX_BLOCKS = 1184  # loss_bpr.cu kLossMaxBlocks
LOSS_THREADS = 256  # loss_bpr.cu kLossThreads; a triple takes D / 4 lanes
REG = 0.05
ORACLE_MAX_BATCH = 40_000  # above this the numpy oracle is too slow for a test; the device float64 reference stands alone
ORACLE_MAX_M = 4096
U32 = 2.0 ** -24  # float32 unit roundoff: half the spacing of floats just above 1


def bpr_cap(d):
    """Triples the BPR kernels cover in one pass of their capped grid."""
    return LOSS_MAX_BLOCKS * (LOSS_THREADS // (d // 4))


@pytest.fixture(scope="module")
def L():
    from hypergraph_diffusion_for_recommendation_b200 import _lib, loss_torch

    _lib.lib()  # raises if libhgr.so is missing: there is no fallback
    return types.SimpleNamespace(loss=loss_torch, lib=_lib)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def powerlaw_ids(rng, n, size):
    """Ids in [0, n) with P(id < k) = (k / n) ** (1/4): row 0 alone draws n ** -1/4 of the batch (5.6 % at n = 10^5)."""
    return np.minimum((n * rng.random(size) ** 4).astype(np.int64), n - 1)


# ------------------------------------------------------------------------------------------------------------- BPR + L2
def bpr_ref64(ut, it, u, p, n, reg, batch_size, w_rec=2.0, w_reg=3.0):
    """util/loss_torch.py's bpr_loss + l2_reg_loss(reg, U, P, N) / batch_size on the gathered rows, in float64 autograd on
    the tables' device, with grad_out = (w_rec, w_reg).  Also returns, per gradient element, the sum over the triples of
    the absolute values of the contributions added there (the scale of the kernel's atomic accumulation)."""
    U = ut.detach().double().requires_grad_(True)
    I = it.detach().double().requires_grad_(True)
    ue, pe, ne = U[u], I[p], I[n]
    x = (ue * pe).sum(1) - (ue * ne).sum(1)
    rec = torch.mean(-torch.log(10e-6 + torch.sigmoid(x)))
    nu, np_, nn = torch.norm(ue, p=2), torch.norm(pe, p=2), torch.norm(ne, p=2)
    regl = (nu + np_ + nn) * reg / batch_size
    (w_rec * rec + w_reg * regl).backward()
    with torch.no_grad():
        s = torch.sigmoid(x)
        gx = (w_rec * s * (1 - s) / (10e-6 + s) / len(u)).abs()[:, None]
        c = w_reg * reg / batch_size
        tiny = torch.finfo(torch.float64).tiny
        # x = <u,p> - <u,n>: a user row receives g p and -g n, which may be rounded apart before they cancel
        tu = gx * (pe.abs() + ne.abs()) + c * ue.abs() / nu.clamp_min(tiny)
        tp = gx * ue.abs() + c * pe.abs() / np_.clamp_min(tiny)
        tn = gx * ue.abs() + c * ne.abs() / nn.clamp_min(tiny)
        su = torch.zeros_like(U).index_add_(0, u, tu)
        si = torch.zeros_like(I).index_add_(0, p, tp).index_add_(0, n, tn)
    return types.SimpleNamespace(rec=rec.detach(), reg=regl.detach(), du=U.grad, di=I.grad, su=su, si=si)


def within_terms(got, want, terms, tau=RTOL):
    """Per element |got - want| <= tau * sum |contributions|.  Each contribution carries a few float32 roundings (under 1e-6
    of itself; the kernel sums the three norms in double) and the atomic accumulation in any order adds rounding of the
    partial sums, which are bounded by the sum of the absolute contributions; 1e-5 covers both with room.  An element
    nothing touched must come out exactly 0."""
    d = (got.detach().double() - want).abs()
    return bool((d <= tau * terms).all())


def bpr_run(L, ut, it, u, p, n, reg, batch_size, w_rec=2.0, w_reg=3.0):
    tu, ti = ut.clone().requires_grad_(True), it.clone().requires_grad_(True)
    rec, regl = L.loss.bpr_l2_from_tables(tu, ti, u, p, n, reg, batch_size)
    (w_rec * rec + w_reg * regl).backward()
    return rec.detach(), regl.detach(), tu.grad, ti.grad


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("where", ["cap-1", "cap", "cap+1", "3cap+17"])
def test_bpr_l2_across_grid_passes(L, d, where):
    """Batches on both sides of one capped grid pass and past three, on 3 000 users x 7 000 items with power-law ids (row 0
    takes over 10 % of the batch, thousands of red.global.add on one row).  The 3cap+17 batch is short: batch_size is twice
    the triples drawn.  Losses to 1e-5, gradients per element and globally; the forward sums in a fixed order, so a second
    run gives the same loss bits."""
    c = bpr_cap(d)
    batch = {"cap-1": c - 1, "cap": c, "cap+1": c + 1, "3cap+17": 3 * c + 17}[where]
    batch_size = 2 * batch if where == "3cap+17" else batch
    rng = np.random.default_rng(d * 10 + len(where))
    ut = (rng.standard_normal((3000, d)) * 0.3).astype(np.float32)
    it = (rng.standard_normal((7000, d)) * 0.3).astype(np.float32)
    u, p, n = powerlaw_ids(rng, 3000, batch), powerlaw_ids(rng, 7000, batch), powerlaw_ids(rng, 7000, batch)
    assert (u == 0).sum() > 1000 and (n == 0).sum() > 500
    gu, gp, gn = cuda(u), cuda(p), cuda(n)
    tu, ti = cuda(ut), cuda(it)
    rec, regl, du, di = bpr_run(L, tu, ti, gu, gp, gn, REG, batch_size)
    ref = bpr_ref64(tu, ti, gu, gp, gn, REG, batch_size)
    assert rel_err(rec, ref.rec) < RTOL and rel_err(regl, ref.reg) < RTOL
    assert within_terms(du, ref.du, ref.su) and within_terms(di, ref.di, ref.si)
    assert grad_err(du, ref.du) < BPR_GRAD and grad_err(di, ref.di) < BPR_GRAD
    rec2, reg2, du2, di2 = bpr_run(L, tu, ti, gu, gp, gn, REG, batch_size)
    assert torch.equal(bits(rec), bits(rec2)) and torch.equal(bits(regl), bits(reg2))
    assert within_terms(du2, ref.du, ref.su) and within_terms(di2, ref.di, ref.si)  # atomics: equal within the bar, not bitwise
    if batch <= ORACLE_MAX_BATCH:
        o_rec, o_reg, o_du, o_di = O.bpr_l2_from_tables(ut, it, u, p, n, REG, batch_size)
        _, _, du0, di0 = O.bpr_l2_from_tables(ut, it, u, p, n, 0.0, batch_size)
        assert rel_err(rec, o_rec) < RTOL and rel_err(regl, o_reg) < RTOL
        assert grad_err(du, 2.0 * du0 + 3.0 * (o_du - du0)) < BPR_GRAD and grad_err(di, 2.0 * di0 + 3.0 * (o_di - di0)) < BPR_GRAD


def test_bpr_l2_headline_batch(L):
    """bench.py's shape: D = 64, a batch of 1 048 576 triples (56 passes of the capped grid) on 10^5 users x 10^5 items
    with power-law ids, through bpr_l2_from_tables and through the window form (bpr_l2_sharded without reduce_sums) at
    world 1, where users and items are one gathered table.  Both forms run the same forward sums, so their losses agree
    bit for bit."""
    d, batch, nu_, ni_ = 64, 1 << 20, 100_000, 100_000
    assert batch > 55 * bpr_cap(d)
    rng = np.random.default_rng(64)
    tu = cuda((rng.standard_normal((nu_, d)) * 0.1).astype(np.float32))
    ti = cuda((rng.standard_normal((ni_, d)) * 0.1).astype(np.float32))
    gu, gp, gn = (cuda(powerlaw_ids(rng, k, batch)) for k in (nu_, ni_, ni_))
    rec, regl, du, di = bpr_run(L, tu, ti, gu, gp, gn, REG, batch)
    ref = bpr_ref64(tu, ti, gu, gp, gn, REG, batch)
    assert rel_err(rec, ref.rec) < RTOL and rel_err(regl, ref.reg) < RTOL
    assert within_terms(du, ref.du, ref.su) and within_terms(di, ref.di, ref.si)
    assert grad_err(du, ref.du) < BPR_GRAD and grad_err(di, ref.di) < BPR_GRAD
    full = torch.cat([tu, ti]).requires_grad_(True)
    rec_w, reg_w = L.loss.bpr_l2_sharded(full, lambda x: x, 0, gu, gp + nu_, gn + nu_, REG, batch)
    (2.0 * rec_w + 3.0 * reg_w).backward()
    assert torch.equal(bits(rec_w), bits(rec)) and torch.equal(bits(reg_w), bits(regl))
    assert within_terms(full.grad, torch.cat([ref.du, ref.di]), torch.cat([ref.su, ref.si]))


def test_bpr_l2_owner_sharded_at_scale_with_an_idle_rank(L):
    """dist.train_step's loss at world 8, replayed on one GPU as in test_gpu_losses.py, on a batch of more than 7 grid passes
    at D = 64.  Rank 5 owns no user of the batch: its four partial sums are exactly 0 and its gradient rows come from
    positives and negatives alone.  The summed loss is the same on every rank and matches the float64 reference."""
    world, n_loc, d, batch, idle = 8, 2000, 64, 140_000, 5
    assert batch >= 7 * bpr_cap(d)
    rng = np.random.default_rng(8)
    n_rows = world * n_loc
    full = cuda((rng.standard_normal((n_rows, d)) * 0.3).astype(np.float32))
    busy = np.setdiff1d(np.arange(n_rows), np.arange(idle * n_loc, (idle + 1) * n_loc))
    u = rng.permutation(busy)[powerlaw_ids(rng, busy.size, batch)]
    perm = rng.permutation(n_rows)
    p, n = perm[powerlaw_ids(rng, n_rows, batch)], perm[powerlaw_ids(rng, n_rows, batch)]
    gu, gp, gn = cuda(u), cuda(p), cuda(n)
    parts = []
    for r in range(world):
        own = full[r * n_loc:(r + 1) * n_loc].clone().requires_grad_(True)
        L.loss.bpr_l2_sharded(own, lambda x: full, r * n_loc, gu, gp, gn, REG, batch, lambda t: parts.append(t.clone()))
    total = torch.stack(parts).sum(0)
    assert torch.equal(parts[idle], torch.zeros_like(parts[idle]))
    assert all(float(q[0]) > 0 for r, q in enumerate(parts) if r != idle)
    losses, grads = [], []
    for r in range(world):
        own = full[r * n_loc:(r + 1) * n_loc].clone().requires_grad_(True)
        rec, regl = L.loss.bpr_l2_sharded(own, lambda x: full, r * n_loc, gu, gp, gn, REG, batch, lambda t: t.copy_(total))
        (2.0 * rec + 3.0 * regl).backward()
        losses.append(torch.stack([rec.detach(), regl.detach()]))
        grads.append(own.grad)
    for q in losses[1:]:
        assert torch.equal(q, losses[0])
    ref = bpr_ref64(full, full, gu, gp, gn, REG, batch)
    want, terms = ref.du + ref.di, ref.su + ref.si  # users and items index the same table
    assert rel_err(losses[0][0], ref.rec) < RTOL and rel_err(losses[0][1], ref.reg) < RTOL
    got = torch.cat(grads)
    assert within_terms(got, want, terms) and grad_err(got, want) < BPR_GRAD
    idle_rows = slice(idle * n_loc, (idle + 1) * n_loc)
    assert float(ref.su[idle_rows].abs().max()) == 0.0 and float(grads[idle].abs().max()) > 0


SAT_X = [0.0, 1e-3, -1e-3, 10.0, -10.0, 20.0, -20.0, 90.0, -90.0, 200.0, -200.0]
SAT_REPS = 64


def saturated_tables(d):
    """SAT_REPS triples per target x = <u,p> - <u,n>, each with its own rows: p is u0 plus noise, n is small noise, and u =
    u0 * x / <u0, p - n>, so x is a product of rows of comparable size, without cancellation.  x = 0 comes from a zero
    user row.  Targets of |x| >= 90 overflow expf(-x) or expf(x) in float32."""
    rng = np.random.default_rng(d + 7)
    k = len(SAT_X) * SAT_REPS
    u0 = rng.standard_normal((k, d))
    pos = u0 + 0.1 * rng.standard_normal((k, d))
    neg = 0.1 * rng.standard_normal((k, d))
    x = np.repeat(SAT_X, SAT_REPS)
    user = u0 * (x / (u0 * (pos - neg)).sum(1))[:, None]
    return user.astype(np.float32), np.concatenate([pos, neg]).astype(np.float32), x


@pytest.mark.parametrize("d", WIDTHS)
def test_bpr_l2_saturated_scores(L, d):
    """Scores from s = 1/2 to s = 0 and s = 1 in float32.  Every loss and gradient is finite.  Per target, the loss over its
    triples is judged per term: for x <= 0 (and |x| = 1e-3) the term is at least log(2) - 1e-3 and keeps the 1e-5 bar; for
    x >= 10 the term is -log(1e-5 + s) with s within 5e-5 of 1, a difference of two numbers near 1 (10e-6f + 1.0f is
    1.0000100136, so a term of -1e-5 is off by 1.4e-3 of itself).  There float32 gets the sigmoid, the add and the log's
    argument each to about one spacing of floats near 1 (2^-23), so the bar is 8 x 2^-24 absolute on top of 1e-5 relative.
    The gradients of the whole batch keep the global 2e-5 bar."""
    ut, it, x = saturated_tables(d)
    k = ut.shape[0]
    tu, ti = cuda(ut), cuda(it)
    gu, gp, gn = (cuda(a) for a in (np.arange(k), np.arange(k), k + np.arange(k)))
    for t in SAT_X:
        sel = torch.from_numpy(np.flatnonzero(x == t)).cuda()
        rec, regl, du, di = bpr_run(L, tu, ti, gu[sel], gp[sel], gn[sel], REG, SAT_REPS)
        ref = bpr_ref64(tu, ti, gu[sel], gp[sel], gn[sel], REG, SAT_REPS)
        assert all(bool(torch.isfinite(v).all()) for v in (rec, regl, du, di)), t
        bar = RTOL * abs(float(ref.rec)) + (8 * U32 if t >= 10 else 0.0)
        assert abs(float(rec) - float(ref.rec)) <= bar, (t, float(rec), float(ref.rec))
        assert rel_err(regl, ref.reg) < RTOL
    rec, regl, du, di = bpr_run(L, tu, ti, gu, gp, gn, REG, k)
    ref = bpr_ref64(tu, ti, gu, gp, gn, REG, k)
    assert all(bool(torch.isfinite(v).all()) for v in (rec, regl, du, di))
    assert rel_err(rec, ref.rec) < RTOL and rel_err(regl, ref.reg) < RTOL
    assert grad_err(du, ref.du) < BPR_GRAD and grad_err(di, ref.di) < BPR_GRAD


@pytest.mark.parametrize("d", WIDTHS)
def test_bpr_l2_zero_rows(L, d):
    """Every negative is a zero row, so ||N|| = 0 with reg > 0: the L2 gradient of those rows is exactly 0 (torch's norm
    backward masks a zero norm), never NaN, and the rest matches float64.  Then a batch of zero rows only: reg loss 0, rec
    loss -log(0.5 + 1e-5), gradients 0."""
    rng = np.random.default_rng(d)
    batch, n_users, n_items, n_zero = 5000, 300, 700, 20
    ut = (rng.standard_normal((n_users, d)) * 0.3).astype(np.float32)
    it = (rng.standard_normal((n_items, d)) * 0.3).astype(np.float32)
    it[:n_zero] = 0.0
    u, p, n = rng.integers(0, n_users, batch), rng.integers(n_zero, n_items, batch), rng.integers(0, n_zero, batch)
    tu, ti = cuda(ut), cuda(it)
    gu, gp, gn = cuda(u), cuda(p), cuda(n)
    rec, regl, du, di = bpr_run(L, tu, ti, gu, gp, gn, REG, batch)
    ref = bpr_ref64(tu, ti, gu, gp, gn, REG, batch)
    assert bool(torch.isfinite(du).all() and torch.isfinite(di).all())
    assert rel_err(rec, ref.rec) < RTOL and rel_err(regl, ref.reg) < RTOL
    assert grad_err(du, ref.du) < BPR_GRAD and grad_err(di, ref.di) < BPR_GRAD
    _, _, du_reg, di_reg = bpr_run(L, tu, ti, gu, gp, gn, REG, batch, w_rec=0.0, w_reg=1.0)  # the L2 term alone
    assert not bool(di_reg[:n_zero].any()) and bool(torch.isfinite(di_reg).all())
    ref_reg = bpr_ref64(tu, ti, gu, gp, gn, REG, batch, w_rec=0.0, w_reg=1.0)
    assert grad_err(du_reg, ref_reg.du) < BPR_GRAD and grad_err(di_reg, ref_reg.di) < BPR_GRAD
    z_u, z_i = torch.zeros_like(tu), torch.zeros_like(ti)
    rec, regl, du, di = bpr_run(L, z_u, z_i, gu, gp, gn, REG, batch)
    assert float(regl) == 0.0 and rel_err(rec, -np.log(0.5 + 1e-5)) < RTOL
    assert not bool(du.any()) and not bool(di.any())


@pytest.mark.parametrize("d", WIDTHS)
def test_bpr_l2_empty_batch(L, d):
    """No triples: both losses 0 and both gradients zero tensors of the tables' shapes, without an error."""
    tu = torch.randn(30, d, device="cuda")
    ti = torch.randn(50, d, device="cuda")
    e = torch.empty(0, dtype=torch.int64, device="cuda")
    rec, regl, du, di = bpr_run(L, tu, ti, e, e, e, REG, 2048)
    torch.cuda.synchronize()
    assert float(rec) == 0.0 and float(regl) == 0.0
    assert du.shape == tu.shape and di.shape == ti.shape and not bool(du.any()) and not bool(di.any())


def test_bpr_l2_bad_index_counter(L):
    """hgr_bpr_l2_fwd_f32 skips a triple with an id outside its table, or negative, and counts it once however many of its
    ids are bad, also in the last grid pass.  The losses are those of the good triples, the rec mean still over the whole
    batch.  (bpr_l2_from_tables turns a nonzero count into a device-side assertion, so the entry point is called directly.)"""
    d = 64
    batch = 3 * bpr_cap(d) + 17
    rng = np.random.default_rng(11)
    n_users, n_items = 3000, 7000
    u, p, n = rng.integers(0, n_users, batch), rng.integers(0, n_items, batch), rng.integers(0, n_items, batch)
    u[5] = -1
    p[batch // 2] = n_items
    n[batch - 1] = -7
    u[batch - 2], p[batch - 2] = n_users, -1  # two bad ids, one bad triple
    n[batch - 3] = n_items + 100
    bad_rows = [5, batch // 2, batch - 1, batch - 2, batch - 3]
    tu = cuda((rng.standard_normal((n_users, d)) * 0.3).astype(np.float32))
    ti = cuda((rng.standard_normal((n_items, d)) * 0.3).astype(np.float32))
    gu, gp, gn = cuda(u), cuda(p), cuda(n)
    lib = L.lib.lib()
    saved = torch.empty(int(lib.hgr_bpr_l2_workspace_bytes(batch)), dtype=torch.uint8, device="cuda")
    out = torch.empty(2, dtype=torch.float32, device="cuda")
    bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    L.lib.check(lib.hgr_bpr_l2_fwd_f32(tu.data_ptr(), ti.data_ptr(), n_users, n_items, d, gu.data_ptr(), gp.data_ptr(), gn.data_ptr(),
                                       batch, REG, float(batch), out.data_ptr(), saved.data_ptr(), saved.numel(), bad.data_ptr(),
                                       L.lib.stream_ptr()))
    assert int(bad.item()) == len(bad_rows)
    good = torch.from_numpy(np.setdiff1d(np.arange(batch), bad_rows)).cuda()
    ref = bpr_ref64(tu, ti, gu[good], gp[good], gn[good], REG, batch)
    assert rel_err(out[0], ref.rec * good.numel() / batch) < RTOL and rel_err(out[1], ref.reg) < RTOL


# --------------------------------------------------------------------------------------------------- contrastLoss / InfoNCE
def ssl_ref64(e1, e2, nodes, temp, kind, b_cos=True, weight=1.0, chunk=4096):
    """float64 autograd of util/loss_torch.py on the device: contrastLoss (kind 0; F.normalize(E + 1e-8) of the whole tables,
    then the picked rows, repeats included) or InfoNCE (kind 1).  The [M, M] logits are formed in row chunks.  Returns
    (loss, dE1, dE2, c) with c = r / (r + 1e-5) per row for InfoNCE."""
    a1 = e1.detach().double().requires_grad_(True)
    a2 = e2.detach().double().requires_grad_(True)
    if kind == 0:
        A, B = F.normalize(a1 + 1e-8, p=2)[nodes], F.normalize(a2 + 1e-8, p=2)[nodes]
    else:
        A, B = (F.normalize(a1, dim=1), F.normalize(a2, dim=1)) if b_cos else (a1, a2)
    m = A.shape[0]
    total, coef = 0.0, []
    for r0 in range(0, m, chunk):
        a, b = A[r0:r0 + chunk], B[r0:r0 + chunk]
        pos = torch.exp((a * b).sum(-1) / temp)
        ttl = torch.exp(a @ B.T / temp).sum(-1)
        if kind == 0:
            term = -torch.log(pos / (ttl + 1e-8))
        else:
            r = pos / ttl
            term = -torch.log(r + 10e-6)
            coef.append((r / (r + 10e-6)).detach())
        total = total + term.sum()
    loss = total / m
    d1, d2 = torch.autograd.grad(weight * loss, [a1, a2])
    return loss.detach(), d1, d2, (torch.cat(coef) if coef else None)


def ssl_views(d, n_rows, seed):
    """Two views with cosine about 0.3: the positive logit stands out without dominating the row sum."""
    rng = np.random.default_rng(seed)
    e1 = rng.standard_normal((n_rows, d)).astype(np.float32) * 0.3
    e2 = (0.3 * e1 + rng.standard_normal((n_rows, d)) * 0.3).astype(np.float32)
    return e1, e2


def ssl_run(L, kind, t1, t2, nodes, temp, b_cos=True, weight=3.0, need=(True, True)):
    a1, a2 = t1.clone().requires_grad_(need[0]), t2.clone().requires_grad_(need[1])
    loss = L.loss.contrastLoss(a1, a2, nodes, temp) if kind == 0 else L.loss.InfoNCE(a1, a2, temp, b_cos)
    (weight * loss).backward()
    return loss.detach(), a1.grad, a2.grad


def ssl_grad_bar(temp):
    """The global 5e-5 gradient bar holds at T = 0.2.  Its error is that of the float32 logits, which scales with 1 / T."""
    return SSL_GRAD * max(1.0, 0.2 / temp)


SSL_M = [2, 63, 64, 65, 1111, 4096, 18881]  # ssl_splits: 1, 1, 1, 2, 8, 5 and 1 slices
SSL_GRID = [(kind, d, m, 0.2) for kind in (0, 1) for d in WIDTHS for m in SSL_M]
SSL_GRID += [(kind, d, m, t) for kind in (0, 1) for d in (32, 128) for m in (65, 18881) for t in (0.05, 1.0)]


@pytest.mark.parametrize("kind,d,m,temp", SSL_GRID)
def test_ssl_losses_grid(L, kind, d, m, temp):
    """contrastLoss (kind 0, unique ids into tables a third larger than the batch) and InfoNCE (kind 1, M rows) at every
    width, at slice counts 1, 2, 8 and 5 and at M = 18 881 where a single slice loops over 296 tiles, and at T = 0.05 and 1.
    Loss to 1e-5, both weighted gradients to the global bar; unique ids give the same bits on a second run."""
    n_rows = m + m // 3 + 7 if kind == 0 else m
    e1, e2 = ssl_views(d, n_rows, seed=m * 7 + d + kind)
    nodes = np.sort(np.random.default_rng(m).permutation(n_rows)[:m]) if kind == 0 else None
    gnodes = cuda(nodes) if kind == 0 else None
    t1, t2 = cuda(e1), cuda(e2)
    loss, d1, d2 = ssl_run(L, kind, t1, t2, gnodes, temp)
    ref_loss, r1, r2, _ = ssl_ref64(t1, t2, gnodes, temp, kind, weight=3.0)
    bar = ssl_grad_bar(temp)
    assert rel_err(loss, ref_loss) < RTOL
    assert grad_err(d1, r1) < bar and grad_err(d2, r2) < bar
    loss2, d1b, d2b = ssl_run(L, kind, t1, t2, gnodes, temp)
    assert torch.equal(bits(loss), bits(loss2)) and torch.equal(bits(d1), bits(d1b)) and torch.equal(bits(d2), bits(d2b))
    if m <= ORACLE_MAX_M:
        o_loss, o_d1, o_d2 = O.contrast_loss(e1, e2, nodes, temp) if kind == 0 else O.info_nce(e1, e2, temp)
        assert rel_err(loss, o_loss) < RTOL and grad_err(d1, 3.0 * o_d1) < bar and grad_err(d2, 3.0 * o_d2) < bar


@pytest.mark.parametrize("d,b_cos", [(32, True), (64, True), (128, True), (32, False), (128, False)])
def test_infonce_disagreeing_views(L, d, b_cos):
    """Independent views at T = 1: r = exp(pos) / sum is about 1/M, so c = r / (r + 1e-5) sits visibly below 1 and the
    backward must carry it.  b_cos = False has no oracle; its rows are scaled so that the logits stay within a few units."""
    m, temp = 4096, 1.0
    rng = np.random.default_rng(d + b_cos)
    scale = 1.0 if b_cos else 0.3
    v1, v2 = (rng.standard_normal((2, m, d)) * scale).astype(np.float32)
    t1, t2 = cuda(v1), cuda(v2)
    loss, d1, d2 = ssl_run(L, 1, t1, t2, None, temp, b_cos)
    ref_loss, r1, r2, coef = ssl_ref64(t1, t2, None, temp, 1, b_cos, weight=3.0)
    assert float(coef.mean()) < 0.99
    assert rel_err(loss, ref_loss) < RTOL
    assert grad_err(d1, r1) < SSL_GRAD and grad_err(d2, r2) < SSL_GRAD


@pytest.mark.parametrize("d", WIDTHS)
def test_contrast_loss_repeated_ids(L, d):
    """A node list with repeats, as the reference evaluates it: duplicate rows and columns of the logits, and each table row
    gets the sum of the gradients of its copies (index backward)."""
    rng = np.random.default_rng(d)
    e1, e2 = ssl_views(d, 500, seed=d)
    nodes = rng.integers(0, 500, 1111)
    assert np.unique(nodes).size < nodes.size
    t1, t2, gnodes = cuda(e1), cuda(e2), cuda(nodes)
    loss, d1, d2 = ssl_run(L, 0, t1, t2, gnodes, 0.2)
    ref_loss, r1, r2, _ = ssl_ref64(t1, t2, gnodes, 0.2, 0, weight=3.0)
    assert rel_err(loss, ref_loss) < RTOL
    assert grad_err(d1, r1) < SSL_GRAD and grad_err(d2, r2) < SSL_GRAD


@pytest.mark.parametrize("kind", [0, 1])
def test_ssl_one_sided_backward(L, kind):
    """Only one operand requires grad: its gradient equals, bit for bit, that half of the two-sided backward."""
    m, d = 1111, 64
    e1, e2 = ssl_views(d, m, seed=kind)
    t1, t2 = cuda(e1), cuda(e2)
    nodes = cuda(np.arange(m)[::-1].copy()) if kind == 0 else None
    _, d1, d2 = ssl_run(L, kind, t1, t2, nodes, 0.2)
    _, only1, none2 = ssl_run(L, kind, t1, t2, nodes, 0.2, need=(True, False))
    _, none1, only2 = ssl_run(L, kind, t1, t2, nodes, 0.2, need=(False, True))
    assert none1 is None and none2 is None
    assert torch.equal(bits(only1), bits(d1)) and torch.equal(bits(only2), bits(d2))


def test_contrast_loss_unequal_tables(L):
    """E1 has more rows than E2; every id is below both.  Rows of E1 beyond the batch get no gradient."""
    d, m = 64, 1111
    rng = np.random.default_rng(3)
    e1 = (rng.standard_normal((10_000, d)) * 0.3).astype(np.float32)
    e2 = (0.3 * e1[:3000] + rng.standard_normal((3000, d)) * 0.3).astype(np.float32)
    nodes = np.sort(rng.permutation(3000)[:m])
    t1, t2, gnodes = cuda(e1), cuda(e2), cuda(nodes)
    loss, d1, d2 = ssl_run(L, 0, t1, t2, gnodes, 0.2)
    ref_loss, r1, r2, _ = ssl_ref64(t1, t2, gnodes, 0.2, 0, weight=3.0)
    assert d1.shape == t1.shape and d2.shape == t2.shape
    assert rel_err(loss, ref_loss) < RTOL
    assert grad_err(d1, r1) < SSL_GRAD and grad_err(d2, r2) < SSL_GRAD
    assert not bool(d1[3000:].any())


@pytest.mark.parametrize("d", [32, 128])
def test_contrast_loss_padded_extremes(L, d):
    """contrastLoss_padded on 4 096 copies of one id (one active slot, 4 095 inactive) and on a batch that covers every row of
    the tables.  The mean runs over the active slots only, and rows outside the batch get no gradient."""
    n_rows = 3000
    e1, e2 = ssl_views(d, n_rows, seed=d)
    t1, t2 = cuda(e1), cuda(e2)
    one = torch.full((4096,), 1234, dtype=torch.int64, device="cuda")
    a1, a2 = t1.clone().requires_grad_(True), t2.clone().requires_grad_(True)
    loss = L.loss.contrastLoss_padded(a1, a2, one, 0.2)
    (3.0 * loss).backward()
    ref_loss, r1, r2, _ = ssl_ref64(t1, t2, one[:1], 0.2, 0, weight=3.0)
    # a single node: loss = log(1 + 1e-8 / e^x), gradients ~ 0 (pure cancellation), as in test_gpu_losses.py
    assert abs(float(loss.detach()) - float(ref_loss)) < 1e-6 and float(a1.grad.abs().max()) < 1e-6
    rest = torch.ones(n_rows, dtype=torch.bool, device="cuda")
    rest[1234] = False
    assert not bool(a1.grad[rest].any()) and not bool(a2.grad[rest].any())
    rng = np.random.default_rng(d)
    every = cuda(rng.permutation(np.concatenate([np.arange(n_rows), rng.integers(0, n_rows, 4096 - n_rows)])))
    a1, a2 = t1.clone().requires_grad_(True), t2.clone().requires_grad_(True)
    loss = L.loss.contrastLoss_padded(a1, a2, every, 0.2)
    (3.0 * loss).backward()
    ref_loss, r1, r2, _ = ssl_ref64(t1, t2, torch.arange(n_rows, device="cuda"), 0.2, 0, weight=3.0)
    assert rel_err(loss, ref_loss) < RTOL
    assert grad_err(a1.grad, r1) < SSL_GRAD and grad_err(a2.grad, r2) < SSL_GRAD


@pytest.mark.parametrize("d", WIDTHS)
def test_contrast_loss_degenerate_rows(L, d):
    """Zero rows (well defined through the + 1e-8: every entry 1e-8, a direction of all ones) and rows with e1 == e2, whose
    positive logit is the row maximum 1 / T.  A zero row's gradient is divided by its norm of 1e-8 sqrt(D), so it is judged
    on its own and the other rows against theirs.  Then an empty node list: loss 0 and zero gradients (torch's mean over
    nothing would be NaN)."""
    n_rows, m = 2000, 1111
    e1, e2 = ssl_views(d, n_rows, seed=d + 1)
    e1[:10] = 0.0
    e2[10:20] = 0.0
    e2[20:520] = e1[20:520]
    rng = np.random.default_rng(d)
    nodes = np.sort(np.concatenate([np.arange(520), 520 + rng.permutation(n_rows - 520)[:m - 520]]))
    t1, t2, gnodes = cuda(e1), cuda(e2), cuda(nodes)
    loss, d1, d2 = ssl_run(L, 0, t1, t2, gnodes, 0.2)
    ref_loss, r1, r2, _ = ssl_ref64(t1, t2, gnodes, 0.2, 0, weight=3.0)
    assert rel_err(loss, ref_loss) < RTOL
    for got, want, zero in ((d1, r1, slice(0, 10)), (d2, r2, slice(10, 20))):
        keep = torch.ones(n_rows, dtype=torch.bool, device="cuda")
        keep[zero] = False
        assert bool(torch.isfinite(got).all())
        assert grad_err(got[zero], want[zero]) < SSL_GRAD and grad_err(got[keep], want[keep]) < SSL_GRAD
    a1, a2 = t1.clone().requires_grad_(True), t2.clone().requires_grad_(True)
    loss = L.loss.contrastLoss(a1, a2, torch.empty(0, dtype=torch.int64, device="cuda"), 0.2)
    (3.0 * loss).backward()
    torch.cuda.synchronize()
    assert float(loss.detach()) == 0.0 and not bool(a1.grad.any()) and not bool(a2.grad.any())
