"""The propagation epilogue, hgconv's autograd and the LayerNorm kernels at every supported width (D = 32, 64, 128), on
whole rows and on split rows reduced by both paths of spmm_heavy_reduce_kernel (one row group for rows of at most 64
chunks, the whole block above), against float64 references.

The epilogue is checked against float64 arithmetic applied to the kernel's own ``pre`` (the product before the
epilogue), which isolates the epilogue from the summation order of the product; ``pre`` itself is checked bit for bit
against the same plan without an epilogue and, on rows that are not split, against the sequential CPU oracle."""
import ctypes as C
import types

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.nn.functional as F

from oracle import hgr_oracle as O

from conftest import rowwise_rel_err as rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
GROUP_REDUCE_MAX = 64  # spmm.cu kGroupReduceMax: split rows with more chunks are summed by the whole block
SENTINEL = 0x7FC0BEEF  # a NaN bit pattern no kernel produces
SLOPE = float(np.float32(0.3))
EPS = float(np.float32(1e-5))  # the epilogue and the LayerNorm kernels take eps as float32
WIDTHS = [32, 64, 128]
PLANS = ["whole", "chunk64", "chunk8", "window"]


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def sentinel(rows, d):
    return torch.full((rows, d), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


def untouched(t):
    return bool((t.view(torch.int32) == SENTINEL).any())


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def column_bar_ok(got, want, terms):
    """Sums of many terms of both signs (dgamma, dbeta): per column, |got - want| <= 1e-5 * sum_rows |term|.  A bar relative
    to the result alone would be either flaky or toothless."""
    got = got.detach().double().cpu()
    return bool(((got - want).abs() <= RTOL * terms.abs().sum(0)).all())


def dgamma_terms(dy, xhat):
    """The size of each term dy * x_hat of dgamma.  float32 knows x_hat = (x - mean) * rstd only to a few ulps of the row's
    scale, not of x_hat itself, so an entry near the row mean counts as |dy| (|x_hat| + 1)."""
    return dy.abs() * (xhat.abs() + 1)


@pytest.fixture(scope="module")
def hgr():
    from hypergraph_diffusion_for_recommendation_b200 import _lib, graph, ops

    assert torch.cuda.is_available()
    _lib.lib()  # raises if libhgr.so is missing: there is no fallback
    return types.SimpleNamespace(lib=_lib, graph=graph, ops=ops)


@pytest.fixture(scope="module")
def big(hgr):
    """An 8 000-node power-law adjacency (rows of up to 2 195 nonzeros) under four plans of the same CSR: no split rows;
    rows cut every 64 nonzeros (at most 35 chunks: group reduce only); every 8 nonzeros and at 512-row window crossings
    (both reduce paths; the window plan gives chunk_start explicit boundaries)."""
    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions

    g = powerlaw_interactions(3000, 5000, 120_000, seed=3)
    csr = O.build_norm_adj(g.train_u, g.train_i, 3000, 5000)
    n = 8000
    mk = lambda **kw: hgr.graph.DeviceCSR.from_host(*csr, (n, n), symmetric=True, **kw)
    plans = {"whole": mk(chunk_nnz=1 << 30), "chunk64": mk(chunk_nnz=64), "chunk8": mk(chunk_nnz=8),
             "window": mk(chunk_nnz=16, split="window:9:8:0")}
    light, paths = {}, {}
    for name, a in plans.items():
        heavy = a.heavy_rows.long().cpu()
        chunks = (a.heavy_chunk_ptr[1:] - a.heavy_chunk_ptr[:-1]).cpu()
        mask = torch.ones(n, dtype=torch.bool)
        mask[heavy] = False
        light[name] = mask
        paths[name] = (int((chunks <= GROUP_REDUCE_MAX).sum()), int((chunks > GROUP_REDUCE_MAX).sum()))
    assert paths["whole"] == (0, 0)
    assert paths["chunk64"][0] > 0 and paths["chunk64"][1] == 0  # 2 195 nonzeros are 35 chunks of 64
    for name in ("chunk8", "window"):
        assert paths[name][0] > 0 and paths[name][1] > 0, (name, paths[name])
    assert plans["window"].desc.chunk_start
    return types.SimpleNamespace(g=g, csr=csr, n=n, plans=plans, light=light, paths=paths, cache={})


def _inputs(big, d):
    """Per width: X, the oracle's product and every plan's product without an epilogue (computed once)."""
    if d not in big.cache:
        x = np.random.default_rng(d).standard_normal((big.n, d)).astype(np.float32)
        big.cache[d] = (x, O.spmm(*big.csr, x), {})
    return big.cache[d]


def epilogue64(pre, slope=None, gamma=None, beta=None, residual=None, addends=(), scale=1.0, scaled=False):
    """finish_row in float64, from the kernel's own pre."""
    a = pre.detach().double().cpu()
    if slope is not None:
        a = torch.where(a > 0, a, a * slope)
    if gamma is not None:
        mu = a.mean(1, keepdim=True)
        var = ((a - mu) ** 2).mean(1, keepdim=True)
        a = (a - mu) / torch.sqrt(var + EPS) * gamma.double().cpu() + beta.double().cpu()
    if residual is not None:
        a = a + residual.double().cpu()
    for t in addends:
        a = a + t.double().cpu()
    if scaled:
        a = a * scale
    return a


# ------------------------------------------------------------------------------------------ A: epilogue x width x plan
@pytest.mark.parametrize("stage", ["full", "ln", "leaky", "scale_always"])
@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("d", WIDTHS)
def test_epilogue_at_every_width_on_every_reduce_path(hgr, big, d, plan, stage):
    a = big.plans[plan]
    x, ref, plain = _inputs(big, d)
    xt = cuda(x)
    if plan not in plain:
        plain[plan] = hgr.ops.spmm_raw(a, xt)
    rng = np.random.default_rng(1000 * d + 10 * PLANS.index(plan) + len(stage))
    rnd = lambda *s: cuda(rng.standard_normal(s).astype(np.float32))
    kw = {}
    if stage == "full":
        kw = dict(slope=SLOPE, gamma=rnd(d), beta=rnd(d), residual=rnd(big.n, d), addends=tuple(rnd(big.n, d) for _ in range(8)),
                  scale=0.25)
        assert len(kw["addends"]) == hgr.lib.HGR_MAX_ADDENDS
    elif stage == "ln":
        kw = dict(gamma=rnd(d), beta=rnd(d), scale=0.25)  # no addends and no scale_always: the scale is not applied
    elif stage == "leaky":
        kw = dict(slope=SLOPE)
    else:
        kw = dict(scale=0.25, scale_always=True)
    outs = []
    for _ in range(2):
        pre, y = sentinel(big.n, d), sentinel(big.n, d)
        hgr.ops.spmm_raw(a, xt, hgr.ops._epilogue(pre=pre, **kw), out=y)
        assert not untouched(pre) and not untouched(y)  # every row written
        outs.append((pre, y))
    (pre, y), (pre2, y2) = outs
    assert torch.equal(bits(pre), bits(pre2)) and torch.equal(bits(y), bits(y2))  # reproducible: no atomics
    assert torch.equal(bits(pre), bits(plain[plan]))  # pre is the product, stored before the epilogue
    light = big.light[plan]
    assert torch.equal(bits(pre).cpu()[light], bits(torch.from_numpy(ref))[light])  # unsplit rows: the oracle's bits
    want = epilogue64(pre, kw.get("slope"), kw.get("gamma"), kw.get("beta"), kw.get("residual"), kw.get("addends", ()), 0.25,
                      stage in ("full", "scale_always"))
    assert rel_err(y, want) < RTOL


@pytest.mark.parametrize("d", WIDTHS)
def test_lightgcn_readout_at_the_addend_limit(hgr, big, d):
    """hgr_lightgcn_forward_f32 with 8 layers: the readout epilogue adds E0 and the 7 stored layers (HGR_MAX_ADDENDS).
    Against float64 layers; and on rows that are not split, every layer and the readout are the bits of the plan without
    split rows applied to the same input."""
    lib = hgr.lib.lib()
    a, whole = big.plans["chunk8"], big.plans["whole"]
    n, L = big.n, 8
    e0 = cuda(np.random.default_rng(77 + d).standard_normal((n, d)).astype(np.float32))
    layers = sentinel((L - 1) * n, d).view(L - 1, n, d)
    out = sentinel(n, d)
    ws = a.workspace(d)
    hgr.lib.check(lib.hgr_lightgcn_forward_f32(C.byref(a.desc), e0.data_ptr(), layers.data_ptr(), out.data_ptr(), L, d, 0, ws.data_ptr(),
                                               ws.numel() * 4, hgr.lib.stream_ptr()))
    assert not untouched(layers) and not untouched(out)
    assert torch.equal(bits(out), bits(hgr.ops.lightgcn_propagate_raw(a, e0, L)))
    ip, ix, dv = big.csr
    m = sp.csr_matrix((dv.astype(np.float64), ix, ip), shape=(n, n))
    e = e0.double().cpu().numpy()
    acc = e.copy()
    for _ in range(L):
        e = m @ e
        acc += e
    assert rel_err(out, acc / (L + 1)) < RTOL
    light = big.light["chunk8"]
    prev = e0
    for k in range(L - 1):
        assert torch.equal(bits(layers[k]).cpu()[light], bits(hgr.ops.spmm_raw(whole, prev)).cpu()[light]), k
        prev = layers[k]
    ep = hgr.ops._epilogue(addends=(e0,) + tuple(layers[k] for k in range(L - 1)), scale=float(np.float32(1) / np.float32(L + 1)))
    assert torch.equal(bits(out).cpu()[light], bits(hgr.ops.spmm_raw(whole, layers[L - 2], ep)).cpu()[light])


# ------------------------------------------------------------------------------------------ B: hgconv autograd
@pytest.fixture(scope="module")
def rect(hgr, big):
    """The row-normalised [users, items] interaction matrix, cut every 8 nonzeros (and its transpose)."""
    g = big.g
    r = hgr.graph.build_interaction_csr(g.train_u, g.train_i, 3000, 5000, row_normalize=True, chunk_nnz=8)
    assert r.desc.n_heavy_rows > 0 and r.t().desc.n_heavy_rows > 0
    return r


def _sparse64(a):
    ip, ix, dv = (t.cpu() for t in (a.indptr, a.indices, a.values))
    rows = torch.repeat_interleave(torch.arange(a.shape[0]), ip[1:] - ip[:-1])
    return torch.sparse_coo_tensor(torch.stack([rows, ix.long()]), dv.double(), a.shape).coalesce()


HGCONV_CASES = {  # name: (slope, layer norm, residual)
    "leaky_ln_residual_is_x": (0.5, True, "x"),
    "leaky_ln_residual": (0.5, True, "separate"),
    "ln_only": (None, True, None),
    "leaky_only": (0.2, False, None),
}


@pytest.mark.parametrize("matrix", ["square", "rectangular"])
@pytest.mark.parametrize("case", list(HGCONV_CASES))
@pytest.mark.parametrize("d", WIDTHS)
def test_hgconv_autograd_at_every_width(hgr, big, rect, d, case, matrix):
    slope, ln, res = HGCONV_CASES[case]
    if matrix == "rectangular" and res == "x":
        pytest.skip("y = f(x) + x needs a square matrix")
    a = big.plans["chunk8"] if matrix == "square" else rect
    n_out, n_in = a.shape[0], a.t().shape[1]
    rng = np.random.default_rng(d + 7 * len(case) + len(matrix))
    f32 = lambda *s: rng.standard_normal(s).astype(np.float32)
    x, gam, bet, r, gr = f32(n_in, d), 1 + 0.1 * f32(d), f32(d), f32(n_out, d), f32(n_out, d)
    xt = cuda(x).requires_grad_(True)
    gt = cuda(gam).requires_grad_(True) if ln else None
    bt = cuda(bet).requires_grad_(True) if ln else None
    rt = cuda(r).requires_grad_(True) if res == "separate" else None
    y = hgr.ops.hgconv(a, xt, slope=slope, ln_weight=gt, ln_bias=bt, residual=xt if res == "x" else rt)
    (y * cuda(gr)).sum().backward()

    # float64 reference
    A = _sparse64(a)
    x64 = torch.from_numpy(x).double().requires_grad_(True)
    g64 = torch.from_numpy(gam).double().requires_grad_(True)
    b64 = torch.from_numpy(bet).double().requires_grad_(True)
    r64 = torch.from_numpy(r).double().requires_grad_(True)
    z = torch.sparse.mm(A, torch.sparse.mm(A.t(), x64))
    if slope is not None:
        # LeakyReLU with the branch the kernel took: an entry within rounding of zero may have the other sign in float64,
        # and the derivative jumps there from 1 to the slope.  The kernel's pre is the same product (same plan, same bits).
        pre = torch.empty(n_out, d, device="cuda")
        hgr.ops.hgconv_raw(a, a.t(), xt.detach(), hgr.ops._epilogue(pre=pre))
        z = z * torch.where(pre.cpu() > 0, 1.0, float(np.float32(slope))).double()
    xhat = None
    if ln:
        xhat = F.layer_norm(z, (d,), eps=EPS)
        z = xhat * g64 + b64
    if res == "x":
        z = z + x64
    elif res == "separate":
        z = z + r64
    G = torch.from_numpy(gr).double()
    (z * G).sum().backward()
    assert rel_err(y, z.detach()) < RTOL
    assert rel_err(xt.grad, x64.grad) < 2e-5
    if res == "separate":
        assert torch.equal(bits(rt.grad), bits(cuda(gr)))
    if ln:
        assert column_bar_ok(gt.grad, g64.grad, dgamma_terms(G, xhat.detach()))
        assert column_bar_ok(bt.grad, b64.grad, G)


# ------------------------------------------------------------------------------------------ C: the LayerNorm kernels
def _ln_reference(x, gamma, beta, dy, slope=None):
    """float64 autograd of LayerNorm(leaky_relu(x)) * gamma + beta: (y, dx, dgamma, dbeta, x_hat)."""
    x64 = x.double().cpu().requires_grad_(True)
    g64 = gamma.double().cpu().requires_grad_(True)
    b64 = beta.double().cpu().requires_grad_(True)
    a = x64 if slope is None else F.leaky_relu(x64, slope)
    xhat = F.layer_norm(a, (x.shape[1],), eps=EPS)
    y = xhat * g64 + b64
    (y * dy.double().cpu()).sum().backward()
    return y.detach(), x64.grad, g64.grad, b64.grad, xhat.detach()


@pytest.mark.parametrize("n", [1, 7, 8257, 100_003])
@pytest.mark.parametrize("d", WIDTHS)
def test_layer_norm_kernels_on_random_rows(hgr, d, n):
    """hgr_layer_norm_f32 and hgr_leaky_ln_bwd_f32 (with and without gamma).  8 257 rows make 130 partial blocks, so each
    thread of the parameter-gradient reduce adds two; 100 003 rows reach the backward's cap of 1 184 blocks."""
    gen = torch.Generator(device="cuda").manual_seed(n + d)
    rnd = lambda *s: torch.randn(*s, generator=gen, device="cuda")
    x, dy = rnd(n, d), rnd(n, d)
    gamma, beta = 1 + 0.1 * rnd(d), rnd(d)
    xg, gg, bg = (t.clone().requires_grad_(True) for t in (x, gamma, beta))
    y = hgr.ops.layer_norm(xg, gg, bg, eps=EPS)
    y.backward(dy)
    want_y, want_dx, want_dg, want_db, xhat = _ln_reference(x, gamma, beta, dy)
    assert rel_err(y, want_y) < RTOL
    assert rel_err(xg.grad, want_dx) < RTOL
    G = dy.double().cpu()
    assert column_bar_ok(gg.grad, want_dg, dgamma_terms(G, xhat)) and column_bar_ok(bg.grad, want_db, G)

    # the backward with LeakyReLU in front, twice: the parameter gradients are reproducible
    dpre, dg, db = hgr.ops.leaky_ln_bwd(x, dy, gamma, EPS, SLOPE)
    dpre2, dg2, db2 = hgr.ops.leaky_ln_bwd(x, dy, gamma, EPS, SLOPE)
    assert torch.equal(bits(dpre), bits(dpre2)) and torch.equal(bits(dg), bits(dg2)) and torch.equal(bits(db), bits(db2))
    _, want_dpre, want_dg, want_db, xhat = _ln_reference(x, gamma, beta, dy, SLOPE)
    assert rel_err(dpre, want_dpre) < RTOL
    assert column_bar_ok(dg, want_dg, dgamma_terms(G, xhat)) and column_bar_ok(db, want_db, G)

    # no LayerNorm: dpre is dy or dy * slope, one float32 product
    dpre, dg, db = hgr.ops.leaky_ln_bwd(x, dy, None, EPS, SLOPE)
    assert dg is None and db is None
    assert torch.equal(bits(dpre), bits(torch.where(x > 0, dy, dy * SLOPE)))


@pytest.mark.parametrize("d", WIDTHS)
def test_layer_norm_forward_at_its_grid_cap(hgr, d):
    """160 001 rows: more than the forward's 2 368 blocks of 64 rows, so the blocks stride over the rows."""
    n = 160_001
    gen = torch.Generator(device="cuda").manual_seed(d)
    x = torch.randn(n, d, generator=gen, device="cuda") * 3 + 1
    gamma, beta = torch.randn(d, generator=gen, device="cuda"), torch.randn(d, generator=gen, device="cuda")
    with torch.no_grad():
        y = hgr.ops.layer_norm(x, gamma, beta, eps=EPS)
    x64 = x.double().cpu()
    assert rel_err(y, F.layer_norm(x64, (d,), gamma.double().cpu(), beta.double().cpu(), eps=EPS)) < RTOL


def _row_errs(got, want):
    """Per row: max_j |got - want| / max_j |want| (rowwise_rel_err before its max over rows)."""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    scale = want.abs().amax(1).clamp(min=1e-30)
    return (got - want).abs().amax(1) / scale


@pytest.mark.parametrize("family", ["offset", "constant"])
@pytest.mark.parametrize("d", WIDTHS)
def test_layer_norm_on_ill_conditioned_rows(hgr, d, family):
    """Rows where float32 itself loses digits: a large common offset (1e3 + N(0, 1e-2)) and constant rows (var = 0).  The
    bar is the reference's own arithmetic: torch's float32 CUDA layer_norm against float64.  Over the rows of the family,
    the kernel's worst error is at most twice torch's worst error (+ 1e-6)."""
    n = 8257
    gen = torch.Generator(device="cuda").manual_seed(d + len(family))
    if family == "offset":
        x = 1e3 + 1e-2 * torch.randn(n, d, generator=gen, device="cuda")
    else:
        x = (10 * torch.randn(n, 1, generator=gen, device="cuda")).expand(n, d).contiguous()
        x[:3] = torch.tensor([0.0, 1e3, -7.25], device="cuda")[:, None]
    dy = torch.randn(n, d, generator=gen, device="cuda")
    gamma, beta = 1 + 0.1 * torch.randn(d, generator=gen, device="cuda"), torch.randn(d, generator=gen, device="cuda")
    want_y, want_dx, want_dg, want_db, xhat = _ln_reference(x, gamma, beta, dy)

    def run(fn):
        xg, gg, bg = (t.clone().requires_grad_(True) for t in (x, gamma, beta))
        y = fn(xg, gg, bg)
        y.backward(dy)
        return y, xg.grad, gg.grad, bg.grad

    got = run(lambda a, g, b: hgr.ops.layer_norm(a, g, b, eps=EPS))
    t32 = run(lambda a, g, b: F.layer_norm(a, (d,), g, b, eps=EPS))
    for what, k, want in (("y", 0, want_y), ("dx", 1, want_dx)):
        mine, theirs = _row_errs(got[k], want).max(), _row_errs(t32[k], want).max()
        assert mine <= 2 * theirs + 1e-6, (what, float(mine), float(theirs))
    for what, k, want, terms in (("dgamma", 2, want_dg, dgamma_terms(dy.double().cpu(), xhat)), ("dbeta", 3, want_db, dy.double().cpu())):
        size = terms.abs().sum(0)
        mine = ((got[k].double().cpu() - want).abs() / size).max()
        theirs = ((t32[k].double().cpu() - want).abs() / size).max()
        assert mine <= 2 * theirs + RTOL, (what, float(mine), float(theirs))
    if family == "constant":  # mean and variance are exact: y = beta, bit for bit
        assert torch.equal(bits(got[0]), bits(beta.expand(n, d)))


@pytest.mark.parametrize("d", WIDTHS)
def test_leaky_ln_bwd_at_the_kink(hgr, d):
    """pre == 0 (both signs): the LeakyReLU derivative there is the slope, as in torch."""
    n = 2049
    gen = torch.Generator(device="cuda").manual_seed(d)
    pre = torch.randn(n, d, generator=gen, device="cuda")
    pick = torch.rand(n, d, generator=gen, device="cuda")
    pre[pick < 0.3] = 0.0
    pre[pick > 0.85] = -0.0
    pre[:4] = 0.0  # whole rows at the kink
    dy = torch.randn(n, d, generator=gen, device="cuda")
    dpre, _, _ = hgr.ops.leaky_ln_bwd(pre, dy, None, EPS, SLOPE)
    assert torch.equal(bits(dpre), bits(torch.where(pre > 0, dy, dy * SLOPE)))
    p = pre.clone().requires_grad_(True)
    F.leaky_relu(p, SLOPE).backward(dy)
    assert torch.equal(bits(dpre), bits(p.grad))  # torch's own float32 derivative
    dpre, _, _ = hgr.ops.leaky_ln_bwd(pre, dy, None, EPS, None)
    assert torch.equal(bits(dpre), bits(dy))
    gamma, beta = 1 + 0.1 * torch.randn(d, generator=gen, device="cuda"), torch.randn(d, generator=gen, device="cuda")
    dpre, dg, db = hgr.ops.leaky_ln_bwd(pre, dy, gamma, EPS, SLOPE)
    _, want_dpre, want_dg, want_db, xhat = _ln_reference(pre, gamma, beta, dy, SLOPE)
    assert rel_err(dpre, want_dpre) < RTOL
    G = dy.double().cpu()
    assert column_bar_ok(dg, want_dg, dgamma_terms(G, xhat)) and column_bar_ok(db, want_db, G)
