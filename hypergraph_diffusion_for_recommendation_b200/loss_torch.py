"""Losses of the reference's ``util/loss_torch.py`` on libhgr.so.

``contrastLoss`` / ``InfoNCE`` (util/loss_torch.py:103-110, 32-40) run on csrc/loss_ssl.cu.

``bpr_l2_from_tables`` is the fused product path: gathers + BPR + L2 in one forward launch and one
backward launch (reference: ``rec_user_emb[user_idx]`` ... ``bpr_loss`` ... ``l2_reg_loss / batch_size``,
model/graph/LightGCN.py:52-55).  ``bpr_loss`` / ``l2_reg_loss`` keep the reference signatures
(util/loss_torch.py:5-9,17-21) for callers that already hold gathered rows.
"""
from __future__ import annotations

import torch

from . import _lib


def _raise_on_bad_index(bad: torch.Tensor, what: str) -> None:
    """The kernels skip ids outside the tables and count them; the reference's ``emb[idx]`` raises IndexError.  Surface the
    counter without a host synchronisation: a device-side assertion (fatal, like the reference's exception; capturable)."""
    torch._assert_async(bad[0] == 0, "libhgr: %s got indices outside the embedding tables (see include/hgr.h)" % what)


def _idx(t: torch.Tensor, device) -> torch.Tensor:
    # the reference's sampler yields CPU LongTensors (util/sampler.py:261-263): one H2D copy here
    return t.to(device=device, dtype=torch.int64, non_blocking=True).contiguous()


class _BprL2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, user_tab, item_tab, u, p, n, reg, batch_size):
        if not (user_tab.is_cuda and item_tab.is_cuda):
            raise _lib.HgrError("embedding tables must be CUDA tensors (no CPU path)")
        user_tab, item_tab = user_tab.contiguous(), item_tab.contiguous()
        if user_tab.dtype != torch.float32 or item_tab.dtype != torch.float32 or user_tab.shape[1] != item_tab.shape[1]:
            raise TypeError("tables must be float32 with equal width")
        dev = user_tab.device
        u, p, n = _idx(u, dev), _idx(p, dev), _idx(n, dev)
        batch = int(u.numel())
        if p.numel() != batch or n.numel() != batch:
            raise ValueError("user / pos / neg index arrays differ in length")
        lib = _lib.lib()
        saved = torch.empty(int(lib.hgr_bpr_l2_workspace_bytes(batch)), dtype=torch.uint8, device=dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.hgr_bpr_l2_fwd_f32(user_tab.data_ptr(), item_tab.data_ptr(), user_tab.shape[0], item_tab.shape[0],
                                          user_tab.shape[1], u.data_ptr(), p.data_ptr(), n.data_ptr(), batch, float(reg),
                                          float(batch_size), out.data_ptr(), saved.data_ptr(), saved.numel(), bad.data_ptr(),
                                          _lib.stream_ptr()))
        _raise_on_bad_index(bad, "bpr_l2_from_tables")
        ctx.save_for_backward(user_tab, item_tab, u, p, n, saved)
        ctx.reg, ctx.batch_size = float(reg), float(batch_size)
        return out

    @staticmethod
    def backward(ctx, grad):
        user_tab, item_tab, u, p, n, saved = ctx.saved_tensors
        du, di = torch.zeros_like(user_tab), torch.zeros_like(item_tab)
        grad = grad.contiguous().to(torch.float32)
        _lib.check(_lib.lib().hgr_bpr_l2_bwd_f32(user_tab.data_ptr(), item_tab.data_ptr(), user_tab.shape[0], item_tab.shape[0],
                                                 user_tab.shape[1], u.data_ptr(), p.data_ptr(), n.data_ptr(), int(u.numel()), ctx.reg,
                                                 ctx.batch_size, saved.data_ptr(), grad.data_ptr(), du.data_ptr(), di.data_ptr(),
                                                 _lib.stream_ptr()))
        return du, di, None, None, None, None, None


class _BprL2Sharded(torch.autograd.Function):
    """BPR + L2 over ONE gathered table of which this rank owns rows ``[row_lo, row_hi)``: the forward gathers the table
    (``gather`` callable: a collective, or the copy a propagation kernel already published), evaluates the loss on the whole
    batch (identical on every rank), and the backward produces only the owned gradient rows (hgr_bpr_l2_bwd_window_f32)."""

    @staticmethod
    def forward(ctx, own, gather, row_lo, u, p, n, reg, batch_size):
        full = gather(own).contiguous()
        dev = full.device
        u, p, n = _idx(u, dev), _idx(p, dev), _idx(n, dev)
        batch = int(u.numel())
        lib = _lib.lib()
        saved = torch.empty(int(lib.hgr_bpr_l2_workspace_bytes(batch)), dtype=torch.uint8, device=dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.hgr_bpr_l2_fwd_f32(full.data_ptr(), full.data_ptr(), full.shape[0], full.shape[0], full.shape[1], u.data_ptr(),
                                          p.data_ptr(), n.data_ptr(), batch, float(reg), float(batch_size), out.data_ptr(),
                                          saved.data_ptr(), saved.numel(), bad.data_ptr(), _lib.stream_ptr()))
        _raise_on_bad_index(bad, "bpr_l2_sharded (ids must index the gathered table: Partition.perm_user / perm_item)")
        ctx.save_for_backward(full, u, p, n, saved)
        ctx.meta = (int(row_lo), int(own.shape[0]), float(reg), float(batch_size))
        return out

    @staticmethod
    def backward(ctx, grad):
        full, u, p, n, saved = ctx.saved_tensors
        row_lo, n_own, reg, batch_size = ctx.meta
        d = torch.zeros((n_own, full.shape[1]), dtype=torch.float32, device=full.device)
        grad = grad.contiguous().to(torch.float32)
        _lib.check(_lib.lib().hgr_bpr_l2_bwd_window_f32(full.data_ptr(), full.shape[0], full.shape[1], u.data_ptr(), p.data_ptr(),
                                                        n.data_ptr(), int(u.numel()), reg, batch_size, saved.data_ptr(), grad.data_ptr(),
                                                        row_lo, row_lo + n_own, d.data_ptr(), _lib.stream_ptr()))
        return d, None, None, None, None, None, None, None


class _BprL2Owned(torch.autograd.Function):
    """The same loss with the forward sharded by OWNER (VERDICT r1, item 5): a rank evaluates the triples whose user row it
    owns (hgr_bpr_l2_fwd_owned_f32: 1/world of the gathers), the four batch sums are added over the ranks with ONE all_reduce of
    32 bytes (``reduce_sums``), hgr_bpr_l2_finish_f32 turns the totals into the two losses -- identical on every rank -- and the
    backward (hgr_bpr_l2_bwd_owned_f32) produces this rank's gradient rows from every triple that touches one of them,
    recomputing ``x`` from the rows it loads anyway.  Nothing crosses ranks but the 32 bytes."""

    @staticmethod
    def forward(ctx, own, gather, row_lo, u, p, n, reg, batch_size, reduce_sums):
        full = gather(own).contiguous()
        dev = full.device
        u, p, n = _idx(u, dev), _idx(p, dev), _idx(n, dev)
        batch = int(u.numel())
        lib = _lib.lib()
        n_own = int(own.shape[0])
        scratch = torch.empty(int(lib.hgr_bpr_l2_workspace_bytes(batch)), dtype=torch.uint8, device=dev)
        sums = torch.empty(4, dtype=torch.float64, device=dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        norms = torch.empty(4, dtype=torch.float32, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.hgr_bpr_l2_fwd_owned_f32(full.data_ptr(), full.shape[0], full.shape[1], u.data_ptr(), p.data_ptr(), n.data_ptr(),
                                                batch, int(row_lo), int(row_lo) + n_own, sums.data_ptr(), scratch.data_ptr(),
                                                scratch.numel(), bad.data_ptr(), _lib.stream_ptr()))
        reduce_sums(sums)
        _lib.check(lib.hgr_bpr_l2_finish_f32(sums.data_ptr(), batch, float(reg), float(batch_size), out.data_ptr(), norms.data_ptr(),
                                             _lib.stream_ptr()))
        _raise_on_bad_index(bad, "bpr_l2_sharded (ids must index the gathered table: Partition.perm_user / perm_item)")
        ctx.save_for_backward(full, u, p, n, norms)
        ctx.meta = (int(row_lo), n_own, float(reg), float(batch_size))
        return out

    @staticmethod
    def backward(ctx, grad):
        full, u, p, n, norms = ctx.saved_tensors
        row_lo, n_own, reg, batch_size = ctx.meta
        d = torch.zeros((n_own, full.shape[1]), dtype=torch.float32, device=full.device)
        grad = grad.contiguous().to(torch.float32)
        _lib.check(_lib.lib().hgr_bpr_l2_bwd_owned_f32(full.data_ptr(), full.shape[0], full.shape[1], u.data_ptr(), p.data_ptr(),
                                                       n.data_ptr(), int(u.numel()), reg, batch_size, norms.data_ptr(), grad.data_ptr(),
                                                       row_lo, row_lo + n_own, d.data_ptr(), _lib.stream_ptr()))
        return d, None, None, None, None, None, None, None, None


def bpr_l2_sharded(own_rows, gather, row_lo, user_idx, pos_idx, neg_idx, reg, batch_size, reduce_sums=None):
    """``(rec_loss, reg_loss)`` for sharded training; ``user_idx / pos_idx / neg_idx`` index the gathered table.  With
    ``reduce_sums`` (a callable that adds a 4-element float64 tensor over the ranks in place) the forward is sharded by owner
    (``_BprL2Owned``); without it every rank evaluates the whole batch (``_BprL2Sharded``)."""
    if reduce_sums is not None:
        out = _BprL2Owned.apply(own_rows, gather, row_lo, user_idx, pos_idx, neg_idx, reg, batch_size, reduce_sums)
    else:
        out = _BprL2Sharded.apply(own_rows, gather, row_lo, user_idx, pos_idx, neg_idx, reg, batch_size)
    return out[0], out[1]


def bpr_l2_from_tables(user_tab, item_tab, user_idx, pos_idx, neg_idx, reg, batch_size):
    """Returns ``(rec_loss, reg_loss)`` as 0-d tensors; ``reg_loss`` already carries ``/ batch_size``."""
    out = _BprL2.apply(user_tab, item_tab, user_idx, pos_idx, neg_idx, reg, batch_size)
    return out[0], out[1]


def bpr_loss(user_emb, pos_item_emb, neg_item_emb):
    """util/loss_torch.py:5-9 on already gathered rows (identity gather through the fused kernel)."""
    b = user_emb.shape[0]
    ar = torch.arange(b, device=user_emb.device)
    items = torch.cat([pos_item_emb, neg_item_emb], 0)
    return _BprL2.apply(user_emb, items, ar, ar, ar + b, 0.0, 1.0)[0]


def l2_reg_loss(reg, *args):
    """util/loss_torch.py:17-21: ``reg * sum_k ||args[k]||_F``."""
    emb_loss = 0
    for emb in args:
        emb_loss = emb_loss + torch.norm(emb, p=2)
    return emb_loss * reg


class _SslLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, e1, e2, nodes, temp, kind, normalize):
        if not (e1.is_cuda and e2.is_cuda):
            raise _lib.HgrError("embedding tables must be CUDA tensors (no CPU path)")
        if e1.dtype != torch.float32 or e2.dtype != torch.float32 or e1.dim() != 2 or e2.dim() != 2 or e1.shape[1] != e2.shape[1]:
            raise TypeError("operands must be 2-D float32 with equal width")
        e1, e2 = e1.contiguous(), e2.contiguous()
        dev = e1.device
        if nodes is not None:
            nodes = _idx(nodes, dev)
            m = int(nodes.numel())
        else:
            if e1.shape[0] != e2.shape[0]:
                raise ValueError("views differ in length")
            m = int(e1.shape[0])
        d = int(e1.shape[1])
        lib = _lib.lib()
        nbytes = int(lib.hgr_ssl_workspace_bytes(m, d))
        saved = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
        off = (-saved.data_ptr()) % 256
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.hgr_ssl_loss_fwd_f32(e1.data_ptr(), e2.data_ptr(), e1.shape[0], e2.shape[0], d, _lib.ptr(nodes), m, float(temp),
                                            int(kind), int(normalize), loss.data_ptr(), saved.data_ptr() + off, nbytes, bad.data_ptr(),
                                            _lib.stream_ptr()))
        ctx.save_for_backward(saved, nodes if nodes is not None else torch.empty(0, device=dev))
        ctx.meta = (e1.shape, e2.shape, d, m, float(temp), int(normalize), off, nbytes, nodes is not None)
        _raise_on_bad_index(bad, "contrastLoss / InfoNCE (a NEGATIVE id is an inactive slot of contrastLoss_padded, an id >= rows is an error)")
        return loss[0]

    @staticmethod
    def backward(ctx, grad):
        saved, nodes = ctx.saved_tensors
        s1, s2, d, m, temp, normalize, off, nbytes, has_nodes = ctx.meta
        dev = saved.device
        d1 = torch.zeros(s1, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        d2 = torch.zeros(s2, dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        g = grad.reshape(1).contiguous().to(torch.float32)
        _lib.check(_lib.lib().hgr_ssl_loss_bwd_f32(s1[0], s2[0], d, nodes.data_ptr() if has_nodes else None, m, temp, normalize,
                                                   saved.data_ptr() + off, nbytes, g.data_ptr(), _lib.ptr(d1), _lib.ptr(d2),
                                                   _lib.stream_ptr()))
        return d1, d2, None, None, None, None


def contrastLoss(embeds1, embeds2, nodes, temp):
    """util/loss_torch.py:103-110.  Only the picked rows are normalised and the [M, M] logits stay on chip.  The reference
    passes ``torch.unique`` ids; a repeated id is evaluated as the reference expression does, as duplicate rows and
    columns of the logits, and its table row gets the sum of the gradients of its copies."""
    return _SslLoss.apply(embeds1, embeds2, nodes, temp, 0, 1)


def unique_padded(idx: torch.Tensor) -> torch.Tensor:
    """``torch.unique(idx)`` at a FIXED size: the ids sorted ascending with every repeat replaced by -1 (an inactive slot of
    ``contrastLoss``).  No host synchronisation and no data-dependent shape, so a training step that uses it can be captured
    in a CUDA graph; the active entries stand in ``torch.unique``'s order."""
    s = torch.sort(idx.reshape(-1)).values
    first = torch.ones_like(s, dtype=torch.bool)
    first[1:] = s[1:] != s[:-1]
    return torch.where(first, s, torch.full_like(s, -1))


def contrastLoss_padded(embeds1, embeds2, batch_idx, temp):
    """``contrastLoss(embeds1, embeds2, torch.unique(batch_idx), temp)`` (the call of HCCF.calcLosses, model/graph/HCCF.py:62-66)
    without the variable-length ``unique``: same loss and gradients to rounding."""
    return _SslLoss.apply(embeds1, embeds2, unique_padded(batch_idx), temp, 0, 1)


def InfoNCE(view1, view2, temperature, b_cos=True):
    """util/loss_torch.py:32-40."""
    return _SslLoss.apply(view1, view2, None, temperature, 1, 1 if b_cos else 0)
