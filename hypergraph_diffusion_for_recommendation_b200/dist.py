"""Row-partitioned propagation across the GPUs of one NVSwitch box (SURVEY.md section 8e).

The reference is single-process (SURVEY.md F2); this module is the scaling axis the north star adds:

* **Partition.**  Users and items are each cut into ``world`` contiguous ranges; rank ``r`` owns user range
  ``r`` and item range ``r``: their CSR rows, embedding rows and optimiser state.  Owned rows are laid out
  ``[own users | own items | padding]`` (``n_loc`` rows, equal on every rank), so the gathered table is the
  concatenation of the ranks' blocks: node ``v`` sits at ``perm(v) = owner(v) * n_loc + offset(v)``.
* **Local matrix.**  ``A_loc = A[own rows, :]`` with columns renumbered by ``perm`` but kept in their
  ORIGINAL ascending order inside a row, so each output row is accumulated in exactly the order of the
  single-GPU kernel: the sharded result is bit-identical to the unsharded one.
* **Exchange.**  Every propagation needs the gathered table of the previous one.  Fused form (default on CUDA): the
  propagation kernel's epilogue stores each finished row into the gathered table of EVERY rank -- symmetric-memory
  buffers mapped over NVLink (``hgr_epilogue_t::gather_out``) -- so the all-gather rides on the kernel that produces
  the rows and overlaps its remaining work; a device-side barrier orders the readers.  Rows that do not come out of a
  propagation kernel (parameters, outputs of dense layers) use one NCCL ``all_gather``.  Then the same
  ``hgr_spmm_f32`` kernel on ``A_loc``.  The normalised adjacency is symmetric, so the backward pass is
  ``dX_own = A_loc . all_gather(dY_own)``: a gather, never a reduction.
* **Loss.**  The final tables are gathered once; every rank evaluates the fused BPR + L2 kernel on the triples whose USER
  it owns, the four batch sums cross the ranks in one 32-byte ``all_reduce`` (identical losses on all ranks), and the backward
  writes the rank's own gradient rows from every triple that touches them.  Gradients of the small
  replicated parameters (LayerNorm, Linear) are summed with one ``all_reduce``.
* **Evaluation** shards the test users: each rank ranks its own users against the gathered item table.

The kernel set is a constructor argument so the host logic (partition maps, gathers, autograd wiring) is
exercised by the world_size-2 ``gloo`` CPU tests with an injected CPU matrix product; the product default is
libhgr.so and nothing else.
"""
from __future__ import annotations

import types
from dataclasses import dataclass

import torch
import torch.distributed as dist


@dataclass
class Partition:
    """Ownership maps of the 1-D row partition: rank ``r`` owns users ``[user_bounds[r], user_bounds[r + 1])`` and items
    ``[item_bounds[r], item_bounds[r + 1])``.  Without bounds the ranges hold equal COUNTS (``ceil(n / world)`` each);
    ``Partition.balanced`` cuts them so that every rank's rows hold about the same number of nonzeros -- the propagation
    kernel's time follows the nonzeros, and a step ends when the slowest rank does.  ``up`` / ``ip`` are the LARGEST range
    sizes: every rank lays its rows out as ``[own users, padded to up | own items, padded to ip]``."""
    n_users: int
    n_items: int
    world: int
    user_bounds: tuple | None = None
    item_bounds: tuple | None = None

    def __post_init__(self):
        def check(bounds, n, what):
            b = tuple(int(v) for v in bounds)
            if len(b) != self.world + 1 or b[0] != 0 or b[-1] != n or any(x > y for x, y in zip(b, b[1:])):
                raise ValueError("%s bounds must be %d ascending ids from 0 to %d" % (what, self.world + 1, n))
            return b

        self.uniform = self.user_bounds is None and self.item_bounds is None
        if self.user_bounds is None:
            up = -(-self.n_users // self.world)
            self.user_bounds = tuple(min(r * up, self.n_users) for r in range(self.world + 1))
        if self.item_bounds is None:
            ip = -(-self.n_items // self.world)
            self.item_bounds = tuple(min(r * ip, self.n_items) for r in range(self.world + 1))
        self.user_bounds = check(self.user_bounds, self.n_users, "user")
        self.item_bounds = check(self.item_bounds, self.n_items, "item")
        if self.uniform:  # (the last ranks of a uniform partition may own fewer rows, or none: the stride stays ceil(n / world))
            self.up = -(-self.n_users // self.world)
            self.ip = -(-self.n_items // self.world)
        else:
            self.up = max(b - a for a, b in zip(self.user_bounds, self.user_bounds[1:]))
            self.ip = max(b - a for a, b in zip(self.item_bounds, self.item_bounds[1:]))
        self.n_loc = -(-(self.up + self.ip) // 4) * 4  # rows per rank, padded
        self.n_glob = self.n_loc * self.world
        self._cuts = {}

    @classmethod
    def balanced(cls, n_users: int, n_items: int, world: int, deg_u: torch.Tensor, deg_i: torch.Tensor) -> "Partition":
        """Ranges with (nearly) equal nonzeros: range r of the users ends where the running sum of the user degrees passes
        ``r / world`` of their total, the same for the items.  A rank's block then holds ~1/world of the user-row nonzeros
        plus ~1/world of the item-row nonzeros whatever the degree distribution (a single item with 1 % of all interactions
        shifts a count-based cut by 6 % at 8 ranks: 245 M vs 260 M nonzeros on the 10 M x 2 M x 1 B graph)."""
        def cuts(deg, n):
            if world == 1 or n == 0:
                return (0,) + (n,) * world
            cum = torch.cumsum(deg.to(torch.int64), 0)
            total = int(cum[-1])
            targets = torch.tensor([(total * r) // world for r in range(1, world)], dtype=torch.int64, device=cum.device)
            b = (torch.searchsorted(cum, targets, right=False) + 1).clamp(max=n).tolist() if total > 0 else [
                min(r * -(-n // world), n) for r in range(1, world)]
            out = [0]
            for v in b:
                out.append(max(int(v), out[-1]))
            return tuple(out + [n])

        return cls(n_users, n_items, world, cuts(deg_u, n_users), cuts(deg_i, n_items))

    def users_of(self, rank):
        return self.user_bounds[rank], self.user_bounds[rank + 1]

    def items_of(self, rank):
        return self.item_bounds[rank], self.item_bounds[rank + 1]

    def _owner(self, ids: torch.Tensor, bounds: tuple, what: str):
        key = (what, ids.device)
        t = self._cuts.get(key)
        if t is None:
            t = self._cuts[key] = torch.tensor(bounds, dtype=torch.int64, device=ids.device)
        r = torch.bucketize(ids, t[1:-1], right=True)
        return r, t[r]

    def perm_user(self, u: torch.Tensor) -> torch.Tensor:
        u = u.to(torch.int64)
        if self.uniform:
            return torch.div(u, self.up, rounding_mode="floor") * self.n_loc + u % self.up
        r, lo = self._owner(u, self.user_bounds, "u")
        return r * self.n_loc + (u - lo)

    def perm_item(self, i: torch.Tensor) -> torch.Tensor:
        i = i.to(torch.int64)
        if self.uniform:
            return torch.div(i, self.ip, rounding_mode="floor") * self.n_loc + self.up + i % self.ip
        r, lo = self._owner(i, self.item_bounds, "i")
        return r * self.n_loc + self.up + (i - lo)


def local_block(part: Partition, rank: int, u: torch.Tensor, i: torch.Tensor, use_builder: bool | None = None):
    """``A[own rows, :]`` of the normalised bipartite adjacency of the interaction list ``(u, i)``, as
    ``(indptr int64 [n_loc + 1], indices int32, values float32)`` with permuted column ids.  The permutation is monotonic inside
    the user range and inside the item range, so ascending permuted ids ARE the original ascending order of a row: every output
    row is accumulated in the single-GPU order.  Values are ``(d[row] * m) * d[col]`` with ``d = np.power(deg, -0.5)`` from the
    host's table and ``m`` the multiplicity of a repeated pair: bit-identical to ``Interaction.norm_adj``.

    On CUDA the block comes out of the product builder (csrc/graph_build.cu: radix sort of THIS RANK's entries only -- the
    interactions whose user or item it owns -- duplicates summed, LUT degree scale); the torch sort / bincount form below is the
    host-logic path of the gloo CPU tests."""
    dev = u.device
    if use_builder is None:
        use_builder = dev.type == "cuda"
    u = u.to(torch.int64)
    i = i.to(torch.int64)
    # degrees count every listed interaction (duplicates included), like the row sums the reference normalises by; in a job
    # whose ranks hold disjoint slices of the list this is the one all_reduce of the build
    deg_u = torch.bincount(u, minlength=part.n_users)
    deg_i = torch.bincount(i, minlength=part.n_items)
    from .graph import host_pow_lut

    max_deg = int(max(deg_u.max().item() if deg_u.numel() else 0, deg_i.max().item() if deg_i.numel() else 0))
    lut = torch.from_numpy(host_pow_lut(max_deg + 1, -0.5)).to(dev)
    du, di = lut[deg_u], lut[deg_i]
    u0, u1 = part.users_of(rank)
    i0, i1 = part.items_of(rank)
    if use_builder:
        from . import graph

        mu = (u >= u0) & (u < u1)
        mi = (i >= i0) & (i < i1)
        rows = torch.cat([u[mu] - u0, part.up + (i[mi] - i0)]).to(torch.int32)
        cols = torch.cat([part.perm_item(i[mu]), part.perm_user(u[mi])]).to(torch.int32)
        del mu, mi
        indptr, indices, values, _ = graph._build("coo", rows, cols, part.n_loc, part.n_glob)
        del rows, cols
        d_rows = torch.zeros(part.n_loc, dtype=torch.float32, device=dev)
        d_rows[:u1 - u0] = du[u0:u1]
        d_rows[part.up:part.up + (i1 - i0)] = di[i0:i1]
        d_cols = torch.zeros(part.n_glob, dtype=torch.float32, device=dev)
        d_cols[part.perm_user(torch.arange(part.n_users, device=dev))] = du
        d_cols[part.perm_item(torch.arange(part.n_items, device=dev))] = di
        graph._scale(indptr, indices, values, part.n_loc, d_rows, d_cols)
        return indptr, indices, values
    # host-logic path (unique pairs): user rows: columns are items, ascending item id
    m = (u >= u0) & (u < u1)
    key = torch.sort((u[m] - u0) * part.n_items + i[m]).values
    ru, ci = torch.div(key, part.n_items, rounding_mode="floor"), key % part.n_items
    # item rows: columns are users, ascending user id
    m = (i >= i0) & (i < i1)
    key = torch.sort((i[m] - i0) * part.n_users + u[m]).values
    ri, cu = torch.div(key, part.n_users, rounding_mode="floor"), key % part.n_users
    del key, m
    counts = torch.zeros(part.n_loc, dtype=torch.int64, device=dev)
    counts[:u1 - u0] = deg_u[u0:u1]
    counts[part.up:part.up + (i1 - i0)] = deg_i[i0:i1]
    indptr = torch.zeros(part.n_loc + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=indptr[1:])
    indices = torch.cat([part.perm_item(ci), part.perm_user(cu)]).to(torch.int32)
    values = torch.cat([du[ru + u0] * di[ci], di[ri + i0] * du[cu]])
    return indptr, indices, values


class LibhgrKernels:
    """The product kernels (libhgr.so).  The gloo CPU tests pass an object with the same three methods built on
    a CPU matrix product to exercise the partition / gather / autograd logic without a GPU."""

    @staticmethod
    def make_block(indptr, indices, values, shape):
        from .graph import DeviceCSR

        return DeviceCSR(indptr, indices, values, shape)  # rows are long-tailed like the global matrix: split plan kept

    @staticmethod
    def spmm(block, x, ep=None, no_local_out=False):
        """``epilogue(block @ x)``; ``ep`` is a dict of ``ops.make_epilogue`` keyword arguments."""
        from . import ops

        return ops.spmm_raw(block, x, ops.make_epilogue(**ep) if ep else None, no_local_out=no_local_out)

    @staticmethod
    def leaky_ln_bwd(pre, dy, gamma, eps, slope, gather_ptrs=(), gather_row_offset=0, gather_mc=0):
        from . import ops

        return ops.leaky_ln_bwd(pre, dy, gamma, eps, slope, gather_ptrs, gather_row_offset, gather_mc)

    @staticmethod
    def publish_rows(x, gather_ptrs, gather_row_offset, gather_mc=0):
        from . import ops

        ops.publish_rows(x, gather_ptrs, gather_row_offset, gather_mc)


class SymmetricPool:
    """Ring of gathered ``[world * n_loc, D]`` tables in symmetric memory: every rank allocates the same buffers,
    ``rendezvous`` maps the peers' copies into this process (NVLink peer access), and the propagation kernel's
    epilogue stores each finished row straight into all of them (``hgr_epilogue_t::gather_out``).  ``barrier``
    is the device-side cross-rank barrier that orders the peers' reads after those stores."""

    def __init__(self, n_glob: int, d: int, device, group, n_buffers: int = 4):
        import torch.distributed._symmetric_memory as symm_mem

        import os

        self.bufs, self.hdls, self.ptrs, self.mc = [], [], [], []
        use_mc = os.environ.get("HGR_MULTICAST", "1") != "0"
        for _ in range(n_buffers):
            t = symm_mem.empty((n_glob, d), dtype=torch.float32, device=device)
            h = symm_mem.rendezvous(t, group=group if group is not None else dist.group.WORLD)
            self.bufs.append(t)
            self.hdls.append(h)
            self.ptrs.append([int(p) for p in h.buffer_ptrs])
            # NVSwitch multicast address of the slot (0 when the fabric / driver has no NVLS): one multimem.st per 16 bytes
            # reaches every rank's copy, the unicast pointers stay as the fallback
            self.mc.append(int(getattr(h, "multicast_ptr", 0) or 0) if use_mc else 0)
        self.multicast = all(m != 0 for m in self.mc) and len(self.mc) > 0
        self.next = 0
        self.wait_events = None

    def take(self, reading: torch.Tensor | None = None) -> int:
        """Next slot of the ring; never the slot the kernel about to run READS (``reading``: its gathered input) -- peers would be
        storing into it meanwhile.  Every rank makes the same calls in the same order, so all ranks skip the same slot."""
        for _ in range(len(self.bufs)):
            k = self.next
            self.next = (k + 1) % len(self.bufs)
            if reading is None or self.bufs[k].data_ptr() != reading.data_ptr():
                return k
        raise RuntimeError("symmetric pool: no free slot")

    def barrier(self, k: int) -> None:
        ev = self.wait_events
        if ev is not None:  # bench: how long this rank sits in the cross-rank barriers of a step
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.hdls[k].barrier(channel=0)
            e1.record()
            ev.append((e0, e1))
        else:
            self.hdls[k].barrier(channel=0)


class _AllGatherRows(torch.autograd.Function):
    """``[n_loc, D]`` owned rows -> ``[world * n_loc, D]``.  ``grad_mode``: ``'slice'`` when every rank holds the
    same full gradient (replicated loss), ``'reduce'`` for a reduce-scatter of per-rank partial gradients."""

    @staticmethod
    def forward(ctx, x, g, grad_mode):
        ctx.g, ctx.grad_mode = g, grad_mode
        return g.all_gather(x)

    @staticmethod
    def backward(ctx, grad):
        g = ctx.g
        if ctx.grad_mode == "slice":
            return grad[g.rank * g.part.n_loc:(g.rank + 1) * g.part.n_loc].contiguous(), None, None
        out = torch.empty((g.part.n_loc, grad.shape[1]), dtype=grad.dtype, device=grad.device)
        dist.reduce_scatter_tensor(out, grad.contiguous(), group=g.group)
        return out, None, None


class _DistSpmm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, g):
        ctx.g = g
        return g.k.spmm(g.block, g.gathered(x.contiguous()))

    @staticmethod
    def backward(ctx, dy):
        g = ctx.g  # A symmetric: dX_own = (A^T dY)[own] = A[own, :] dY
        return g.k.spmm(g.block, g.gathered(dy.contiguous())), None


class DistGraph:
    """The rank's block of the adjacency + the communicator.  Quacks like the ``DeviceCSR`` the encoders hold
    (``shape``, ``_nnz``, ``t``) and routes ``ops.spmm / hgconv / lightgcn_propagate`` to the sharded forms."""

    def __init__(self, part: Partition, rank: int, indptr, indices, values, group=None, kernels=None):
        self.part, self.rank, self.world, self.group = part, rank, part.world, group
        self.k = kernels or LibhgrKernels
        self.block = self.k.make_block(indptr, indices, values, (part.n_loc, part.n_glob))
        self.shape = (part.n_glob, part.n_glob)
        self.symmetric = True
        self.device = indptr.device
        self._nnz_local = int(indices.numel())
        self.gather_events = None  # bench: list of (start, end) CUDA events around every all_gather
        # fused all-gather (propagation epilogue stores into every rank's gathered table): CUDA + libhgr only
        import os

        self.fused = (self.k is LibhgrKernels and self.world > 1 and indptr.is_cuda and self.world <= 8
                      and os.environ.get("HGR_FUSED_GATHER", "1") != "0")
        # a block whose kernel publishes its rows to many ranks spreads the whole rows through the work list, so the exchange
        # leaves at a steady rate instead of in the first windows (graph._spread_schedule)
        if self.fused and part.n_glob * 256 >= (1 << 30) and hasattr(self.block, "set_schedule"):
            self.block.set_schedule("spread")
        self._pools = {}     # D -> SymmetricPool
        self._published = {}  # pool slot -> (tensor kept alive, version): local rows whose gathered copy sits in that slot
        self.publish_copy = os.environ.get("HGR_PUBLISH_COPY", "1") != "0"
        self.n_fused, self.n_collective, self.n_published = 0, 0, 0
        self.copy_events = []

    def _nnz(self):
        return self._nnz_local

    def t(self):
        return self

    def to(self, *a, **k):
        return self

    cuda = to

    # ---- fused all-gather ---------------------------------------------------------------------
    def pool(self, d: int):
        p = self._pools.get(d)
        if p is None and self.fused:
            try:
                p = SymmetricPool(self.part.n_glob, d, self.device, self.group)
            except Exception as e:  # no peer access / symmetric memory on this box: keep the NCCL exchange
                import warnings

                warnings.warn("symmetric memory unavailable (%s): sharded propagation falls back to NCCL all_gather" % (e,))
                self.fused = False
                return None
            self._pools[d] = p
        return p

    def spmm_published(self, full_in: torch.Tensor, ep: dict | None = None, want_local: bool = True):
        """``y_own = epilogue(A_loc @ full_in)`` whose rows are stored, by the kernel's own epilogue, into slot ``k`` of
        the symmetric pool on EVERY rank (fused all-gather).  Returns ``(gathered [n_glob, D], y_own or None)``."""
        pool = self.pool(full_in.shape[1])
        k = pool.take(reading=full_in)
        self._published.pop(k, None)  # the slot is being rewritten: forget what it held
        self.multicast = pool.multicast
        ep = dict(ep or {}, gather_ptrs=pool.ptrs[k], gather_row_offset=self.rank * self.part.n_loc,
                  gather_mc=pool.mc[k] if pool.multicast else 0)
        y = self.k.spmm(self.block, full_in, ep, no_local_out=not want_local)
        pool.barrier(k)  # every rank's rows have landed here, and every rank is done reading the slot's old contents
        if y is not None:
            self._published[k] = (y, y._version)
        self.n_fused += 1
        return pool.bufs[k], y

    def leaky_ln_bwd_published(self, pre, dy, gamma, eps, slope):
        """LayerNorm / LeakyReLU backward whose ``dz`` rows land in every rank's gathered table as they are computed (the
        sharded backward propagation that follows needs exactly that table).  Returns ``(dz, dgamma, dbeta, gathered dz)``."""
        pool = self.pool(dy.shape[1])
        k = pool.take()
        self._published.pop(k, None)
        dz, dgamma, dbeta = self.k.leaky_ln_bwd(pre, dy, gamma, eps, slope, pool.ptrs[k], self.rank * self.part.n_loc,
                                                pool.mc[k] if pool.multicast else 0)
        pool.barrier(k)
        self._published[k] = (dz, dz._version)
        self.n_fused += 1
        return dz, dgamma, dbeta, pool.bufs[k]

    def publish_by(self, d: int, produce):
        """Let a row-wise kernel that is NOT a propagation carry the exchange: ``produce(gather)`` runs it with
        ``gather = (peer pointers, row offset, multicast pointer)`` of a free pool slot and returns its ``[n_loc, d]`` output, whose
        gathered copy is then registered like a propagation's (``ops.linear(publish=...)``, ``ops.add_rows(publish=...)``)."""
        pool = self.pool(d)
        if pool is None:
            return produce(None)
        k = pool.take()
        self._published.pop(k, None)
        y = produce((pool.ptrs[k], self.rank * self.part.n_loc, pool.mc[k] if pool.multicast else 0))
        pool.barrier(k)
        self._published[k] = (y, y._version)
        self.n_fused += 1
        return y

    def publish(self, x: torch.Tensor) -> torch.Tensor:
        """Rows that do not come out of a libhgr kernel (dense layers, elementwise ops): one copy kernel stores them into
        every rank's table over NVLink (757 GB/s measured at 2 ranks against 428 GB/s for the NCCL all_gather)."""
        pool = self.pool(x.shape[1])
        k = pool.take()
        self._published.pop(k, None)
        if pool.wait_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.k.publish_rows(x, pool.ptrs[k], self.rank * self.part.n_loc, pool.mc[k] if pool.multicast else 0)
            e1.record()
            self.copy_events.append((e0, e1))
        else:
            self.k.publish_rows(x, pool.ptrs[k], self.rank * self.part.n_loc, pool.mc[k] if pool.multicast else 0)
        pool.barrier(k)
        self._published[k] = (x, x._version)
        self.n_published += 1
        return pool.bufs[k]

    def gathered(self, x: torch.Tensor) -> torch.Tensor:
        """Gathered table of the owned rows ``x``: the pool slot a previous kernel already filled, else a peer-store copy
        (``HGR_PUBLISH_COPY=0``: an NCCL collective)."""
        if self.fused:
            pool = self._pools.get(x.shape[1])
            for k, (t, ver) in self._published.items():
                # same storage AND unmodified since it was published (an optimizer step on a parameter bumps _version)
                if t.data_ptr() == x.data_ptr() and t.shape == x.shape and t._version == ver == x._version:
                    return pool.bufs[k]
            if self.publish_copy and x.dim() == 2 and x.shape[0] == self.part.n_loc and x.dtype == torch.float32 \
                    and x.shape[1] % 4 == 0 and self.pool(x.shape[1]) is not None:
                return self.publish(x.contiguous())
        return self.all_gather(x)

    def all_gather(self, x: torch.Tensor) -> torch.Tensor:
        self.n_collective += 1
        x = x.contiguous()
        out = torch.empty((self.world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
        if self.gather_events is not None and x.is_cuda:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dist.all_gather_into_tensor(out, x, group=self.group)
            e1.record()
            self.gather_events.append((e0, e1))
        else:
            dist.all_gather_into_tensor(out, x, group=self.group)
        return out

    # ---- sharded operators (same signatures as ops.*) ------------------------------------------
    def spmm(self, x):
        return _DistSpmm.apply(x, self)

    def lightgcn_propagate(self, ego, n_layers, sum_readout=False):
        """``mean_k A^k E`` on owned rows: one gather + one local propagation per layer; the last layer's
        readout (sum of the layer tables, scale) is fused into its kernel epilogue as in the local form."""
        return _DistLightGCN.apply(ego, self, n_layers, sum_readout)

    def hgconv(self, x, slope=None, ln_weight=None, ln_bias=None, residual=None, eps=1e-5):
        return _DistHGConv.apply(x, ln_weight, ln_bias, residual, self, slope, eps)

    def gather_tables(self, own: torch.Tensor, grad_mode="slice") -> torch.Tensor:
        return _AllGatherRows.apply(own, self, grad_mode)


def _lightgcn_rows(g: DistGraph, e0, n_layers, sum_readout, publish_last=False):
    if n_layers == 0:
        return e0.clone()
    layers = [e0]
    cur = e0
    full = g.gathered(e0)
    for k in range(n_layers):
        if k + 1 < n_layers:
            if g.fused and g.pool(e0.shape[1]) is not None:
                full, cur = g.spmm_published(full, None, want_local=True)  # next layer's input arrives with this kernel
            else:
                cur = g.k.spmm(g.block, full)
                full = g.all_gather(cur)
            layers.append(cur)
        else:
            ep = dict(addends=layers, scale=1.0 if sum_readout else 1.0 / (n_layers + 1))
            if publish_last and g.fused and g.pool(e0.shape[1]) is not None:
                _, cur = g.spmm_published(full, ep, want_local=True)  # the loss (or the evaluation) gathers these rows next
            else:
                cur = g.k.spmm(g.block, full, ep)
    return cur


class _DistLightGCN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, e0, g, n_layers, sum_readout):
        ctx.g, ctx.n_layers, ctx.sum_readout = g, n_layers, sum_readout
        return _lightgcn_rows(g, e0.contiguous(), n_layers, sum_readout, publish_last=True)

    @staticmethod
    def backward(ctx, dout):
        # out = c sum_k A^k e0 and A symmetric: the same sharded recurrence applied to dout
        return _lightgcn_rows(ctx.g, dout.contiguous(), ctx.n_layers, ctx.sum_readout), None, None, None


class _DistHGConv(torch.autograd.Function):
    """Sharded ``[LN](leaky(A (A x))) [+ residual]``: two gathers + two local propagations; activation,
    LayerNorm and residual stay fused in the second kernel's epilogue (they are row-local)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, residual, g, slope, eps):
        need_pre = (slope is not None or gamma is not None) and any(ctx.needs_input_grad[:3])
        x = x.contiguous()
        pre = torch.empty_like(x) if need_pre else None
        gm = gamma.contiguous() if gamma is not None else None
        bt = beta.contiguous() if beta is not None else None
        rs = residual.contiguous() if residual is not None else None
        ep = dict(slope=slope, gamma=gm, beta=bt, eps=eps, residual=rs, pre=pre)
        if g.fused and g.pool(x.shape[1]) is not None:
            # node -> hyperedge stage publishes its rows into every rank's table; the node stage publishes y too,
            # for the propagation that consumes it next (EquivSetConv chains two of these)
            full_t, _ = g.spmm_published(g.gathered(x), None, want_local=False)
            _, y = g.spmm_published(full_t, ep, want_local=True)
        else:
            t = g.k.spmm(g.block, g.all_gather(x))
            y = g.k.spmm(g.block, g.all_gather(t), ep)
        ctx.g, ctx.slope, ctx.eps = g, slope, eps
        ctx.has_ln, ctx.has_res = gamma is not None, residual is not None
        ctx.save_for_backward(pre, gm)
        return y

    @staticmethod
    def backward(ctx, dy):
        pre, gamma = ctx.saved_tensors
        g = ctx.g
        dy = dy.contiguous()
        dgamma = dbeta = None
        fused = g.fused and g.pool(dy.shape[1]) is not None
        full_dz = None
        if pre is not None:
            if fused and ctx.needs_input_grad[0]:
                dz, dgamma, dbeta, full_dz = g.leaky_ln_bwd_published(pre, dy, gamma if ctx.has_ln else None, ctx.eps, ctx.slope)
            else:
                dz, dgamma, dbeta = g.k.leaky_ln_bwd(pre, dy, gamma if ctx.has_ln else None, ctx.eps, ctx.slope)
        else:
            dz = dy
        dx = None
        if ctx.needs_input_grad[0]:
            if fused:
                full_t, _ = g.spmm_published(full_dz if full_dz is not None else g.gathered(dz), None, want_local=False)
                dx = g.k.spmm(g.block, full_t)
            else:
                t = g.k.spmm(g.block, g.all_gather(dz))
                dx = g.k.spmm(g.block, g.all_gather(t))
        return dx, dgamma, dbeta, (dy if ctx.has_res else None), None, None, None


# ------------------------------------------------------------------------------------------------
# construction + training step
# ------------------------------------------------------------------------------------------------
def build_partitioned(u, i, n_users, n_items, rank, world, device=None, group=None, kernels=None, balanced=None):
    """Every rank holds the same interaction list (synthetic generator, same seed) and keeps its own rows; the ranges are cut
    by nonzeros (``Partition.balanced``; ``balanced=False`` or ``HGR_BALANCED_PARTITION=0``: by count).
    Returns a namespace with ``adj`` (DistGraph), ``data`` (what the encoders read: local ``n_users`` /
    ``n_items`` and the adjacency handle) and ``part``."""
    if balanced is None:
        import os

        balanced = os.environ.get("HGR_BALANCED_PARTITION", "1") != "0"
    if balanced and world > 1:
        # every rank computes the same cuts from the same degree tables (in a job whose ranks hold slices of the list, the
        # degree tables are the one all_reduce of the build)
        part = Partition.balanced(n_users, n_items, world, torch.bincount(u.to(torch.int64), minlength=n_users),
                                  torch.bincount(i.to(torch.int64), minlength=n_items))
    else:
        part = Partition(n_users, n_items, world)
    indptr, indices, values = local_block(part, rank, u, i)
    adj = DistGraph(part, rank, indptr, indices, values, group=group, kernels=kernels)
    data = types.SimpleNamespace(n_users=part.up, n_items=part.n_loc - part.up, norm_adj=None, norm_adj_device=adj)
    return types.SimpleNamespace(adj=adj, data=data, part=part)


def sync_replicated_grads(model, owned_names=("embedding_dict.user_emb", "embedding_dict.item_emb"), group=None):
    """Sum the gradients of the parameters every rank holds a copy of (LayerNorm, Linear); the embedding rows
    are owned, not replicated.  One flat all_reduce."""
    grads = [p.grad for n, p in model.named_parameters() if p.grad is not None and not n.endswith(owned_names)]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, group=group)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


def _unsplit(out_u: torch.Tensor, out_i: torch.Tensor) -> torch.Tensor:
    """The encoders return ``(rows[:n_users], rows[n_users:])``: when both are views covering one table, use that table
    itself (so a gathered copy published by the kernel that produced it can be found) instead of concatenating them."""
    base = out_u._base
    if (base is not None and base is out_i._base and base.dim() == 2 and base.is_contiguous() and out_u.data_ptr() == base.data_ptr()
            and out_u.shape[0] + out_i.shape[0] == base.shape[0] and out_u.shape[1] == base.shape[1]
            and out_i.data_ptr() == base.data_ptr() + out_u.numel() * base.element_size()):
        return base
    return torch.cat([out_u, out_i], 0)


def train_step(model, optimizer, g: DistGraph, user_idx, pos_idx, neg_idx, reg: float, batch_size: int, loss_fn=None):
    """One sharded step of the reference's training loop (model/graph/LightGCN.py:49-66): propagate the owned
    rows, gather the final tables, fused BPR + L2 on the whole batch, backward, summed replicated gradients,
    optimiser step on the owned rows.  ``user_idx / pos_idx / neg_idx`` are GLOBAL dense ids."""
    marks = []

    def mark(name):  # bench: CUDA events between the phases of the step (g.phase_events = [] switches it on)
        if getattr(g, "phase_events", None) is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))

    mark("start")
    out_u, out_i = model()[:2]
    mark("encoder forward")
    own = _unsplit(out_u, out_i)
    part = g.part
    pu, pp, pn = part.perm_user(user_idx), part.perm_item(pos_idx), part.perm_item(neg_idx)
    if loss_fn is None:
        # product path: the gathered table comes from the last propagation's epilogue when it published it; the backward
        # produces only this rank's gradient rows
        from .loss_torch import bpr_l2_sharded

        import os

        reduce_sums = None
        if g.world > 1 and os.environ.get("HGR_OWNER_SHARDED_LOSS", "1") != "0":
            def reduce_sums(t):  # the loss's only exchange: 4 doubles
                dist.all_reduce(t, group=g.group)
        rec_loss, reg_loss = bpr_l2_sharded(own, g.gathered, g.rank * part.n_loc, pu, pp, pn, reg, batch_size, reduce_sums)
    else:
        full = g.gather_tables(own)
        rec_loss, reg_loss = loss_fn(full, full, pu, pp, pn, reg, batch_size)
    mark("loss forward")
    optimizer.zero_grad(set_to_none=True)
    (rec_loss + reg_loss).backward()
    mark("backward")
    if g.world > 1:
        sync_replicated_grads(model, group=g.group)
    mark("replicated-gradient all_reduce")
    optimizer.step()
    mark("optimizer")
    if marks:
        g.phase_events.append(marks)
    return torch.stack([rec_loss.detach(), reg_loss.detach()])


def fullrank_topk_sharded(g: DistGraph, out_u: torch.Tensor, out_i: torch.Tensor, test_users_local: torch.Tensor,
                          train_indptr_own: torch.Tensor, train_indices_own: torch.Tensor, n_items: int, k: int,
                          mode: str = "exact", engine: str = "auto", return_stats: bool = False):
    """Full-ranking evaluation sharded by user (SURVEY.md 8e): every rank ranks ITS users (``test_users_local`` index the
    rank's own user rows ``out_u``; ``train_indptr_own / train_indices_own`` is the training matrix of those rows with GLOBAL
    item ids) against the whole item table, which is assembled once from the gathered rows.  Returns this rank's
    ``(ids, scores[, stats])`` with global item ids; recommendation lists never cross ranks (metric sums do, as scalars).
    ``k`` and ``mode`` have the range of ``evaluation.fullrank_topk`` (up to 256 in both modes)."""
    from . import evaluation

    with torch.no_grad():
        full = g.gathered(_unsplit(out_u, out_i))
        item_tab = full[g.part.perm_item(torch.arange(n_items, device=full.device))].contiguous()  # rows back in item-id order
        u_tab = out_u[:train_indptr_own.numel() - 1].contiguous()  # the training matrix may cover a prefix of the owned users
        return evaluation.fullrank_topk(u_tab, item_tab, test_users_local, train_indptr_own, train_indices_own, k, mode=mode,
                                        engine=engine, return_stats=return_stats)
