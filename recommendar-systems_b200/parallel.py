"""Multi-GPU paths that shard naturally (SURVEY.md section 8e). One process per GPU,
torch.distributed (NCCL over NVLink/NVSwitch on the B200 box, gloo in the CPU tests).

* Propagation: nodes are cut into P contiguous row ranges balanced by non-zeros; rank p owns the
  CSR rows of its range (all columns) and computes those rows of every layer; one all-gather per
  layer rebuilds the full embedding table. Ranges have different lengths, so nodes are renumbered
  into a *padded* layout (`pid = owner * R + local`, R = longest range): every rank writes its
  slice of the next layer in place and `all_gather_into_tensor` needs no packing or compaction;
  the local CSR's column indices are rewritten to padded ids once.
  Backward (training with replicated loss): the same loop on the gradient (A_hat symmetric).
* Bipartite propagation (`ShardedBipartite`, the path bench.py scales): the all-gather above moves
  the WHOLE table every layer (4 N d bytes per rank whatever P is: 3 GB at 10M x 2M, d = 64), so
  it stops scaling at P = 2. A user-item graph only ever needs ITEM vectors to move: rank p owns a
  range of users; per layer it computes its users' rows from the (replicated) item table and, with
  the transpose of the same edge block, the contribution of its users to EVERY item; one
  all-reduce of the [I, d] item table (0.5 GB; NVLS reduces in the switch) finishes the layer and
  overlaps with the user-side SpMM. User vectors never leave their owner, the item table ends up
  replicated -- exactly what the item-sharded evaluation wants -- and the batch's user rows are
  fetched with a [Bu, d] all-reduce.
* Evaluation: items are cut into P equal ranges; every rank runs the fused score + mask + top-K
  kernel on its item slice (global ids via `item_offset`), the [n, K] (score, id) lists are
  all-gathered and merged with `mmrec_topk_merge` (same tie rule: lower id first).
* Evaluation of the user-sharded LightGCN (`ShardedEvalData`, `ShardedLightGCN.eval_metric_sums`):
  after the propagation a rank holds the whole item table, its users' rows, their training edges
  (the mask, `sb.R`) and their held-out edges (the ground truth), so it scores only its own users,
  with the mask rows looked up by user id in `sb.R` (mmrec_score_mask_topk_rows_f32). The only
  collective of a pass besides the propagation is one all-reduce of the [5, K] metric sums.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import graph as G
from . import ops


def partition_by_nnz(row_ptr_host: np.ndarray, world: int) -> np.ndarray:
    """Row boundaries b[0..world] with ~equal (nnz + rows) per part. row_ptr_host: int64 [n+1]."""
    n = len(row_ptr_host) - 1
    cost = row_ptr_host.astype(np.int64) + np.arange(n + 1, dtype=np.int64)   # nnz + one unit per row
    targets = cost[-1] * np.arange(1, world, dtype=np.float64) / world
    cuts = np.searchsorted(cost, targets, side="left")
    b = np.concatenate(([0], cuts, [n])).astype(np.int64)
    return np.maximum.accumulate(b)


class PaddedLayout:
    """Node id <-> padded id for row ranges of unequal length."""

    def __init__(self, bounds: np.ndarray):
        self.bounds = np.asarray(bounds, dtype=np.int64)
        self.world = len(self.bounds) - 1
        self.sizes = np.diff(self.bounds)
        self.R = int(max(1, self.sizes.max()))
        self.n = int(self.bounds[-1])

    def to_padded(self, ids: torch.Tensor) -> torch.Tensor:
        b = torch.as_tensor(self.bounds, device=ids.device)
        owner = torch.searchsorted(b, ids.to(torch.int64), right=True) - 1
        return owner * self.R + (ids.to(torch.int64) - b[owner])

    def pad(self, X: torch.Tensor) -> torch.Tensor:
        """[n, d] -> [world * R, d] (rows of rank p at p*R...)."""
        out = X.new_zeros(self.world * self.R, X.shape[1])
        for p in range(self.world):
            lo, hi = int(self.bounds[p]), int(self.bounds[p + 1])
            out[p * self.R: p * self.R + hi - lo] = X[lo:hi]
        return out

    def unpad(self, Xp: torch.Tensor) -> torch.Tensor:
        parts = [Xp[p * self.R: p * self.R + int(self.sizes[p])] for p in range(self.world)]
        return torch.cat(parts, dim=0)


class ShardedUIGraph:
    """This rank's row slice of a (symmetric) CSRGraph in the padded numbering."""

    def __init__(self, full: G.CSRGraph, rank: int, world: int, bounds=None):
        rp = full.row_ptr.cpu().numpy().astype(np.int64)
        self.layout = PaddedLayout(partition_by_nnz(rp, world) if bounds is None else bounds)
        self.rank, self.world = rank, world
        lo, hi = int(self.layout.bounds[rank]), int(self.layout.bounds[rank + 1])
        self.lo, self.hi = lo, hi
        a, b = int(rp[lo]), int(rp[hi])
        row_ptr = (full.row_ptr[lo: hi + 1] - a).contiguous()
        col = self.layout.to_padded(full.col_idx[a:b]).to(torch.int32).contiguous()
        vals = full.vals[a:b].contiguous()
        self.local = G.CSRGraph(row_ptr, col, vals, hi - lo, self.layout.world * self.layout.R)
        self.local.t = self.local          # A_hat symmetric: the backward uses the same rows

    @property
    def n_local(self):
        return self.hi - self.lo


def _all_gather_rows(buf: torch.Tensor, rank: int, R: int, group=None):
    """In-place all-gather of the [R, d] slices of `buf` ([world * R, d])."""
    dist.all_gather_into_tensor(buf, buf[rank * R: (rank + 1) * R], group=group)


def _local_spmm(sg, x_pad, y_slice, acc_in, acc_out, scale):
    ops.spmm_raw(sg.local, x_pad, Y=y_slice, acc_in=acc_in, acc_out=acc_out, acc_scale=scale)


def _propagate_padded(sg: ShardedUIGraph, x0_pad, n_layers, scale_last, acc0, group=None,
                      local_spmm=_local_spmm):
    """acc <- (acc0 + sum_{l=1..L} A^l x0) * scale_last on the padded layout. acc0 is the local
    [n_local, d] slice to start the running sum from (x0's own rows for the forward mean, the
    gradient for the backward Horner chain... see callers). Returns the full padded result."""
    R, rank, nl = sg.layout.R, sg.rank, sg.n_local
    x = x0_pad
    acc = torch.zeros(R, x0_pad.shape[1], dtype=x0_pad.dtype, device=x0_pad.device)
    for l in range(1, n_layers + 1):
        last = l == n_layers
        nxt = None
        y_slice = None
        if not last:
            nxt = torch.zeros_like(x0_pad)
            y_slice = nxt[rank * R: rank * R + nl]
        local_spmm(sg, x, y_slice, acc0 if l == 1 else acc[:nl], acc[:nl], scale_last if last else 1.0)
        if not last:
            _all_gather_rows(nxt, rank, R, group)
            x = nxt
    out = torch.zeros_like(x0_pad)
    out[rank * R: rank * R + nl] = acc[:nl]
    _all_gather_rows(out, rank, R, group)
    return out


class _ShardedPropagateMean(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X0, sg, n_layers, group, local_spmm):
        ctx.sg, ctx.n_layers, ctx.group, ctx.local_spmm = sg, n_layers, group, local_spmm
        if n_layers == 0:
            return X0.clone()
        x0_pad = sg.layout.pad(X0.contiguous())
        own = x0_pad[sg.rank * sg.layout.R: sg.rank * sg.layout.R + sg.n_local]
        out = _propagate_padded(sg, x0_pad, n_layers, 1.0 / (n_layers + 1), own, group, local_spmm)
        return sg.layout.unpad(out)

    @staticmethod
    def backward(ctx, dOut):
        sg, L = ctx.sg, ctx.n_layers
        if L == 0:
            return dOut, None, None, None, None
        # replicated loss: dOut is identical on every rank. Horner: t <- g + A t, L times.
        g_pad = sg.layout.pad(dOut.contiguous())
        R, rank, nl = sg.layout.R, sg.rank, sg.n_local
        own = g_pad[rank * R: rank * R + nl]
        t = g_pad
        for l in range(L):
            nxt = torch.zeros_like(g_pad)
            ctx.local_spmm(sg, t, None, own, nxt[rank * R: rank * R + nl], 1.0 / (L + 1) if l == L - 1 else 1.0)
            _all_gather_rows(nxt, rank, R, ctx.group)
            t = nxt
        return sg.layout.unpad(t), None, None, None, None


def sharded_propagate_mean(sg: ShardedUIGraph, X0, n_layers, group=None, local_spmm=_local_spmm):
    """mean_{l=0..L} A^l X0 with rows sharded over the process group; every rank passes the full
    X0 [n, d] and gets the full result (SURVEY 8e row 1)."""
    return _ShardedPropagateMean.apply(X0, sg, n_layers, group, local_spmm)


def item_range(n_items: int, rank: int, world: int):
    per = -(-n_items // world)
    lo = min(n_items, rank * per)
    return lo, min(n_items, lo + per)


@torch.no_grad()
def sharded_score_topk(user_emb, users, item_emb_local, item_lo, k, mask_rowptr=None, mask_cols=None,
                       group=None, local_topk=None, merge=None):
    """Item-sharded full-rank top-K: local fused top-K on this rank's item slice, all-gather of the
    (score, id) lists, K-way merge. Every rank returns the same ids int64 [n, k]."""
    world = dist.get_world_size(group)
    if local_topk is None:
        ids, vals = ops.score_mask_topk(user_emb, users, item_emb_local, k, mask_rowptr, mask_cols,
                                        item_offset=item_lo, return_scores=True)
    else:
        ids, vals = local_topk(user_emb, users, item_emb_local, item_lo, k, mask_rowptr, mask_cols)
    n = users.numel()
    all_v = torch.empty(world * n, k, dtype=torch.float32, device=vals.device)
    all_i = torch.empty(world * n, k, dtype=torch.int32, device=vals.device)
    dist.all_gather_into_tensor(all_v, vals.contiguous(), group=group)
    dist.all_gather_into_tensor(all_i, ids.to(torch.int32).contiguous(), group=group)
    all_v, all_i = all_v.view(world, n, k), all_i.view(world, n, k)
    if merge is None:
        return ops.topk_merge(all_v, all_i)[0]
    return merge(all_v, all_i)


# ------------------------------------------------------------------ user-partitioned bipartite
def _spmm_cuda(g, X, Y=None, acc_in=None, acc_out=None, scale=1.0, narrow=False, y16=None):
    ops.spmm_raw(g, X, Y=Y, acc_in=acc_in, acc_out=acc_out, acc_scale=scale, narrow=narrow, y16=y16)


PRECISIONS = ("fp32", "bf16")


def _check_precision(precision):
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {PRECISIONS}, got {precision!r}")


class ShardedBipartite:
    """Rank p's share of a symmetric user-item graph: users [lo, hi) (balanced by non-zeros) with
    R_p = A[lo:hi, U:] (zero-copy view of the full CSR) and R_p^T (items x local users)."""

    def __init__(self, full: G.CSRGraph, rank: int, world: int, bounds=None, csr_from_coo=None):
        U, I = int(full.n_users), int(full.n_items)
        rp = full.row_ptr[:U + 1].cpu().numpy().astype(np.int64)
        self.bounds = partition_by_nnz(rp, world) if bounds is None else np.asarray(bounds, dtype=np.int64)
        self.rank, self.world, self.U, self.I = rank, world, U, I
        lo, hi = int(self.bounds[rank]), int(self.bounds[rank + 1])
        self.lo, self.hi = lo, hi
        self.R = G.CSRGraph(full.row_ptr[lo: hi + 1], full.col_idx, full.vals, hi - lo, I, col_offset=U)
        a, b = int(rp[lo]), int(rp[hi])
        dev = full.vals.device
        counts = (full.row_ptr[lo + 1: hi + 1] - full.row_ptr[lo: hi]).to(torch.int64)
        rows_local = torch.repeat_interleave(torch.arange(hi - lo, device=dev), counts)
        items = full.col_idx[a:b].to(torch.int64) - U
        build = csr_from_coo or G.csr_from_coo
        self.Rt = build(items, rows_local, full.vals[a:b], I, hi - lo, with_transpose=False)
        self.Rt_blocked = None
        self.nnz_local = b - a
        self._rt_chunks = {}

    @classmethod
    def from_local_edges(cls, users, items, bounds, rank, world, n_users, n_items, recipe="f64eps", group=None,
                         csr_from_coo=None, rt_block_users=None):
        """Build rank p's share WITHOUT ever holding the full graph: `users` / `items` are this
        rank's unique training edges (global ids, users in [bounds[rank], bounds[rank + 1])).
        Values follow graph.build_ui_graph's recipe (D^-1/2 A D^-1/2 with the reference's own host
        arithmetic through a degree LUT); the item degrees are the only global quantity and come
        from one all-reduce of the [I] histogram."""
        self = cls.__new__(cls)
        U, I = int(n_users), int(n_items)
        self.bounds = np.asarray(bounds, dtype=np.int64)
        self.rank, self.world, self.U, self.I = rank, world, U, I
        lo, hi = int(self.bounds[rank]), int(self.bounds[rank + 1])
        self.lo, self.hi = lo, hi
        dev = users.device
        rows_local = users.to(torch.int64) - lo
        items = items.to(torch.int64)
        deg_u = torch.bincount(rows_local, minlength=hi - lo)
        deg_i = torch.bincount(items, minlength=I)
        if world > 1:
            dist.all_reduce(deg_i, group=group)
        max_deg = torch.stack([deg_u.max() if deg_u.numel() else deg_i.new_zeros(()), deg_i.max()]).max()
        lut_np, _ = G._degree_lut(recipe, int(max_deg.item()) + 1)
        lut = torch.from_numpy(np.asarray(lut_np, dtype=np.float64)).to(dev)
        vals = (lut[deg_u[rows_local]] * lut[deg_i[items]]).to(torch.float32)
        if recipe != "f64eps":                  # float32 recipes multiply in float32
            vals = lut[deg_u[rows_local]].to(torch.float32) * lut[deg_i[items]].to(torch.float32)
        build = csr_from_coo or G.csr_from_coo
        self.R = build(rows_local, items, vals, hi - lo, I, with_transpose=False)
        self.nnz_local = int(users.numel())
        self._rt_chunks = {}
        self.Rt_blocked = None
        if rt_block_users and hi - lo > rt_block_users:
            # the local user table does not fit L2: R_p^T in user (column) blocks, see
            # graph.ColumnBlockedCSR. `users` must be ascending (edge lists sorted by user are).
            self.Rt = None
            self.Rt_blocked = G.ColumnBlockedCSR.from_col_sorted_coo(items, rows_local, vals, I, hi - lo,
                                                                     int(rt_block_users), build=build)
        else:
            self.Rt = build(items, rows_local, vals, I, hi - lo, with_transpose=False)
        return self

    def rt_chunks(self, n_chunks):
        """R_p^T cut into `n_chunks` item ranges (zero-copy row-pointer views with their own work
        lists): the unit of the chunked all-reduce in bipartite_propagate_mean."""
        n_chunks = max(1, min(int(n_chunks), self.I))
        if n_chunks not in self._rt_chunks:
            per = -(-self.I // n_chunks)
            out = []
            for c in range(n_chunks):
                a, b = min(self.I, c * per), min(self.I, (c + 1) * per)
                if b > a:
                    g = G.CSRGraph(self.Rt.row_ptr[a: b + 1], self.Rt.col_idx, self.Rt.vals, b - a, self.Rt.n_cols,
                                   col_offset=self.Rt.col_offset)
                    out.append((g, a, b))
            self._rt_chunks[n_chunks] = out
        return self._rt_chunks[n_chunks]


@torch.no_grad()
def bipartite_propagate_mean(sb: ShardedBipartite, Xu_local, Xi, n_layers, group=None, spmm_fn=_spmm_cuda,
                             chunks=4, timing=None, reduce_items=False, after_first_exchange=None,
                             precision="fp32"):
    """mean_{l=0..L} A^l X0 for a bipartite graph, users sharded / items replicated.
    Xu_local [hi - lo, d]: this rank's user rows of X0; Xi [I, d]: the item rows (same on every
    rank). Returns (users' rows of this rank, all item rows).
    reduce_items=True: Xi is this rank's PARTIAL of the item rows (the backward, where each rank
    holds the item gradient of its own triples); their sum over the group is the operand. Its
    chunked all-reduce is issued first and waited for like a layer's yi: (a) of layer 1 runs under
    it, (b) of layer 1 waits.
    after_first_exchange: called once, right after layer 1's item-table all-reduce is issued, to
    queue another collective on the group's stream behind the exchanges issued so far (with
    reduce_items: the operand's and layer 1's), so that it runs under (b) of layer 1 and (a) of
    layer 2 instead of delaying the operand's reduction that (b) of layer 1 waits for.

    Per layer l a rank computes (a) what its users add to every item, yi_l = R_p^T xu_{l-1}, and
    (b) its users' rows, yu_l = R_p xi_{l-1}; the only exchange is the all-reduce of yi_l. The item
    table is cut into `chunks` item ranges: the all-reduce of range c is issued (on NCCL's stream)
    as soon as its SpMM is enqueued and runs under the SpMM of range c + 1, under (b) of the same
    layer and -- because (a) of layer l + 1 needs only yu_l, which never leaves the rank -- under
    (a) of the next layer as well: the compute stream waits for the reduced yi_l only right before
    (b) of layer l + 1. With P ranks (a) + (b) is ~2 nnz / P of gather work per layer against one
    4 I d all-reduce, so the exchange hides completely while it is the shorter of the two.
    `timing` (dict of lists of (start, end) CUDA events per phase) is filled when given.

    precision="bf16": the operand every SpMM gathers from is bfloat16 (half the bytes per gathered
    row), everything else stays in the dtype of the inputs. Layer 1 gathers Xu_local / Xi rounded
    once (with reduce_items: the reduced item operand, rounded after its all-reduce); layer l > 1
    gathers layer l - 1's output rounded to nearest even: the user rows by the SpMM that computes
    them (`y16`; no full-precision copy is written), the item rows after their all-reduce, from the
    reduced values (the same on every rank). The running sums add the unrounded layer outputs to
    the unrounded Xu_local / Xi. `spmm_fn` then receives bfloat16 X and, on the user side, y16=
    instead of Y=."""
    _check_precision(precision)
    lowp = precision == "bf16"
    L = n_layers
    multi = sb.world > 1
    if L == 0:
        xi0 = Xi.clone()
        if reduce_items and multi:
            dist.all_reduce(xi0, group=group)
        if after_first_exchange is not None:
            after_first_exchange()
        return Xu_local.clone(), xi0
    scale = 1.0 / (L + 1)
    acc_u, acc_i = Xu_local, Xi.clone()
    xu, xi = Xu_local.contiguous(), Xi.contiguous()
    if lowp:
        xu = xu.to(torch.bfloat16)
        if not reduce_items:                                  # else rounded once reduced, in layer 1
            xi = xi.to(torch.bfloat16)
    d = acc_i.shape[1]
    blocked = getattr(sb, "Rt_blocked", None)
    parts = sb.rt_chunks(chunks) if blocked is None else None

    def mark(name):
        if timing is None:
            return None
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        timing.setdefault(name, []).append(ev)
        ev[0].record()
        return ev

    def done(ev):
        if ev is not None:
            ev[1].record()

    pending = None                                            # (works, yi) of the previous layer
    if reduce_items:
        xi = acc_i                                            # reduced in place; read by (b) of layer 1 only
        works = []
        if multi:
            ranges = [(0, sb.I)] if parts is None else [(a, b) for _, a, b in parts]
            works = [dist.all_reduce(acc_i[a:b], group=group, async_op=True) for a, b in ranges]
        pending = (works, None)
    for l in range(1, L + 1):
        last = l == L
        yi = torch.empty(sb.I, d, dtype=acc_i.dtype, device=acc_i.device)
        works = []
        ev = mark("rt_spmm")
        if blocked is not None:
            # user table larger than L2: one launch per user block (its vectors stay L2-resident), the
            # item table accumulates across blocks and is reduced whole; the exchange still hides
            # under (b) of this layer and (a) of the next
            kw = {"narrow": True} if spmm_fn is _spmm_cuda else {}
            for bi, g in enumerate(blocked.blocks):
                if bi == 0:
                    spmm_fn(g, xu, Y=yi, **kw)
                else:
                    spmm_fn(g, xu, acc_in=yi, acc_out=yi, **kw)
            if multi:
                works.append(dist.all_reduce(yi, group=group, async_op=True))
        else:
            for g, a, b in parts:
                spmm_fn(g, xu, Y=yi[a:b])                     # (a): this rank's users -> item range [a, b)
                if multi:
                    works.append(dist.all_reduce(yi[a:b], group=group, async_op=True))
        done(ev)
        if l == 1 and after_first_exchange is not None:
            after_first_exchange()
        if pending is not None:                               # (b) needs the reduced item table of layer l - 1
            ev = mark("exposed_all_reduce")
            for w in pending[0]:
                w.wait()
            done(ev)
            if pending[1] is not None:
                acc_i.add_(pending[1])
                xi = pending[1]
            if lowp:                                          # round the reduced item rows
                xi = xi.to(torch.bfloat16)
        yu = None if last else torch.empty_like(xu)
        acc_new = torch.empty_like(acc_u if lowp else xu)
        ev = mark("r_spmm")
        if lowp:
            spmm_fn(sb.R, xi, acc_in=acc_u, acc_out=acc_new, scale=scale if last else 1.0, y16=yu)
        else:
            spmm_fn(sb.R, xi, Y=yu, acc_in=acc_u, acc_out=acc_new, scale=scale if last else 1.0)
        done(ev)
        acc_u = acc_new
        pending = (works, yi)
        xu = yu
    ev = mark("exposed_all_reduce")
    for w in pending[0]:
        w.wait()
    done(ev)
    acc_i.add_(pending[1])
    acc_i.mul_(scale)
    return acc_u, acc_i


@torch.no_grad()
def bipartite_score_topk(sb: ShardedBipartite, out_u_local, out_i, users, k, group=None, local_topk=None,
                         merge=None):
    """Full-rank top-K for global user ids `users` on the outputs of bipartite_propagate_mean:
    the batch's user rows come from their owners (one [Bu, d] all-reduce), items are scored in P
    ranges and the lists merged. Every rank returns the same ids."""
    users = users.to(torch.int64)
    ub = torch.zeros(users.numel(), out_u_local.shape[1], dtype=out_u_local.dtype, device=out_u_local.device)
    mine = (users >= sb.lo) & (users < sb.hi)
    ub[mine] = out_u_local[users[mine] - sb.lo]
    dist.all_reduce(ub, group=group)
    lo, hi = item_range(sb.I, sb.rank, sb.world)
    rows = torch.arange(users.numel(), device=users.device)
    return sharded_score_topk(ub, rows, out_i[lo:hi].contiguous(), lo, k, group=group, local_topk=local_topk,
                              merge=merge)


# ------------------------------------------------------------------ training on the user-sharded graph
def _span(timing, name):
    """(start, end) CUDA events of one phase, appended to timing[name]; None when not timing."""
    if timing is None:
        return None
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    timing.setdefault(name, []).append(ev)
    ev[0].record()
    return ev


def _end(ev):
    if ev is not None:
        ev[1].record()


class _BipartitePropagateMean(torch.autograd.Function):
    """bipartite_propagate_mean with a backward. mean_{l=0..L} A^l is symmetric, so the backward
    is the same operator on (dU_local, dI); dI is this rank's partial (the item gradient of the
    triples it owns) and is summed over the group by the operator's first, overlapped, exchange."""

    @staticmethod
    def forward(ctx, Xu_local, Xi, sb, n_layers, group, spmm_fn, chunks, timing, backward_exchange_hook, precision):
        ctx.args = (sb, n_layers, group, spmm_fn, chunks, timing, backward_exchange_hook, precision)
        ev = _span(timing, "forward_propagation")
        out = bipartite_propagate_mean(sb, Xu_local.detach(), Xi.detach(), n_layers, group, spmm_fn, chunks, timing,
                                       precision=precision)
        _end(ev)
        return out

    @staticmethod
    def backward(ctx, dU, dI):
        sb, L, group, spmm_fn, chunks, timing, hook, precision = ctx.args
        ev = _span(timing, "backward_propagation")
        gu, gi = bipartite_propagate_mean(sb, dU.contiguous(), dI.contiguous(), L, group, spmm_fn, chunks, timing,
                                          reduce_items=True, after_first_exchange=hook, precision=precision)
        _end(ev)
        return gu, gi, None, None, None, None, None, None, None, None


def bipartite_propagate(sb: ShardedBipartite, Xu_local, Xi, n_layers, group=None, spmm_fn=_spmm_cuda, chunks=4,
                        timing=None, backward_exchange_hook=None, precision="fp32"):
    """Differentiable bipartite_propagate_mean. Backward exchanges: one chunked all-reduce of the
    partial item gradient, then one per layer as in the forward (1 + L); the returned item
    gradient is the group's total, identical on every rank. `backward_exchange_hook` is the
    backward's `after_first_exchange` (see bipartite_propagate_mean). `precision` applies to the
    forward and to the backward, which runs the same operator (rounding the incoming gradients
    where the forward rounds the tables; the item gradient after its reduction)."""
    _check_precision(precision)
    return _BipartitePropagateMean.apply(Xu_local, Xi, sb, n_layers, group, spmm_fn, chunks, timing,
                                         backward_exchange_hook, precision)


def _xavier_rows(n, d, lo, hi, seed, device):
    """Rows [lo, hi) of an xavier-uniform [n, d] table (fan n + d, models.LightGCN's init),
    generated in fixed 1M-row blocks so the values do not depend on how the rows are sharded."""
    bound = (6.0 / (n + d)) ** 0.5
    blk = 1 << 20
    out = [torch.empty(0, d, device=device)]
    for b0 in range(lo // blk * blk, hi, blk):
        b1 = min(n, b0 + blk)
        g = torch.Generator(device=device).manual_seed(seed + b0 // blk)
        x = (torch.rand(b1 - b0, d, generator=g, device=device) * 2 - 1) * bound
        out.append(x[max(lo, b0) - b0: min(hi, b1) - b0])
    return torch.cat(out).contiguous()


def _loss_fns_cuda():
    return ops.lightgcn_loss_fwd, ops.lightgcn_loss_bwd


class _ShardedLightGCNLoss(torch.autograd.Function):
    """LightGCN's loss over the union of every rank's triples from this rank's share: partial sums
    on the local triples, one all-reduce of [bpr, |U|^2, |P|^2, |N|^2, B_p], the global loss and the
    backward coefficients formed on the device (no host round trip)."""

    @staticmethod
    def forward(ctx, user_out, item_out, user_ego, item_ego, users, pos, neg, model):
        fwd, _ = model.loss_fns
        ev = _span(model.timing, "loss")
        out4, dx = fwd(user_out.detach(), item_out.detach(), user_ego.detach(), item_ego.detach(), users, pos, neg,
                       model.gamma)
        # B_p travels with the sums (exact in float32 up to 2^24 triples per step)
        red = torch.cat([out4, out4.new_full((1,), float(users.numel()))])
        if model.sb.world > 1:
            dist.all_reduce(red, group=model.group)
        B = red[4].clamp(min=1.0)
        norms = red[1:4].sqrt()
        rw = model.reg_weight
        loss = red[0] / B + rw * (norms.sum() / B)
        # d|x|/dx = x / |x|, and 0 at x = 0 as torch.norm's backward
        reg = torch.where(norms > 0, rw / (B * norms.clamp(min=torch.finfo(norms.dtype).tiny)),
                          torch.zeros_like(norms))
        ctx.coef4 = torch.cat([(1.0 / B).reshape(1), reg]).to(out4.dtype)
        ctx.model = model
        ctx.save_for_backward(user_out, item_out, user_ego, item_ego, users, pos, neg, dx)
        _end(ev)
        return loss

    @staticmethod
    def backward(ctx, g):
        user_out, item_out, user_ego, item_ego, users, pos, neg, dx = ctx.saved_tensors
        model = ctx.model
        _, bwd = model.loss_fns
        ev = _span(model.timing, "loss")
        grads = [torch.zeros_like(t) for t in (user_out, item_out, user_ego, item_ego)]
        bwd(user_out, item_out, user_ego, item_ego, users, pos, neg, dx, ctx.coef4 * g, *grads)
        _end(ev)
        model._hold_item_reg_grad(grads[3])
        return grads[0], grads[1], grads[2], None, None, None, None, None


class ShardedLightGCN(torch.nn.Module):
    """LightGCN (lightgcn.py, the reference's loss semantics) trained on the user-sharded bipartite
    graph: rank p holds the ego rows of its users [lo, hi) and the whole (replicated) item table;
    `sb` is its ShardedBipartite (e.g. from `ShardedBipartite.from_local_edges`).

    Per step: L item-table all-reduces in the forward propagation, one scalar all-reduce of the loss
    sums, 1 + L in the backward propagation and one of the item-table regulariser gradient. The
    latter is queued on the group's stream right after the backward's layer-1 exchange (behind the
    reduction of the partial item gradient that layer 1 waits for, not in front of it) and waited
    for when the item table's gradient is complete (just before the optimizer step). The item table and its optimizer state stay bit-identical on every
    rank: every operation after a reduction runs on replicated, reduced values in a fixed order.

    `user_emb` / `item_emb`: initial tables (this rank's user rows, all item rows); default: xavier
    uniform per table, from fixed seeded 1M-row blocks (the same values at every world size).
    `precision` ("fp32" or "bf16"): the operand precision of the propagation's SpMMs in the
    training forward, its backward and the evaluation forward (see bipartite_propagate_mean);
    parameters, optimizer state, loss and scoring stay float32 either way.
    `spmm_fn` / `loss_fns` = (fwd, bwd) replace the CUDA operators (ops.lightgcn_loss_fwd / _bwd
    signatures), e.g. by float64 CPU arithmetic in tests; so does `eval_fns` = (topk, metric_sums)
    for the evaluation (signatures of _topk_rows_cuda and ops.topk_metric_sums).

    Evaluation (`eval_metric_sums`, driven by trainer.Trainer.evaluate with a ShardedEvalData): the
    forward runs once per pass, cached in eval mode and dropped by train(); each rank scores its own
    users against the item table with its training CSR `sb.R` as the mask."""

    def __init__(self, sb: ShardedBipartite, embedding_size=64, n_layers=4, reg_weight=1e-2, group=None,
                 user_emb=None, item_emb=None, seed=2024, chunks=4, gamma=1e-10, spmm_fn=_spmm_cuda, loss_fns=None,
                 device=None, eval_fns=None, precision="fp32"):
        super().__init__()
        _check_precision(precision)
        self.precision = precision
        self.sb, self.group, self.n_layers, self.reg_weight = sb, group, int(n_layers), float(reg_weight)
        self.chunks, self.gamma, self.spmm_fn = chunks, float(gamma), spmm_fn
        self.loss_fns = loss_fns or _loss_fns_cuda()
        self.n_users, self.n_items, self.latent_dim = sb.U, sb.I, int(embedding_size)
        dev = torch.device(device) if device is not None else sb.R.vals.device
        if user_emb is None:
            user_emb = _xavier_rows(sb.U, self.latent_dim, sb.lo, sb.hi, seed, dev)
        if item_emb is None:
            item_emb = _xavier_rows(sb.I, self.latent_dim, 0, sb.I, seed + (1 << 20), dev)
        if user_emb.shape != (sb.hi - sb.lo, self.latent_dim) or item_emb.shape != (sb.I, self.latent_dim):
            raise ValueError("ShardedLightGCN: user_emb must be [hi - lo, d] (this rank's rows), item_emb [I, d]")
        self.embedding_dict = torch.nn.ParameterDict({
            "user_emb": torch.nn.Parameter(user_emb.detach().clone().contiguous()),
            "item_emb": torch.nn.Parameter(item_emb.detach().clone().contiguous())})
        self.embedding_dict["item_emb"].register_post_accumulate_grad_hook(self._finish_item_grad)
        self._pending_item_reg = None
        self.timing = None            # dict: CUDA-event spans per phase (scripts/sharded_train.py)
        self.eval_fns = eval_fns or (_topk_rows_cuda, ops.topk_metric_sums)
        self._eval_cache = None
        self._mask = None

    def train(self, mode=True):
        self._eval_cache = None
        return super().train(mode)

    def pre_epoch_processing(self):
        pass

    def post_epoch_processing(self):
        pass

    def forward(self):
        """-> (this rank's rows of the final user table, the final item table)."""
        e = self.embedding_dict
        return bipartite_propagate(self.sb, e["user_emb"], e["item_emb"], self.n_layers, self.group, self.spmm_fn,
                                   self.chunks, self.timing, backward_exchange_hook=self._issue_item_reg,
                                   precision=self.precision)

    def calculate_loss(self, interaction):
        """interaction: this rank's [3, B_p] triples (users as LOCAL row ids, global item ids; B_p
        may be 0). Returns the loss of the union of all ranks' triples, identical on every rank."""
        users, pos, neg = interaction[0], interaction[1], interaction[2]
        uo, io = self.forward()
        e = self.embedding_dict
        return _ShardedLightGCNLoss.apply(uo, io, e["user_emb"], e["item_emb"], users, pos, neg, self)

    def _hold_item_reg_grad(self, d_item_ego):
        """Loss backward: this rank's partial of the item-ego gradient; reduced by _issue_item_reg."""
        self._pending_item_reg = {"grad": d_item_ego, "work": None, "issued": False}

    def _issue_item_reg(self):
        """Propagation backward, after its layer-1 exchange: queue the regulariser all-reduce."""
        pend = self._pending_item_reg
        if pend is not None and not pend["issued"]:
            if self.sb.world > 1:
                pend["work"] = dist.all_reduce(pend["grad"], group=self.group, async_op=True)
            pend["issued"] = True

    def _finish_item_grad(self, p):
        """The item table's gradient is complete: add the reduced regulariser gradient."""
        self._issue_item_reg()
        pend, self._pending_item_reg = self._pending_item_reg, None
        if pend is None:
            return
        ev = _span(self.timing, "exposed_all_reduce")
        if pend["work"] is not None:
            pend["work"].wait()
        _end(ev)
        p.grad.add_(pend["grad"])

    @torch.no_grad()
    def full_sort_topk(self, users, k):
        """Top-k item ids (unmasked) for GLOBAL user ids `users`, the same on every rank."""
        uo, io = self.forward()
        return bipartite_score_topk(self.sb, uo, io, users, k, group=self.group)

    @torch.no_grad()
    def restore_embeddings(self):
        """(this rank's final user rows, the final item table) of the evaluation forward: computed
        once per evaluation pass in eval mode (its L item-table all-reduces run on every rank)."""
        if self.training or self._eval_cache is None:
            uo, io = self.forward()
            if self.training:
                return uo, io
            self._eval_cache = (uo.contiguous(), io.contiguous())
        return self._eval_cache

    def _mask_csr(self):
        """This rank's training CSR as the evaluation mask: (row_ptr, col_idx, col_offset). The
        kernels walk a mask row with an ascending cursor, so the columns are checked to ascend
        strictly within every row (once)."""
        if self._mask is None:
            R = self.sb.R
            rp = R.row_ptr
            a, b = int(rp[0]), int(rp[-1])
            cols = R.col_idx[a:b]
            if cols.numel() > 1:
                up = cols[1:] > cols[:-1]
                starts = rp[1:-1].to(torch.int64) - a                 # where a row begins, the order may restart
                up[starts[(starts > 0) & (starts < cols.numel())] - 1] = True
                if not bool(up.all()):
                    raise ValueError("ShardedLightGCN: the training CSR's columns must ascend within each row")
            self._mask = (rp, R.col_idx, R.col_offset)
        return self._mask

    @torch.no_grad()
    def eval_topk(self, users, k):
        """Top-k item ids, training items masked, for LOCAL user ids `users` of this rank, from the
        evaluation forward. No collective besides that forward's."""
        uo, io = self.restore_embeddings()
        rp, cols, off = self._mask_csr()
        # a CSR whose columns carry an offset (a view of the full graph's user rows) masks with the
        # offset ids: score them under those ids and map back
        ids = self.eval_fns[0](uo, users, io, k, rp, cols, off)
        return ids - off if off else ids

    @torch.no_grad()
    def eval_metric_sums(self, eval_data, k):
        """This rank's [5, k] float64 metric sums (ops.topk_metric_sums rows) over its evaluated
        users `eval_data` (a ShardedEvalData), scored `eval_data.step` users at a time. Every rank
        must call it: the evaluation forward has collectives. Trainer.evaluate reduces the sums."""
        uo, io = self.restore_embeddings()
        rowptr, items = eval_data.gt_csr()
        n = eval_data.eval_u.numel()
        sums = torch.zeros(5, k, dtype=torch.float64, device=io.device)
        for a in range(0, n, eval_data.step):
            b = min(n, a + eval_data.step)
            ids = self.eval_topk(eval_data.eval_u[a:b], k)
            sums += self.eval_fns[1](ids, rowptr[a:b + 1], items)
        return sums


def _topk_rows_cuda(user_emb, users, item_emb, k, mask_rowptr, mask_cols, item_offset):
    return ops.score_mask_topk_rows(user_emb, users, item_emb, k, mask_rowptr, mask_cols, item_offset=item_offset)


class ShardedEvalData:
    """One rank's share of a held-out split (valid or test) for ShardedLightGCN's evaluation, built
    on the device from this rank's held-out edges (`users`: global ids in [sb.lo, sb.hi); `items`):
    * `eval_u`: LOCAL ids of the rank's users with at least one held-out edge, ascending (int64);
    * `gt_csr()`: their ground truth as EvalDataLoader.gt_csr gives it (int32 row pointers,
      ascending int32 item ids);
    * `n_users_global` / `total_pos`: evaluated users and held-out interactions over the whole
      group (one all-reduce here), the denominators of TopKEvaluator's metrics;
    * `reduce_metric_sums`: sums a rank's [5, K] metric sums over the group, so every rank forms the
      same result dict (and makes the same early-stopping decision in Trainer.fit).
    `batch_users`: evaluated users per scoring launch (bounds the [n, K] workspaces)."""

    def __init__(self, sb: ShardedBipartite, users, items, group=None, batch_users=1 << 17):
        users = users.to(torch.int64) - sb.lo
        items = items.to(torch.int64)
        if users.numel() and (int(users.min()) < 0 or int(users.max()) >= sb.hi - sb.lo):
            raise ValueError("ShardedEvalData: held-out edges of users this rank does not own")
        key = torch.sort(users * sb.I + items)[0]
        self.eval_u, counts = torch.unique_consecutive(key // sb.I, return_counts=True)
        rowptr = torch.zeros(self.eval_u.numel() + 1, dtype=torch.int64, device=key.device)
        rowptr[1:] = torch.cumsum(counts, 0)
        self._gt = (rowptr.to(torch.int32), (key % sb.I).to(torch.int32))
        cnt = torch.tensor([self.eval_u.numel(), key.numel()], dtype=torch.int64, device=key.device)
        if sb.world > 1:
            dist.all_reduce(cnt, group=group)
        self.n_users_global, self.total_pos = int(cnt[0]), float(cnt[1])
        self.world, self.group, self.step = sb.world, group, int(batch_users)

    def gt_csr(self):
        return self._gt

    def reduce_metric_sums(self, sums):
        if self.world > 1:
            sums = sums.clone()
            dist.all_reduce(sums, group=self.group)
        return sums


# ------------------------------------------------------------------ item-range sharded modality tables
# SURVEY 8e row 2: the trainable [I, 4096] / [I, 384] feature tables (smore.py:76-77, mgcn.py:62-72,
# freedom.py:48-55), their projection (smore.py:256-257), its gradients and the Adam state are the
# largest HBM consumers of a SMORE / MGCN / FREEDOM step and are independent per item row. Rank p
# keeps rows [lo_p, hi_p) of every table (parameter + exp_avg + exp_avg_sq: 12 of the 16 bytes per
# element stay local for good); per projection
#   forward : Y_p = X_p W^T + b on the local rows, all-gather of the [I/P, d] slices -> Y [I, d];
#   backward: dY is replicated (everything downstream of the projection is replicated), so
#             dX_p = dY[lo:hi] W stays local, dW = all-reduce(dY[lo:hi]^T X_p), db likewise.
# Slices are padded to the longest range so that all_gather_into_tensor needs no packing.
def _linear_cuda(x, W, b):
    return ops.linear(x, W, b)


class ShardedRows:
    """Contiguous, near-equal row ranges of an [n, *] table over the ranks of a process group."""

    def __init__(self, n_rows: int, rank: int, world: int):
        self.n, self.rank, self.world = int(n_rows), int(rank), int(world)
        self.per = -(-self.n // self.world)
        self.lo = min(self.n, self.rank * self.per)
        self.hi = min(self.n, self.lo + self.per)

    def local(self, table: torch.Tensor) -> torch.Tensor:
        return table[self.lo: self.hi]


class _ShardedProjection(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_local, W, b, rows, group, linear_fn):
        y_local = linear_fn(x_local.detach(), W.detach(), None if b is None else b.detach())
        d = y_local.shape[1]
        buf = torch.empty(rows.world * rows.per, d, dtype=y_local.dtype, device=y_local.device)
        if y_local.shape[0] == rows.per:
            mine = y_local.contiguous()
        else:                                   # the last range is shorter: pad its slice
            mine = torch.zeros(rows.per, d, dtype=y_local.dtype, device=y_local.device)
            mine[: y_local.shape[0]] = y_local
        dist.all_gather_into_tensor(buf, mine, group=group)
        ctx.save_for_backward(x_local, W)
        ctx.rows, ctx.group, ctx.has_bias = rows, group, b is not None
        return buf[: rows.n]

    @staticmethod
    def backward(ctx, dY):
        x_local, W = ctx.saved_tensors
        rows = ctx.rows
        dy = dY[rows.lo: rows.hi].contiguous()
        dx = dy @ W if ctx.needs_input_grad[0] else None
        # dW and db travel in one buffer: one all-reduce per projection
        n_out, n_in = W.shape
        pack = torch.empty(n_out, n_in + 1, dtype=W.dtype, device=W.device)
        pack[:, :n_in] = dy.t() @ x_local
        pack[:, n_in] = dy.sum(0)
        dist.all_reduce(pack, group=ctx.group)
        dW = pack[:, :n_in].contiguous()
        db = pack[:, n_in].contiguous() if ctx.has_bias else None
        return dx, dW, db, None, None, None


class _ShardedProjectionCuda(_ShardedProjection):
    """Same exchange, local products on the 3xTF32 GEMMs of the library."""

    @staticmethod
    def backward(ctx, dY):
        x_local, W = ctx.saved_tensors
        rows = ctx.rows
        dy = dY[rows.lo: rows.hi].contiguous()
        M, K = x_local.shape
        N = W.shape[0]
        dx = ops.gemm(dy, True, W, False, M, K, N) if ctx.needs_input_grad[0] else None
        pack = torch.empty(N, K + 1, dtype=W.dtype, device=W.device)
        pack[:, :K] = ops.gemm(dy, False, x_local, False, N, K, M)
        pack[:, K] = dy.sum(0)
        dist.all_reduce(pack, group=ctx.group)
        return dx, pack[:, :K].contiguous(), (pack[:, K].contiguous() if ctx.has_bias else None), None, None, None


def sharded_projection(x_local, W, b, rows: ShardedRows, group=None, linear_fn=None):
    """`Linear(table)` with the table's rows sharded over the group: every rank passes its
    [I/P, F] slice and gets the full [I, d] projection; gradients as described above."""
    if linear_fn is None:
        return _ShardedProjectionCuda.apply(x_local, W, b, rows, group, _linear_cuda)
    return _ShardedProjection.apply(x_local, W, b, rows, group, linear_fn)


def sharded_sumsq(replicated, sharded, group=None):
    """Sum of squares over a parameter (or gradient) list of which `sharded` tensors hold only this
    rank's rows: local sums of the sharded part are all-reduced, the replicated part counts once.
    Used by the mirror-gradient step for its global grad / param RMS (trainer.py:289-305)."""
    dev = (replicated or sharded)[0].device
    s = torch.zeros((), dtype=torch.float32, device=dev)
    if sharded:
        s = torch.stack(torch._foreach_norm(list(sharded))).pow(2).sum()
        dist.all_reduce(s, group=group)
    if replicated:
        s = s + torch.stack(torch._foreach_norm(list(replicated))).pow(2).sum()
    return s
