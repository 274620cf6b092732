"""torch.autograd wrappers over the C ABI: the operator layer the models are written against.

Each Function replaces a family of torch call sites in the reference models (file:line cited per
op). Everything runs on CUDA through libmmrec_b200.so; there is no CPU or eager fallback.
"""
from __future__ import annotations

import ctypes

import torch

from . import lib
from .graph import CSRGraph

_counters = {}


def _counter(device):
    """Zero-initialised arrival counter shared by the self-resetting last-block reductions."""
    key = (device.type, device.index)
    if key not in _counters:
        _counters[key] = torch.zeros(1024, dtype=torch.int32, device=device)
    return _counters[key]


# Index range checks (a host sync per call): off in production, on with MMREC_CHECK_IDS=1. The
# gather / scatter kernels trust their int64 ids the way a raw CUDA kernel does -- where torch
# indexing would raise IndexError they would read or `red.add` out of bounds -- and
# compute-sanitizer is not available on the GPU pool, so this is the memcheck of the id arguments.
CHECK_IDS = __import__("os").environ.get("MMREC_CHECK_IDS", "0") == "1"


def _check_ids(idx, n, what):
    if CHECK_IDS and idx is not None and idx.numel():
        lo, hi = int(idx.min()), int(idx.max())
        if lo < 0 or hi >= n:
            raise IndexError(f"{what}: index range [{lo}, {hi}] outside [0, {n})")


def _f32c(t):
    if t.dtype != torch.float32:
        raise RuntimeError(f"expected float32, got {t.dtype}")
    return t.contiguous()


L2_BYTES = 126 << 20
SPMM_NARROW, SPMM_STREAM = 1, 2
# Measured on the 10M x 2M x 486M graph (profiles/r02_config5_spmm_experiments.txt): the eviction
# hints change nothing (129.6 vs 130.1 ms for four layers), so they stay off unless asked for.
_STREAM_DEFAULT = __import__("os").environ.get("MMREC_SPMM_STREAM", "0") == "1"
_NARROW_ALL = __import__("os").environ.get("MMREC_SPMM_NARROW", "0") == "1"          # A/B switch


def spmm_raw(g: CSRGraph, X, Y=None, acc_in=None, acc_out=None, acc_scale=1.0, cos_ref=None,
             cos_w=None, y_pre=None, narrow=False, stream_policy=None, y16=None):
    """mmrec_spmm_csr_f32 on already-allocated tensors (no autograd). narrow=True: the tiling for
    graphs of very short rows; stream_policy: L2 eviction hints for operands larger than the cache
    (default: on when the gathered table exceeds half of L2) -- mmrec_spmm_csr_ex_f32.
    A bfloat16 X runs mmrec_spmm_csr_bf16_f32 (fp32 arithmetic, fp32 Y / acc); `y16` (bfloat16
    [n_rows, d]) then receives y rounded to nearest even."""
    lib.require_cuda(X)
    d = X.shape[1]
    if X.shape[0] < g.n_cols:
        raise RuntimeError(f"spmm: X has {X.shape[0]} rows, graph has {g.n_cols} columns")
    if X.dtype == torch.bfloat16:
        _spmm_bf16(g, X, Y, y16, acc_in, acc_out, acc_scale, cos_ref, cos_w, y_pre, narrow, stream_policy)
        return
    if X.dtype != torch.float32 or y16 is not None:
        raise RuntimeError(f"spmm: X must be float32 or bfloat16 (y16 only with bfloat16), got {X.dtype}")
    if stream_policy is None:
        stream_policy = _STREAM_DEFAULT and cos_ref is None and 4 * d * g.n_cols > L2_BYTES // 2
    flags = (SPMM_NARROW if (narrow or _NARROW_ALL) else 0) | (SPMM_STREAM if stream_policy else 0)
    if flags:
        lib.call("mmrec_spmm_csr_ex_f32", lib.ptr(g.row_ptr), lib.ptr(g.col_idx), lib.ptr(g.vals),
                 lib.ptr(g.tasks), g.n_tasks, lib.ptr(g.slot_base), lib.ptr(g.counters),
                 lib.ptr(g.scratch(d)), g.col_offset, lib.ptr(X), d, lib.ptr(Y),
                 lib.ptr(acc_in), lib.ptr(acc_out), float(acc_scale), lib.ptr(cos_ref), lib.ptr(cos_w),
                 lib.ptr(y_pre), flags, lib.stream())
        return
    lib.call("mmrec_spmm_csr_f32", lib.ptr(g.row_ptr), lib.ptr(g.col_idx),
             lib.ptr(g.vals), lib.ptr(g.tasks), g.n_tasks, lib.ptr(g.slot_base), lib.ptr(g.counters),
             lib.ptr(g.scratch(d)), g.col_offset, lib.ptr(X), d, lib.ptr(Y),
             lib.ptr(acc_in), lib.ptr(acc_out), float(acc_scale), lib.ptr(cos_ref), lib.ptr(cos_w),
             lib.ptr(y_pre), lib.stream())


def _spmm_bf16(g, X, Y, y16, acc_in, acc_out, acc_scale, cos_ref, cos_w, y_pre, narrow, stream_policy):
    d = X.shape[1]
    if not X.is_contiguous():
        raise RuntimeError("spmm_bf16: X must be contiguous")
    for name, t, dt in (("Y", Y, torch.float32), ("y16", y16, torch.bfloat16), ("acc_in", acc_in, torch.float32),
                        ("acc_out", acc_out, torch.float32)):
        if t is None:
            continue
        lib.require_cuda(t)
        if t.dtype != dt or tuple(t.shape) != (g.n_rows, d) or not t.is_contiguous():
            raise RuntimeError(f"spmm_bf16: {name} must be a contiguous {dt} [{g.n_rows}, {d}] tensor, "
                               f"got {t.dtype} {tuple(t.shape)}")
    flags = (SPMM_NARROW if (narrow or _NARROW_ALL) else 0) | (SPMM_STREAM if stream_policy else 0)
    lib.call("mmrec_spmm_csr_bf16_f32", lib.ptr(g.row_ptr), lib.ptr(g.col_idx), lib.ptr(g.vals),
             lib.ptr(g.tasks), g.n_tasks, lib.ptr(g.slot_base), lib.ptr(g.counters),
             lib.ptr(g.scratch(d)), g.col_offset, lib.ptr(X), d, lib.ptr(Y), lib.ptr(y16),
             lib.ptr(acc_in), lib.ptr(acc_out), float(acc_scale), lib.ptr(cos_ref), lib.ptr(cos_w),
             lib.ptr(y_pre), flags, lib.stream())


def spmm_blocked_raw(bg, X, Y):
    """Y = A X for a graph.ColumnBlockedCSR: one launch per column block, the first writes Y, the
    others accumulate into it (the X slice of the block in flight stays L2-resident)."""
    for b, g in enumerate(bg.blocks):
        if b == 0:
            spmm_raw(g, X, Y=Y, narrow=True)
        else:
            spmm_raw(g, X, acc_in=Y, acc_out=Y, narrow=True)


class _SpMM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X, g):
        X = _f32c(X)
        Y = torch.empty(g.n_rows, X.shape[1], dtype=torch.float32, device=X.device)
        spmm_raw(g, X, Y=Y)
        ctx.g = g
        return Y

    @staticmethod
    def backward(ctx, dY):
        g = ctx.g
        if g.t is None:
            raise RuntimeError("spmm backward needs the transposed CSR (build with_transpose=True)")
        dY = _f32c(dY)
        dX = torch.empty(g.t.n_rows, dY.shape[1], dtype=torch.float32, device=dY.device)
        spmm_raw(g.t, dY, Y=dX)
        return dX, None


def spmm_multi_raw(graphs, Xs, Ys=None, acc_ins=None, acc_outs=None):
    """mmrec_spmm_csr_multi_f32: up to 4 independent SpMMs of the same width in one launch."""
    n = len(graphs)
    d = Xs[0].shape[1]
    arr = (lib.SpmmProblem * n)()
    keep = []
    seen = {}
    for i, (g, X) in enumerate(zip(graphs, Xs)):
        lib.require_cuda(X)
        if X.shape[1] != d or X.shape[0] < g.n_cols:
            raise RuntimeError("spmm_multi: operand shapes do not match the graphs")
        slot = seen.get(id(g), 0)                 # same graph twice in one launch: own scratch
        seen[id(g)] = slot + 1
        scratch, counters = g.scratch(d, slot), g.counters_for(slot)
        keep += [scratch, counters]
        p = arr[i]
        p.row_ptr, p.col_idx, p.vals = lib.ptr(g.row_ptr), lib.ptr(g.col_idx), lib.ptr(g.vals)
        p.tasks, p.n_tasks, p.slot_base = lib.ptr(g.tasks), g.n_tasks, lib.ptr(g.slot_base)
        p.counters, p.scratch, p.col_offset = lib.ptr(counters), lib.ptr(scratch), g.col_offset
        p.X = lib.ptr(X)
        p.Y = lib.ptr(Ys[i]) if Ys is not None else None
        p.acc_in = lib.ptr(acc_ins[i]) if acc_ins is not None else None
        p.acc_out = lib.ptr(acc_outs[i]) if acc_outs is not None else None
        p.acc_scale = 1.0
    import ctypes
    lib.call("mmrec_spmm_csr_multi_f32", ctypes.byref(arr), n, d, lib.stream())


class _SpMMMulti(torch.autograd.Function):
    """Y_i = A_i X_i for several (graph, X) pairs in one launch; backward dX_i = A_i^T dY_i in one."""

    @staticmethod
    def forward(ctx, graphs, *Xs):
        Xs = [_f32c(x) for x in Xs]
        Ys = [torch.empty(g.n_rows, x.shape[1], dtype=torch.float32, device=x.device)
              for g, x in zip(graphs, Xs)]
        spmm_multi_raw(graphs, Xs, Ys=Ys)
        ctx.graphs = graphs
        return tuple(Ys)

    @staticmethod
    def backward(ctx, *dYs):
        gts = []
        for g in ctx.graphs:
            if g.t is None:
                raise RuntimeError("spmm backward needs the transposed CSR (build with_transpose=True)")
            gts.append(g.t)
        ref = next(d for d in dYs if d is not None)
        dYs = [_f32c(dy) if dy is not None else
               torch.zeros(g.n_rows, ref.shape[1], dtype=torch.float32, device=ref.device)
               for dy, g in zip(dYs, ctx.graphs)]
        dXs = [torch.empty(gt.n_rows, dy.shape[1], dtype=torch.float32, device=dy.device)
               for gt, dy in zip(gts, dYs)]
        spmm_multi_raw(gts, dYs, Ys=dXs)
        return (None, *dXs)


class _ModalityViews(torch.autograd.Function):
    """The modality views of MGCN / SMORE (mgcn.py:170-184, smore.py:289-317) for all modalities at
    once: x <- A_m x (n_layers item-item hops), u = R x, view_m = cat([u, x]). The last item hop
    writes straight into rows [U, N) of the view and the R hop into rows [0, U): no torch.cat; the
    backward adds the direct gradient of the item rows inside the R^T launch (accumulate epilogue)
    instead of a separate add per view."""

    @staticmethod
    def forward(ctx, item_graphs, R, n_layers, *xs):
        xs = [_f32c(x) for x in xs]
        n = len(xs)
        U, I, d = R.n_rows, R.n_cols, xs[0].shape[1]
        dev = xs[0].device
        outs = [torch.empty(U + I, d, dtype=torch.float32, device=dev) for _ in range(n)]
        cur = xs
        for layer in range(n_layers):
            last = layer == n_layers - 1
            ys = [o[U:] for o in outs] if last else [torch.empty_like(x) for x in cur]
            spmm_multi_raw(item_graphs, cur, Ys=ys)
            cur = ys
        spmm_multi_raw([R] * n, cur, Ys=[o[:U] for o in outs])
        ctx.item_graphs, ctx.R, ctx.n_layers = item_graphs, R, n_layers
        return tuple(outs)

    @staticmethod
    def backward(ctx, *douts):
        R, n_layers = ctx.R, ctx.n_layers
        U, I = R.n_rows, R.n_cols
        ref = next(g for g in douts if g is not None)
        douts = [torch.zeros_like(ref) if g is None else _f32c(g) for g in douts]
        n = len(douts)
        gts = []
        for g in ctx.item_graphs:
            if g.t is None:
                raise RuntimeError("modality views backward needs the transposed item graphs")
            gts.append(g.t)
        # d x = R^T d u + (direct gradient of the item rows), one launch for all views
        cur = [torch.empty(I, ref.shape[1], dtype=torch.float32, device=ref.device) for _ in range(n)]
        spmm_multi_raw([R.t] * n, [g[:U] for g in douts], acc_ins=[g[U:] for g in douts], acc_outs=cur)
        for _ in range(n_layers):
            nxt = [torch.empty_like(c) for c in cur]
            spmm_multi_raw(gts, cur, Ys=nxt)
            cur = nxt
        return (None, None, None, *cur)


def modality_views(item_graphs, R, n_layers, xs):
    """[cat([R x_m', x_m'])] with x_m' = A_m^n_layers x_m, for up to 4 modalities; see _ModalityViews."""
    return list(_ModalityViews.apply(list(item_graphs), R, int(n_layers), *xs))


def spmm_multi(graphs, Xs):
    """[torch.sparse.mm(A_i, X_i)] for independent pairs (at most 4) in one launch each way."""
    graphs = list(graphs)
    if len(graphs) == 1:
        return [spmm(graphs[0], Xs[0])]
    return list(_SpMMMulti.apply(graphs, *Xs))


def spmm(g: CSRGraph, X):
    """Y = A X; replaces torch.sparse.mm(A, X) (layergcn.py:133, freedom.py:169,174,
    mgcn.py:162-184, smore.py:282-317, lightgcn.py:122). Backward: dX = A^T dY."""
    return _SpMM.apply(X, g)


def _horner(g, G, n_layers, scale_last):
    """t <- G + A t, n_layers times, starting from t = G; last step scaled."""
    t = G
    for l in range(n_layers):
        out = torch.empty_like(G)
        spmm_raw(g, t, acc_in=G, acc_out=out, acc_scale=scale_last if l == n_layers - 1 else 1.0)
        t = out
    return t


class _PropagateMean(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X0, g, n_layers):
        X0 = _f32c(X0)
        ctx.g, ctx.n_layers = g, n_layers
        if n_layers == 0:
            return X0.clone()
        inv = 1.0 / (n_layers + 1)
        acc = torch.empty_like(X0)
        x = X0
        for l in range(1, n_layers + 1):
            last = l == n_layers
            y = None if last else torch.empty_like(X0)
            spmm_raw(g, x, Y=y, acc_in=X0 if l == 1 else acc, acc_out=acc,
                     acc_scale=inv if last else 1.0)
            x = y
        return acc

    @staticmethod
    def backward(ctx, dOut):
        g, L = ctx.g, ctx.n_layers
        dOut = _f32c(dOut)
        if L == 0:
            return dOut, None, None
        gt = g.t
        if gt is None:
            raise RuntimeError("propagate_mean backward needs the transposed CSR")
        # d X0 = 1/(L+1) * sum_l (A^T)^l dOut, evaluated as a Horner chain
        return _horner(gt, dOut, L, 1.0 / (L + 1)), None, None


def propagate_mean(g: CSRGraph, X0, n_layers):
    """mean_{l=0..L} A^l X0 with the running sum fused into the SpMM epilogue; replaces the
    layer loop + stack + mean at freedom.py:171-179, mgcn.py:159-167, smore.py:278-287,
    lightgcn.py:118-128."""
    return _PropagateMean.apply(X0, g, n_layers)


class _LayerGCNPropagate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X0, g, n_layers):
        X0 = _f32c(X0)
        n, d = X0.shape
        P = torch.empty(n_layers, n, d, dtype=torch.float32, device=X0.device)
        W = torch.empty(n_layers, n, dtype=torch.float32, device=X0.device)
        acc = torch.empty_like(X0)
        x = X0
        for l in range(n_layers):
            y = torch.empty_like(X0) if l < n_layers - 1 else None
            spmm_raw(g, x, Y=y, acc_in=None if l == 0 else acc, acc_out=acc, acc_scale=1.0,
                     cos_ref=X0, cos_w=W[l], y_pre=P[l])
            x = y
        ctx.g, ctx.n_layers = g, n_layers
        ctx.save_for_backward(X0, P, W)
        return acc

    @staticmethod
    def backward(ctx, dOut):
        X0, P, W = ctx.saved_tensors
        g, L = ctx.g, ctx.n_layers
        gt = g.t
        dOut = _f32c(dOut)
        n, d = X0.shape
        dE0 = torch.zeros_like(X0)
        dE = dOut
        for l in range(L - 1, -1, -1):
            dP = torch.empty_like(X0)
            lib.call("mmrec_layergcn_cos_bwd_f32", lib.ptr(dE), lib.ptr(P[l]), lib.ptr(X0),
                     lib.ptr(W[l]), n, d, lib.ptr(dP), lib.ptr(dE0), lib.stream())
            if l > 0:
                nxt = torch.empty_like(X0)
                spmm_raw(gt, dP, acc_in=dOut, acc_out=nxt)       # dE_{l-1} = dOut + A^T dP_l
                dE = nxt
            else:
                spmm_raw(gt, dP, acc_in=dE0, acc_out=dE0)        # dX0 = dE0 + A^T dP_1
        return dE0, None, None


def layergcn_propagate(g: CSRGraph, X0, n_layers):
    """LayerGCN.forward's layer loop (layergcn.py:127-140): SpMM, cosine re-weighting against the
    ego layer and the layer sum fused in one kernel per layer."""
    return _LayerGCNPropagate.apply(X0, g, n_layers)


# ----------------------------------------------------------------------------------------- BPR
def _bpr_fwd(ue, ie, users, pos, neg):
    B, d = users.numel(), ue.shape[1]
    _check_ids(users, ue.shape[0], "bpr users")
    _check_ids(pos, ie.shape[0], "bpr positive items")
    _check_ids(neg, ie.shape[0], "bpr negative items")
    out = torch.empty(2, dtype=torch.float32, device=ue.device)
    sig = torch.empty(B, dtype=torch.float32, device=ue.device)
    partial = torch.empty(2 * B, dtype=torch.float32, device=ue.device)
    lib.call("mmrec_bpr_fwd_f32", lib.ptr(ue), lib.ptr(ie), d, lib.ptr(users), lib.ptr(pos),
             lib.ptr(neg), B, lib.ptr(out), lib.ptr(sig), lib.ptr(partial),
             lib.ptr(_counter(ue.device)), lib.stream())
    return out, sig


class _BPRSplit(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ue, ie, users, pos, neg):
        ue, ie = _f32c(ue), _f32c(ie)
        out, sig = _bpr_fwd(ue, ie, users, pos, neg)
        ctx.save_for_backward(ue, ie, users, pos, neg, sig)
        return out

    @staticmethod
    def backward(ctx, g):
        ue, ie, users, pos, neg, sig = ctx.saved_tensors
        g = _f32c(g)
        due, die = torch.zeros_like(ue), torch.zeros_like(ie)
        lib.call("mmrec_bpr_bwd_f32", lib.ptr(ue), lib.ptr(ie), ue.shape[1], lib.ptr(users),
                 lib.ptr(pos), lib.ptr(neg), users.numel(), lib.ptr(sig), lib.ptr(g), lib.ptr(due),
                 lib.ptr(die), lib.stream())
        return due, die, None, None, None


class _BPRTable(torch.autograd.Function):
    @staticmethod
    def forward(ctx, emb, n_users, users, pos, neg):
        emb = _f32c(emb)
        out, sig = _bpr_fwd(emb[:n_users], emb[n_users:], users, pos, neg)
        ctx.n_users = n_users
        ctx.save_for_backward(emb, users, pos, neg, sig)
        return out

    @staticmethod
    def backward(ctx, g):
        emb, users, pos, neg, sig = ctx.saved_tensors
        nu = ctx.n_users
        g = _f32c(g)
        d_emb = torch.zeros_like(emb)
        lib.call("mmrec_bpr_bwd_f32", lib.ptr(emb[:nu]), lib.ptr(emb[nu:]), emb.shape[1],
                 lib.ptr(users), lib.ptr(pos), lib.ptr(neg), users.numel(), lib.ptr(sig), lib.ptr(g),
                 lib.ptr(d_emb[:nu]), lib.ptr(d_emb[nu:]), lib.stream())
        return d_emb, None, None, None, None


def bpr(user_emb, item_emb, users, pos, neg):
    """-> tensor[2] = (sum_b -logsigmoid(<u,p> - <u,n>), sum_b 0.5(|u|^2+|p|^2+|n|^2)).
    Replaces the gather + mul + sum + logsigmoid chains at layergcn.py:142-163,
    freedom.py:182-189, mgcn.py:210-222, smore.py:366-378."""
    return _BPRSplit.apply(user_emb, item_emb, users, pos, neg)


def bpr_table(all_emb, n_users, users, pos, neg):
    """Same, for a stacked [users; items] table (one dense gradient instead of two slices)."""
    return _BPRTable.apply(all_emb, n_users, users, pos, neg)


# ------------------------------------------------------------------------------- LightGCN loss
def _lightgcn_loss_args(what, user_out, item_out, user_ego, item_ego, users, pos, neg):
    """Checks shared by the forward and the backward: float32 CUDA tables of matching shapes,
    int64 CUDA ids of one length inside their tables (range checked with MMREC_CHECK_IDS=1)."""
    user_out, item_out, user_ego, item_ego = (_f32c(t) for t in (user_out, item_out, user_ego, item_ego))
    lib.require_cuda(user_out, item_out, user_ego, item_ego, users, pos, neg)
    B, d = users.numel(), user_out.shape[1]
    if pos.numel() != B or neg.numel() != B or users.dtype != torch.int64 or pos.dtype != torch.int64 \
            or neg.dtype != torch.int64:
        raise RuntimeError(f"{what}: users / pos / neg must be int64 tensors of one length")
    if not (item_out.shape[1] == user_ego.shape[1] == item_ego.shape[1] == d) or \
            user_ego.shape[0] != user_out.shape[0] or item_ego.shape[0] != item_out.shape[0]:
        raise RuntimeError(f"{what}: final and ego tables must have matching shapes")
    _check_ids(users, user_out.shape[0], f"{what} users")
    _check_ids(pos, item_out.shape[0], f"{what} positive items")
    _check_ids(neg, item_out.shape[0], f"{what} negative items")
    return user_out, item_out, user_ego, item_ego, users.contiguous(), pos.contiguous(), neg.contiguous()


def lightgcn_loss_fwd(user_out, item_out, user_ego, item_ego, users, pos, neg, gamma=1e-10):
    """Partial sums of LightGCN's loss (lightgcn.py:133-159) over these triples (no autograd):
    -> (out4 = [sum -log(gamma + sigmoid(x)), sum |u0|^2, sum |p0|^2, sum |n0|^2], dx [B]);
    `users` index the user tables, `pos` / `neg` the item tables (int64; B may be 0)."""
    user_out, item_out, user_ego, item_ego, users, pos, neg = _lightgcn_loss_args(
        "lightgcn_loss_fwd", user_out, item_out, user_ego, item_ego, users, pos, neg)
    B, d = users.numel(), user_out.shape[1]
    dev = user_out.device
    out4 = torch.empty(4, dtype=torch.float32, device=dev)
    dx = torch.empty(B, dtype=torch.float32, device=dev)
    partial = torch.empty(lib.load().mmrec_lightgcn_loss_fwd_workspace_floats(B), dtype=torch.float32, device=dev)
    lib.call("mmrec_lightgcn_loss_fwd_f32", lib.ptr(user_out), lib.ptr(item_out), lib.ptr(user_ego),
             lib.ptr(item_ego), d, lib.ptr(users), lib.ptr(pos), lib.ptr(neg), B, float(gamma), lib.ptr(out4),
             lib.ptr(dx), lib.ptr(partial), lib.ptr(_counter(dev)), lib.stream())
    return out4, dx


def lightgcn_loss_bwd(user_out, item_out, user_ego, item_ego, users, pos, neg, dx, coef4,
                      d_user_out, d_item_out, d_user_ego, d_item_ego):
    """Scatter-adds the gradients of the loss formed from `lightgcn_loss_fwd`'s sums into the four
    zeroed float32 outputs (shapes of the four tables). coef4 (device float32 [4]) =
    (dL/d sum_bpr, dL/d|U| / |U|, dL/d|P| / |P|, dL/d|N| / |N|), see include/mmrec_b200.h."""
    user_out, item_out, user_ego, item_ego, users, pos, neg = _lightgcn_loss_args(
        "lightgcn_loss_bwd", user_out, item_out, user_ego, item_ego, users, pos, neg)
    outs = (d_user_out, d_item_out, d_user_ego, d_item_ego)
    lib.require_cuda(dx, coef4, *outs)
    for o, t in zip(outs, (user_out, item_out, user_ego, item_ego)):
        if o.shape != t.shape or o.dtype != torch.float32 or not o.is_contiguous():
            raise RuntimeError("lightgcn_loss_bwd: outputs must be contiguous float32 tensors shaped like the tables")
    if dx.dtype != torch.float32 or dx.numel() != users.numel() or coef4.numel() != 4:
        raise RuntimeError("lightgcn_loss_bwd: dx must be float32 [B] (from lightgcn_loss_fwd), coef4 [4]")
    lib.call("mmrec_lightgcn_loss_bwd_f32", lib.ptr(user_out), lib.ptr(item_out), lib.ptr(user_ego),
             lib.ptr(item_ego), user_out.shape[1], lib.ptr(users), lib.ptr(pos), lib.ptr(neg), users.numel(),
             lib.ptr(dx.contiguous()), lib.ptr(_f32c(coef4)), lib.ptr(d_user_out), lib.ptr(d_item_out),
             lib.ptr(d_user_ego), lib.ptr(d_item_ego), lib.stream())


# ------------------------------------------------------------------------------------- InfoNCE
class _InfoNCEPair(torch.autograd.Function):
    """cl_items + cl_users of MGCN/SMORE.calculate_loss (mgcn.py:248-251, smore.py:403-408) on
    stacked [users; items] tables."""

    @staticmethod
    def forward(ctx, side, content, n_users, users, pos_items, temperature, reduce=True):
        side, content = _f32c(side), _f32c(content)
        _check_ids(users, n_users, "infonce users")
        _check_ids(pos_items, side.shape[0] - n_users, "infonce items")
        dev, d = side.device, side.shape[1]
        inv_t = 1.0 / temperature
        saved = []
        losses = torch.empty(2, dtype=torch.float32, device=dev)
        slots = ((n_users, pos_items), (0, users))
        pair = users.numel() == pos_items.numel() and bool(lib.load().mmrec_infonce_pair_supported(d))
        if pair:                                 # both problems in one launch per stage
            B = users.numel()
            n_ws = lib.load().mmrec_infonce_fwd_workspace_floats(B)
            V1 = [torch.empty(B, d, dtype=torch.float32, device=dev) for _ in slots]
            V2 = [torch.empty(B, d, dtype=torch.float32, device=dev) for _ in slots]
            inv_norm = [torch.empty(2 * B, dtype=torch.float32, device=dev) for _ in slots]
            ttl = [torch.empty(B, dtype=torch.float32, device=dev) for _ in slots]
            partial = [torch.empty(n_ws, dtype=torch.float32, device=dev) for _ in slots]
            T1 = [side[row0:] for row0, _ in slots]
            T2 = [content[row0:] for row0, _ in slots]
            idxs = [idx for _, idx in slots]
            outs = [losses[0:], losses[1:]]
            lib.call("mmrec_infonce_pair_fwd_f32", _ptr_array(T1), _ptr_array(T2), d, _ptr_array(idxs), B, inv_t,
                     _ptr_array(outs), _ptr_array(V1), _ptr_array(V2), _ptr_array(inv_norm), _ptr_array(ttl),
                     _ptr_array(partial), lib.stream())
            for s_ in range(2):
                saved += [V1[s_], V2[s_], inv_norm[s_], ttl[s_], idxs[s_]]
            slots = ()
        for slot, (row0, idx) in enumerate(slots):
            B = idx.numel()
            V1 = torch.empty(B, d, dtype=torch.float32, device=dev)
            V2 = torch.empty_like(V1)
            inv_norm = torch.empty(2 * B, dtype=torch.float32, device=dev)
            ttl = torch.empty(B, dtype=torch.float32, device=dev)
            partial = torch.empty(lib.load().mmrec_infonce_fwd_workspace_floats(B), dtype=torch.float32,
                                  device=dev)
            lib.call("mmrec_infonce_fwd_f32", lib.ptr(side[row0:]), lib.ptr(content[row0:]), d,
                     lib.ptr(idx), B, inv_t, lib.ptr(losses[slot:]), lib.ptr(V1), lib.ptr(V2),
                     lib.ptr(inv_norm), lib.ptr(ttl), lib.ptr(partial), lib.ptr(_counter(dev)),
                     lib.stream())
            saved += [V1, V2, inv_norm, ttl, idx]
        ctx.n_users, ctx.inv_t, ctx.shape, ctx.reduce, ctx.pair = n_users, inv_t, side.shape, reduce, pair
        ctx.save_for_backward(*saved)
        return losses.sum() if reduce else losses

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        n, d = ctx.shape
        dev = g.device
        g = _f32c(g)
        coefs = (g.reshape(1), g.reshape(1)) if ctx.reduce else (g[0:1], g[1:2])
        d_both = torch.zeros(2, n, d, dtype=torch.float32, device=dev)      # one fill for both scatter targets
        d_side, d_content = d_both[0], d_both[1]
        rows0 = (ctx.n_users, 0)
        if ctx.pair:
            B = saved[4].numel()
            S = lib.load().mmrec_infonce_splits(B)
            V1, V2, inv_norm, ttl, idxs = ([saved[5 * s_ + j] for s_ in range(2)] for j in range(5))
            ws1 = [torch.empty(S, B, d, dtype=torch.float32, device=dev) for _ in range(2)]
            ws2 = [torch.empty(S, B, d, dtype=torch.float32, device=dev) for _ in range(2)]
            lib.call("mmrec_infonce_pair_bwd_f32", _ptr_array(V1), _ptr_array(V2), _ptr_array(inv_norm),
                     _ptr_array(ttl), d, _ptr_array(idxs), B, ctx.inv_t, _ptr_array(list(coefs)), S,
                     _ptr_array(ws1), _ptr_array(ws2), _ptr_array([d_side[r:] for r in rows0]),
                     _ptr_array([d_content[r:] for r in rows0]), lib.stream())
            rows0 = ()
        for slot, row0 in enumerate(rows0):
            V1, V2, inv_norm, ttl, idx = saved[5 * slot: 5 * slot + 5]
            B = idx.numel()
            S = lib.load().mmrec_infonce_splits(B)
            ws1 = torch.empty(S, B, d, dtype=torch.float32, device=dev)
            ws2 = torch.empty_like(ws1)
            lib.call("mmrec_infonce_bwd_f32", lib.ptr(V1), lib.ptr(V2), lib.ptr(inv_norm),
                     lib.ptr(ttl), d, lib.ptr(idx), B, ctx.inv_t, lib.ptr(coefs[slot]), S, lib.ptr(ws1),
                     lib.ptr(ws2), lib.ptr(d_side[row0:]), lib.ptr(d_content[row0:]), lib.stream())
        return d_side, d_content, None, None, None, None, None


def infonce_pair(side, content, n_users, users, pos_items, temperature, reduce=True):
    """cl_items + cl_users (reduce=False: the two losses as a [2] tensor, items first)."""
    return _InfoNCEPair.apply(side, content, n_users, users, pos_items, temperature, reduce)


class _LossHead(torch.autograd.Function):
    """bpr/B + reg_weight * reg/batch_size + cl_weight * (cl_i + cl_u) in one launch each way
    (mgcn.py:241-253, smore.py:396-411), bit-identical to the tensor expression."""

    @staticmethod
    def forward(ctx, o2, cl2, inv_b, rw, inv_bs, clw):
        o2, cl2 = _f32c(o2), _f32c(cl2)
        out = torch.empty(1, dtype=torch.float32, device=o2.device)
        ctx.c = (float(inv_b), float(rw), float(inv_bs), float(clw))
        lib.call("mmrec_loss_head_fwd_f32", lib.ptr(o2), lib.ptr(cl2), *ctx.c, lib.ptr(out), lib.stream())
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        g = _f32c(g).reshape(1)
        d_o2 = torch.empty(2, dtype=torch.float32, device=g.device)
        d_cl2 = torch.empty(2, dtype=torch.float32, device=g.device)
        lib.call("mmrec_loss_head_bwd_f32", lib.ptr(g), *ctx.c, lib.ptr(d_o2), lib.ptr(d_cl2), lib.stream())
        return d_o2, d_cl2, None, None, None, None


def loss_head(o2, cl2, batch, reg_weight, train_batch_size, cl_weight):
    """o2 = bpr_table(...) sums, cl2 = infonce_pair(..., reduce=False); float32 reciprocals as torch's
    division by a host scalar."""
    import numpy as np
    lib.require_cuda(o2, cl2)
    inv_b = float(np.float32(1.0) / np.float32(batch))
    inv_bs = float(np.float32(1.0) / np.float32(train_batch_size))
    return _LossHead.apply(o2, cl2, inv_b, reg_weight, inv_bs, cl_weight)


# ------------------------------------------------------------------------------------ spectral
class _Spectral(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, txt, w_img, w_txt, w_fus, weight_norm):
        img, txt = _f32c(img), _f32c(txt)
        w_img, w_txt, w_fus = _f32c(w_img), _f32c(w_txt), _f32c(w_fus)
        n, d = img.shape
        taps = torch.empty(3 * d, dtype=torch.float32, device=img.device)
        ic, tc, fc = torch.empty_like(img), torch.empty_like(img), torch.empty_like(img)
        lib.call("mmrec_spectral_fwd_f32", lib.ptr(img), lib.ptr(txt), n, d, lib.ptr(w_img),
                 lib.ptr(w_txt), lib.ptr(w_fus), int(weight_norm), lib.ptr(taps), lib.ptr(ic),
                 lib.ptr(tc), lib.ptr(fc), lib.stream())
        ctx.weight_norm = int(weight_norm)
        ctx.save_for_backward(img, txt, w_img, w_txt, w_fus, taps)
        return ic, tc, fc

    @staticmethod
    def backward(ctx, g_ic, g_tc, g_fc):
        img, txt, w_img, w_txt, w_fus, taps = ctx.saved_tensors
        n, d = img.shape
        g_ic, g_tc, g_fc = _f32c(g_ic), _f32c(g_tc), _f32c(g_fc)
        d_img, d_txt = torch.empty_like(img), torch.empty_like(txt)
        dh = torch.zeros(3 * d, dtype=torch.float32, device=img.device)
        dwi, dwt, dwf = torch.empty_like(w_img), torch.empty_like(w_txt), torch.empty_like(w_fus)
        lib.call("mmrec_spectral_bwd_f32", lib.ptr(img), lib.ptr(txt), n, d, lib.ptr(w_img),
                 lib.ptr(w_txt), lib.ptr(w_fus), ctx.weight_norm, lib.ptr(taps), lib.ptr(g_ic),
                 lib.ptr(g_tc), lib.ptr(g_fc), lib.ptr(d_img), lib.ptr(d_txt), lib.ptr(dh),
                 lib.ptr(dwi), lib.ptr(dwt), lib.ptr(dwf), lib.stream())
        return d_img, d_txt, dwi, dwt, dwf, None


def spectrum_convolution(img, txt, w_img, w_txt, w_fus, weight_norm=True):
    """SMORE.spectrum_convolution (smore.py:209-238) -> (image_conv, text_conv, fusion_conv)."""
    return _Spectral.apply(img, txt, w_img, w_txt, w_fus, weight_norm)


# --------------------------------------------------------------------------------- dense linear
def gemm(A, a_kcontig, B, b_kcontig, M, N, K, bias=None):
    """mmrec_gemm_tf32x3_f32: C[M,N] = op(A) op(B) (+bias), fp32-accurate on tensor cores."""
    L = lib.load()
    splits = L.mmrec_gemm_splits(M, N, K, int(a_kcontig), int(b_kcontig))
    C = torch.empty(M, N, dtype=torch.float32, device=A.device)
    ws = torch.empty(splits, M, N, dtype=torch.float32, device=A.device) if splits > 1 else None
    lib.call("mmrec_gemm_tf32x3_f32", lib.ptr(A), int(a_kcontig), lib.ptr(B), int(b_kcontig),
             lib.ptr(bias), lib.ptr(C), M, N, K, splits, lib.ptr(ws), lib.stream())
    return C


@torch.no_grad()
def score_matrix(user_rows, item_emb):
    """`user_rows @ item_emb.T` -> [Bu, n_items] on the library GEMM (3xTF32): the dense
    `full_sort_predict` of layergcn.py:186-188, freedom.py:219-222, mgcn.py:260-263, smore.py:419-422
    for callers that want the score matrix itself (the trainer uses the fused top-K instead).
    Rows of the output are 16-byte vectors, so the item count is padded to a multiple of 4 with
    zero rows and the view of the first n_items columns is returned."""
    lib.require_cuda(user_rows, item_emb)
    u, v = _f32c(user_rows), _f32c(item_emb)
    n_items, d = v.shape
    pad = (-n_items) % 4
    if pad:
        v = torch.cat([v, v.new_zeros(pad, d)], dim=0)
    out = gemm(u, True, v, True, u.shape[0], n_items + pad, d)
    return out[:, :n_items] if pad else out


class _Inject3(torch.autograd.Function):
    """item + scale * g_m for three gates (smore.py:269-272), one launch each way."""

    @staticmethod
    def forward(ctx, item, g0, g1, g2, scale):
        item, g0, g1, g2 = _f32c(item), _f32c(g0), _f32c(g1), _f32c(g2)
        outs = [torch.empty_like(item) for _ in range(3)]
        lib.call("mmrec_inject3_fwd_f32", lib.ptr(item), lib.ptr(g0), lib.ptr(g1), lib.ptr(g2), float(scale),
                 item.numel(), lib.ptr(outs[0]), lib.ptr(outs[1]), lib.ptr(outs[2]), lib.stream())
        ctx.scale = float(scale)
        return tuple(outs)

    @staticmethod
    def backward(ctx, d0, d1, d2):
        d0, d1, d2 = _f32c(d0), _f32c(d1), _f32c(d2)
        outs = [torch.empty_like(d0) for _ in range(4)]
        lib.call("mmrec_inject3_bwd_f32", lib.ptr(d0), lib.ptr(d1), lib.ptr(d2), ctx.scale, d0.numel(),
                 lib.ptr(outs[0]), lib.ptr(outs[1]), lib.ptr(outs[2]), lib.ptr(outs[3]), lib.stream())
        return outs[0], outs[1], outs[2], outs[3], None


def inject3(item, g0, g1, g2, scale):
    """(item + scale * g0, item + scale * g1, item + scale * g2) for [I, d] tensors, d % 4 == 0."""
    lib.require_cuda(item, g0, g1, g2)
    return _Inject3.apply(item, g0, g1, g2, scale)


def colsum(x):
    """x.sum(0) of a row-major [M, N] CUDA matrix (N % 4 == 0) in one launch (mmrec_colsum_f32)."""
    lib.require_cuda(x)
    x = _f32c(x)
    out = torch.empty(x.shape[1], dtype=torch.float32, device=x.device)
    nb = lib.load().mmrec_colsum_workspace_bytes(x.shape[0], x.shape[1])
    ws = torch.empty(nb // 4, dtype=torch.float32, device=x.device) if nb else None
    lib.call("mmrec_colsum_ws_f32", lib.ptr(x), x.shape[0], x.shape[1], lib.ptr(out), lib.ptr(ws), lib.stream())
    return out


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W, b):
        x, W = _f32c(x), _f32c(W)
        ctx.save_for_backward(x, W)
        ctx.has_bias = b is not None
        return gemm(x, True, W, True, x.shape[0], W.shape[0], W.shape[1], None if b is None else _f32c(b))

    @staticmethod
    def backward(ctx, dy):
        x, W = ctx.saved_tensors
        dy = _f32c(dy)
        M, K = x.shape
        N = W.shape[0]
        dx = gemm(dy, True, W, False, M, K, N) if ctx.needs_input_grad[0] else None
        dW = gemm(dy, False, x, False, N, K, M) if ctx.needs_input_grad[1] else None
        db = colsum(dy) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dW, db


class LowRankGrad:
    """Gradient of a feature table X that enters the model only through Y = X W^T + b: the rank-d
    product G = dY @ W, kept as its two factors (dY [I, d], W [d, F]) and never materialised. The
    optimizer (optim.FusedAdam) and the mirror-gradient step (trainer.py) consume it tile by tile
    inside the tcgen05 kernels of mmrec_table_adam_lowrank_f32 / mmrec_table_lowrank_sumsq_f64."""
    __slots__ = ("dY", "W")

    def __init__(self, dY, W):
        self.dY, self.W = dY, W

    def dense(self):
        """The [I, F] gradient itself (tests / fallbacks only)."""
        return gemm(self.dY, True, self.W, False, self.dY.shape[0], self.W.shape[1], self.dY.shape[1])


def table_lowrank_supported(table, W):
    return (table.is_cuda and table.dim() == 2 and W.dim() == 2 and
            bool(lib.load().mmrec_table_lowrank_supported(table.shape[0], table.shape[1], W.shape[0])))


class _TableProject(torch.autograd.Function):
    """`trs(emb.weight)` for a trainable feature table (smore.py:257-259, mgcn.py:148-150,
    freedom.py:207-210) whose [I, F] gradient is never written: backward returns dW and db, and
    leaves the table's gradient on the parameter as `_mmrec_lowrank = LowRankGrad(dY, W)`.

    `delta = (coef, dY1, W1)` evaluates the projection at the mirror-gradient point
    X' = X - coef * dY1 @ W1 (trainer.py:307-310) without touching the table:
        Y'  = X W^T - coef * dY1 (W1 W^T) + b
        dW' = dY^T X - coef * (dY^T dY1) W1
    (two d x d products and two thin GEMMs instead of a read-modify-write of the 115 MB table
    before the pass and another one after it)."""

    @staticmethod
    def forward(ctx, X, W, b, holder, delta):
        X, W = _f32c(X), _f32c(W)
        I, F = X.shape
        d = W.shape[0]
        Y = gemm(X, True, W, True, I, d, F, None if b is None else _f32c(b))
        if delta is not None:
            coef, dY1, W1 = delta
            S = gemm(W1, True, W, True, d, d, F)                    # W1 W^T
            corr = gemm(dY1, True, S, False, I, d, d)               # dY1 (W1 W^T)
            from .optim import axpy_multi
            axpy_multi([Y], [corr], coef, sign=-1.0)
        ctx.holder, ctx.delta, ctx.has_bias = holder, delta, b is not None
        ctx.save_for_backward(X, W)
        return Y

    @staticmethod
    def backward(ctx, dY):
        X, W = ctx.saved_tensors
        dY = _f32c(dY)
        I, F = X.shape
        d = W.shape[0]
        dW = gemm(dY, False, X, False, d, F, I) if ctx.needs_input_grad[1] else None
        if dW is not None and ctx.delta is not None:
            coef, dY1, W1 = ctx.delta
            T = gemm(dY, False, dY1, False, d, d, I)                # dY^T dY1
            corr = gemm(T, True, W1, False, d, F, d)                # (dY^T dY1) W1
            from .optim import axpy_multi
            axpy_multi([dW], [corr], coef, sign=-1.0)
        db = colsum(dY) if ctx.has_bias and ctx.needs_input_grad[2] else None
        param = ctx.holder.weight
        if getattr(param, "_mmrec_lowrank", None) is not None:
            raise RuntimeError("table_project: the table already carries a low-rank gradient (used twice in one "
                               "backward, or zero_grad was not called); accumulate is not supported")
        param._mmrec_lowrank = LowRankGrad(dY.detach(), W.detach())     # factors only: no autograd history
        return None, dW, db, None, None


def table_project(emb, W, b):
    """`F.linear(emb.weight, W, b)` with the table's gradient kept low-rank (see _TableProject).
    `emb` is the nn.Embedding that owns the table; a pending mirror-gradient displacement is read
    from `emb.weight._mmrec_delta`."""
    lib.require_cuda(emb.weight, W)
    return _TableProject.apply(emb.weight, W, b, emb, getattr(emb.weight, "_mmrec_delta", None))


def linear(x, W, b=None):
    """F.linear(x, W, b) for 2-D x on the 3xTF32 tensor-core GEMM (K4). There is no library
    fallback: shapes the kernel does not cover (rows are moved as 16-byte vectors, so both widths
    must be multiples of 4) raise."""
    lib.require_cuda(x, W)
    if x.dim() != 2 or W.shape[0] % 4 or W.shape[1] % 4:
        raise RuntimeError(f"mmrec_b200.linear: unsupported shape x{tuple(x.shape)} W{tuple(W.shape)} "
                           "(2-D input, in/out widths multiples of 4); there is no cuBLAS fallback")
    return _Linear.apply(x, W, b)


class Linear(torch.nn.Linear):
    """nn.Linear with the same parameters / init / state_dict keys, forward on `linear`."""

    def forward(self, x):
        return linear(x, self.weight, self.bias)


_ACT_CODE = {None: 0, "tanh": 1, "sigmoid": 2}


def _dense_workspace(K, N, dev):
    """Scratch for the per-CTA dW/db partial sums of mmrec_dense_act_bwd_f32 (caching allocator)."""
    nbytes = lib.load().mmrec_dense_act_bwd_workspace_bytes(K, N)
    return torch.empty(nbytes // 4, dtype=torch.float32, device=dev)


class _DenseAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W, b, act):
        x, W = _f32c(x), _f32c(W)
        b = None if b is None else _f32c(b)
        M, K = x.shape
        N = W.shape[0]
        y = torch.empty(M, N, dtype=torch.float32, device=x.device)
        lib.call("mmrec_dense_act_fwd_f32", lib.ptr(x), lib.ptr(W), lib.ptr(b), lib.ptr(y), M, K, N,
                 act, lib.stream())
        ctx.act, ctx.has_bias = act, b is not None
        ctx.save_for_backward(x, W, y)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, y = ctx.saved_tensors
        dy = _f32c(dy)
        M, K = x.shape
        N = W.shape[0]
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dW = torch.empty_like(W)
        db = torch.empty(N, dtype=torch.float32, device=x.device) if ctx.has_bias else None
        lib.call("mmrec_dense_act_bwd_f32", lib.ptr(dy), lib.ptr(y), lib.ptr(x), lib.ptr(W), lib.ptr(dx),
                 lib.ptr(dW), lib.ptr(db), lib.ptr(_dense_workspace(K, N, x.device)), M, K, N, ctx.act,
                 lib.stream())
        return dx, dW, db, None


class _DenseActTC(torch.autograd.Function):
    """act(F.linear(x, W, b)) over many rows on the tcgen05 GEMM (activation in its epilogue);
    backward = dz = dy * act'(y), dx = dz W, dW = dz^T x (tcgen05 as well), db = colsum(dz)."""

    @staticmethod
    def forward(ctx, x, W, b, act):
        x, W = _f32c(x), _f32c(W)
        b = None if b is None else _f32c(b)
        M, K = x.shape
        N = W.shape[0]
        y = torch.empty(M, N, dtype=torch.float32, device=x.device)
        lib.call("mmrec_linear_act_tc_f32", lib.ptr(x), lib.ptr(W), lib.ptr(b), lib.ptr(y), M, K, N, act, lib.stream())
        ctx.act, ctx.has_bias = act, b is not None
        ctx.save_for_backward(x, W, y)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, y = ctx.saved_tensors
        dy = _f32c(dy)
        M, K = x.shape
        N = W.shape[0]
        if ctx.act:
            dz = torch.empty_like(dy)
            lib.call("mmrec_act_bwd_f32", lib.ptr(dy), lib.ptr(y), dy.numel(), ctx.act, lib.ptr(dz), lib.stream())
        else:
            dz = dy
        dx = gemm(dz, True, W, False, M, K, N) if ctx.needs_input_grad[0] else None
        dW = gemm(dz, False, x, False, N, K, M) if ctx.needs_input_grad[1] else None
        db = colsum(dz) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dW, db, None


def dense_act_tc_supported(M, K, N):
    return bool(lib.load().mmrec_linear_act_tc_supported(int(M), int(K), int(N)))


def dense_act(x, W, b=None, act=None):
    """act(F.linear(x, W, b)) for the d x d side-network layers in ONE launch (forward) and one
    launch + a partial-sum reduce (backward: dX, dW, db and the activation derivative together);
    3xTF32 tensor-core products (fp32-class accuracy). Other shapes: `linear` + torch activation."""
    if x.dim() == 2 and x.is_cuda and W.shape[0] == 128 and dense_act_tc_supported(x.shape[0], W.shape[1], W.shape[0]):
        return _DenseActTC.apply(x, W, b, _ACT_CODE[act])       # many rows x (128 x 128): tcgen05
    if x.dim() == 2 and x.is_cuda and lib.load().mmrec_dense_act_supported(W.shape[1], W.shape[0]):
        return _DenseAct.apply(x, W, b, _ACT_CODE[act])
    y = linear(x, W, b)
    return y if act is None else (torch.tanh(y) if act == "tanh" else torch.sigmoid(y))


class _DenseActBatch(torch.autograd.Function):
    """n independent act(F.linear(x_i, W_i, b_i)) of one shape in one launch each way.
    apply(act, n, x_0.., W_0.., b_0..) -> n outputs."""

    @staticmethod
    def forward(ctx, act, n, *t):
        xs = [_f32c(v) for v in t[:n]]
        Ws = [_f32c(v) for v in t[n:2 * n]]
        bs = [None if v is None else _f32c(v) for v in t[2 * n:3 * n]]
        M, K = xs[0].shape
        N = Ws[0].shape[0]
        ys = [torch.empty(M, N, dtype=torch.float32, device=xs[0].device) for _ in range(n)]
        lib.call("mmrec_dense_act_batch_fwd_f32", _ptr_array(xs), _ptr_array(Ws), _ptr_array(bs), _ptr_array(ys),
                 n, M, K, N, act, lib.stream())
        ctx.act, ctx.n, ctx.has_bias = act, n, [b is not None for b in bs]
        ctx.save_for_backward(*xs, *Ws, *ys)
        return tuple(ys)

    @staticmethod
    def backward(ctx, *dys):
        n = ctx.n
        t = ctx.saved_tensors
        xs, Ws, ys = t[:n], t[n:2 * n], t[2 * n:3 * n]
        M, K = xs[0].shape
        N = Ws[0].shape[0]
        dev = xs[0].device
        dys = [torch.zeros(M, N, dtype=torch.float32, device=dev) if g is None else _f32c(g) for g in dys]
        dxs = [torch.empty_like(x) if ctx.needs_input_grad[2 + i] else None for i, x in enumerate(xs)]
        dWs = [torch.empty_like(W) for W in Ws]
        dbs = [torch.empty(N, dtype=torch.float32, device=dev) if hb else None for hb in ctx.has_bias]
        ws = torch.empty(n * (lib.load().mmrec_dense_act_bwd_workspace_bytes(K, N) // 4), dtype=torch.float32,
                         device=dev)
        lib.call("mmrec_dense_act_batch_bwd_f32", _ptr_array(dys), _ptr_array(ys), _ptr_array(xs), _ptr_array(Ws),
                 _ptr_array(dxs), _ptr_array(dWs), _ptr_array(dbs), lib.ptr(ws), n, M, K, N, ctx.act, lib.stream())
        return (None, None, *dxs, *dWs, *dbs)


def dense_stack_batch(stacks, xs):
    """[stack_i(x_i)] for DenseStacks that are each one Linear(d, d) (+ Tanh / Sigmoid) of the same
    shape, as one batched launch (SMORE / MGCN modality gates); anything else runs stack by stack."""
    def one_layer(st):
        mods = list(st)
        if not mods or not isinstance(mods[0], torch.nn.Linear) or len(mods) > 2:
            return None
        act = None
        if len(mods) == 2:
            act = "tanh" if isinstance(mods[1], torch.nn.Tanh) else "sigmoid" if isinstance(mods[1], torch.nn.Sigmoid) else 0
            if act == 0:
                return None
        return mods[0], act
    info = [one_layer(st) for st in stacks]
    if all(i is not None for i in info) and all(x.dim() == 2 and x.is_cuda for x in xs) and all(
            i[0].weight.shape[0] == 128 and dense_act_tc_supported(x.shape[0], i[0].weight.shape[1], 128)
            for i, x in zip(info, xs)):
        return [dense_act(x, i[0].weight, i[0].bias, i[1]) for i, x in zip(info, xs)]
    ok = (1 < len(stacks) <= 4 and all(i is not None for i in info) and len({i[1] for i in info}) == 1
          and len({tuple(i[0].weight.shape) for i in info}) == 1 and len({tuple(x.shape) for x in xs}) == 1
          and all(x.dim() == 2 and x.is_cuda for x in xs)
          and lib.load().mmrec_dense_act_supported(info[0][0].weight.shape[1], info[0][0].weight.shape[0])
          and len({i[0].bias is None for i in info}) == 1)
    if not ok:
        return [st(x) for st, x in zip(stacks, xs)]
    lins = [i[0] for i in info]
    return list(_DenseActBatch.apply(_ACT_CODE[info[0][1]], len(xs), *xs, *[l.weight for l in lins],
                                     *[l.bias for l in lins]))


class DenseStack(torch.nn.Sequential):
    """nn.Sequential of Linear / Tanh / Sigmoid with the reference's module indices (so the
    state_dict keys `gate_v.0.weight`, `query_v.2.weight` ... are unchanged) whose forward fuses
    every Linear with the activation that follows it."""

    def forward(self, x):
        mods = list(self)
        i = 0
        while i < len(mods):
            m = mods[i]
            nxt = mods[i + 1] if i + 1 < len(mods) else None
            if isinstance(m, torch.nn.Linear):
                act = "tanh" if isinstance(nxt, torch.nn.Tanh) else "sigmoid" if isinstance(nxt, torch.nn.Sigmoid) else None
                x = dense_act(x, m.weight, m.bias, act)
                i += 2 if act else 1
            else:
                x = m(x)
                i += 1
        return x


# ------------------------------------------------------------------- SMORE side network (fused)
_ptr_array = lib.ptr_array


class _SmoreSide(torch.autograd.Function):
    """smore.py:321-341 in one forward / one backward launch (mmrec_smore_side_*_f32).
    apply(F, V, T, C, masks, drop, W0, b0, ..., W6, b6) -> (all_embeds, side_embeds).
    `drop` = (p, seed, counter) or None: the dropout multipliers are generated inside both kernels
    (lib.Dropout) instead of being read from `masks`."""

    @staticmethod
    def forward(ctx, F, V, T, C_, masks, drop, *wb):
        F, V, T, C_ = _f32c(F), _f32c(V), _f32c(T), _f32c(C_)
        Ws = [_f32c(w) for w in wb[0::2]]
        bs = [None if b is None else _f32c(b) for b in wb[1::2]]
        masks = None if masks is None else _f32c(masks)
        n, d = F.shape
        # nothing is kept for a backward that cannot come (evaluation forward under no_grad)
        need_bwd = any(ctx.needs_input_grad)
        saved = torch.empty(7, n, d, dtype=torch.float32, device=F.device) if need_bwd else None
        side, all_e = torch.empty_like(F), torch.empty_like(F)
        if drop is not None and masks is not None:
            raise RuntimeError("smore_side: pass either mask tensors or an in-kernel dropout spec")
        tc_ws = lib.load().mmrec_smore_side_fwd_tc_workspace_bytes(n, d) if masks is None else 0
        if tc_ws:
            # tcgen05 forward (d = 64): weights pre-split into UMMA images in a 224 KB workspace
            ws = torch.empty(tc_ws + 1024, dtype=torch.uint8, device=F.device)
            ws_ptr = (ws.data_ptr() + 1023) & ~1023
            lib.call("mmrec_smore_side_fwd_tc_f32", lib.ptr(F), lib.ptr(V), lib.ptr(T), lib.ptr(C_),
                     _ptr_array(Ws), _ptr_array(bs), ctypes.byref(lib.Dropout.make(*drop)) if drop is not None else None,
                     lib.ptr(saved), lib.ptr(side), lib.ptr(all_e), n, d, ws_ptr, lib.stream())
        elif drop is not None:
            lib.call("mmrec_smore_side_fwd_drop_f32", lib.ptr(F), lib.ptr(V), lib.ptr(T), lib.ptr(C_),
                     _ptr_array(Ws), _ptr_array(bs), ctypes.byref(lib.Dropout.make(*drop)), lib.ptr(saved), lib.ptr(side),
                     lib.ptr(all_e), n, d, lib.stream())
        else:
            lib.call("mmrec_smore_side_fwd_f32", lib.ptr(F), lib.ptr(V), lib.ptr(T), lib.ptr(C_),
                     _ptr_array(Ws), _ptr_array(bs), lib.ptr(masks), lib.ptr(saved), lib.ptr(side),
                     lib.ptr(all_e), n, d, lib.stream())
        ctx.drop = drop
        ctx.has_mask = masks is not None
        ctx.has_bias = [b is not None for b in bs]
        if need_bwd:
            ctx.save_for_backward(F, V, T, C_, saved, *Ws, *[b for b in bs if b is not None],
                                  *([masks] if masks is not None else []))
        return all_e, side

    @staticmethod
    def backward(ctx, g_all, g_side):
        t = ctx.saved_tensors
        F, V, T, C_, saved = t[:5]
        Ws = list(t[5:12])
        rest = list(t[12:])
        bs = [rest.pop(0) if hb else None for hb in ctx.has_bias]
        masks = rest.pop(0) if ctx.has_mask else None
        n, d = F.shape
        g_all = None if g_all is None else _f32c(g_all)
        g_side = None if g_side is None else _f32c(g_side)
        dF, dV, dT, dC = (torch.empty_like(F) for _ in range(4))
        dWs = [torch.empty_like(w) for w in Ws]
        dbs = [None if b is None else torch.empty_like(b) for b in bs]
        ws = torch.empty(lib.load().mmrec_smore_side_bwd_workspace_bytes(n, d) // 4, dtype=torch.float32,
                         device=F.device)
        if ctx.drop is not None:
            lib.call("mmrec_smore_side_bwd_drop_f32", lib.ptr(g_all), lib.ptr(g_side), lib.ptr(F), lib.ptr(V),
                     lib.ptr(T), lib.ptr(C_), _ptr_array(Ws), _ptr_array(bs), ctypes.byref(lib.Dropout.make(*ctx.drop)),
                     lib.ptr(saved), lib.ptr(dF), lib.ptr(dV), lib.ptr(dT), lib.ptr(dC), _ptr_array(dWs),
                     _ptr_array(dbs), lib.ptr(ws), n, d, lib.stream())
        else:
            lib.call("mmrec_smore_side_bwd_f32", lib.ptr(g_all), lib.ptr(g_side), lib.ptr(F), lib.ptr(V),
                     lib.ptr(T), lib.ptr(C_), _ptr_array(Ws), _ptr_array(bs), lib.ptr(masks), lib.ptr(saved),
                     lib.ptr(dF), lib.ptr(dV), lib.ptr(dT), lib.ptr(dC), _ptr_array(dWs), _ptr_array(dbs),
                     lib.ptr(ws), n, d, lib.stream())
        grads = []
        for dw, db in zip(dWs, dbs):
            grads += [dw, db]
        return (dF, dV, dT, dC, None, None, *grads)


def smore_side_supported(d):
    """Widths the models route through the fused kernel. The library also instantiates d = 128
    (tested), but there the fp32-FMA kernel holds one 255-register CTA per SM and is slower than
    the unfused path (Clothing, d = 128: 20.6 vs 18.5 ms/step): that width waits for the
    tensor-core version."""
    import os
    widths = (32, 64, 128) if os.environ.get("MMREC_SIDE128", "0") == "1" else (32, 64)
    return int(d) in widths and bool(lib.load().mmrec_smore_side_supported(int(d)))


def dropout_mask(planes, n, d, drop, device=None):
    """The [planes, n, d] multipliers (0 or 1/(1-p)) an in-kernel dropout spec `drop` = (p, seed,
    counter) generates (mmrec_dropout_mask_f32) -- for tests and diagnostics; the kernels never
    materialise them."""
    dev = drop[2].device if drop[2] is not None else (device or torch.device("cuda", torch.cuda.current_device()))
    out = torch.empty(planes, n, d, dtype=torch.float32, device=dev)
    lib.call("mmrec_dropout_mask_f32", lib.ptr(out), planes, n, d, ctypes.byref(lib.Dropout.make(*drop)), lib.stream())
    return out


def smore_side(fusion, image, text, content, layers, masks=None, drop=None):
    """Fused modality-aware preference module. `layers` = the seven nn.Linear modules in the
    order query_v.0, query_v.2, query_t.0, query_t.2, gate_image_prefer.0, gate_text_prefer.0,
    gate_fusion_prefer.0; masks = [3, n, d] dropout multipliers or None; drop = (p, seed, counter[,
    row_ids, n_total]) for dropout generated inside the kernels (no mask tensor; see lib.Dropout --
    with row_ids the call runs on gathered rows and drops what the dense call would drop there).
    Returns (content + side, side)."""
    lib.require_cuda(fusion, image, text, content)
    wb = []
    for m in layers:
        wb += [m.weight, m.bias]
    return _SmoreSide.apply(fusion, image, text, content, masks, drop, *wb)


# ------------------------------------------- batch rows of node tables (row-local modules in training)
class _GatherBatchRows(torch.autograd.Function):
    """apply(users, pos, neg, n_users, *tables) -> (row_ids, *compact tables): rows users | n_users + pos |
    n_users + neg of every [N, d] table as [3 B, d] tables (mmrec_gather_batch_rows_f32). Backward: the
    compact gradients scatter-added into dense zero tables (mmrec_scatter_batch_rows_add_f32)."""

    @staticmethod
    def forward(ctx, users, pos, neg, n_users, *tables):
        tables = [_f32c(t) for t in tables]
        lib.require_cuda(users, pos, neg, *tables)
        if not (users.dtype == pos.dtype == neg.dtype == torch.int64) or not (users.numel() == pos.numel() == neg.numel()):
            raise RuntimeError("gather_batch_rows: users / pos / neg must be int64 tensors of one length")
        B, (N, d) = users.numel(), tables[0].shape
        if any(t.shape != (N, d) for t in tables) or not 1 <= len(tables) <= 4:
            raise RuntimeError("gather_batch_rows: 1..4 tables of one shape")
        if CHECK_IDS:
            _check_ids(users, n_users, "batch users")
            _check_ids(pos, N - n_users, "batch pos items")
            _check_ids(neg, N - n_users, "batch neg items")
        idx = torch.empty(3 * B, dtype=torch.int64, device=users.device)
        outs = [torch.empty(3 * B, d, dtype=torch.float32, device=users.device) for _ in tables]
        lib.call("mmrec_gather_batch_rows_f32", _ptr_array(tables), len(tables), lib.ptr(users.contiguous()),
                 lib.ptr(pos.contiguous()), lib.ptr(neg.contiguous()), B, int(n_users), d, _ptr_array(outs), lib.ptr(idx),
                 lib.stream())
        ctx.shape, ctx.n_tables = (N, d), len(tables)
        ctx.save_for_backward(idx)
        ctx.mark_non_differentiable(idx)
        return (idx, *outs)

    @staticmethod
    def backward(ctx, _d_idx, *d_outs):
        (idx,) = ctx.saved_tensors
        N, d = ctx.shape
        dense = torch.zeros(ctx.n_tables, N, d, dtype=torch.float32, device=idx.device)      # one fill for all tables
        srcs = [None if g is None else _f32c(g) for g in d_outs]
        if any(g is not None for g in srcs):
            lib.call("mmrec_scatter_batch_rows_add_f32", _ptr_array(srcs), ctx.n_tables, lib.ptr(idx), idx.numel(), d,
                     _ptr_array([dense[t] for t in range(ctx.n_tables)]), lib.stream())
        return (None, None, None, None, *[dense[t] if ctx.needs_input_grad[4 + t] else None for t in range(ctx.n_tables)])


def gather_batch_rows(tables, users, pos, neg, n_users):
    """(row_ids int64 [3 B], [table[row_ids] for table in tables]) with row_ids = users | n_users + pos |
    n_users + neg -- the rows of a training batch, for modules that are row-local (see csrc/batch_rows.cu)."""
    out = _GatherBatchRows.apply(users, pos, neg, int(n_users), *tables)
    return out[0], list(out[1:])


class _GatherBatchViews(torch.autograd.Function):
    """apply(R, users, pos, neg, content, *item_tables) -> (row_ids, content_c, *views_c): the batch rows of
    the modality views cat([R x', x']) without forming them -- user rows are rows of R times x' (only for the
    users of the batch), item rows are copied (mmrec_gather_batch_views_f32). Backward: scatter-add along the
    same non-zeros into dense zero tables."""

    @staticmethod
    def forward(ctx, R, users, pos, neg, content, *tables):
        tables = [_f32c(t) for t in tables]
        content = _f32c(content)
        lib.require_cuda(users, pos, neg, content, *tables)
        if not (users.dtype == pos.dtype == neg.dtype == torch.int64) or not (users.numel() == pos.numel() == neg.numel()):
            raise RuntimeError("gather_batch_views: users / pos / neg must be int64 tensors of one length")
        B, (I, d) = users.numel(), tables[0].shape
        if any(t.shape != (I, d) for t in tables) or not 1 <= len(tables) <= 3 or I != R.n_cols or \
                content.shape != (R.n_rows + I, d):
            raise RuntimeError("gather_batch_views: 1..3 item tables [I, d] and a content table [U + I, d]")
        if CHECK_IDS:
            _check_ids(users, R.n_rows, "batch users")
            _check_ids(pos, I, "batch pos items")
            _check_ids(neg, I, "batch neg items")
        users, pos, neg = users.contiguous(), pos.contiguous(), neg.contiguous()
        dev = users.device
        idx = torch.empty(3 * B, dtype=torch.int64, device=dev)
        content_c = torch.empty(3 * B, d, dtype=torch.float32, device=dev)
        outs = [torch.empty(3 * B, d, dtype=torch.float32, device=dev) for _ in tables]
        lib.call("mmrec_gather_batch_views_f32", lib.ptr(R.row_ptr), lib.ptr(R.col_idx), lib.ptr(R.vals), R.col_offset,
                 _ptr_array(tables), len(tables), lib.ptr(content), lib.ptr(users), lib.ptr(pos), lib.ptr(neg), B,
                 R.n_rows, d, _ptr_array(outs), lib.ptr(content_c), lib.ptr(idx), lib.stream())
        ctx.R, ctx.dims, ctx.n_tables = R, (I, d), len(tables)
        ctx.save_for_backward(users, pos, neg)
        ctx.mark_non_differentiable(idx)
        return (idx, content_c, *outs)

    @staticmethod
    def backward(ctx, _d_idx, d_content, *d_outs):
        users, pos, neg = ctx.saved_tensors
        R, (I, d), n = ctx.R, ctx.dims, ctx.n_tables
        dev = users.device
        d_tables = torch.zeros(n, I, d, dtype=torch.float32, device=dev)
        d_dense_content = torch.zeros(R.n_rows + I, d, dtype=torch.float32, device=dev)
        srcs = [None if g is None else _f32c(g) for g in d_outs]
        dc = None if d_content is None else _f32c(d_content)
        lib.call("mmrec_scatter_batch_views_add_f32", lib.ptr(R.row_ptr), lib.ptr(R.col_idx), lib.ptr(R.vals),
                 R.col_offset, _ptr_array(srcs), n, lib.ptr(dc), lib.ptr(users), lib.ptr(pos), lib.ptr(neg),
                 users.numel(), R.n_rows, d, _ptr_array([d_tables[t] for t in range(n)]),
                 lib.ptr(d_dense_content) if dc is not None else None, lib.stream())
        return (None, None, None, None, d_dense_content if ctx.needs_input_grad[4] else None,
                *[d_tables[t] if ctx.needs_input_grad[5 + t] else None for t in range(n)])


def gather_batch_views(R, item_tables, content, users, pos, neg):
    """(row_ids [3 B], content[row_ids], [cat([R x, x])[row_ids] for x in item_tables]) for the rows users |
    n_users + pos | n_users + neg of a training batch, without the user-side SpMM over all users."""
    out = _GatherBatchViews.apply(R, users, pos, neg, content, *item_tables)
    return out[0], out[1], list(out[2:])


# ------------------------------------------- SMORE preference module, row part (wide embeddings)
class _SmoreCombine(torch.autograd.Function):
    """smore.py:321-341 after the seven Linear layers: apply(zv, zt, V, T, F, C, gi, gt, gf, masks)
    -> (content + side, side); see mmrec_smore_combine_*_f32."""

    @staticmethod
    def forward(ctx, zv, zt, V, T, F, C_, gi, gt, gf, masks, drop=None):
        zv, zt, V, T, F, C_, gi, gt, gf = (_f32c(t) for t in (zv, zt, V, T, F, C_, gi, gt, gf))
        masks = None if masks is None else _f32c(masks)
        n, d = F.shape
        side, all_e = torch.empty_like(F), torch.empty_like(F)
        if drop is not None and masks is not None:
            raise RuntimeError("smore_combine: pass either mask tensors or an in-kernel dropout spec")
        lib.call("mmrec_smore_combine_fwd_f32" if drop is None else "mmrec_smore_combine_fwd_drop_f32",
                 lib.ptr(zv), lib.ptr(zt), lib.ptr(V), lib.ptr(T), lib.ptr(F), lib.ptr(C_), lib.ptr(gi), lib.ptr(gt),
                 lib.ptr(gf), lib.ptr(masks) if drop is None else ctypes.byref(lib.Dropout.make(*drop)), n, d,
                 lib.ptr(side), lib.ptr(all_e), lib.stream())
        ctx.drop = drop
        ctx.has_mask = masks is not None
        ctx.save_for_backward(zv, zt, V, T, F, gi, gt, gf, *([masks] if masks is not None else []))
        return all_e, side

    @staticmethod
    def backward(ctx, g_all, g_side):
        t = ctx.saved_tensors
        zv, zt, V, T, F, gi, gt, gf = t[:8]
        masks = t[8] if ctx.has_mask else None
        n, d = F.shape
        g_all = None if g_all is None else _f32c(g_all)
        g_side = None if g_side is None else _f32c(g_side)
        outs = [torch.empty_like(F) for _ in range(9)]          # dzv dzt dV dT dF dC dgi dgt dgf
        lib.call("mmrec_smore_combine_bwd_f32" if ctx.drop is None else "mmrec_smore_combine_bwd_drop_f32",
                 lib.ptr(g_all), lib.ptr(g_side), lib.ptr(zv), lib.ptr(zt), lib.ptr(V), lib.ptr(T), lib.ptr(F),
                 lib.ptr(gi), lib.ptr(gt), lib.ptr(gf),
                 lib.ptr(masks) if ctx.drop is None else ctypes.byref(lib.Dropout.make(*ctx.drop)), n, d,
                 *[lib.ptr(o) for o in outs], lib.stream())
        dzv, dzt, dV, dT, dF, dC, dgi, dgt, dgf = outs
        return dzv, dzt, dV, dT, dF, dC, dgi, dgt, dgf, None, None


def smore_combine_supported(d):
    return bool(lib.load().mmrec_smore_combine_supported(int(d)))


def smore_combine(zv, zt, image, text, fusion, content, gi, gt, gf, masks=None, drop=None):
    """Row part of SMORE's preference module: (content + side, side) from the pre-softmax query
    outputs, the three views, the content embeddings and the three sigmoid gates (+ dropout: mask
    tensors, or drop = (p, seed, counter) generated in the kernels)."""
    lib.require_cuda(zv, zt, image, text, fusion, content, gi, gt, gf)
    return _SmoreCombine.apply(zv, zt, image, text, fusion, content, gi, gt, gf, masks, drop)


# ------------------------------------------------------------------- MGCN attention fuser (fused)
class _MgcnFuse(torch.autograd.Function):
    """mgcn.py:188-205 after the d x d layers: apply(Hi, Ht, w2, Ei, Et, Pi, Pt, C) -> (all, side)."""

    @staticmethod
    def forward(ctx, Hi, Ht, w2, Ei, Et, Pi, Pt, C_):
        Hi, Ht, Ei, Et, Pi, Pt, C_ = (_f32c(t) for t in (Hi, Ht, Ei, Et, Pi, Pt, C_))
        w2c = _f32c(w2).reshape(-1)
        n, d = Ei.shape
        att = torch.empty(n, 2, dtype=torch.float32, device=Ei.device)
        side, all_e = torch.empty_like(Ei), torch.empty_like(Ei)
        lib.call("mmrec_mgcn_fuse_fwd_f32", lib.ptr(Hi), lib.ptr(Ht), lib.ptr(w2c), lib.ptr(Ei), lib.ptr(Et),
                 lib.ptr(Pi), lib.ptr(Pt), lib.ptr(C_), n, d, lib.ptr(att), lib.ptr(side), lib.ptr(all_e),
                 lib.stream())
        ctx.w2_shape = tuple(w2.shape)
        ctx.save_for_backward(Hi, Ht, w2c, Ei, Et, Pi, Pt, att)
        return all_e, side

    @staticmethod
    def backward(ctx, g_all, g_side):
        Hi, Ht, w2c, Ei, Et, Pi, Pt, att = ctx.saved_tensors
        n, d = Ei.shape
        g_all = None if g_all is None else _f32c(g_all)
        g_side = None if g_side is None else _f32c(g_side)
        dHi, dHt, dEi, dEt, dPi, dPt, dC = (torch.empty_like(Ei) for _ in range(7))
        nb = lib.load().mmrec_mgcn_fuse_bwd_blocks(n, d)
        part = torch.empty(nb, d, dtype=torch.float32, device=Ei.device)
        dw2 = torch.empty(d, dtype=torch.float32, device=Ei.device)
        lib.call("mmrec_mgcn_fuse_bwd_f32", lib.ptr(g_all), lib.ptr(g_side), lib.ptr(Hi), lib.ptr(Ht), lib.ptr(w2c),
                 lib.ptr(Ei), lib.ptr(Et), lib.ptr(Pi), lib.ptr(Pt), lib.ptr(att), n, d, lib.ptr(dHi), lib.ptr(dHt),
                 lib.ptr(dEi), lib.ptr(dEt), lib.ptr(dPi), lib.ptr(dPt), lib.ptr(dC), lib.ptr(part), lib.ptr(dw2),
                 lib.stream())
        return dHi, dHt, dw2.reshape(ctx.w2_shape), dEi, dEt, dPi, dPt, dC


def mgcn_fuse_supported(d):
    return bool(lib.load().mmrec_mgcn_fuse_supported(int(d)))


def mgcn_fuse(h_img, h_txt, w2, image_embeds, text_embeds, p_img, p_txt, content):
    """MGCN's attention fuser (mgcn.py:188-205) -> (content + side, side); h_m =
    tanh(query_common.0(m_embeds)), w2 = query_common.2.weight, p_m = sigmoid(gate_m_prefer.0(content))."""
    lib.require_cuda(h_img, h_txt, w2, image_embeds, text_embeds, p_img, p_txt, content)
    return _MgcnFuse.apply(h_img, h_txt, w2, image_embeds, text_embeds, p_img, p_txt, content)


def dense_act_batch(xs, linears, act):
    """[act(F.linear(x_i, W_i, b_i))] for nn.Linear modules of one shape in one launch each way (the
    same module may appear more than once: autograd sums its gradients)."""
    lins = list(linears)
    return list(_DenseActBatch.apply(_ACT_CODE[act], len(xs), *xs, *[l.weight for l in lins],
                                     *[l.bias for l in lins]))


# ------------------------------------------------------------------------------ item kNN graphs
@torch.no_grad()
def knn_graph(feat, k, mode, neighbors=None):
    """(rows, cols, weights) of the cosine top-k item graph on the device (SURVEY 8a row a5).
    mode 'sym'     : build_sim + build_knn_normalized_graph(sparse, 'sym') + get_sparse_laplacian
                     (utils/utils.py:134-184) -- MGCN / SMORE;
    mode 'freedom' : FREEDOM.get_knn_adj_mat + compute_normalized_laplacian (freedom.py:79-100).
    Row normalisation, the [I, I] cosine GEMM (3xTF32), the per-row top-k (ties -> lower id) and
    the edge weights all run in the library; rows / cols come back int64 like the reference's
    index tensors, in (row, rank) order. `neighbors` ([n, k] integer tensor) replaces the top-k
    selection by given neighbour lists -- parity tests pin the edge set to the reference's, whose
    float32 near-ties depend on the BLAS build -- the similarities and weights are still computed
    here."""
    feat = _f32c(feat)
    lib.require_cuda(feat)
    n, F = feat.shape
    dev = feat.device
    if F % 4:                                   # GEMM rows are 16-byte vectors: zero-pad the features
        feat = torch.nn.functional.pad(feat, (0, 4 - F % 4))
        F = feat.shape[1]
    n_pad = (n + 3) // 4 * 4                    # ... and so are the rows of the cosine matrix
    nrm = torch.zeros(n_pad, F, dtype=torch.float32, device=dev)
    lib.call("mmrec_row_normalize_f32", lib.ptr(feat), n, F, lib.ptr(nrm), lib.stream())
    sim = gemm(nrm, True, nrm, True, n_pad, n_pad, F)
    if neighbors is None:
        val = torch.empty(n, k, dtype=torch.float32, device=dev)
        idx = torch.empty(n, k, dtype=torch.int32, device=dev)
        lib.call("mmrec_row_topk_f32", lib.ptr(sim), n, n, n_pad, k, lib.ptr(val), lib.ptr(idx), lib.stream())
    else:
        idx = torch.as_tensor(neighbors).to(dev).to(torch.int32).contiguous()
        if tuple(idx.shape) != (n, k):
            raise RuntimeError(f"knn_graph: neighbors must be [{n}, {k}], got {tuple(idx.shape)}")
        val = sim[:n].gather(1, idx.to(torch.int64)).contiguous()
    del sim
    w = torch.empty(n, k, dtype=torch.float32, device=dev)
    dis = torch.empty(n, dtype=torch.float32, device=dev)
    lib.call("mmrec_knn_weights_f32", lib.ptr(idx), lib.ptr(val), n, k, {"sym": 0, "freedom": 1}[mode],
             lib.ptr(dis), lib.ptr(w), lib.stream())
    rows = torch.arange(n, device=dev).unsqueeze(1).expand(-1, k).flatten()
    return rows, idx.flatten().to(torch.int64), w.flatten()


# -------------------------------------------------------------------------------- score + top-K
def choose_splits(n_users, n_items):
    """Item-range splits so that (user tiles x splits) is close to one wave of 148 CTAs (the
    tensor-core kernel runs one 128-user CTA per SM); never fewer than 256 items per split."""
    tiles = (n_users + 127) // 128
    want = max(1, 148 // tiles)
    return int(max(1, min(want, 32, (n_items + 255) // 256)))


@torch.no_grad()
def score_mask_topk(user_emb, users, item_emb, k, mask_rowptr=None, mask_cols=None, item_offset=0,
                    n_splits=None, return_scores=False, merge=True, simt=False):
    """Fused `u @ item_e.T` + `scores[mask] = -1e10` + top-K (smore.py:421 / trainer.py:522-526).
    Returns ids int64 [n_users, k] (+ scores). With merge=False returns the per-split partial
    lists (vals [S, n, k], ids int32 [S, n, k]) for a cross-rank merge."""
    user_emb, item_emb = _f32c(user_emb), _f32c(item_emb)
    lib.require_cuda(user_emb, item_emb, users)
    n, n_items, d = users.numel(), item_emb.shape[0], item_emb.shape[1]
    _check_ids(users, user_emb.shape[0], "score_mask_topk users")
    dev = user_emb.device
    S = n_splits or choose_splits(n, n_items)
    ws_val = torch.empty(S, n, k, dtype=torch.float32, device=dev)
    ws_idx = torch.empty(S, n, k, dtype=torch.int32, device=dev)
    out_val = torch.empty(n, k, dtype=torch.float32, device=dev)
    out_idx = torch.empty(n, k, dtype=torch.int64, device=dev)
    lib.call("mmrec_score_mask_topk_simt_f32" if simt else "mmrec_score_mask_topk_f32",
             lib.ptr(user_emb), lib.ptr(users), n, lib.ptr(item_emb),
             n_items, item_offset, d, lib.ptr(mask_rowptr), lib.ptr(mask_cols), k, S,
             lib.ptr(ws_val), lib.ptr(ws_idx), lib.ptr(out_val), lib.ptr(out_idx), lib.stream())
    if not merge:
        return ws_val, ws_idx
    return (out_idx, out_val) if return_scores else out_idx


@torch.no_grad()
def score_mask_topk_rows(user_emb, users, item_emb, k, mask_rowptr, mask_cols, item_offset=0, n_splits=None,
                         return_scores=False):
    """score_mask_topk with the mask as a CSR over the rows of `user_emb` (mmrec_score_mask_topk_rows_f32):
    the mask of entry b is row users[b] of (mask_rowptr int32 [user_emb.shape[0] + 1], mask_cols int32,
    ascending global item ids inside each row), e.g. a rank's training CSR; no per-batch mask is built."""
    user_emb, item_emb = _f32c(user_emb), _f32c(item_emb)
    lib.require_cuda(user_emb, item_emb, users, mask_rowptr, mask_cols)
    if mask_rowptr.dtype != torch.int32 or mask_cols.dtype != torch.int32:
        raise RuntimeError("score_mask_topk_rows: the mask CSR must be int32")
    if mask_rowptr.numel() != user_emb.shape[0] + 1:
        raise RuntimeError(f"score_mask_topk_rows: mask_rowptr has {mask_rowptr.numel()} entries, the user table "
                           f"{user_emb.shape[0]} rows")
    n, n_items, d = users.numel(), item_emb.shape[0], item_emb.shape[1]
    _check_ids(users, user_emb.shape[0], "score_mask_topk_rows users")
    dev = user_emb.device
    S = n_splits or choose_splits(n, n_items)
    ws_val = torch.empty(S, n, k, dtype=torch.float32, device=dev)
    ws_idx = torch.empty(S, n, k, dtype=torch.int32, device=dev)
    out_val = torch.empty(n, k, dtype=torch.float32, device=dev)
    out_idx = torch.empty(n, k, dtype=torch.int64, device=dev)
    lib.call("mmrec_score_mask_topk_rows_f32", lib.ptr(user_emb), lib.ptr(users.contiguous()), n, lib.ptr(item_emb),
             n_items, item_offset, d, lib.ptr(mask_rowptr.contiguous()), lib.ptr(mask_cols.contiguous()), k, S,
             lib.ptr(ws_val), lib.ptr(ws_idx), lib.ptr(out_val), lib.ptr(out_idx), lib.stream())
    return (out_idx, out_val) if return_scores else out_idx


@torch.no_grad()
def topk_merge(vals, idx):
    """K-way merge of [L, n, k] descending lists (ties -> lower id)."""
    L, n, k = vals.shape
    out_val = torch.empty(n, k, dtype=torch.float32, device=vals.device)
    out_idx = torch.empty(n, k, dtype=torch.int64, device=vals.device)
    lib.call("mmrec_topk_merge", lib.ptr(vals.contiguous()), lib.ptr(idx.contiguous()), L, n, k,
             lib.ptr(out_val), lib.ptr(out_idx), lib.stream())
    return out_idx, out_val


# ------------------------------------------------------------------------------ top-K metrics
_METRIC_ROWS = {"recall": 0, "recall2": 1, "precision": 2, "ndcg": 3, "map": 4}
_METRIC_TABLES = {}


@torch.no_grad()
def topk_metric_sums(topk, gt_rowptr, gt_items, return_hits=False):
    """mmrec_topk_metrics_f64: per-rank sums over users of recall / cumulative hits / precision /
    ndcg / map (float64 [5, k] on the device) for `topk` int64 [n, k] against the ascending
    ground-truth CSR. Replaces TopKEvaluator's hit-matrix loop + numpy reductions."""
    import numpy as np
    lib.require_cuda(topk, gt_rowptr, gt_items)
    topk = topk.contiguous()
    n, k = topk.shape
    dev = topk.device
    if (k, dev) not in _METRIC_TABLES:         # constants: built once, outside any graph capture
        disc_np = 1.0 / np.log2(np.arange(1, k + 1, dtype=np.float64) + 1)     # metrics.py:35-64
        _METRIC_TABLES[(k, dev)] = (torch.from_numpy(disc_np).to(dev), torch.from_numpy(np.cumsum(disc_np)).to(dev))
    disc, idcg = _METRIC_TABLES[(k, dev)]
    sums = torch.empty(5, k, dtype=torch.float64, device=dev)
    hits = torch.empty(n, k, dtype=torch.uint8, device=dev) if return_hits else None
    ws = torch.empty(lib.load().mmrec_topk_metrics_workspace_bytes(n), dtype=torch.uint8, device=dev)
    lib.call("mmrec_topk_metrics_f64", lib.ptr(topk), n, k, lib.ptr(gt_rowptr), lib.ptr(gt_items),
             lib.ptr(disc), lib.ptr(idcg), lib.ptr(hits), lib.ptr(sums), lib.ptr(ws), lib.stream())
    return (sums, hits) if return_hits else sums
