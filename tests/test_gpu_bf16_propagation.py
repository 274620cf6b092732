"""B200 tests of the bf16 propagation mode of the user-sharded LightGCN: the bf16-operand SpMM
(mmrec_spmm_csr_bf16_f32) against float64 and against the fp32 kernel on the widened operand,
parallel.bipartite_propagate_mean / bipartite_propagate (precision="bf16") against the float64
restatement of tests/bf16_ref.py, ShardedLightGCN(precision="bf16") training and evaluation at
world 1, and 2 ranks over NCCL against world 1 where the box has two GPUs.

Tolerances against the float64 restatement. The restatement rounds the same values at the same
points; what differs is the accumulation (fp32 in CSR order on the GPU, float64 there) and, rarely,
a value that lies within that accumulation error of a bf16 rounding midpoint and so rounds to the
other neighbour: one element moves by one bf16 ulp (2^-8 relative) and carries that into the
later layers. Emulating the kernel's fp32 accumulation on the CPU on graphs of this size puts the
normwise distance at 4e-8 (3 layers) to 7e-7 (4 layers); bf16 against exact propagation is
~3e-4. PROP_TOL = 2e-5 leaves a factor 30 above the first and 15 below the second."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from bf16_ref import PropagateBf16, propagate_bf16
from conftest import pkg
from oracle import ops as oops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GAMMA = 1e-10
U, I, E = 3000, 500, 60000
PROP_TOL = 2e-5
BF16_U = 2.0 ** -9          # unit roundoff of bfloat16


def _nrm(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


# ------------------------------------------------------------------ the kernel
def _random_csr(n_rows, n_cols, seed, lead, col_offset):
    """CSR with empty rows, light rows and heavy rows (> 64 non-zeros: split across tasks), whose
    row pointers are a view starting at row `lead` of a larger CSR (so row_ptr[0] != 0), column ids
    shifted by `col_offset`. Returns (CSRGraph, dense float64 [n_rows, n_cols])."""
    G = pkg("graph")
    g = torch.Generator().manual_seed(seed)
    rows = lead + n_rows
    deg = torch.randint(1, 40, (rows,), generator=g)
    deg[torch.rand(rows, generator=g) < 0.15] = 0
    heavy = torch.rand(rows, generator=g) < 0.06
    deg[heavy] = torch.randint(65, 400, (int(heavy.sum()),), generator=g)
    rp = torch.zeros(rows + 1, dtype=torch.int64)
    rp[1:] = torch.cumsum(deg, 0)
    nnz = int(rp[-1])
    cols = torch.randint(0, n_cols, (nnz,), generator=g)
    vals = torch.randn(nnz, generator=g)
    dense = torch.zeros(n_rows, n_cols, dtype=torch.float64)
    r = torch.repeat_interleave(torch.arange(rows), deg)
    keep = r >= lead
    dense.index_put_((r[keep] - lead, cols[keep]), vals[keep].double(), accumulate=True)
    rp_dev = rp.to(torch.int32).to(DEV)
    csr = G.CSRGraph(rp_dev[lead:], (cols + col_offset).to(torch.int32).to(DEV), vals.to(DEV), n_rows, n_cols,
                     col_offset=col_offset)
    assert int(csr.row_ptr[0]) != 0 and csr.slot_base.numel() > 0 and (deg[lead:] == 0).any()
    return csr, dense


@pytest.mark.parametrize("d", [32, 64, 128])
@pytest.mark.parametrize("narrow", [False, True])
def test_bf16_spmm_kernel(d, narrow):
    ops = pkg("ops")
    n_rows, n_cols = 300, 450
    g, A = _random_csr(n_rows, n_cols, seed=d + narrow, lead=37, col_offset=1000)
    gen = torch.Generator(device=DEV).manual_seed(d)
    X = (torch.randn(n_cols, d, generator=gen, device=DEV) * 0.5).to(torch.bfloat16)
    acc0 = torch.randn(n_rows, d, generator=gen, device=DEV)
    y_ref = A @ X.double().cpu()
    scale = 0.3

    def run(mode):
        Y = y16 = acc_in = acc_out = None
        if mode in ("Y", "Y+acc"):
            Y = torch.full((n_rows, d), float("nan"), device=DEV)
        if mode in ("Y+acc", "acc+Y16"):
            acc_in, acc_out = acc0.clone(), torch.full((n_rows, d), float("nan"), device=DEV)
        if mode == "aliased":
            acc_in = acc_out = acc0.clone()
        if mode in ("acc+Y16", "aliased"):
            y16 = torch.full((n_rows, d), float("nan"), device=DEV, dtype=torch.bfloat16)
        ops.spmm_raw(g, X, Y=Y, acc_in=acc_in, acc_out=acc_out, acc_scale=scale, narrow=narrow, y16=y16)
        # the fp32 kernel on the widened operand, same arguments
        Yf = None if Y is None else torch.empty_like(Y)
        accf_in = None if acc_in is None else acc0.clone()
        accf_out = None if acc_out is None else (accf_in if mode == "aliased" else torch.empty_like(acc_out))
        ops.spmm_raw(g, X.float(), Y=Yf, acc_in=accf_in, acc_out=accf_out, acc_scale=scale, narrow=narrow)
        return Y, y16, acc_out, Yf, accf_out

    Y_only = None
    for mode in ("Y", "Y+acc", "acc+Y16", "aliased"):
        Y, y16, acc_out, Yf, accf_out = run(mode)
        again = run(mode)
        for a, b in zip((Y, y16, acc_out), again[:3]):
            assert a is None or torch.equal(a, b), mode                      # bit-reproducible
        if Y is not None:
            assert _nrm(Y, y_ref) < 1e-6, mode
            assert torch.equal(Y, Yf), mode
            Y_only = Y
        if acc_out is not None:
            assert _nrm(acc_out, (acc0.double().cpu() + y_ref) * scale) < 1e-6, mode
            assert torch.equal(acc_out, accf_out), mode
        if y16 is not None:
            assert torch.equal(y16, Y_only.to(torch.bfloat16)), mode


def test_bf16_spmm_rejects_what_it_does_not_cover():
    ops = pkg("ops")
    g, _ = _random_csr(64, 80, seed=3, lead=5, col_offset=0)
    d = 64
    X = torch.zeros(80, d, device=DEV, dtype=torch.bfloat16)
    Y = torch.zeros(64, d, device=DEV)
    for bad_d in (48, 256):                                                  # widths
        with pytest.raises(RuntimeError, match="code -1"):
            ops.spmm_raw(g, torch.zeros(80, bad_d, device=DEV, dtype=torch.bfloat16),
                         Y=torch.zeros(64, bad_d, device=DEV))
    buf = torch.zeros(80 * d + 1, device=DEV, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="code -2"):                       # misaligned X
        ops.spmm_raw(g, buf[1:].view(80, d), Y=Y)
    fbuf = torch.zeros(64 * d + 1, device=DEV)
    with pytest.raises(RuntimeError, match="code -2"):                       # misaligned output
        ops.spmm_raw(g, X, Y=fbuf[1:].view(64, d))
    with pytest.raises(RuntimeError):                                        # host tensors
        ops.spmm_raw(g, X.cpu(), Y=Y)
    with pytest.raises(RuntimeError):
        ops.spmm_raw(g, X, y16=torch.zeros(64, d, dtype=torch.bfloat16))
    with pytest.raises(RuntimeError):                                        # fp16 operands
        ops.spmm_raw(g, X.half(), Y=Y)
    with pytest.raises(RuntimeError):
        ops.spmm_raw(g, X, y16=torch.zeros(64, d, device=DEV, dtype=torch.float16))
    with pytest.raises(RuntimeError):
        ops.spmm_raw(g, X.float(), Y=Y, y16=torch.zeros(64, d, device=DEV, dtype=torch.bfloat16))
    with pytest.raises(RuntimeError, match="code -1"):                       # no cosine epilogue
        ops.spmm_raw(g, X, Y=Y, cos_ref=torch.zeros(64, d, device=DEV), cos_w=torch.zeros(64, device=DEV))
    with pytest.raises(RuntimeError, match="code -1"):                       # no streaming variant
        ops.spmm_raw(g, X, Y=Y, stream_policy=True)


# ------------------------------------------------------------------ propagation
def _graph(blocked):
    par, synth = pkg("parallel"), pkg("synth")
    u, i = synth.make_scaled_edges(DEV, U, I, E, block=1024)
    sb = par.ShardedBipartite.from_local_edges(u, i, np.array([0, U]), 0, 1, U, I, "f64eps",
                                               rt_block_users=1000 if blocked else None)
    assert (sb.Rt_blocked is not None) == blocked
    R = sb.R
    rp = R.row_ptr.long().cpu()
    rows = torch.repeat_interleave(torch.arange(U), rp[1:] - rp[:-1])
    cols = R.col_idx.long().cpu() - R.col_offset + U
    vals = R.vals.double().cpu()
    A = torch.sparse_coo_tensor(torch.stack([torch.cat([rows, cols]), torch.cat([cols, rows])]),
                                torch.cat([vals, vals]), (U + I, U + I)).coalesce()
    return sb, A


@pytest.mark.parametrize("blocked", [False, True])
def test_bf16_propagation_matches_restatement(blocked):
    par = pkg("parallel")
    sb, A = _graph(blocked)
    d, L = 64, 3
    gen = torch.Generator(device=DEV).manual_seed(11)
    Xu, Xi = (torch.randn(U, d, generator=gen, device=DEV) * 0.1), (torch.randn(I, d, generator=gen, device=DEV) * 0.1)
    ou, oi = par.bipartite_propagate_mean(sb, Xu, Xi, L, precision="bf16")
    assert ou.dtype == oi.dtype == torch.float32
    ou2, oi2 = par.bipartite_propagate_mean(sb, Xu, Xi, L, precision="bf16")
    assert torch.equal(ou, ou2) and torch.equal(oi, oi2)
    ref = propagate_bf16(A, torch.cat([Xu, Xi]).double().cpu(), L)
    got = torch.cat([ou, oi])
    assert _nrm(got, ref) < PROP_TOL, _nrm(got, ref)
    fu, fi = par.bipartite_propagate_mean(sb, Xu, Xi, L)                    # fp32 mode
    dist_fp32 = _nrm(got, torch.cat([fu, fi]))
    assert 2 * PROP_TOL < dist_fp32 < L * BF16_U, dist_fp32
    # backward: the same rounded operator on the gradients (the item part through reduce_items)
    xu, xi = Xu.clone().requires_grad_(True), Xi.clone().requires_grad_(True)
    gu, gi = torch.randn(U, d, generator=gen, device=DEV), torch.randn(I, d, generator=gen, device=DEV)
    pu, pi = par.bipartite_propagate(sb, xu, xi, L, precision="bf16")
    assert torch.equal(pu, ou) and torch.equal(pi, oi)
    ((pu * gu).sum() + (pi * gi).sum()).backward()
    ref_g = propagate_bf16(A, torch.cat([gu, gi]).double().cpu(), L)
    assert _nrm(torch.cat([xu.grad, xi.grad]), ref_g) < PROP_TOL


# ------------------------------------------------------------------ training and evaluation
def _lightgcn_env():
    from parity_util import make_env
    env = make_env("LightGCN", DEV)
    m, train = env["model"], env["train"]
    batches = []
    for b in train:
        batches.append(b.clone())
        if len(batches) == 5:
            break
    train.pr = 0
    return env, m, batches


def _sharded_world1(m, cfg, precision):
    par = pkg("parallel")
    sb = par.ShardedBipartite.from_local_edges(m._edge_u, m._edge_i, np.array([0, m.n_users]), 0, 1, m.n_users,
                                               m.n_items, "f64eps")
    e = m.embedding_dict
    return par.ShardedLightGCN(sb, cfg["embedding_size"], cfg["n_layers"], cfg["reg_weight"],
                               user_emb=e["user_emb"].detach(), item_emb=e["item_emb"].detach(), precision=precision)


def _adjacency(sb):
    R = sb.R
    nU = sb.U
    rp = R.row_ptr.long().cpu()
    rows = torch.repeat_interleave(torch.arange(nU), rp[1:] - rp[:-1])
    cols = R.col_idx.long().cpu()[int(rp[0]): int(rp[-1])] - R.col_offset + nU
    vals = R.vals.double().cpu()[int(rp[0]): int(rp[-1])]
    return torch.sparse_coo_tensor(torch.stack([torch.cat([rows, cols]), torch.cat([cols, rows])]),
                                   torch.cat([vals, vals]), (nU + sb.I, nU + sb.I)).coalesce()


def test_bf16_sharded_lightgcn_training_matches_restatement(capsys):
    FusedAdam = pkg("optim").FusedAdam
    env, m, batches = _lightgcn_env()
    cfg = env["config"]
    sm = _sharded_world1(m, cfg, "bf16")
    fm = _sharded_world1(m, cfg, "fp32")
    A = _adjacency(sm.sb)
    nU, L, rw, lr = sm.n_users, cfg["n_layers"], cfg["reg_weight"], cfg["learning_rate"]
    P = [t.detach().double().cpu().requires_grad_(True) for t in (sm.embedding_dict["user_emb"],
                                                                   sm.embedding_dict["item_emb"])]
    ref_opt = torch.optim.Adam(P, lr=lr)
    opt, fopt = FusedAdam(sm.parameters(), lr=lr), FusedAdam(fm.parameters(), lr=lr)
    for step, b in enumerate(batches):
        for o, mod in ((opt, sm), (fopt, fm)):
            o.zero_grad(set_to_none=True)
            loss = mod.calculate_loss(b)
            loss.backward()
            o.step()
            if mod is sm:
                got = loss.item()
        u, p, n = (t.cpu() for t in b[:3])
        ref_opt.zero_grad(set_to_none=True)
        X = PropagateBf16.apply(torch.cat(P), A, L)
        ref = oops.bpr_gamma_mean(X[:nU][u], X[nU:][p], X[nU:][n], GAMMA) + rw * oops.emb_loss(P[0][u], P[1][p],
                                                                                                P[1][n])
        ref.backward()
        ref_opt.step()
        assert abs(got - ref.item()) <= 1e-5 * abs(ref.item()), (step, got, ref.item())
    for k, t in zip(("user_emb", "item_emb"), P):
        assert _rel(sm.embedding_dict[k].detach(), t.detach()) < 3e-4, k
    with capsys.disabled():
        print("\nbf16 vs fp32 model after 5 steps (max-abs rel):",
              {k: _rel(sm.embedding_dict[k].detach(), fm.embedding_dict[k].detach()) for k in ("user_emb", "item_emb")},
              "bf16 vs float64 restatement:",
              {k: _rel(sm.embedding_dict[k].detach(), t.detach()) for k, t in zip(("user_emb", "item_emb"), P)})


def test_bf16_sharded_evaluation():
    par, synth, data_m, trm, cfgm, ops = (pkg(x) for x in ("parallel", "synth", "data", "trainer", "config", "ops"))
    u, i = synth.make_scaled_edges(DEV, U, I, E, block=1024)
    lab = synth.scaled_edge_labels(u, i)
    t = lab == 0
    sb = par.ShardedBipartite.from_local_edges(u[t], i[t], np.array([0, U]), 0, 1, U, I, "f64eps")
    sm = par.ShardedLightGCN(sb, 64, 4, 1e-2, precision="bf16")
    cfg = cfgm.Config("LightGCN", "scaled", {"device": torch.device(DEV), "cuda_graph": False,
                                             "metrics": ["Recall", "Recall2", "Precision", "NDCG", "MAP"],
                                             "topk": [10, 20, 50]})
    tr = trm.Trainer(cfg, sm)
    loader = data_m.DeviceTrainLoader(u[t], i[t], U, I, 4096, seed=5, rank=0, world=1, user_lo=0)
    tr._train_epoch([b for _, b in zip(range(3), loader)], 0)
    sev = par.ShardedEvalData(sb, u[lab == 1], i[lab == 1], batch_users=700)
    first = tr.evaluate(sev)
    assert tr.evaluate(sev) == first
    sm.eval()
    uo, io = sm.restore_embeddings()
    got = sm.eval_topk(sev.eval_u, 50)
    want = ops.score_mask_topk_rows(uo, sev.eval_u, io, 50, sb.R.row_ptr, sb.R.col_idx, item_offset=0)
    assert torch.equal(got.long(), want.long())
    sm.train()


# ------------------------------------------------------------------ two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = f"cuda:{rank}"
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(dev))
    try:
        global DEV
        DEV = dev
        par, FusedAdam = pkg("parallel"), pkg("optim").FusedAdam
        env, m, batches = _lightgcn_env()
        cfg = env["config"]
        ref = _sharded_world1(m, cfg, "bf16")                            # world-1 model, no collectives
        nU, nI = m.n_users, m.n_items
        eu, ei = m._edge_u.to(torch.int64), m._edge_i.to(torch.int64)
        rp = np.concatenate(([0], np.cumsum(np.bincount(eu.cpu().numpy(), minlength=nU))))
        bounds = par.partition_by_nnz(rp, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        mine = (eu >= lo) & (eu < hi)
        sb = par.ShardedBipartite.from_local_edges(eu[mine], ei[mine], bounds, rank, world, nU, nI, "f64eps")
        e = m.embedding_dict
        sm = par.ShardedLightGCN(sb, cfg["embedding_size"], cfg["n_layers"], cfg["reg_weight"],
                                 user_emb=e["user_emb"].detach()[lo:hi], item_emb=e["item_emb"].detach(),
                                 precision="bf16")
        opt_ref = FusedAdam(ref.parameters(), lr=cfg["learning_rate"])
        opt = FusedAdam(sm.parameters(), lr=cfg["learning_rate"])
        for step, b in enumerate(batches):
            own = (b[0] >= lo) & (b[0] < hi)
            part = b[:, own].clone()
            part[0] -= lo
            for o, mod, x in ((opt_ref, ref, b), (opt, sm, part)):
                o.zero_grad(set_to_none=True)
                loss = mod.calculate_loss(x)
                loss.backward()
                o.step()
                if mod is ref:
                    want = loss.item()
            assert abs(loss.item() - want) <= 1e-5 * abs(want), (step, loss.item(), want)
        assert _rel(sm.embedding_dict["item_emb"].detach(), ref.embedding_dict["item_emb"].detach()) < 3e-4
        assert _rel(sm.embedding_dict["user_emb"].detach(), ref.embedding_dict["user_emb"].detach()[lo:hi]) < 3e-4
        it = sm.embedding_dict["item_emb"].detach().contiguous()
        allit = torch.empty(world, *it.shape, device=dev)
        dist.all_gather_into_tensor(allit, it)
        st = opt.state[sm.embedding_dict["item_emb"]]
        allm = torch.empty(world, *it.shape, device=dev)
        dist.all_gather_into_tensor(allm, st["exp_avg_sq"].contiguous())
        torch.cuda.synchronize()
        assert all(torch.equal(allit[r], allit[0]) and torch.equal(allm[r], allm[0]) for r in range(world))
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_bf16_sharded_lightgcn_nccl_2gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = _free_port()
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(2))
