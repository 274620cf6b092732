"""B200 tests of LightGCN training on the user-sharded bipartite graph: the LightGCN loss kernels
against float64 torch, parallel.ShardedLightGCN (world 1, and 2 ranks over NCCL where the box has
two GPUs) against models.LightGCN + FusedAdam on the same batches, and the per-rank loader's CUDA
negatives against oracle/sampler.py."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import pkg
from oracle import sampler as osampler

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GAMMA = 1e-10


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def _ref_loss(uo, io, ue, ie, u, p, n, rw):
    x = (uo[u] * io[p]).sum(1) - (uo[u] * io[n]).sum(1)
    B = max(u.numel(), 1)
    mf = -torch.log(GAMMA + torch.sigmoid(x)).sum() / B
    return mf + rw * (torch.norm(ue[u]) + torch.norm(ie[p]) + torch.norm(ie[n])) / B


@pytest.mark.parametrize("d", [32, 64, 128])
@pytest.mark.parametrize("batch", [0, 1, 777])
def test_lightgcn_loss_kernels(d, batch):
    ops = pkg("ops")
    g = torch.Generator(device=DEV).manual_seed(d + batch)
    nu, ni, rw = 37, 29, 1e-2
    uo, ue = (torch.randn(nu, d, generator=g, device=DEV) * 0.3 for _ in range(2))
    io, ie = (torch.randn(ni, d, generator=g, device=DEV) * 0.3 for _ in range(2))
    u = torch.randint(0, nu, (batch,), generator=g, device=DEV)          # users and items repeat
    p = torch.randint(0, ni, (batch,), generator=g, device=DEV)
    n = torch.randint(0, ni, (batch,), generator=g, device=DEV)
    n[::5] = p[::5]                                                      # pos == neg
    out4, dx = ops.lightgcn_loss_fwd(uo, io, ue, ie, u, p, n, GAMMA)
    out4b, _ = ops.lightgcn_loss_fwd(uo, io, ue, ie, u, p, n, GAMMA)
    assert torch.equal(out4, out4b)                                      # fixed-order reduction
    T = [t.double().requires_grad_(True) for t in (uo, io, ue, ie)]
    if batch == 0:
        assert torch.equal(out4.cpu(), torch.zeros(4))
    else:
        want = _ref_loss(*T, u, p, n, rw)
        want.backward()
    B = max(batch, 1)
    o = out4.double()
    norms = o[1:].sqrt()
    got = o[0] / B + rw * norms.sum() / B
    if batch:
        assert abs(float(got) - float(want.detach())) <= 1e-6 * abs(float(want.detach()))
    coef = torch.cat([torch.tensor([1.0 / B], device=DEV, dtype=torch.float64),
                      torch.where(norms > 0, rw / (B * norms), torch.zeros_like(norms))]).float()
    grads = [torch.zeros_like(t) for t in (uo, io, ue, ie)]
    ops.lightgcn_loss_bwd(uo, io, ue, ie, u, p, n, dx, coef, *grads)
    for gr, t in zip(grads, T):
        if batch == 0:
            assert not bool(gr.any())
        else:
            assert _rel(gr, t.grad) < 1e-5


def test_lightgcn_loss_rejects_bad_arguments():
    ops = pkg("ops")
    t = torch.zeros(4, 6, device=DEV)                                   # d % 4 != 0
    ids = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(RuntimeError):
        ops.lightgcn_loss_fwd(t, t, t, t, ids, ids, ids)
    t8 = torch.zeros(4, 8, device=DEV)
    with pytest.raises(RuntimeError):
        ops.lightgcn_loss_fwd(t8, t8, t8, t8, ids, ids, ids.to(torch.int32))


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


def _sharded_world1(m, cfg):
    par = pkg("parallel")
    U, I = m.n_users, m.n_items
    sb = par.ShardedBipartite.from_local_edges(m._edge_u, m._edge_i, np.array([0, U]), 0, 1, U, I, "f64eps")
    e = m.embedding_dict
    return par.ShardedLightGCN(sb, cfg["embedding_size"], cfg["n_layers"], cfg["reg_weight"],
                               user_emb=e["user_emb"].detach(), item_emb=e["item_emb"].detach())


def test_sharded_lightgcn_world1_matches_lightgcn(tmp_path):
    dist.init_process_group("nccl", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        _world1(pkg("optim").FusedAdam)
    finally:
        dist.destroy_process_group()


def _world1(FusedAdam):
    env, m, batches = _lightgcn_env()
    cfg = env["config"]
    sm = _sharded_world1(m, cfg)
    opt_ref = FusedAdam(m.parameters(), lr=cfg["learning_rate"])
    opt = FusedAdam(sm.parameters(), lr=cfg["learning_rate"])
    m.train()
    for step, b in enumerate(batches):
        opt_ref.zero_grad(set_to_none=True)
        opt.zero_grad(set_to_none=True)
        ref = m.calculate_loss(b)
        ref.backward()
        loss = sm.calculate_loss(b)
        loss.backward()
        if step == 0:
            for k in ("user_emb", "item_emb"):
                assert _rel(sm.embedding_dict[k].grad, m.embedding_dict[k].grad) < 2e-5, k
        assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item()), (step, loss.item(), ref.item())
        opt_ref.step()
        opt.step()
    for k in ("user_emb", "item_emb"):
        assert _rel(sm.embedding_dict[k].detach(), m.embedding_dict[k].detach()) < 3e-4, k
    users = torch.arange(0, m.n_users, 3, device=DEV)
    with torch.no_grad():
        uo, io = sm.forward()
    assert torch.equal(sm.full_sort_topk(users, 20).long(), pkg("ops").score_mask_topk(uo, users, io, 20).long())
    # Trainer drives the model unchanged (eager steps, FusedAdam over both tables)
    trm, cfgm = pkg("trainer"), pkg("config")
    tc = cfgm.Config("LightGCN", "tiny", {"device": torch.device(DEV), "cuda_graph": False})
    tr = trm.Trainer(tc, sm)
    assert type(tr.optimizer).__name__ == "FusedAdam"
    total, losses = tr._train_epoch(batches, 0)
    assert len(losses) == len(batches) and np.isfinite(total)


def test_rank_loader_negatives_match_oracle():
    data_m, synth = pkg("data"), pkg("synth")
    U, I, lo, hi = 3000, 500, 1000, 2200
    su, si = synth.make_scaled_edges(DEV, U, I, 60000, block=1024)
    mine = (su >= lo) & (su < hi)
    dl = data_m.DeviceTrainLoader(su[mine], si[mine], hi - lo, I, batch_size=4096, seed=7, rank=1, world=1,
                                  user_lo=lo)
    assert dl.seed == data_m.rank_seed(7, 1) != 7
    rp, hc = dl.hist_rowptr.cpu().numpy(), dl.hist_cols.cpu().numpy()
    n = int(mine.sum())
    sizes = []
    for step, batch in enumerate(dl):
        assert int(batch[0].min()) >= 0 and int(batch[0].max()) < hi - lo
        sizes.append(batch.shape[1])
        if step < 3:
            want = osampler.neg_sample_counter(batch[0].cpu().numpy(), None, I, rp, hc, dl.seed, step)
            assert np.array_equal(batch[2].cpu().numpy(), want)
    assert len(sizes) == -(-n // 4096) and sum(sizes) == n and max(sizes) - min(sizes) <= 1


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
        ref = _sharded_world1(m, cfg)                                   # world-1 model, no collectives
        U, I = m.n_users, m.n_items
        eu, ei = m._edge_u.to(torch.int64), m._edge_i.to(torch.int64)
        rp = np.concatenate(([0], np.cumsum(np.bincount(eu.cpu().numpy(), minlength=U))))
        bounds = par.partition_by_nnz(rp, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        mine = (eu >= lo) & (eu < hi)
        sb = par.ShardedBipartite.from_local_edges(eu[mine], ei[mine], bounds, rank, world, U, I, "f64eps")
        e = m.embedding_dict
        sm = par.ShardedLightGCN(sb, cfg["embedding_size"], cfg["n_layers"], cfg["reg_weight"], group=None,
                                 user_emb=e["user_emb"].detach()[lo:hi], item_emb=e["item_emb"].detach())
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
        ids = sm.full_sort_topk(torch.arange(0, U, 7, device=dev), 10)
        allids = torch.empty(world, *ids.shape, dtype=ids.dtype, device=dev)
        dist.all_gather_into_tensor(allids, ids.contiguous())
        assert all(torch.equal(allids[r], allids[0]) for r in range(world))
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_sharded_lightgcn_nccl_2gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = _free_port()
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(2))


def _empty_slice_worker(rank, world, port, out_dir):
    """Rank 0 holds fewer interactions than there are steps: its empty slices go through the CUDA
    sampler and the loss kernels like any other."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        data_m, ops, synth = pkg("data"), pkg("ops"), pkg("synth")
        U, I, B = 3000, 500, 512
        su, si = synth.make_scaled_edges(DEV, U, I, 60000, block=1024)
        lo, hi = (0, 2) if rank == 0 else (2, U)
        mine = torch.nonzero((su >= lo) & (su < hi)).flatten()
        if rank == 0:
            mine = mine[:5]
        dl = data_m.DeviceTrainLoader(su[mine], si[mine], hi - lo, I, B, seed=3, rank=rank, user_lo=lo)
        with pytest.raises(ValueError):
            data_m.DeviceTrainLoader(su[mine], si[mine], hi - lo, I, B, rank=rank, world=world + 1, user_lo=lo)
        S = len(dl)
        n = mine.numel()
        assert sum(dl.nnz_per_rank) == int(((su >= 0) & (su < 2)).sum().clamp(max=5)) + int((su >= 2).sum())
        assert rank != 0 or n < S
        rp, hc = dl.hist_rowptr.cpu().numpy(), dl.hist_cols.cpu().numpy()
        g = torch.Generator(device=DEV).manual_seed(rank)
        uo, ue = (torch.randn(hi - lo, 32, generator=g, device=DEV) for _ in range(2))
        io, ie = (torch.randn(I, 32, generator=g, device=DEV) for _ in range(2))
        coef = torch.ones(4, device=DEV)
        sizes = []
        for step, b in enumerate(dl):
            sizes.append(b.shape[1])
            assert b.is_cuda and b.dtype == torch.int64
            if rank == 0 or step < 3:
                want = osampler.neg_sample_counter(b[0].cpu().numpy(), None, I, rp, hc, dl.seed, step)
                assert np.array_equal(b[2].cpu().numpy(), want)
            out4, dx = ops.lightgcn_loss_fwd(uo, io, ue, ie, b[0], b[1], b[2])
            grads = [torch.zeros_like(t) for t in (uo, io, ue, ie)]
            ops.lightgcn_loss_bwd(uo, io, ue, ie, b[0], b[1], b[2], dx, coef, *grads)
            if b.shape[1] == 0:
                assert not bool(out4.any()) and not any(bool(x.any()) for x in grads)
        torch.cuda.synchronize()
        assert len(sizes) == S and sum(sizes) == n and max(sizes) - min(sizes) <= 1
        assert rank != 0 or sizes.count(0) == S - n
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_rank_loader_empty_slices_cuda(tmp_path):
    port = _free_port()
    mp.spawn(_empty_slice_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(2))
