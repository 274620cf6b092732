"""world_size-2/3 gloo tests (CPU) of LightGCN training on the user-sharded bipartite graph
(parallel.ShardedLightGCN, per-rank batches of data.DeviceTrainLoader). The per-rank arithmetic is
injected in float64: the SpMM on torch.sparse, the loss restated from oracle.ops.bpr_gamma_mean /
emb_loss; the CUDA kernels are covered by tests/test_gpu_sharded_train.py."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import TINY, pkg
from oracle import graph as ograph
from oracle import models as omodels
from oracle import ops as oops
from oracle import sampler as osampler

GAMMA = 1e-10


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _csr_from_coo(rows, cols, vals, n_rows, n_cols, with_transpose=False):
    o = np.lexsort((cols.numpy(), rows.numpy()))
    rp = np.concatenate(([0], np.cumsum(np.bincount(rows.numpy(), minlength=n_rows)))).astype(np.int32)
    return pkg("graph").CSRGraph(torch.from_numpy(rp), cols[o].to(torch.int32), vals[o], n_rows, n_cols)


def _spmm_f64(g, X, Y=None, acc_in=None, acc_out=None, scale=1.0):
    rp = g.row_ptr.long()
    base = int(rp[0])
    A = torch.sparse_csr_tensor(rp - base, g.col_idx.long()[base: int(rp[-1])] - g.col_offset,
                                g.vals.double()[base: int(rp[-1])], size=(g.n_rows, g.n_cols))
    y = torch.sparse.mm(A, X.double()[: g.n_cols]).to(X.dtype)
    if Y is not None:
        Y.copy_(y)
    if acc_out is not None:
        acc_out.copy_(((acc_in + y) if acc_in is not None else y) * scale)


def _loss_fwd_f64(uo, io, ue, ie, users, pos, neg, gamma):
    """Partial sums of bpr_gamma_mean * B and of the squared EmbLoss norms; dx by autograd of the
    per-triple term of bpr_gamma_mean."""
    with torch.enable_grad():
        ps, ns = oops.bpr_scores(uo[users], io[pos], io[neg])
        x = (ps - ns).detach().requires_grad_(True)
        per = -torch.log(gamma + torch.sigmoid(x))
        (dx,) = torch.autograd.grad(per.sum(), x) if users.numel() else (torch.zeros_like(x),)
    out4 = torch.stack([per.detach().sum(), ue[users].pow(2).sum(), ie[pos].pow(2).sum(), ie[neg].pow(2).sum()])
    return out4, dx


def _loss_bwd_f64(uo, io, ue, ie, users, pos, neg, dx, coef4, d_uo, d_io, d_ue, d_ie):
    s = (coef4[0] * dx)[:, None]
    d_uo.index_add_(0, users, s * (io[pos] - io[neg]))
    d_io.index_add_(0, pos, s * uo[users])
    d_io.index_add_(0, neg, -s * uo[users])
    d_ue.index_add_(0, users, coef4[1] * ue[users])
    d_ie.index_add_(0, pos, coef4[2] * ie[pos])
    d_ie.index_add_(0, neg, coef4[3] * ie[neg])


def _setup(rank, world, bounds=None):
    par, synth = pkg("parallel"), pkg("synth")
    data = synth.make_dataset("tiny", **TINY)
    u, i = data.split(0)
    U, I = data.n_users, data.n_items
    eu, ei = torch.from_numpy(np.asarray(u, np.int64)), torch.from_numpy(np.asarray(i, np.int64))
    if bounds is None:
        rp = np.concatenate(([0], np.cumsum(np.bincount(u, minlength=U))))
        bounds = par.partition_by_nnz(rp, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    mine = (eu >= lo) & (eu < hi)
    sb = par.ShardedBipartite.from_local_edges(eu[mine], ei[mine], bounds, rank, world, U, I, recipe="f32",
                                               csr_from_coo=_csr_from_coo)
    return dict(u=u, i=i, U=U, I=I, eu=eu, ei=ei, mine=mine, sb=sb, lo=lo, hi=hi)


def _loader(env, rank, world, batch_size, seed=5):
    U_loc = env["hi"] - env["lo"]
    return pkg("data").DeviceTrainLoader(env["eu"][env["mine"]], env["ei"][env["mine"]], U_loc, env["I"], batch_size,
                                         seed=seed, rank=rank, world=world, user_lo=env["lo"],
                                         sampler=osampler.neg_sample_counter)


def _train_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        par = pkg("parallel")
        env = _setup(rank, world)
        sb, U, I, lo, hi = env["sb"], env["U"], env["I"], env["lo"], env["hi"]
        d, L, rw, lr = 16, 3, 1e-2, 1e-2
        gen = torch.Generator().manual_seed(7)
        U0 = (torch.rand(U, d, generator=gen, dtype=torch.float64) - 0.5) * 0.4
        I0 = (torch.rand(I, d, generator=gen, dtype=torch.float64) - 0.5) * 0.4
        model = par.ShardedLightGCN(sb, d, L, rw, user_emb=U0[lo:hi], item_emb=I0, spmm_fn=_spmm_f64,
                                    loss_fns=(_loss_fwd_f64, _loss_bwd_f64), gamma=GAMMA)
        opt = torch.optim.Adam(model.parameters(), lr=lr)
        # the same model in one process on the union batches (oracle)
        r, c, v = ograph.norm_adj_f32(env["u"], env["i"], U, I)
        Gr = {"norm_adj": ograph.to_torch_csr(r, c, v, (U + I, U + I), torch.float64)}
        P = {"embedding_dict.user_emb": U0.clone().requires_grad_(True),
             "embedding_dict.item_emb": I0.clone().requires_grad_(True)}
        ref_opt = torch.optim.Adam(list(P.values()), lr=lr)
        cfg = {"n_layers": L, "reg_weight": rw}
        loader = _loader(env, rank, world, batch_size=256)
        assert len(loader) == -(-len(env["u"]) // 256)
        it = iter(loader)
        for step in range(3):
            batch = next(it)
            slices = [None] * world
            dist.all_gather_object(slices, (batch + torch.tensor([[lo], [0], [0]])).numpy())
            union = torch.from_numpy(np.concatenate(slices, axis=1))
            opt.zero_grad(set_to_none=True)
            loss = model.calculate_loss(batch)
            loss.backward()
            opt.step()
            ref_opt.zero_grad(set_to_none=True)
            ref = omodels.lightgcn_loss(P, Gr, cfg, union)
            ref.backward()
            ref_opt.step()
            assert abs(loss.item() - ref.item()) <= 1e-9 * abs(ref.item()), (step, loss.item(), ref.item())
            assert model.embedding_dict["item_emb"].grad is not None
        users_all = [None] * world
        items_all = [None] * world
        dist.all_gather_object(users_all, model.embedding_dict["user_emb"].detach())
        dist.all_gather_object(items_all, model.embedding_dict["item_emb"].detach())
        assert torch.allclose(torch.cat(users_all), P["embedding_dict.user_emb"].detach(), rtol=0, atol=1e-9)
        assert torch.allclose(items_all[rank], P["embedding_dict.item_emb"].detach(), rtol=0, atol=1e-9)
        assert all(torch.equal(t, items_all[0]) for t in items_all)
        st = opt.state[model.embedding_dict["item_emb"]]
        states = [None] * world
        dist.all_gather_object(states, (st["exp_avg"], st["exp_avg_sq"]))
        assert all(torch.equal(a, states[0][0]) and torch.equal(b, states[0][1]) for a, b in states)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_lightgcn_matches_single_process(world, tmp_path):
    port = _free_port()
    mp.spawn(_train_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def _uneven_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        data_m, par, cfgm, trm = pkg("data"), pkg("parallel"), pkg("config"), pkg("trainer")
        bounds = np.array([0, 1, 240]) if world == 2 else np.array([0, 2, 120, 240])
        env = _setup(rank, world, bounds)
        B = 64
        loader = _loader(env, rank, world, B, seed=11)
        E, n_p = len(env["u"]), int(env["mine"].sum())
        S = -(-E // B)
        assert len(loader) == S and loader.nnz_per_rank[rank] == n_p and sum(loader.nnz_per_rank) == E
        if rank == 0:
            assert n_p < S                        # this rank has empty steps
        # the world size is the process group's: omitted it is derived, a wrong one is refused
        args = (env["eu"][env["mine"]], env["ei"][env["mine"]], env["hi"] - env["lo"], env["I"], B)
        assert len(data_m.DeviceTrainLoader(*args, rank=rank, user_lo=env["lo"],
                                            sampler=osampler.neg_sample_counter)) == S
        with pytest.raises(ValueError):
            data_m.DeviceTrainLoader(*args, rank=rank, world=world + 1, user_lo=env["lo"],
                                     sampler=osampler.neg_sample_counter)
        assert loader.seed == data_m.rank_seed(11, rank) and (rank == 0) == (loader.seed == 11)
        # local history CSR, built here independently, for the oracle sampler
        lu = (env["eu"][env["mine"]] - env["lo"]).numpy()
        li = env["ei"][env["mine"]].numpy()
        o = np.lexsort((li, lu))
        hrp = np.concatenate(([0], np.cumsum(np.bincount(lu, minlength=env["hi"] - env["lo"]))))
        hcols = li[o]
        for epoch in range(2):
            sizes, seen = [], []
            for s, batch in enumerate(loader):
                sizes.append(batch.shape[1])
                seen.append(batch[:2].T.numpy())
                want = osampler.neg_sample_counter(batch[0].numpy(), None, env["I"], hrp, hcols,
                                                   data_m.rank_seed(11, rank), epoch * S + s)
                assert np.array_equal(batch[2].numpy(), want)
            assert len(sizes) == S and max(sizes) - min(sizes) <= 1 and sum(sizes) == n_p
            got = np.concatenate(seen)
            got = got[np.lexsort((got[:, 1], got[:, 0]))]
            ref = np.stack([lu, li], 1)[o]
            assert np.array_equal(got, ref)       # every local interaction once per epoch, local user ids
        # one epoch through the Trainer (empty steps on some ranks still meet every collective)
        d = 8
        gen = torch.Generator().manual_seed(3)
        model = par.ShardedLightGCN(env["sb"], d, 2, 1e-2,
                                    user_emb=torch.rand(env["hi"] - env["lo"], d, generator=gen, dtype=torch.float64),
                                    item_emb=torch.rand(env["I"], d, generator=torch.Generator().manual_seed(4),
                                                        dtype=torch.float64),
                                    spmm_fn=_spmm_f64, loss_fns=(_loss_fwd_f64, _loss_bwd_f64))
        cfg = cfgm.Config("LightGCN", "tiny", {"device": torch.device("cpu"), "cuda_graph": False, "epochs": 1})
        tr = trm.Trainer(cfg, model)
        total, losses = tr._train_epoch(loader, 0)
        assert len(losses) == S and np.isfinite(total)
        all_losses = [None] * world
        dist.all_gather_object(all_losses, [float(x) for x in losses])
        assert all(x == all_losses[0] for x in all_losses)
        items = [None] * world
        dist.all_gather_object(items, model.embedding_dict["item_emb"].detach())
        assert all(torch.equal(t, items[0]) for t in items)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_rank_batches_uneven_nnz(world, tmp_path):
    port = _free_port()
    mp.spawn(_uneven_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_rank_seed():
    data_m = pkg("data")
    assert data_m.rank_seed(999, 0) == 999
    assert len({data_m.rank_seed(999, r) for r in range(8)}) == 8
    assert all(0 <= data_m.rank_seed(2 ** 64 - 1, r) < 2 ** 64 for r in range(8))
