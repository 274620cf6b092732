"""B200 tests of full-rank evaluation on the user-sharded bipartite graph: the mask-rows-by-user-id
entry point (mmrec_score_mask_topk_rows_f32) against the per-batch-CSR one, world-1
parallel.ShardedLightGCN evaluation against models.LightGCN through Trainer.evaluate and
EvalDataLoader on the same split, and 2 ranks over NCCL against world 1 where the box has two GPUs."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
METRICS = ["Recall", "Recall2", "Precision", "NDCG", "MAP"]
TOPK = [10, 20, 50]
U, I, E = 3000, 500, 60000


def _mask_table(n_rows, n_items, item_offset, gen):
    """Random ascending mask rows over a user table, a fifth of them empty."""
    lens = torch.randint(0, 61, (n_rows,), generator=gen)
    lens[torch.rand(n_rows, generator=gen) < 0.2] = 0
    rows = [torch.sort(torch.randperm(n_items, generator=gen)[: int(n)])[0] + item_offset for n in lens]
    rowptr = torch.zeros(n_rows + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(lens, 0)
    return rowptr, rows


@pytest.mark.parametrize("d", [32, 64, 128])
@pytest.mark.parametrize("n_users,k,item_offset", [(1, 1, 0), (129, 20, 0), (1000, 50, 1000), (300, 7, 37)])
def test_rows_entry_matches_batch_csr(d, n_users, k, item_offset):
    _rows_vs_batch(d, n_users, k, item_offset)


@pytest.mark.parametrize("d,k", [(32, 100), (128, 64)])
def test_rows_entry_matches_batch_csr_simt(d, k):
    """K beyond the tensor-core tiling's shared memory: both entry points run the CUDA-core kernel."""
    _rows_vs_batch(d, 257, k, 5)


def _rows_vs_batch(d, n_users, k, item_offset):
    ops = pkg("ops")
    gen = torch.Generator().manual_seed(d * 1000 + n_users + k)
    n_rows, n_items = 700, 3000
    ue = torch.randn(n_rows, d, generator=gen).to(DEV)
    ie = torch.randn(n_items, d, generator=gen).to(DEV)
    rowptr, rows = _mask_table(n_rows, n_items, item_offset, gen)
    users = torch.randint(0, n_rows, (n_users,), generator=gen)               # repeats allowed
    cols = torch.cat(rows).to(torch.int32)
    # the per-batch CSR the existing entry point needs: row b = mask row of users[b]
    blens = torch.tensor([len(rows[u]) for u in users.tolist()], dtype=torch.int64)
    brp = torch.zeros(n_users + 1, dtype=torch.int64)
    brp[1:] = torch.cumsum(blens, 0)
    # one unreferenced trailing entry: an all-empty batch would otherwise pass no column array at all
    bcols = torch.cat([rows[u] for u in users.tolist()] + [torch.zeros(1, dtype=torch.int64)]).to(torch.int32)
    want_i, want_v = ops.score_mask_topk(ue, users.to(DEV), ie, k, brp.to(torch.int32).to(DEV), bcols.to(DEV),
                                         item_offset=item_offset, return_scores=True)
    got_i, got_v = ops.score_mask_topk_rows(ue, users.to(DEV), ie, k, rowptr.to(torch.int32).to(DEV), cols.to(DEV),
                                            item_offset=item_offset, return_scores=True)
    assert torch.equal(got_i, want_i)
    assert torch.equal(got_v, want_v)
    # masked items only where the row leaves fewer than k unmasked ones
    for b, u in enumerate(users.tolist()[:50]):
        if n_items - len(rows[u]) >= k:
            assert not bool(torch.isin(got_i[b].cpu(), rows[u]).any())


def test_rows_entry_rejects_a_mask_of_another_shape():
    ops = pkg("ops")
    ue = torch.zeros(10, 32, device=DEV)
    ie = torch.zeros(40, 32, device=DEV)
    users = torch.arange(10, device=DEV)
    rp = torch.zeros(10, dtype=torch.int32, device=DEV)                       # one row pointer short
    with pytest.raises(RuntimeError):
        ops.score_mask_topk_rows(ue, users, ie, 5, rp, torch.zeros(0, dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError):
        ops.score_mask_topk_rows(ue, users, ie, 5, torch.zeros(11, dtype=torch.int64, device=DEV),
                                 torch.zeros(0, dtype=torch.int32, device=DEV))


def _split(dev):
    synth = pkg("synth")
    u, i = synth.make_scaled_edges(dev, U, I, E, block=1024)
    return u, i, synth.scaled_edge_labels(u, i)


def _config(**kw):
    cd = {"device": torch.device(DEV), "data_path": None, "is_multimodal_model": False, "metrics": METRICS,
          "topk": TOPK, "eval_batch_size": 256}
    cd.update(kw)
    return pkg("config").Config("LightGCN", "scaled", cd)


def test_split_on_the_device_equals_the_host_split():
    u, i, lab = _split(DEV)
    assert torch.equal(pkg("synth").scaled_edge_labels(u.cpu(), i.cpu()), lab.cpu())


def test_sharded_world1_evaluation_matches_lightgcn():
    data_m, models, par, trm = pkg("data"), pkg("models"), pkg("parallel"), pkg("trainer")
    u, i, lab = _split(DEV)
    config = _config()
    ds = data_m.RecDataset(config, u.cpu().numpy(), i.cpu().numpy(), lab.cpu().numpy(), user_num=U, item_num=I)
    tr, va, te = ds.split()
    train = data_m.TrainDataLoader(config, tr, batch_size=2048, shuffle=True)
    train.pretrain_setup()
    m = models.LightGCN(config, train).to(DEV)
    ref_tr = trm.Trainer(config, m)
    sb = par.ShardedBipartite.from_local_edges(u[lab == 0], i[lab == 0], np.array([0, U]), 0, 1, U, I, "f64eps")
    e = m.embedding_dict
    sm = par.ShardedLightGCN(sb, config["embedding_size"], config["n_layers"], config["reg_weight"],
                             user_emb=e["user_emb"].detach(), item_emb=e["item_emb"].detach())
    sh_tr = trm.Trainer(_config(cuda_graph=False), sm)
    for label, part in ((1, va), (2, te)):
        loader = data_m.EvalDataLoader(config, part, additional_dataset=tr, batch_size=config["eval_batch_size"])
        sev = par.ShardedEvalData(sb, u[lab == label], i[lab == label], batch_users=700)
        # same evaluated users, their ground truth in the same format
        order = torch.argsort(loader.eval_u)
        assert torch.equal(loader.eval_u[order], sev.eval_u)
        ref = ref_tr.evaluate(loader)
        assert ref_tr.evaluate(loader) == ref                                 # graph-replayed pass
        got = sh_tr.evaluate(sev)
        assert got == ref, (got, ref)
        ref_ids = torch.cat(ref_tr.evaluate_topk(loader))[order]
        sm.eval()
        got_ids = sm.eval_topk(sev.eval_u, max(TOPK))
        assert torch.equal(got_ids, ref_ids)
        assert sev.n_users_global == loader.eval_u.numel() and sev.total_pos == float(loader.eval_len_list.sum())
    assert sm._eval_cache is not None
    sm.train()
    assert sm._eval_cache is None


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
        par, trm, cfgm = pkg("parallel"), pkg("trainer"), pkg("config")
        synth = pkg("synth")
        cfg = cfgm.Config("LightGCN", "scaled", {"device": torch.device(dev), "cuda_graph": False,
                                                 "metrics": METRICS, "topk": TOPK})
        u, i = synth.make_scaled_edges(dev, U, I, E, block=1024)
        lab = synth.scaled_edge_labels(u, i)
        t = lab == 0
        # world 1 on this rank, no collectives
        sb1 = par.ShardedBipartite.from_local_edges(u[t], i[t], np.array([0, U]), 0, 1, U, I, "f64eps")
        one = trm.Trainer(cfg, par.ShardedLightGCN(sb1, 64, 4, 1e-2))
        want = [one.evaluate(par.ShardedEvalData(sb1, u[lab == x], i[lab == x])) for x in (1, 2)]
        rp = np.concatenate(([0], np.cumsum(np.bincount(u[t].cpu().numpy(), minlength=U))))
        bounds = par.partition_by_nnz(rp, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        su, si = synth.make_scaled_edges(dev, U, I, E, user_range=(lo, hi), block=1024)
        sl = synth.scaled_edge_labels(su, si)
        sb = par.ShardedBipartite.from_local_edges(su[sl == 0], si[sl == 0], bounds, rank, world, U, I, "f64eps")
        tr = trm.Trainer(cfg, par.ShardedLightGCN(sb, 64, 4, 1e-2))
        got = [tr.evaluate(par.ShardedEvalData(sb, su[sl == x], si[sl == x])) for x in (1, 2)]
        assert got == want, (rank, got, want)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_sharded_evaluation_nccl_2gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = _free_port()
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(2))
