"""CPU tests of full-rank evaluation on the user-sharded bipartite graph: the held-out split of the
scaled graph (synth.scaled_edge_labels), parallel.ShardedEvalData + ShardedLightGCN.eval_metric_sums
through trainer.Trainer at world 2 and 3 over gloo, against TopKEvaluator's numpy hit-matrix path
in one process, and Trainer.fit's early stopping on every rank. The per-rank arithmetic is
injected in float64 (SpMM, loss, score + mask + top-K, metric sums); the CUDA kernels are covered
by tests/test_gpu_sharded_eval.py."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import pkg
from oracle import graph as ograph
from oracle import models as omodels
from oracle import sampler as osampler
from test_sharded_train_gloo import _csr_from_coo, _loss_bwd_f64, _loss_fwd_f64, _spmm_f64

METRICS = ["Recall", "Recall2", "Precision", "NDCG", "MAP"]
SHAPE = dict(U=600, I=150, E=9000, block=128)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _edges(lo=None, hi=None):
    synth = pkg("synth")
    rng = None if lo is None else (lo, hi)
    u, i = synth.make_scaled_edges("cpu", SHAPE["U"], SHAPE["I"], SHAPE["E"], user_range=rng, block=SHAPE["block"])
    return u, i, synth.scaled_edge_labels(u, i)


# ------------------------------------------------------------------------------------ the split
def _labels_numpy(u, i, seed=2024):
    """scaled_edge_labels restated in uint64 numpy."""
    m = (1 << 64) - 1

    def mix(x):
        x = x ^ (x >> np.uint64(30))
        x = x * np.uint64(0xBF58476D1CE4E5B9)
        x = x ^ (x >> np.uint64(27))
        x = x * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))

    with np.errstate(over="ignore"):
        salt = int(mix(np.array([(seed ^ 0x5851F42D4C957F2D) & m], dtype=np.uint64))[0])
        x = (u.astype(np.uint64) << np.uint64(32)) + i.astype(np.uint64) + np.uint64(salt)
        r = (mix(x) >> np.uint64(40)).astype(np.int64)
    lab = (r >= round(0.8 * (1 << 24))).astype(np.int64) + (r >= round(0.9 * (1 << 24))).astype(np.int64)
    first = np.ones(len(u), dtype=bool)
    first[1:] = u[1:] != u[:-1]
    lab[first] = 0
    return lab


def test_split_rules_and_hash():
    synth = pkg("synth")
    u, i = synth.make_scaled_edges("cpu", 20000, 2000, 400000, block=4096)
    lab = synth.scaled_edge_labels(u, i)
    un, iN, ln = u.numpy(), i.numpy(), lab.numpy()
    assert np.array_equal(ln, _labels_numpy(un, iN))
    assert set(np.unique(ln)) == {0, 1, 2}                              # three disjoint parts cover every edge
    first = np.ones(len(un), dtype=bool)
    first[1:] = un[1:] != un[:-1]
    assert first.sum() == 20000                                        # every user once
    assert (ln[first] == 0).all()                                      # its lowest item: train
    assert (iN[first] == np.minimum.reduceat(iN, np.flatnonzero(first))).all()
    frac = np.bincount(ln[~first], minlength=3) / (~first).sum()
    assert np.abs(frac - np.array([0.8, 0.1, 0.1])).max() < 0.005, frac
    assert not torch.equal(synth.scaled_edge_labels(u, i, seed=7), lab)


@pytest.mark.parametrize("world", [2, 3])
def test_split_of_rank_edges_is_slice_of_one_rank_split(world):
    par = pkg("parallel")
    u, i, lab = _edges()
    rp = np.concatenate(([0], np.cumsum(np.bincount(u.numpy(), minlength=SHAPE["U"]))))
    bounds = par.partition_by_nnz(rp, world)
    for r in range(world):
        lo, hi = int(bounds[r]), int(bounds[r + 1])
        lu, li, ll = _edges(lo, hi)
        m = (u >= lo) & (u < hi)
        assert torch.equal(lu, u[m]) and torch.equal(li, i[m]) and torch.equal(ll, lab[m])


# ------------------------------------------------------------------------------ injected operators
def _topk_f64(ue, users, ie, k, rowptr, cols, item_offset):
    """Score + mask + top-K in float64: stable descending sort, ties -> lower id (the kernels' rule)."""
    s = ue[users].double() @ ie.double().T
    for r, u in enumerate(users.tolist()):
        c = cols[int(rowptr[u]): int(rowptr[u + 1])].long() - item_offset
        s[r, c] = -1e10
    return torch.sort(s, dim=1, descending=True, stable=True)[1][:, :k] + item_offset


def _sums_f64(topk, gt_rowptr, gt_items):
    """ops.topk_metric_sums' rows (sums over users) from the reference's metric formulas."""
    tr = pkg("trainer")
    base = int(gt_rowptr[0])
    rp = (gt_rowptr.long() - base).numpy()
    items = gt_items.long().numpy()[base:]
    pos = [items[rp[j]: rp[j + 1]] for j in range(len(rp) - 1)]
    hits = tr.TopKEvaluator.hit_matrix(pos, topk.numpy())
    pl = np.diff(rp)
    n = len(pl)
    rows = [tr.recall_(hits, pl) * n, np.cumsum(hits, axis=1).sum(axis=0), tr.precision_(hits, pl) * n,
            tr.ndcg_(hits, pl) * n, tr.map_(hits, pl) * n]
    return torch.from_numpy(np.stack(rows).astype(np.float64))


def _config(**kw):
    cd = {"device": torch.device("cpu"), "cuda_graph": False, "metrics": METRICS, "topk": [10, 20]}
    cd.update(kw)
    return pkg("config").Config("LightGCN", "scaled", cd)


class _Groups:
    """Held-out items per user in TopKEvaluator's eval_data interface (one process, global users)."""

    def __init__(self, users, items):
        self.users = np.unique(users)
        self.items = [np.sort(items[users == x]) for x in self.users]

    def get_eval_len_list(self):
        return np.array([len(p) for p in self.items], dtype=np.int64)

    def get_eval_items(self):
        return self.items


def _oracle_results(u, i, lab, U0, I0, L):
    """Every metric in one process on the unsharded graph: oracle propagation, float64 top-K with
    all training items masked, TopKEvaluator's numpy hit matrix."""
    tr = pkg("trainer")
    U, I = SHAPE["U"], SHAPE["I"]
    t = lab == 0
    tu, ti = u[t].numpy(), i[t].numpy()
    r, c, v = ograph.norm_adj_f32(tu, ti, U, I)
    G = {"norm_adj": ograph.to_torch_csr(r, c, v, (U + I, U + I), torch.float64)}
    with torch.no_grad():
        uo, io = omodels.lightgcn_forward({"embedding_dict.user_emb": U0, "embedding_dict.item_emb": I0}, G,
                                          {"n_layers": L})
    o = np.lexsort((ti, tu))
    mrp = torch.from_numpy(np.concatenate(([0], np.cumsum(np.bincount(tu, minlength=U)))))
    mcols = torch.from_numpy(ti[o])
    ev = tr.TopKEvaluator(_config())
    out = []
    for label in (1, 2):
        m = (lab == label).numpy()
        g = _Groups(u.numpy()[m], i.numpy()[m])
        ids = _topk_f64(uo, torch.from_numpy(g.users), io, 20, mrp, mcols, 0)
        out.append(ev.evaluate([ids], g))
    return out


def _rank_model(rank, world, L=2, d=16, seed=7):
    par = pkg("parallel")
    U, I = SHAPE["U"], SHAPE["I"]
    u, i, lab = _edges()
    t = lab == 0
    rp = np.concatenate(([0], np.cumsum(np.bincount(u[t].numpy(), minlength=U))))
    bounds = par.partition_by_nnz(rp, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    su, si, sl = _edges(lo, hi)                       # this rank's users only, labelled here
    tr_ = sl == 0
    sb = par.ShardedBipartite.from_local_edges(su[tr_], si[tr_], bounds, rank, world, U, I, recipe="f32",
                                               csr_from_coo=_csr_from_coo)
    gen = torch.Generator().manual_seed(seed)
    U0 = (torch.rand(U, d, generator=gen, dtype=torch.float64) - 0.5) * 0.4
    I0 = (torch.rand(I, d, generator=gen, dtype=torch.float64) - 0.5) * 0.4
    model = par.ShardedLightGCN(sb, d, L, 1e-2, user_emb=U0[lo:hi], item_emb=I0, spmm_fn=_spmm_f64,
                                loss_fns=(_loss_fwd_f64, _loss_bwd_f64), eval_fns=(_topk_f64, _sums_f64))
    valid = par.ShardedEvalData(sb, su[sl == 1], si[sl == 1], batch_users=37)     # several batches per rank
    test = par.ShardedEvalData(sb, su[sl == 2], si[sl == 2], batch_users=37)
    return dict(u=u, i=i, lab=lab, U0=U0, I0=I0, L=L, lo=lo, hi=hi, su=su, si=si, sl=sl, sb=sb, model=model,
                valid=valid, test=test)


def _eval_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        trm = pkg("trainer")
        env = _rank_model(rank, world)
        valid, lab = env["valid"], env["lab"]
        # global denominators from every rank's share
        assert valid.n_users_global == len(np.unique(env["u"][lab == 1].numpy()))
        assert valid.total_pos == float((lab == 1).sum())
        rowptr, items = valid.gt_csr()
        assert rowptr.dtype == torch.int32 and items.dtype == torch.int32
        assert int(valid.eval_u.min()) >= 0 and int(valid.eval_u.max()) < env["hi"] - env["lo"]
        tr = trm.Trainer(_config(), env["model"])
        got = [tr.evaluate(env["valid"]), tr.evaluate(env["test"])]
        assert env["model"]._eval_cache is not None
        env["model"].train()
        assert env["model"]._eval_cache is None
        everyone = [None] * world
        dist.all_gather_object(everyone, got)
        assert all(x == everyone[0] for x in everyone)
        want = _oracle_results(env["u"], env["i"], lab, env["U0"], env["I0"], env["L"])
        assert got == want, (got, want)
        assert set(got[0]) == {f"{m.lower()}@{k}" for m in METRICS for k in (10, 20)}
        assert got[0]["recall@20"] > 0
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_evaluation_matches_single_process(world, tmp_path):
    port = _free_port()
    mp.spawn(_eval_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def _fit_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        data_m, trm = pkg("data"), pkg("trainer")
        env = _rank_model(rank, world)
        t = env["sl"] == 0
        loader = data_m.DeviceTrainLoader(env["su"][t], env["si"][t], env["hi"] - env["lo"], SHAPE["I"], 2048,
                                          seed=5, rank=rank, world=world, user_lo=env["lo"],
                                          sampler=osampler.neg_sample_counter)
        # a large learning rate overshoots after a few epochs, so the validation metric stalls and
        # early stopping ends the run before the last epoch
        tr = trm.Trainer(_config(epochs=12, stopping_step=0, learning_rate=0.5, valid_metric="NDCG@20"),
                         env["model"])
        best, best_valid, best_test = tr.fit(loader, env["valid"], env["test"], verbose=False)
        mine = (sorted(tr.train_loss_dict), best, best_valid, best_test, tr.cur_step)
        everyone = [None] * world
        dist.all_gather_object(everyone, mine)
        assert all(x == everyone[0] for x in everyone)
        assert len(mine[0]) < 12 and best_valid["ndcg@20"] == best > 0
        items = [None] * world
        dist.all_gather_object(items, env["model"].embedding_dict["item_emb"].detach())
        assert all(torch.equal(x, items[0]) for x in items)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_fit_stops_at_the_same_epoch_on_every_rank(world, tmp_path):
    port = _free_port()
    mp.spawn(_fit_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))
