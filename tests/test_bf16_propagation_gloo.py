"""world_size-2/3 gloo tests (CPU) of the bf16 propagation mode of the user-sharded LightGCN
(parallel.ShardedLightGCN(precision="bf16")). The SpMM is injected in float64: it reads the bfloat16
operand exactly and writes the rounded user rows to y16, so the only rounding is the contract's;
the one-process oracle is tests/bf16_ref.py on the whole graph. The CUDA kernel is covered by
tests/test_gpu_bf16_propagation.py."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from bf16_ref import PropagateBf16
from conftest import pkg
from oracle import graph as ograph
from oracle import models as omodels
from oracle import ops as oops
from test_sharded_train_gloo import GAMMA, _free_port, _loader, _loss_bwd_f64, _loss_fwd_f64, _setup


def _spmm_f64_bf16(g, X, Y=None, acc_in=None, acc_out=None, scale=1.0, y16=None):
    """The CUDA operator's contract in float64: X must be bfloat16 (every gathered operand is),
    y16 receives y rounded to bfloat16."""
    assert X.dtype == torch.bfloat16, X.dtype
    rp = g.row_ptr.long()
    base = int(rp[0])
    A = torch.sparse_csr_tensor(rp - base, g.col_idx.long()[base: int(rp[-1])] - g.col_offset,
                                g.vals.double()[base: int(rp[-1])], size=(g.n_rows, g.n_cols))
    y = torch.sparse.mm(A, X.double()[: g.n_cols])
    if Y is not None:
        Y.copy_(y)
    if y16 is not None:
        assert y16.dtype == torch.bfloat16
        y16.copy_(y)
    if acc_out is not None:
        acc_out.copy_(((acc_in + y) if acc_in is not None else y) * scale)


def _oracle_loss(P, A, L, rw, union, U):
    X = PropagateBf16.apply(torch.cat([P["embedding_dict.user_emb"], P["embedding_dict.item_emb"]]), A, L)
    ue, ie = X[:U], X[U:]
    u, p, n = union[0], union[1], union[2]
    reg = oops.emb_loss(P["embedding_dict.user_emb"][u], P["embedding_dict.item_emb"][p],
                        P["embedding_dict.item_emb"][n])
    return oops.bpr_gamma_mean(ue[u], ie[p], ie[n], GAMMA) + rw * reg


def _bf16_worker(rank, world, port, out_dir):
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
        model = par.ShardedLightGCN(sb, d, L, rw, user_emb=U0[lo:hi], item_emb=I0, spmm_fn=_spmm_f64_bf16,
                                    loss_fns=(_loss_fwd_f64, _loss_bwd_f64), gamma=GAMMA, precision="bf16")
        assert model.precision == "bf16"
        opt = torch.optim.Adam(model.parameters(), lr=lr)
        r, c, v = ograph.norm_adj_f32(env["u"], env["i"], U, I)
        A = ograph.to_torch_csr(r, c, v, (U + I, U + I), torch.float64)
        P = {"embedding_dict.user_emb": U0.clone().requires_grad_(True),
             "embedding_dict.item_emb": I0.clone().requires_grad_(True)}
        ref_opt = torch.optim.Adam(list(P.values()), lr=lr)
        it = iter(_loader(env, rank, world, batch_size=256))
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
            ref = _oracle_loss(P, A, L, rw, union, U)
            if step == 0:                      # the mode rounds: the fp32-mode loss is a different number
                with torch.no_grad():
                    exact = omodels.lightgcn_loss(P, {"norm_adj": A}, {"n_layers": L, "reg_weight": rw}, union)
                assert abs(exact.item() - ref.item()) > 1e-7 * abs(ref.item())
            ref.backward()
            ref_opt.step()
            assert abs(loss.item() - ref.item()) <= 1e-9 * abs(ref.item()), (step, loss.item(), ref.item())
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
        # the evaluation forward of the same model (eval mode, no autograd) gives the same item table on
        # every rank as well
        model.eval()
        uo, io = model.restore_embeddings()
        outs = [None] * world
        dist.all_gather_object(outs, io)
        assert all(torch.equal(t, outs[0]) for t in outs)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_bf16_sharded_lightgcn_matches_single_process(world, tmp_path):
    port = _free_port()
    mp.spawn(_bf16_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_unknown_precision_rejected():
    par = pkg("parallel")
    env = _setup(0, 1)
    sb, d = env["sb"], 8
    Xu = torch.zeros(env["hi"] - env["lo"], d, dtype=torch.float64)
    Xi = torch.zeros(env["I"], d, dtype=torch.float64)
    for bad in ("fp16", "bfloat16", None):
        with pytest.raises(ValueError):
            par.ShardedLightGCN(sb, d, 2, user_emb=Xu, item_emb=Xi, loss_fns=(None, None), precision=bad)
        with pytest.raises(ValueError):
            par.bipartite_propagate_mean(sb, Xu, Xi, 2, spmm_fn=_spmm_f64_bf16, precision=bad)
        with pytest.raises(ValueError):
            par.bipartite_propagate(sb, Xu, Xi, 2, spmm_fn=_spmm_f64_bf16, precision=bad)
