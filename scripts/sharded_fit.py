"""LightGCN trained AND evaluated on config 5's graph (scaled power-law, 10M users x 2M items x ~486M
interactions, d = 64, 4 layers) with parallel.ShardedLightGCN, one process per GPU:

    python scripts/sharded_fit.py --gpus N [--epochs 2] [--scale 1.0] [--batch 1048576] [--precision bf16]

The generated edges are split into train / valid / test (synth.scaled_edge_labels, 0.8 / 0.1 /
0.1, each user's first edge train); every rank labels only its own users' edges. The normalised
graph and the per-rank loader are built from the training edges, the per-rank evaluation data
(parallel.ShardedEvalData) from the held-out ones, and trainer.Trainer.fit runs the reference's
loop: an epoch of eager steps, then full-rank Recall / Recall2 / Precision / NDCG / MAP on valid
and test (training items masked, top-K over all items), early stopping on valid Recall@20.
Prints one JSON line: per-epoch training loss and ms/step, the valid and test result dicts, the
best-valid epoch, seconds and evaluated users/s per evaluation pass, peak memory per rank (GiB
allocated by torch) and the GPU's name, power limit and clocks read in the same run."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402  (ClockSampler, quiet_nccl, emit, pkg)
from sharded_train import BATCH_NOTE, gpu_info  # noqa: E402

METRICS = ["Recall", "Recall2", "Precision", "NDCG", "MAP"]
TOPK = [10, 20, 50]


def worker(rank, world, args):
    import numpy as np
    import torch
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    torch.cuda.set_device(rank)
    dev = f"cuda:{rank}"
    if world > 1:
        bench.quiet_nccl()
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(dev))
    par, synth, data_m, trm, cfgm = (bench.pkg(m) for m in ("parallel", "synth", "data", "trainer", "config"))
    bench.pkg("lib").load()
    U, I, E = int(10_000_000 * args.scale), int(2_000_000 * args.scale), int(500_000_000 * args.scale)
    d, L = 64, 4
    sampler = bench.ClockSampler(rank)
    sampler.start()
    t_setup = time.perf_counter()
    deg = synth.scaled_degrees(dev, U, E)
    rp = np.concatenate(([0], np.cumsum(deg.cpu().numpy())))
    bounds = par.partition_by_nnz(rp, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    del deg
    su, si = synth.make_scaled_edges(dev, U, I, E, user_range=(lo, hi))
    lab = synth.scaled_edge_labels(su, si)
    counts = torch.bincount(lab, minlength=3)
    t = lab == 0
    sb = par.ShardedBipartite.from_local_edges(su[t], si[t], bounds, rank, world, U, I, "f64eps",
                                               rt_block_users=args.rt_block_users)
    loader = data_m.DeviceTrainLoader(su[t], si[t], hi - lo, I, args.batch, seed=999, rank=rank, world=world,
                                      user_lo=lo)
    valid = par.ShardedEvalData(sb, su[lab == 1], si[lab == 1], batch_users=args.eval_users)
    test = par.ShardedEvalData(sb, su[lab == 2], si[lab == 2], batch_users=args.eval_users)
    del su, si, lab, t
    model = par.ShardedLightGCN(sb, d, L, 1e-2, chunks=args.chunks, precision=args.precision)
    cfg = cfgm.Config("LightGCN", "scaled", {"device": torch.device(dev), "cuda_graph": False, "epochs": args.epochs,
                                             "eval_step": 1, "stopping_step": args.stopping_step, "metrics": METRICS,
                                             "topk": TOPK, "valid_metric": "Recall@20"})
    trainer = trm.Trainer(cfg, model)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup
    torch.cuda.empty_cache()
    setup_peak = torch.cuda.max_memory_allocated() / 2 ** 30
    torch.cuda.reset_peak_memory_stats()

    # Trainer.fit unchanged; its epoch and evaluation calls are timed from the outside
    epochs, passes = [], []
    train_epoch, evaluate = trainer._train_epoch, trainer.evaluate

    def timed_epoch(data, epoch_idx, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss, batches = train_epoch(data, epoch_idx, **kw)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        epochs.append({"epoch": epoch_idx, "train_loss": float(loss), "steps": len(batches),
                       "ms_per_step": dt * 1e3 / max(1, len(batches)), "seconds": dt})
        return loss, batches

    def timed_eval(eval_data, *a, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = evaluate(eval_data, *a, **kw)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        passes.append({"split": "valid" if eval_data is valid else "test", "epoch": epochs[-1]["epoch"],
                       "seconds": dt, "eval_users_per_s": eval_data.n_users_global / dt, "result": res})
        return res

    trainer._train_epoch, trainer.evaluate = timed_epoch, timed_eval
    best_score, best_valid, best_test = trainer.fit(loader, valid, test, verbose=False)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    peak = torch.cuda.max_memory_allocated() / 2 ** 30
    pk = torch.tensor([setup_peak, peak], dtype=torch.float64, device=dev)
    peaks = [[setup_peak, peak]]
    t_max = torch.tensor([e["ms_per_step"] for e in epochs] + [p["seconds"] for p in passes], dtype=torch.float64,
                         device=dev)
    cnt = torch.stack([counts.to(dev), torch.tensor([sb.nnz_local, 0, 0], device=dev)])
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt)
        allpk = torch.empty(world, 2, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allpk, pk)
        peaks = allpk.tolist()
    t_max = t_max.tolist()
    for e, v in zip(epochs, t_max[:len(epochs)]):
        e["ms_per_step"] = v                          # slowest rank
    for p, v in zip(passes, t_max[len(epochs):]):
        p["seconds"] = v
        p["eval_users_per_s"] = (valid if p["split"] == "valid" else test).n_users_global / v
    info = gpu_info(rank)
    if rank == 0:
        vpass = [p for p in passes if p["split"] == "valid"]
        key = "recall@20"
        best_epoch = None
        best = -1.0
        for p in vpass:                               # early_stopping's rule: strictly better
            if p["result"][key] > best:
                best, best_epoch = p["result"][key], p["epoch"]
        n_split = cnt[0].tolist()
        line = {"metric": "LightGCN fit with full-rank evaluation on the user-sharded graph (config 5)",
                "n_gpus": world, "epochs_run": len(epochs), "epochs_max": args.epochs,
                "workload": f"{U} users x {I} items x {sum(n_split)} interactions (scale {args.scale}) split "
                            f"train / valid / test = {n_split}, d={d}, {L} layers, reg_weight 1e-2, FusedAdam "
                            f"lr {cfg['learning_rate']}",
                "global_batch": args.batch, "batch_note": BATCH_NOTE,
                "epochs": epochs, "eval_passes": passes,
                "eval_note": "seconds per pass = evaluation forward (4 layers) + score / mask / top-K of every "
                             "evaluated user against all items + metrics + one [5, K] all-reduce, slowest rank; "
                             "the first pass also checks the mask CSR",
                "valid_eval_users": valid.n_users_global, "test_eval_users": test.n_users_global,
                "best_valid_epoch": best_epoch, "best_valid_result": best_valid, "best_test_upon_valid": best_test,
                "valid_metric": "recall@20", "best_valid_score": best_score, "setup_seconds_rank0": setup_s,
                "peak_mem_gib_setup_per_rank": [p[0] for p in peaks],
                "peak_mem_gib_fit_per_rank": [p[1] for p in peaks], "chunks": args.chunks,
                "rt_block_users": args.rt_block_users, "precision": args.precision,
                "eval_users_per_launch": args.eval_users,
                "gpu": info, "clocks": clocks}
        bench.emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--epochs", type=int, default=2)
    ap.add_argument("--stopping-step", type=int, default=20)
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--chunks", type=int, default=4)
    ap.add_argument("--rt-block-users", type=int, default=393216)
    ap.add_argument("--precision", choices=["fp32", "bf16"], default="fp32",
                    help="operand precision of the propagation SpMMs (parallel.bipartite_propagate_mean)")
    ap.add_argument("--eval-users", type=int, default=1 << 17)
    args = ap.parse_args()
    if args.gpus == 1:
        worker(0, 1, args)
        return
    import torch.multiprocessing as mp
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(s.getsockname()[1])
    s.close()
    mp.spawn(worker, args=(args.gpus, args), nprocs=args.gpus, join=True)


if __name__ == "__main__":
    main()
