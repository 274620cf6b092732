"""LightGCN training on config 5's graph (scaled power-law, 10M users x 2M items x ~486M
interactions, d = 64, 4 layers) with parallel.ShardedLightGCN, one process per GPU:

    python scripts/sharded_train.py --gpus N [--steps 10] [--warmup 3] [--batch 1048576] [--precision bf16]

Every rank generates and keeps only its own users' edges (as bench.scaled_block does, including
the L2-resident user blocks of R^T), draws per-rank batches with data.DeviceTrainLoader and is
driven by trainer.Trainer's eager step (FusedAdam over the local user rows + the replicated item
table). Prints one JSON line: ms/step, interactions/s, parallel efficiency against the committed
1-GPU line (profiles/r03_sharded_train_1gpu.json), a phase split from CUDA events, peak memory per
rank (GiB allocated by torch: of the set-up -- graph build, loader sort -- and of the training
steps) and the GPU's name, power limit and clocks read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (ClockSampler, quiet_nccl, emit, pkg)

BATCH_NOTE = ("global batch 2^20 interactions: with the reference's 2048 an epoch of ~486M interactions would be "
              "~237k steps, each a full-graph propagation forward and backward")


def gpu_info(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except (OSError, subprocess.TimeoutExpired):
        return {"name": None}


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
    deg = synth.scaled_degrees(dev, U, E)
    rp = np.concatenate(([0], np.cumsum(deg.cpu().numpy())))
    bounds = par.partition_by_nnz(rp, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    su, si = synth.make_scaled_edges(dev, U, I, E, user_range=(lo, hi))
    del deg
    sb = par.ShardedBipartite.from_local_edges(su, si, bounds, rank, world, U, I, "f64eps",
                                               rt_block_users=args.rt_block_users)
    loader = data_m.DeviceTrainLoader(su, si, hi - lo, I, args.batch, seed=999, rank=rank, world=world, user_lo=lo)
    del su, si
    model = par.ShardedLightGCN(sb, d, L, 1e-2, chunks=args.chunks, precision=args.precision)
    cfg = cfgm.Config("LightGCN", "scaled", {"device": torch.device(dev), "cuda_graph": False})
    trainer = trm.Trainer(cfg, model)
    torch.cuda.empty_cache()
    setup_peak = torch.cuda.max_memory_allocated() / 2 ** 30
    torch.cuda.reset_peak_memory_stats()
    it = iter(loader)
    nnz_local = loader.users.numel()

    def run(n, timing):
        model.timing = timing
        opt = trainer.optimizer
        hooks = []
        if timing is not None:
            span = {}
            hooks = [opt.register_step_pre_hook(lambda *a: span.update(ev=par._span(timing, "adam"))),
                     opt.register_step_post_hook(lambda *a: par._end(span["ev"]))]
        losses, inter = [], 0
        for _ in range(n):
            batch = next(it)
            inter += batch.shape[1]
            losses.append(trainer._train_batch(batch))
        for h in hooks:
            h.remove()
        model.timing = None
        return losses, inter

    run(args.warmup, None)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    timing = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    losses, inter = run(args.steps, timing)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    phases = {k: sum(a.elapsed_time(b) for a, b in v) / args.steps for k, v in timing.items()}
    keys = sorted(phases)
    peak = torch.cuda.max_memory_allocated() / 2 ** 30
    t = torch.tensor([ms] + [phases[k] for k in keys], dtype=torch.float64, device=dev)
    cnt = torch.tensor([inter, nnz_local], dtype=torch.int64, device=dev)
    pk = torch.tensor([setup_peak, peak], dtype=torch.float64, device=dev)
    peaks = [[setup_peak, peak]]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt)
        allpk = torch.empty(world, 2, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allpk, pk)
        peaks = allpk.tolist()
    ms = float(t[0])
    phases = dict(zip(keys, t[1:].tolist()))
    last_loss = float(losses[-1].item())
    info = gpu_info(rank)
    if rank == 0:
        inter_total, nnz_total = int(cnt[0]), int(cnt[1])
        eff = None
        ref = os.path.join(ROOT, "profiles", "r03_sharded_train_1gpu.json")
        if world > 1 and os.path.exists(ref):
            ms1 = json.load(open(ref))["ms_per_step"]
            eff = ms1 / (world * ms)
        line = {"metric": "LightGCN training step on the user-sharded graph (config 5), ms/step", "n_gpus": world,
                "ms_per_step": ms, "interactions_per_s": inter_total / args.steps / (ms / 1e3),
                "parallel_efficiency_vs_1gpu": 1.0 if world == 1 else eff,
                "steps": args.steps, "warmup": args.warmup, "global_batch": args.batch, "batch_note": BATCH_NOTE,
                "steps_per_epoch": len(loader),
                "workload": f"{U} users x {I} items x {nnz_total} training interactions (scale {args.scale}), d={d}, "
                            f"{L} layers, reg_weight 1e-2, FusedAdam",
                "phases_ms_per_step_max_over_ranks": phases,
                "phase_note": "forward_propagation / backward_propagation are enqueue-to-completion spans of the "
                              "propagation (rt_spmm / r_spmm are its SpMMs, forward and backward together); loss is the "
                              "loss kernels + the scalar all-reduce; exposed_all_reduce is the time the compute stream "
                              "waited for NCCL (inside the propagation spans, plus the item regulariser gradient); adam "
                              "is the FusedAdam step",
                "peak_mem_gib_setup_per_rank": [p[0] for p in peaks],
                "peak_mem_gib_steps_per_rank": [p[1] for p in peaks], "last_loss": last_loss, "chunks": args.chunks,
                "rt_block_users": args.rt_block_users, "precision": args.precision, "gpu": info, "clocks": clocks}
        bench.emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--chunks", type=int, default=4)
    ap.add_argument("--rt-block-users", type=int, default=393216)
    ap.add_argument("--precision", choices=["fp32", "bf16"], default="fp32",
                    help="operand precision of the propagation SpMMs (parallel.bipartite_propagate_mean)")
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
