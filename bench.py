#!/usr/bin/env python
"""bench.py -- the reference's headline workload on B200 (see DESIGN.md "Measurement").

Workload (BASELINE.json configs[1]): SMORE on a synthetic Amazon-Baby-shaped dataset
(19,445 users x 7,050 items x 160,792 interactions, 4096-d image / 384-d text features, d = 64,
train batch 2048, the reference trainer's mirror-gradient schedule). One "step" = one iteration of
Trainer._train_epoch's batch loop: in steady state 3 forward+backward passes and 2 Adam steps.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

* `value`   : training interactions/s over all ranks, device-timed (CUDA events, max over ranks)
              with the K batches already resident in HBM.
* `e2e`     : the same metric through the public API (TrainDataLoader -> Trainer._train_batch):
              host negative sampling, pinned H2D copy of every [3, B] batch and a D2H read of the
              loss inside the timed region.
* extras    : train_epoch_s, eval_users_per_s (Trainer.evaluate on the validation users),
              per-kernel rooflines (SpMM GB/s vs measured HBM peak), cpu_baseline,
              torch_cuda_reference (the oracle port on stock torch CUDA kernels, N = 1).
* N > 1     : the training step at Baby size does not shard (single-digit-microsecond kernels): the
              headline value runs replicas (one hyper-parameter grid point per GPU, the reference's
              own outer loop; no collective, weak scaling). The paths that DO shard (SURVEY 8e) run
              in the same invocation, at every N including 1, and are reported under
              `config.sharded_config5` (10M x 2M x 500M graph: user-sharded propagation with a
              chunked, overlapped item-table all-reduce + item-sharded top-50 and merge; strong
              scaling, phase split, clock record, top-K checksum) and `config.sharded_config4`
              (SMORE / Clothing d = 128 with item-range sharded feature tables).
* --impl reference : the reference's CPU implementation of the same step (oracle port on torch
              CPU with all host threads), rank 0 only; builds its inputs without the product.
* --dump-outputs DIR : after the K timed steps, rank 0 writes what the last of them handed its caller
              (see dump_outputs) as DIR/<name>.npy. Data, parameters and batches are seeded, so two builds
              run with the same arguments can be compared output for output.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "recommendar-systems_b200"


def pkg(sub):
    return importlib.import_module(PKG + "." + sub)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            v = json.load(open(os.path.join(ROOT, "profiles", name)))["dram_bytes_per_launch"].get(kernel)
        except (OSError, ValueError, KeyError):
            v = None
        if v is not None:
            return v
    return None


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


_REAL_STDOUT = None


def quiet_nccl():
    """stdout carries exactly one JSON line. NCCL writes its version banner (and whatever else it
    logs) to file descriptor 1 from C, whatever NCCL_DEBUG_FILE says: until the result is printed,
    descriptor 1 points at stderr; `emit` restores it for the one line."""
    global _REAL_STDOUT
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    """Print the result line on the real stdout."""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def build_env(device, seed=999, model_name="SMORE", shape="baby", overrides=None):
    import torch
    synth, cfgm, data_m, models = pkg("synth"), pkg("config"), pkg("data"), pkg("models")
    data = synth.make_dataset(shape)
    cd = {"device": torch.device(device), "data_path": None, "v_feat": data.image_feat,
          "t_feat": data.text_feat, "seed": seed}
    cd.update(overrides or {})
    config = cfgm.Config(model_name, shape, cd)
    ds = data_m.RecDataset(config, data.users, data.items, data.labels)
    tr, va, te = ds.split()
    train = data_m.TrainDataLoader(config, tr, batch_size=config["train_batch_size"], shuffle=True)
    valid = data_m.EvalDataLoader(config, va, additional_dataset=tr, batch_size=config["eval_batch_size"])
    cfgm.init_seed(seed)
    train.pretrain_setup()
    model = models.get_model(model_name)(config, train).to(config["device"])
    return dict(config=config, data=data, tr=tr, train=train, valid=valid, model=model)


def take_batches(loader, n):
    out = []
    while len(out) < n:
        for b in loader:
            out.append(b)
            if len(out) == n:
                loader.pr = 0
                break
    return out


DUMP_MAX_BYTES = 64 << 20       # whole dump
DUMP_MAX_ELEMS = 1 << 20        # one array; a larger parameter is cut to a sample of its rows


def dump_outputs(out_dir, loss, model):
    """Write what a training step hands its caller -- the loss it returned and every parameter it
    updated -- as float32 `<name>.npy` files (`loss.npy`, `<parameter name>.npy`) under `out_dir`.
    A parameter of more than DUMP_MAX_ELEMS elements keeps a sample of its rows, the same in every
    run: ascending row ids drawn by a generator seeded with 0 that is used for nothing else, so the
    training's own random streams are not advanced."""
    import numpy as np
    import torch
    arrays = {"loss": loss.detach().float().reshape(-1)}
    for name, p in model.named_parameters():
        t = p.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            keep = max(1, DUMP_MAX_ELEMS * t.shape[0] // t.numel())
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        arrays[name] = t.float()
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def time_kernel(fn, flush, iters=20, warm=3):
    """Mean device time (ms) of fn() with the L2 flushed before every timed launch."""
    import torch
    for _ in range(warm):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        flush.zero_()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / iters


# L2 -> SM crossbar peak of the B200 as ncu reports it (derived__lts__lts2xbar_bytes.sum.peak_sustained in
# profiles/r02_kernels_ncu_raw.csv): the bound of the row gathers of a CSR SpMM, which move nnz * 4 d bytes
# through the L2 whatever the HBM traffic is (on the 600k x 120k graph ncu measures 10.7 TB/s = 91 % of it)
L2_XBAR_PEAK_GBS = 11776.0


def _l2_view(g, d, ms, extra_rows=0):
    """Bytes a row-gather SpMM pulls through the L2 (every gathered row, the CSR arrays, the output and
    epilogue rows) against the crossbar peak."""
    b = g.nnz * (8 + 4 * d) + 4 * (g.n_rows + 1) + 4 * d * g.n_rows * (1 + extra_rows)
    return {"l2_bytes": b, "l2_achieved": b / ms / 1e6, "l2_peak": L2_XBAR_PEAK_GBS,
            "l2_frac": b / ms / 1e6 / L2_XBAR_PEAK_GBS}


def kernel_rooflines(env, peak):
    """Per-kernel achieved algorithmic GB/s (SURVEY 8d byte formulas), L2 flushed per launch."""
    import torch
    ops = pkg("ops")
    model, dev = env["model"], env["config"]["device"]
    d = model.embedding_dim
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # 2 x L2
    out = []
    g = model.norm_adj
    X = torch.randn(g.n_cols, d, device=dev)
    Y = torch.empty(g.n_rows, d, device=dev)
    ms = time_kernel(lambda: ops.spmm_raw(g, X, Y=Y), flush)
    b = g.algorithmic_bytes(d)
    out.append({"kernel": "spmm_csr_kernel (UI graph, one layer)", "bytes": b, "ms": ms,
                "achieved": b / ms / 1e6, "frac": b / ms / 1e6 / peak, **_l2_view(g, d, ms)})
    acc = torch.empty_like(X)
    ms = time_kernel(lambda: ops.spmm_raw(g, X, Y=Y, acc_in=X, acc_out=acc), flush)
    # SURVEY 8(d): a fused L-layer propagation = L x the SpMM bytes + ONE 4 d N write of the
    # accumulated output; per launch that is b + 4 d N / L (the running sum the epilogue re-reads and
    # re-writes every layer is not algorithmic traffic)
    L = int(model.n_ui_layers)
    b2 = b + 4 * d * g.n_rows // max(L, 1)
    out.append({"kernel": "spmm_csr_kernel (UI graph, fused layer-sum)", "bytes": b2, "ms": ms,
                "achieved": b2 / ms / 1e6, "frac": b2 / ms / 1e6 / peak, **_l2_view(g, d, ms, extra_rows=2)})
    gi = model.fusion_adj
    Xi = torch.randn(gi.n_cols, d, device=dev)
    Yi = torch.empty(gi.n_rows, d, device=dev)
    ms = time_kernel(lambda: ops.spmm_raw(gi, Xi, Y=Yi), flush)
    b = gi.algorithmic_bytes(d)
    out.append({"kernel": "spmm_csr_kernel (fusion item-item graph)", "bytes": b, "ms": ms,
                "achieved": b / ms / 1e6, "frac": b / ms / 1e6 / peak})
    # spectral: 2 rows in, 3 rows out
    n = model.n_items
    img, txt = torch.randn(n, d, device=dev), torch.randn(n, d, device=dev)
    w = [model.image_complex_weight[0].detach(), model.text_complex_weight[0].detach(),
         model.fusion_complex_weight[0].detach()]
    ms = time_kernel(lambda: ops.spectrum_convolution(img, txt, *w, True), flush)
    b = 4 * n * d * 5
    out.append({"kernel": "spectral_fwd_kernel", "bytes": b, "ms": ms, "achieved": b / ms / 1e6,
                "frac": b / ms / 1e6 / peak})
    # the table-sized projection GEMMs (image table 7050 x 4096 fp32 = 115 MB, streamed once)
    table = model.image_embedding.weight.detach()
    Wt, bt = model.image_trs.weight.detach(), model.image_trs.bias.detach()
    n, F = table.shape
    dy = torch.randn(n, d, device=dev)
    b = 4 * (n * F + d * F + n * d)
    for name, fn in (("gemm_tc05_kernel (image projection forward)", lambda: ops.gemm(table, True, Wt, True, n, d, F, bt)),
                     ("gemm_tc05_kernel (image projection dW)", lambda: ops.gemm(dy, False, table, False, d, F, n)),
                     ("gemm_tc05_kernel (image projection dX)", lambda: ops.gemm(dy, True, Wt, False, n, F, d))):
        ms = time_kernel(fn, flush)
        out.append({"kernel": name, "bytes": b, "ms": ms, "achieved": b / ms / 1e6, "frac": b / ms / 1e6 / peak})
    # the optimizer pass: p, g, m, v read + p, m, v written = 28 bytes per parameter
    opt = pkg("optim").FusedAdam([torch.nn.Parameter(torch.randn(n, F, device=dev))], lr=1e-3)
    opt.param_groups[0]["params"][0].grad = torch.randn(n, F, device=dev)
    opt.step()
    ms = time_kernel(lambda: opt.step(), flush)
    b = 28 * n * F
    out.append({"kernel": "adam_kernel (image table)", "bytes": b, "ms": ms, "achieved": b / ms / 1e6,
                "frac": b / ms / 1e6 / peak})
    # the same table updated from the factors of its gradient (never materialised): 24 B / parameter
    par = torch.nn.Parameter(torch.randn(n, F, device=dev))
    opt2 = pkg("optim").FusedAdam([par], lr=1e-3)

    def lowrank_step():
        par._mmrec_lowrank = ops.LowRankGrad(dy, Wt)
        opt2.step()
        par._mmrec_lowrank = None
    ms = time_kernel(lowrank_step, flush)
    b = 24 * n * F
    out.append({"kernel": "gemm_tc05_kernel<adam> (image table, low-rank gradient, TMA-streamed)", "bytes": b,
                "ms": ms, "achieved": b / ms / 1e6, "frac": b / ms / 1e6 / peak})
    del opt, opt2, par, dy
    # a user-item graph whose embedding table (184 MB) does not fit the 126 MB L2
    del X, Y, acc
    su, si = pkg("synth").make_scaled_edges(dev, 600_000, 120_000, 30_000_000)
    gl = pkg("graph").build_ui_graph(su, si, 600_000, 120_000, "f64eps")
    del su, si
    X = torch.randn(gl.n_cols, d, device=dev)
    Y = torch.empty(gl.n_rows, d, device=dev)
    ms = time_kernel(lambda: ops.spmm_raw(gl, X, Y=Y), flush, iters=10)
    b = gl.algorithmic_bytes(d)
    gather = gl.nnz * (8 + 4 * d) + 4 * (gl.n_rows + 1) + 4 * d * gl.n_rows
    out.append({"kernel": f"spmm_csr_kernel (scaled UI graph 600k x 120k, nnz {gl.nnz}, > L2)", "bytes": b,
                "ms": ms, "achieved": b / ms / 1e6, "frac": b / ms / 1e6 / peak,
                "no_reuse_gather_bytes": gather, "no_reuse_gather_gbps": gather / ms / 1e6, **_l2_view(gl, d, ms)})
    for o in out:
        o["unit"] = "GB/s"
    return out


def in_step_kernel_times(trainer, batches, patterns):
    """Average device duration (ms) and launches per step of the kernels whose name contains one
    of `patterns`, measured with the profiler's CUDA activity records (CUPTI) over extra replays of
    the SAME captured step the timed region ran: the live in-step figure, L2 state and co-running
    kernels included."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for b in batches:
                trainer._train_batch_graphed(b)
            torch.cuda.synchronize()
        out = {}
        for pat in patterns:
            evs = [e for e in prof.key_averages() if pat in e.key and e.device_time_total > 0]
            n = sum(e.count for e in evs)
            if n:
                out[pat] = {"ms": sum(e.device_time_total for e in evs) / n / 1e3, "per_step": n / len(batches)}
        return out
    except Exception as exc:                    # profiler unavailable: the isolated figures stand
        sys.stderr.write(f"in-step kernel timing skipped: {exc}\n")
        return {}


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        # stdout carries exactly one JSON line: keep NCCL's version banner off it
        quiet_nccl()
        dist.init_process_group("nccl", device_id=torch.device(dev))
    lib = pkg("lib")
    lib.load()
    trainer_m = pkg("trainer")
    env = build_env(dev, seed=999 + rank)                # one grid point (seed) per replica
    model, config = env["model"], env["config"]
    trainer = trainer_m.Trainer(config, model)
    B = config["train_batch_size"]
    K, W = args.steps, args.warmup
    batches = take_batches(env["train"], W + K)
    model.train()
    # clocks / throttle reasons are sampled every 50 ms from before the warm-up until the end of the
    # end-to-end loop (the device-timed K steps alone last a few tens of ms: too short for nvidia-smi)
    sampler = ClockSampler(local)
    sampler.start()
    # The steady-state step is replayed from a CUDA graph that is captured on the 5th step (two eager
    # runs per control-flow variant first): with W < 6 a few extra untimed steps go in front, so that
    # the K timed steps are the steady state whatever W the caller chose.
    for b in take_batches(env["train"], max(0, 6 - W)) + batches[:W]:
        trainer._train_batch_graphed(b)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    l0 = lib.launch_count() + trainer.replayed_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("timed_steps")          # ncu --nvtx --nvtx-include "timed_steps/"
    e0.record()
    for b in batches[W:]:
        loss = trainer._train_batch_graphed(b)
    e1.record()
    torch.cuda.nvtx.range_pop()
    barrier()
    launches = lib.launch_count() + trainer.replayed_launches - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * K * B / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model)     # before the end-to-end epochs train on

    # ---- end to end through the public API: loader (host sampling, pinned H2D) + loss D2H
    # Trainer._train_epoch with the reference's per-batch `loss.item()` (sync_free off): every step
    # draws its batch in the loader, copies it from pinned memory and reads its loss back
    # Whole epochs (the unit the reference's trainer works in: one shuffle of the interactions per
    # epoch, 65 steps at Baby size), at least K steps; three times, median -- one host hiccup in a
    # ~170 ms window would otherwise decide the number.
    trainer.sync_free = False
    n_train_rows = len(env["tr"])
    steps_per_epoch_e2e = -(-n_train_rows // B)
    n_epochs_e2e = max(1, -(-K // steps_per_epoch_e2e))
    for _e in range(3):                     # untimed: the ragged last batch of an epoch gets its own step graph
        trainer._train_epoch(env["train"], 0)   # (captured the third time its shape is seen, like every variant)
    reps = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        done = 0
        for _e in range(n_epochs_e2e):
            _, lb = trainer._train_epoch(env["train"], 0)
            done += len(lb)
        barrier()
        reps.append(time.perf_counter() - t0)
    e2e_rows = n_epochs_e2e * n_train_rows  # interactions actually trained on in the timed region
    e2e_s = sorted(reps)[1]
    e2e_steps = done
    trainer.sync_free = True
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * e2e_rows / e2e_s

    # ---- full-rank evaluation (valid users): e2e (incl. D2H + host metrics) and device only
    n_eval = int(env["valid"].eval_u.shape[0])
    for _ in range(3):                       # eager pass, capture pass, first replay
        trainer.evaluate(env["valid"])
    barrier()
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        metrics = trainer.evaluate(env["valid"])          # Trainer.evaluate: result dict on the host
    torch.cuda.synchronize()
    eval_s = (time.perf_counter() - t0) / reps
    a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("timed_eval")
    a.record()
    trainer.evaluate(env["valid"])
    b_.record()
    torch.cuda.nvtx.range_pop()
    torch.cuda.synchronize()
    eval_dev_ms = a.elapsed_time(b_)

    # ---- the paths that shard, on these same N ranks (config 5, then config 4); rank 0 gets the blocks
    del batches
    sharded5 = sharded4 = None
    if not args.no_sharded_blocks:
        try:
            sharded5 = scaled_block(dev, rank, world, local, scale=args.scale, eval_users=args.eval_users,
                                    steps=10, warmup=3, chunks=args.chunks, partition=args.partition,
                                    rt_block_users=args.rt_block_users)
        except Exception as exc:                      # never lose the headline line to an auxiliary block
            sharded5 = {"error": repr(exc)[:300]} if rank == 0 else None
            if world > 1:
                raise
        torch.cuda.empty_cache()
        try:
            sharded4 = clothing_block(dev, rank, world)
        except Exception as exc:
            sharded4 = {"error": repr(exc)[:300]} if rank == 0 else None
            if world > 1:
                raise
        torch.cuda.empty_cache()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    batches = take_batches(env["train"], W + K)
    peak, peak_src = measured_peaks()
    live = in_step_kernel_times(trainer, batches[W:W + min(K, 5)], ["spmm_csr_kernel<", "adam_kernel", "gemm_tc05_kernel"])
    kr = kernel_rooflines(env, peak)
    dom = dict(kr[1])   # the launch propagate_mean issues: SpMM + fused layer sum over the UI graph
    dom["isolated_ms"], dom["isolated_frac"] = dom["ms"], dom["frac"]
    if "spmm_csr_kernel<" in live:
        # every UI-graph launch of a training step carries the layer-sum epilogue: same bytes
        dom["ms"] = live["spmm_csr_kernel<"]["ms"]
        dom["achieved"] = dom["bytes"] / dom["ms"] / 1e6
        dom["frac"] = dom["achieved"] / peak
        dom["launches_per_step"] = live["spmm_csr_kernel<"]["per_step"]
    n_train = len(env["tr"])
    steps_per_epoch = -(-n_train // B)
    line = {
        "metric": METRIC,
        "value": value, "unit": "interactions/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "l2": "per-step working set (~1.7 GB of tables/optimizer state) exceeds the 126 MB L2; "
                         "kernel rooflines flush L2 before every timed launch",
                   "multi_gpu": "headline value: replicas (one seed per GPU), no collective -- the Baby-sized step "
                                "does not shard; the sharded designs are measured in sharded_config5 / sharded_config4",
                   "sharded_config5": sharded5, "sharded_config4": sharded4},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "interactions/s", "h2d_bytes_per_step": 3 * B * 8,
                "d2h_bytes_per_step": 4, "steps_timed": int(e2e_steps),
                "how": "whole epochs through Trainer._train_epoch (loader shuffle + native negative sampling, pinned "
                       "H2D of every [3, B] batch, loss.item() per step), wall clock, median of 3"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak,
                     "peak_source": peak_src, "unit": "GB/s", "frac": dom["frac"], "traffic": ncu_traffic(dom["kernel"]),
                     "traffic_source": "ncu --set full capture committed under profiles/ (r02_ncu_traffic.json, else r01)",
                     "algorithmic_bytes_per_launch": dom["bytes"], "ms_per_launch": dom["ms"],
                     "timing": "average duration of the kernel's launches inside replays of the timed step "
                               "(CUPTI activity records); isolated_* = one launch after an L2 flush, CUDA events",
                     "launches_per_step": dom.get("launches_per_step"),
                     "isolated_ms_per_launch": dom["isolated_ms"], "isolated_frac": dom["isolated_frac"],
                     "in_step": live,
                     "l2_bound": {"note": "what bounds this kernel is not HBM: every gathered row crosses the L2 -> SM "
                                          "crossbar (nnz * 4 d bytes per launch whatever the DRAM traffic); peak = ncu "
                                          "derived__lts__lts2xbar_bytes.sum.peak_sustained",
                                  "bytes_per_launch": dom.get("l2_bytes"), "peak": L2_XBAR_PEAK_GBS, "unit": "GB/s",
                                  "achieved": (dom["l2_bytes"] / dom["ms"] / 1e6) if dom.get("l2_bytes") else None,
                                  "frac": (dom["l2_bytes"] / dom["ms"] / 1e6 / L2_XBAR_PEAK_GBS) if dom.get("l2_bytes") else None}},
        "kernels": kr,
        "train_epoch_s": steps_per_epoch * ms / K / 1e3,
        "train_epoch_s_e2e": e2e_s / n_epochs_e2e,
        "eval_users_per_s": n_eval / eval_s, "eval_users_per_s_device": n_eval / (eval_dev_ms / 1e3),
        "eval_users": n_eval, "eval_recall@20": metrics.get("recall@20"),
    }
    # whole-step roofline of SURVEY 8(d): ~5.0 GB of algorithmic traffic per steady-state step
    line["step_roofline"] = {"algorithmic_gb_per_step": 5.0, "achieved_gbs": 5.0e9 / (ms / K / 1e3) / 1e9, "peak": peak,
                             "frac": 5.0e9 / (ms / K / 1e3) / 1e9 / peak,
                             "note": "SURVEY 8(d) epoch roofline: 3 x 0.77 GB fwd+bwd + 2 x 0.94 GB Adam + 0.8 GB mirror "
                                     "passes; the low-rank table gradients remove ~1.3 GB of that from what is actually moved"}
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(env, steps=20, warmup=3)
        try:
            del env, trainer, model
            torch.cuda.empty_cache()
            line["torch_cuda_reference"] = torch_cuda_reference(dev)
        except Exception as exc:
            line["torch_cuda_reference"] = {"error": repr(exc)[:300]}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


WORKLOAD = ("SMORE, synthetic Amazon-Baby-shaped (19445 users x 7050 items x 160792 interactions, 4096-d image / "
            "384-d text, d=64, batch 2048, mirror-gradient schedule: steady-state step = 3 fwd+bwd + 2 Adam)")
METRIC = "train interactions/s (SMORE, Baby-shaped; epoch s and eval users/s in extras)"


def oracle_trainer_for(env):
    """The reference's CPU path for the same step: oracle port on torch CPU (our arm's cpu_baseline:
    same parameters and batches as the model that was just timed)."""
    import torch
    from oracle import build as obuild
    from oracle.train import OracleTrainer
    data, tr, config = env["data"], env["tr"], env["config"]
    cfg = {k: config[k] for k in ("n_ui_layers", "n_layers", "image_knn_k", "text_knn_k", "reg_weight",
                                  "cl_loss", "train_batch_size")}
    G, _ = obuild.build_graphs("SMORE", tr.users, tr.items, data.n_users, data.n_items, data.image_feat,
                               data.text_feat, cfg)
    P = {k: v.detach().cpu() for k, v in env["model"].state_dict().items()}
    drop = torch.nn.Dropout(p=config["dropout_rate"])
    return OracleTrainer("SMORE", P, G, cfg, lr=config["learning_rate"],
                         lr_scheduler=tuple(config["learning_rate_scheduler"]), dropout=drop)


def cpu_baseline(env, steps, warmup):
    import torch
    torch.set_num_threads(os.cpu_count())
    ot = oracle_trainer_for(env)
    B = env["config"]["train_batch_size"]
    batches = [b.cpu() for b in take_batches(env["train"], warmup + steps)]
    for b in batches[:warmup]:
        ot.step(b)
    t0 = time.perf_counter()
    for b in batches[warmup:]:
        ot.step(b)
    dt = time.perf_counter() - t0
    return {"value": steps * B / dt, "unit": "interactions/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{steps} steady-state (mirror-gradient) SMORE training steps of the same workload "
                      f"after {warmup} warm-up steps, oracle port on torch CPU; {dt / steps:.2f} s/step"}


# ---- the reference arm: inputs built WITHOUT the product (no model, no CUDA library) ------------
def oracle_smore_inputs(seed=999, n_batches=8):
    """Synthetic Baby-shaped data, the oracle's graphs, SMORE parameters initialised like the model
    (xavier id embeddings, nn.Linear defaults, randn spectral weights) and [3, B] training batches
    -- from synth.py (numpy), config.py (constants) and oracle/ only: the reference arm never maps
    the product's shared library."""
    import numpy as np
    import torch
    import torch.nn as nn
    from oracle import build as obuild
    synth, cfgm = pkg("synth"), pkg("config")
    data = synth.make_dataset("baby")
    tu, ti = data.split(0)
    mc = dict(cfgm.OVERALL)
    mc.update(cfgm.MODEL_DEFAULTS["SMORE"])
    cfg = {k: mc[k] for k in ("n_ui_layers", "n_layers", "image_knn_k", "text_knn_k", "reg_weight", "cl_loss",
                              "train_batch_size")}
    G, parts = obuild.build_graphs("SMORE", tu, ti, data.n_users, data.n_items, data.image_feat, data.text_feat, cfg)
    torch.manual_seed(seed)
    d = mc["embedding_size"]
    P = {"user_embedding.weight": nn.init.xavier_uniform_(torch.empty(data.n_users, d)),
         "item_id_embedding.weight": nn.init.xavier_uniform_(torch.empty(data.n_items, d)),
         "image_embedding.weight": torch.from_numpy(data.image_feat).clone(),
         "text_embedding.weight": torch.from_numpy(data.text_feat).clone()}

    def lin(name, n_in, n_out, bias=True):
        m = nn.Linear(n_in, n_out, bias=bias)
        P[name + ".weight"] = m.weight.detach().clone()
        if bias:
            P[name + ".bias"] = m.bias.detach().clone()
    lin("image_trs", data.image_feat.shape[1], d)
    lin("text_trs", data.text_feat.shape[1], d)
    for q in ("query_v", "query_t"):
        lin(q + ".0", d, d)
        lin(q + ".2", d, d, bias=False)
    for gname in ("gate_v", "gate_t", "gate_f", "gate_image_prefer", "gate_text_prefer", "gate_fusion_prefer"):
        lin(gname + ".0", d, d)
    for w in ("image_complex_weight", "text_complex_weight", "fusion_complex_weight"):
        P[w] = torch.randn(1, d // 2 + 1, 2)
    # batches: shuffled training edges + one uniform negative per row outside the user's history
    rng = np.random.default_rng(seed)
    B = cfg["train_batch_size"]
    order = rng.permutation(len(tu))
    key = np.sort(tu.astype(np.int64) * data.n_items + ti)
    batches = []
    for b in range(n_batches):
        sel = order[(b * B) % len(tu):][:B]
        if len(sel) < B:
            sel = order[:B]
        u, pos = tu[sel].astype(np.int64), ti[sel].astype(np.int64)
        neg = rng.integers(0, data.n_items, size=B)
        for _ in range(50):
            k = u * data.n_items + neg
            at = np.minimum(np.searchsorted(key, k), len(key) - 1)
            bad = key[at] == k
            if not bad.any():
                break
            neg[bad] = rng.integers(0, data.n_items, size=int(bad.sum()))
        batches.append(torch.from_numpy(np.stack([u, pos, neg])))
    return dict(data=data, cfg=cfg, mc=mc, G=G, parts=parts, P=P, batches=batches, n_train=len(tu))


def _oracle_trainer(inp, P, G):
    import torch
    from oracle.train import OracleTrainer
    mc = inp["mc"]
    return OracleTrainer("SMORE", P, G, inp["cfg"], lr=mc["learning_rate"],
                         lr_scheduler=tuple(mc["learning_rate_scheduler"]), dropout=torch.nn.Dropout(p=mc["dropout_rate"]))


def torch_cuda_reference(dev, steps=10, warmup=4):
    """The honest neighbour of the GPU-over-CPU ratio (BASELINE.md section 3): the same oracle port
    -- the reference's torch expressions: torch.sparse.mm on uncoalesced COO adjacencies, nn.Linear,
    torch.fft, torch Adam -- on stock torch CUDA kernels on this B200."""
    import numpy as np
    import torch
    inp = oracle_smore_inputs()
    n, I, U = inp["data"].n_users + inp["data"].n_items, inp["data"].n_items, inp["data"].n_users
    shapes = {"norm_adj": (n, n), "R": (U, I)}
    G = {}
    for k, (r, c, v) in inp["parts"].items():
        idx = torch.from_numpy(np.vstack([r, c]).astype(np.int64))
        G[k] = torch.sparse_coo_tensor(idx, torch.as_tensor(v), shapes.get(k, (I, I))).to(dev)   # uncoalesced, like the reference
    P = {k: v.to(dev) for k, v in inp["P"].items()}
    ot = _oracle_trainer(inp, P, G)
    batches = [b.to(dev) for b in inp["batches"]]
    B = inp["cfg"]["train_batch_size"]
    for s_ in range(warmup):
        ot.step(batches[s_ % len(batches)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s_ in range(steps):
        ot.step(batches[s_ % len(batches)])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": steps * B / dt, "unit": "interactions/s", "ms_per_step": dt / steps * 1e3,
            "what": "oracle port of the reference's SMORE step on stock torch CUDA kernels (cuSPARSE COO SpMM, "
                    f"cuBLAS, cuFFT, torch.optim.Adam), {steps} steady-state steps after {warmup} warm-up, wall clock "
                    "with synchronize on both sides"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count())
    K, W = args.steps, args.warmup
    inp = oracle_smore_inputs(n_batches=max(8, min(W + K, 32)))
    B = inp["cfg"]["train_batch_size"]
    ot = _oracle_trainer(inp, inp["P"], inp["G"])
    batches = inp["batches"]
    for s_ in range(W):
        ot.step(batches[s_ % len(batches)])
    t0 = time.perf_counter()
    for s_ in range(K):
        ot.step(batches[(W + s_) % len(batches)])
    dt = time.perf_counter() - t0
    value = K * B / dt
    line = {"impl": "reference", "metric": METRIC,
            "value": value, "unit": "interactions/s", "n_gpus": int(os.environ.get("WORLD_SIZE", 1)),
            "steps": K, "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "arm": "reference CPU path: oracle port (restatement of the reference's torch expressions) on "
                              "torch CPU, all host threads; inputs built from synth + oracle only"},
            "cpu_baseline": {"value": value, "unit": "interactions/s", "cores": torch.get_num_threads(),
                             "kind": "port", "sample": f"{K} training steps after {W} warm-up steps"},
            "e2e": {"value": value, "unit": "interactions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "train_epoch_s": -(-inp["n_train"] // B) * dt / K}
    print(json.dumps(line))


# ---- the paths that shard (SURVEY 8e): run inside every `--gpus N` invocation -------------------
def _phase_ms(timing, steps):
    import torch
    torch.cuda.synchronize()
    return {k: sum(a.elapsed_time(b) for a, b in v) / steps for k, v in timing.items()}


def scaled_block(dev, rank, world, local, scale=1.0, eval_users=16384, steps=10, warmup=3, chunks=4,
                 partition="auto", rt_block_users=393216):
    """Config 5: scaled power-law graph (scale 1.0 = 10M users x 2M items x ~500M interactions),
    LightGCN-style 4-layer propagation + full-rank top-50 for `eval_users` users per step. Strong
    scaling: N = 1 runs the single-GPU operators on the whole graph; N > 1 shards users by non-zeros
    (every rank generates and keeps ONLY its own edges), replicates the item table through a chunked
    all-reduce that runs under the SpMMs, and scores items in N ranges with a K-way merge.
    Returns the result block on rank 0 (None elsewhere)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    ops, G, par, synth, lib = pkg("ops"), pkg("graph"), pkg("parallel"), pkg("synth"), pkg("lib")
    U, I, E = int(10_000_000 * scale), int(2_000_000 * scale), int(500_000_000 * scale)
    d, L, k, Bu = 64, 4, 50, eval_users
    sampler = ClockSampler(local)      # from the graph build on: the timed steps alone last < 0.3 s at 8 GPUs
    sampler.start()
    if partition == "auto":
        # best measured layout per N (profiles/r02_config5_spmm_experiments.txt): one GPU runs the
        # symmetric CSR over the stacked table in one launch per layer; several GPUs shard users
        partition = "full" if world == 1 else "bipartite"
    gen = torch.Generator(device=dev).manual_seed(999)
    bound = (6.0 / (U + I + d)) ** 0.5
    users = torch.randint(0, U, (Bu,), generator=gen, device=dev)

    def x0_rows(lo, hi):
        """Rows [lo, hi) of the xavier-uniform [U + I, d] table, generated in fixed 1M-row blocks
        (the same values whatever the sharding)."""
        out = []
        blk = 1 << 20
        for b0 in range(lo // blk * blk, hi, blk):
            b1 = min(U + I, b0 + blk)
            g = torch.Generator(device=dev).manual_seed(4000 + b0 // blk)
            x = (torch.rand(b1 - b0, d, generator=g, device=dev) * 2 - 1) * bound
            out.append(x[max(lo, b0) - b0: min(hi, b1) - b0])
        return torch.cat(out)

    if world == 1 and partition == "full":
        su, si = synth.make_scaled_edges(dev, U, I, E)
        nnz_local = int(su.numel())
        full = G.build_ui_graph(su, si, U, I, "f64eps")
        del su, si
        X0 = x0_rows(0, U + I)
    elif partition == "rows":
        su, si = synth.make_scaled_edges(dev, U, I, E)
        nnz_local = int(su.numel())
        full = G.build_ui_graph(su, si, U, I, "f64eps")
        del su, si
        sg = par.ShardedUIGraph(full, rank, world)
        lo_i, hi_i = par.item_range(I, rank, world)
        del full
        X0 = x0_rows(0, U + I)
    else:
        deg = synth.scaled_degrees(dev, U, E)
        rp = np.concatenate(([0], np.cumsum(deg.cpu().numpy())))
        bounds = par.partition_by_nnz(rp, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        su, si = synth.make_scaled_edges(dev, U, I, E, user_range=(lo, hi))
        nnz_local = int(su.numel())
        sb = par.ShardedBipartite.from_local_edges(su, si, bounds, rank, world, U, I, "f64eps",
                                                   rt_block_users=rt_block_users)
        del su, si, deg
        Xu, Xi = x0_rows(lo, hi), x0_rows(U, U + I)
    torch.cuda.empty_cache()
    timing = {}

    def ev(name):
        e = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        timing.setdefault(name, []).append(e)
        e[0].record()
        return e

    def step(tm):
        if world == 1 and partition == "full":
            e = ev("propagate_spmm_x4") if tm is not None else None
            out = ops.propagate_mean(full, X0, L)
            if e:
                e[1].record()
            e = ev("score_topk") if tm is not None else None
            ids = ops.score_mask_topk(out[:U], users, out[U:], k)
            if e:
                e[1].record()
            return ids
        if partition == "rows":
            out = par.sharded_propagate_mean(sg, X0, L)
            return par.sharded_score_topk(out[:U], users, out[U + lo_i: U + hi_i].contiguous(), lo_i, k)
        ou, oi = par.bipartite_propagate_mean(sb, Xu, Xi, L, chunks=chunks, timing=tm)
        e = ev("score_topk_merge") if tm is not None else None
        ids = ops.score_mask_topk(ou, users, oi, k) if world == 1 else par.bipartite_score_topk(sb, ou, oi, users, k)
        if e:
            e[1].record()
        return ids

    with torch.no_grad():
        for _ in range(warmup):
            ids = step(None)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ids = step(timing)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        launches = lib.launch_count() - l0
        clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    phases = _phase_ms(timing, steps)
    checksum = int(ids.sum().item())
    nnz_total = nnz_local
    if world > 1:
        t = torch.tensor([ms] + [phases[k_] for k_ in sorted(phases)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0].item())
        phases = {k_: float(v) for k_, v in zip(sorted(phases), t[1:].tolist())}
        chk = torch.tensor([float(checksum)], device=dev, dtype=torch.float64)
        lo_, hi_ = chk.clone(), chk.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        assert lo_.item() == hi_.item(), "ranks disagree on the merged top-K"
        nz = torch.tensor([nnz_local], device=dev, dtype=torch.int64)
        dist.all_reduce(nz)
        nnz_total = int(nz.item())
    if rank != 0:
        return None
    peak, peak_src = measured_peaks()
    n = U + I
    nnz = 2 * nnz_total                                     # symmetric adjacency: both directions
    spmm_bytes = L * (8 * nnz + 4 * (n + 1) + 8 * d * n)    # SURVEY 8(d): L x one SpMM over the whole graph
    spmm_ms = phases.get("propagate_spmm_x4") or (phases.get("rt_spmm", 0.0) + phases.get("r_spmm", 0.0))
    block = {"workload": f"LightGCN-style propagation (4 layers) + full-rank top-50, {U} users x {I} items x {nnz_total} "
                         f"interactions (scale {scale}), d=64, {Bu} eval users per step",
             "metric": "eval users/s", "value": Bu * steps / (ms / 1e3), "n_gpus": world, "scaling": "strong",
             "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "phases_ms_per_step_max_over_ranks": phases,
             "rt_block_users": rt_block_users if partition == "bipartite" else None,
             "partition": ("single GPU, symmetric CSR over the stacked table" if partition == "full" else
                           "single GPU, bipartite: R (users x items) row-split; R^T (items x users) in user blocks of "
                           f"{rt_block_users} rows whose vectors stay L2-resident") if world == 1 else
                          ("rows by nnz + all-gather of the whole table per layer" if partition == "rows" else
                           f"users by nnz (each rank builds only its own edges), items replicated: item-table all-reduce in "
                           f"{chunks} chunks per layer issued under the SpMMs (waited for right before the next layer's user-side "
                           "SpMM); evaluation: items by range + all-gather of (score, id) lists + K-way merge"),
             "collective_note": "rt_spmm / r_spmm are enqueue-to-completion spans on the compute stream; exposed_all_reduce is "
                                "the time the compute stream spent waiting for NCCL beyond them",
             "clocks": clocks, "gpu_launches": int(launches), "checksum_ids": checksum}
    if spmm_ms > 0:
        gbs = spmm_bytes / (spmm_ms / 1e3) / 1e9
        block["spmm_roofline"] = {"algorithmic_bytes_per_step": spmm_bytes, "spmm_ms_per_step": spmm_ms,
                                  "achieved_gbs_all_gpus": gbs, "peak_gbs_per_gpu": peak, "peak_source": peak_src,
                                  "frac_of_n_gpu_peak": gbs / (peak * world)}
    return block


def clothing_block(dev, rank, world, steps=10, warmup=8):
    """Config 4: SMORE on the Clothing-shaped dataset, d = 128; N > 1 shards the [I, 4096] / [I, 384]
    feature tables, their projections, gradients and Adam state by item range (SURVEY 8e row 2)."""
    import torch
    import torch.distributed as dist
    over = {"embedding_size": 128}
    if world > 1:
        over["table_shard"] = (rank, world)
    env = build_env(dev, model_name="SMORE", shape="clothing", overrides=over)
    trainer = pkg("trainer").Trainer(env["config"], env["model"])
    batches = take_batches(env["train"], warmup + steps)
    env["model"].train()
    env["model"].pre_epoch_processing()
    losses = []
    for b in batches[:warmup]:
        losses.append(trainer._train_batch_graphed(b))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for b in batches[warmup:]:
        losses.append(trainer._train_batch_graphed(b))
    e.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(e) / steps], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    last = float(torch.stack(losses).float()[-1].item())
    B = env["config"]["train_batch_size"]
    del env, trainer
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    return {"workload": "SMORE, synthetic Clothing-shaped (39387 x 23033 x 278677), d=128, batch 2048, mirror-gradient "
                        "schedule", "n_gpus": world, "steps": steps, "warmup": warmup,
            "partition": "single GPU (low-rank table gradients, fused table Adam)" if world == 1 else
                         "item-range sharded feature tables (projection all-gather, dW all-reduce); the rest replicated",
            "ms_per_step": float(t.item()), "value": B / float(t.item()) * 1e3, "metric": "train interactions/s",
            "scaling": "strong", "last_loss": last}


def run_scaled(args):
    """`--workload scaled`: config 5 alone (see scaled_block)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        quiet_nccl()
        dist.init_process_group("nccl", device_id=torch.device(dev))
    pkg("lib").load()
    blk = scaled_block(dev, rank, world, local, scale=args.scale, eval_users=args.eval_users, steps=args.steps,
                       warmup=args.warmup, chunks=args.chunks, partition=args.partition,
                       rt_block_users=args.rt_block_users)
    if rank == 0:
        line = {"metric": "propagate (4 layers) + full-rank top-50, eval users/s (scaled power-law graph)",
                "value": blk["value"], "unit": "users/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": blk["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": blk, "clocks": blk["clocks"],
                "gpu_launches": blk["gpu_launches"]}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="smore_baby", choices=["smore_baby", "scaled"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--eval-users", type=int, default=16384)
    ap.add_argument("--partition", default="auto", choices=["auto", "bipartite", "rows", "full"])
    ap.add_argument("--rt-block-users", type=int, default=393216,
                    help="user rows per L2-resident column block of R^T (0 = unblocked)")
    ap.add_argument("--chunks", type=int, default=4)
    ap.add_argument("--no-sharded-blocks", action="store_true",
                    help="skip the config-5 / config-4 blocks of the default workload (quick runs, ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and parameters after the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "smore_baby"):
        ap.error("--dump-outputs applies to the default workload (--impl ours --workload smore_baby)")
    if args.workload == "scaled" and args.impl == "ours":
        run_scaled(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
