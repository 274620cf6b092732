"""CPU tests: loaders / sampler / evaluator vs the reference's golden vectors, C-ABI exports."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import REPO, TINY, golden, pkg


def _env(model="LightGCN", overrides=None):
    synth, cfgm, data_m = pkg("synth"), pkg("config"), pkg("data")
    data = synth.make_dataset("tiny", **TINY)
    cd = {"device": torch.device("cpu"), "train_batch_size": 512, "eval_batch_size": 64,
          "data_path": None}
    cd.update(overrides or {})
    config = cfgm.Config(model, "tiny", cd)
    ds = data_m.RecDataset(config, data.users, data.items, data.labels)
    tr, va, te = ds.split()
    train = data_m.TrainDataLoader(config, tr, batch_size=512, shuffle=True)
    valid = data_m.EvalDataLoader(config, va, additional_dataset=tr, batch_size=64)
    test = data_m.EvalDataLoader(config, te, additional_dataset=tr, batch_size=64)
    return config, data, train, valid, test


def test_train_loader_replays_reference_batches():
    """Same shuffle (numpy global RNG) and same negatives (Python random) as the reference."""
    g = golden("tiny_lightgcn")
    config, data, train, valid, test = _env()
    pkg("config").init_seed(999)
    train.pretrain_setup()
    assert train.all_items == g["all_items_shuffled"].tolist()
    it = iter(train)
    b0, b1 = next(it), next(it)
    assert b0.dtype == torch.int64 and tuple(b0.shape) == (3, 512)
    assert np.array_equal(b0.numpy(), g["batch0"])
    assert np.array_equal(b1.numpy(), g["batch1"])
    n = 2 + sum(1 for _ in it)
    assert n == len(train) == int(np.ceil(len(train.dataset) / 512))


def test_negatives_never_in_history():
    config, data, train, valid, test = _env()
    pkg("config").init_seed(3)
    train.pretrain_setup()
    for b in train:
        u, neg = b[0].tolist(), b[2].tolist()
        assert all(n not in train.history_items_per_u[x] for x, n in zip(u, neg))


def test_native_sampler_replays_cpython_random():
    """mmrec_neg_sample_mt19937_host draws the same negatives as random.sample(all_items, 1)[0]
    with history rejection and leaves Python's global Mersenne Twister in the same state."""
    import random
    config, data, train, valid, test = _env()
    for seed in (999, 7):
        pkg("config").init_seed(seed)
        train.pretrain_setup()
        st = random.getstate()
        users = train.dataset.users[:1500]
        want = train._sample_neg_ids(users.tolist())
        after_py = random.getstate()
        random.setstate(st)
        got = train._sample_neg_ids_native(users)
        assert got.tolist() == want
        assert random.getstate() == after_py
        assert random.random() == (random.setstate(after_py) or random.random())
    # tiny item universes exercise the rejection loop of _randbelow (n not a power of two)
    L = pkg("lib")
    items = np.array([5, 3, 9], dtype=np.int64)
    rowptr = np.array([0, 1, 1], dtype=np.int64)
    cols = np.array([3], dtype=np.int64)
    u = np.array([0, 1] * 200, dtype=np.int64)
    random.seed(11)
    st = random.getstate()
    ref = []
    for x in u.tolist():
        iid = random.sample(items.tolist(), 1)[0]
        while x == 0 and iid == 3:
            iid = random.sample(items.tolist(), 1)[0]
        ref.append(iid)
    mt = np.array(st[1], dtype=np.uint32)
    out = np.empty(len(u), dtype=np.int64)
    L.call("mmrec_neg_sample_mt19937_host", mt.ctypes.data, items.ctypes.data, 3, rowptr.ctypes.data,
           cols.ctypes.data, 2, u.ctypes.data, len(u), out.ctypes.data)
    assert out.tolist() == ref
    assert tuple(mt.tolist()) == random.getstate()[1]
    # error behaviour: a user who has seen everything cannot be sampled for
    full = np.array([0, 3], dtype=np.int64)
    with pytest.raises(RuntimeError):
        L.call("mmrec_neg_sample_mt19937_host", mt.ctypes.data, items.ctypes.data, 3, full.ctypes.data,
               np.array([3, 5, 9], dtype=np.int64).ctypes.data, 1, np.zeros(1, np.int64).ctypes.data, 1,
               out.ctypes.data)


def test_eval_loader_matches_reference():
    g = golden("tiny_lightgcn")
    config, data, train, valid, test = _env()
    b = next(iter(valid))
    valid.pr = valid.inter_pr = 0
    assert np.array_equal(b[0].numpy(), g["eval_batch_users"])
    assert np.array_equal(b[1].numpy(), g["eval_batch_mask"])
    # the CSR view of the same mask: ascending item ids per user
    rp, cols = valid.mask_csr(0, 64)
    rp, cols = rp.numpy(), cols.numpy()
    m = g["eval_batch_mask"]
    for r in range(64):
        assert sorted(m[1][m[0] == r].tolist()) == cols[rp[r]:rp[r + 1]].tolist()
    # iteration covers every eval user exactly once, ragged last batch included
    seen = torch.cat([bb[0] for bb in valid])
    assert torch.equal(seen, valid.eval_u) and len(valid) == int(np.ceil(len(seen) / 64))


@pytest.mark.parametrize("tag", ["tiny_lightgcn", "tiny_smore", "tiny_freedom"])
def test_evaluator_metrics_match_reference(tag):
    g = golden(tag)
    config, data, train, valid, test = _env()
    ev = pkg("trainer").TopKEvaluator(config)
    topk = g["fit/valid_topk"]
    hits = ev.hit_matrix(valid.get_eval_items(), topk)
    slow = np.asarray([[i in set(m.tolist()) for i in n] for m, n in zip(valid.get_eval_items(), topk)])
    assert np.array_equal(hits, slow)
    raw = ev._calculate_metrics(valid.get_eval_len_list(), hits)
    assert list(g["fit/metric_names"]) == ev.metrics
    np.testing.assert_allclose(raw, g["fit/valid_metrics_raw"], rtol=1e-12, atol=0)
    out = ev.evaluate([torch.from_numpy(topk)], valid)
    keys = [str(k) for k in g["fit/metric_keys"]]
    assert [out[k] for k in keys] == pytest.approx(g["fit/valid"][-1].tolist(), abs=1e-12)


def test_evaluator_rejects_bad_args():
    config, *_ = _env()
    config["metrics"] = ["Recall", "Nope"]
    with pytest.raises(ValueError):
        pkg("trainer").TopKEvaluator(config)
    config["metrics"], config["topk"] = ["Recall"], [0]
    with pytest.raises(ValueError):
        pkg("trainer").TopKEvaluator(config)


def test_tsv_round_trip(tmp_path):
    synth, cfgm, data_m = pkg("synth"), pkg("config"), pkg("data")
    data = synth.make_dataset("tiny", **TINY)
    d = synth.write_reference_layout(data, str(tmp_path))
    config = cfgm.Config("LightGCN", "tiny", {"device": torch.device("cpu")})
    ds = data_m.RecDataset(config, path=os.path.join(d, "tiny.inter"))
    assert ds.user_num == data.n_users and ds.item_num == data.n_items
    assert np.array_equal(ds.users, data.users) and np.array_equal(ds.labels, data.labels)


def test_synth_shapes():
    synth = pkg("synth")
    for name in ("tiny", "small"):
        d = synth.make_dataset(name, features=False)
        U, I, E = synth.SHAPES[name]
        assert len(d.users) == E and d.users.max() == U - 1 and d.items.max() == I - 1
        assert len(np.unique(d.users * I + d.items)) == E
        first = np.concatenate(([0], np.flatnonzero(np.diff(d.users)) + 1))
        assert (d.labels[first] == 0).all()


def test_c_abi_exports_every_declared_symbol():
    """The library loads without a GPU and exports exactly what include/mmrec_b200.h declares."""
    lib = pkg("lib")
    hdr = open(os.path.join(REPO, "include", "mmrec_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(mmrec_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    L = lib.load()
    for name in declared:
        assert hasattr(L, name)
    assert L.mmrec_abi_version() == 1


def test_ctypes_signatures_have_the_header_arity():
    """Every prototype of include/mmrec_b200.h and its ctypes mirror (lib.SIGNATURES) take the same number of
    arguments, pointer arguments are bound as pointers and `void *stream` comes last where the header has it: a
    miscounted argtypes list would otherwise only show up as a wrong result on the GPU."""
    import ctypes
    lib = pkg("lib")
    hdr = open(os.path.join(REPO, "include", "mmrec_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    hdr = re.sub(r"//[^\n]*", "", hdr)
    protos = re.findall(r"\b(mmrec_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", hdr)
    assert len(protos) == len(lib.SIGNATURES)
    for name, args in protos:
        args = [a.strip() for a in args.split(",")] if args.strip() not in ("", "void") else []
        res, argtypes = lib.SIGNATURES[name]
        assert len(args) == len(argtypes), (name, len(args), len(argtypes))
        for a, t in zip(args, argtypes):
            assert ("*" in a) == (t is ctypes.c_void_p), (name, a, t)
        if args and re.search(r"void\s*\*\s*stream$", args[-1]):
            assert argtypes[-1] is ctypes.c_void_p, name


def test_product_does_not_import_oracle():
    root = os.path.join(REPO, "recommendar-systems_b200")
    for fn in os.listdir(root):
        if fn.endswith(".py"):
            src = open(os.path.join(root, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_ops_fail_loudly_without_cuda():
    """No CPU / eager fallback anywhere on the product path: host tensors are an error."""
    ops, graph = pkg("ops"), pkg("graph")
    with pytest.raises(RuntimeError):
        graph.build_ui_graph(torch.zeros(4, dtype=torch.int64), torch.zeros(4, dtype=torch.int64), 2, 2, "f32")
    x = torch.randn(8, 64)
    W, b = torch.randn(64, 64), torch.randn(64)
    idx = torch.zeros(4, dtype=torch.int64)
    calls = [
        lambda: ops.linear(x, W, b),
        lambda: ops.colsum(x),
        lambda: ops.inject3(x, x, x, x, 0.7),
        lambda: ops.knn_graph(x, 2, "sym"),
        lambda: ops.spectrum_convolution(x, x, torch.randn(33, 2), torch.randn(33, 2), torch.randn(33, 2)),
        lambda: ops.bpr_table(x, 4, idx, idx, idx),
        lambda: ops.infonce_pair(x, x, 4, idx, idx, 0.2),
        lambda: ops.score_mask_topk(x, idx, x, 2),
        lambda: ops.loss_head(torch.zeros(2), torch.zeros(2), 4, 0.1, 4, 0.1),
        lambda: ops.gather_batch_rows([x], idx, idx, idx, 4),
    ]
    for i, fn in enumerate(calls):
        with pytest.raises((RuntimeError, ValueError), match=None):
            fn()


def test_accelerate_passes_cpu_calls_through_untouched():
    """The interception mode only takes CUDA float32 calls; on the host it must be transparent."""
    acc = pkg("accelerate")
    idx = torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]])
    a = torch.sparse_coo_tensor(idx, torch.tensor([1.0, 2.0, 3.0, 4.0]), (3, 3))
    x = torch.arange(12, dtype=torch.float32).reshape(3, 4)
    want = torch.sparse.mm(a, x)
    with acc.accelerate() as mode:
        got = torch.sparse.mm(a, x)
    assert torch.equal(got, want) and mode.stats == {"spmm": 0, "converted": 0, "passed": 1}


class _FakeLoader:
    """Yields [3, B] LongTensors and records when batches are drawn (trainer.py:186 loop contract)."""

    def __init__(self, n):
        self.n, self.pr, self.drawn = n, 0, []

    def __iter__(self):
        self.pr = 0
        return self

    def __next__(self):
        if self.pr >= self.n:
            self.pr = 0
            raise StopIteration
        self.pr += 1
        self.drawn.append(self.pr - 1)
        return torch.full((3, 4), self.pr - 1, dtype=torch.long)


class _FakeModel(torch.nn.Module):
    def __init__(self, nan_at=None):
        super().__init__()
        self.w = torch.nn.Parameter(torch.ones(1))
        self.nan_at, self.seen = nan_at, []

    def calculate_loss(self, interaction):
        b = int(interaction[0, 0])
        self.seen.append(b)
        loss = (self.w * float(b + 1)).sum()
        return loss * float("nan") if b == self.nan_at else loss

    def pre_epoch_processing(self):
        pass


def _host_trainer(model, sync_free):
    cfg = pkg("config").Config("LightGCN", "tiny", {"device": torch.device("cpu"), "learner": "sgd",
                                                    "learning_rate": 0.0, "sync_free": sync_free})
    return pkg("trainer").Trainer(cfg, model)


@pytest.mark.parametrize("sync_free", [True, False])
def test_train_epoch_pipelined_loop_keeps_the_reference_contract(sync_free):
    """trainer.py:186-203: every batch is trained once and in order, the epoch loss is the sum of the
    per-batch losses, whether the loss is read back per batch (one step behind) or once per epoch."""
    model, loader = _FakeModel(), _FakeLoader(7)
    tr = _host_trainer(model, sync_free)
    total, batches = tr._train_epoch(loader, 0)
    assert model.seen == list(range(7)) and loader.drawn == list(range(7)) and len(batches) == 7
    assert abs(total - sum(range(1, 8))) < 1e-6
    # an abandoned epoch stops after max_batches and leaves the loader ready for a clean restart
    model.seen.clear()
    total, batches = tr._train_epoch(loader, 0, max_batches=3)
    assert model.seen == [0, 1, 2] and len(batches) == 3 and abs(total - 6.0) < 1e-6 and loader.pr == 0


def test_train_epoch_nan_aborts_like_the_reference_one_batch_late_at_most():
    """trainer.py:201-203: a NaN loss ends the epoch with (loss, tensor(0.0)); with the lagged
    read-back the abort comes at most one batch after the NaN."""
    model, loader = _FakeModel(nan_at=2), _FakeLoader(7)
    tr = _host_trainer(model, sync_free=False)
    loss, flag = tr._train_epoch(loader, 0)
    assert torch.is_tensor(loss) and bool(torch.isnan(loss)) and float(flag) == 0.0
    assert model.seen[:3] == [0, 1, 2] and len(model.seen) <= 4
    model2 = _FakeModel(nan_at=2)
    tr2 = _host_trainer(model2, sync_free=True)
    loss2, _ = tr2._train_epoch(_FakeLoader(7), 0)
    assert torch.is_tensor(loss2) and bool(torch.isnan(loss2))


def test_epoch_shuffle_prefetch_draws_the_same_permutations(tiny_data):
    """Trainer._train_epoch shuffles for the NEXT epoch while the device runs the last steps of the
    current one (TrainDataLoader.prefetch_shuffle): the loader then skips its shuffle at iter(). Same
    numpy draws in the same order -> the same batches as without the prefetch, epoch after epoch, and
    never a second shuffle; the last epoch of a run draws nothing extra."""
    import random
    cfgm, data_m = pkg("config"), pkg("data")
    seen = {}
    for prefetch in (False, True):
        cfg = cfgm.Config("LightGCN", "tiny", {"device": torch.device("cpu"), "learner": "sgd", "learning_rate": 0.0,
                                                "sync_free": True, "epochs": 3, "prefetch_epoch_shuffle": prefetch,
                                                "is_multimodal_model": False, "data_path": None})
        ds = data_m.RecDataset(cfg, tiny_data.users, tiny_data.items, tiny_data.labels)
        tr_split = ds.split()[0]
        loader = data_m.TrainDataLoader(cfg, tr_split, batch_size=cfg["train_batch_size"], shuffle=True)
        cfgm.init_seed(999)
        loader.pretrain_setup()

        class Rec(torch.nn.Module):
            def __init__(self):
                super().__init__()
                self.w = torch.nn.Parameter(torch.ones(1))
                self.batches = []

            def calculate_loss(self, interaction):
                self.batches.append(interaction.clone())
                return (self.w * 1.0).sum()

            def pre_epoch_processing(self):
                pass

        model = Rec()
        tr = pkg("trainer").Trainer(cfg, model)
        shuffles = []
        orig = loader._shuffle
        loader._shuffle = lambda: (shuffles.append(len(model.batches)), orig())[1]
        for epoch in range(3):
            tr._train_epoch(loader, epoch)
        n_per = len(loader)
        # one shuffle per epoch; with the prefetch they happen when the previous epoch's batches are all drawn
        assert len(shuffles) == 3
        assert shuffles == ([0, n_per, 2 * n_per] if prefetch else [0, n_per, 2 * n_per])
        seen[prefetch] = (torch.stack([b for b in model.batches if b.shape[1] == model.batches[0].shape[1]]),
                          np.random.get_state()[1].copy(), random.getstate())
    assert torch.equal(seen[False][0], seen[True][0])
    assert np.array_equal(seen[False][1], seen[True][1]) and seen[False][2] == seen[True][2]


def test_bench_dump_outputs_is_a_seeded_float32_sample(tmp_path):
    """bench.py --dump-outputs: the loss and every parameter as float32 .npy; a parameter above the per-array
    limit keeps the same ascending sample of its rows on every call, and the global numpy / torch random
    streams the training draws from are not advanced."""
    import bench
    model = torch.nn.Module()
    n_rows = bench.DUMP_MAX_ELEMS // 8 + 3
    model.big = torch.nn.Parameter(torch.arange(n_rows, dtype=torch.float32).repeat_interleave(8).reshape(n_rows, 8))
    model.small = torch.nn.Linear(3, 2).double()
    np.random.seed(5)
    torch.manual_seed(5)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.5), model)
    assert np.random.randint(1 << 30) == np.random.RandomState(5).randint(1 << 30)
    assert torch.equal(torch.rand(4), torch.rand(4, generator=torch.Generator().manual_seed(5)))
    names = {"loss.npy", "big.npy", "small.weight.npy", "small.bias.npy"}
    assert set(os.listdir(tmp_path / "a")) == names
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.load(tmp_path / "a" / "loss.npy").tolist() == [1.5]
    assert np.array_equal(np.load(tmp_path / "a" / "small.weight.npy"), model.small.weight.detach().float().numpy())
    big = np.load(tmp_path / "a" / "big.npy")
    assert big.size <= bench.DUMP_MAX_ELEMS and big.shape[1] == 8
    rows = big[:, 0]
    assert np.all(np.diff(rows) > 0) and rows[-1] < n_rows and np.array_equal(big, np.repeat(rows[:, None], 8, 1))
