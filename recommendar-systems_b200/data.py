"""Dataset and loaders with the reference's batch formats and RNG call sequence.

Mirror of /root/reference/src/utils/dataset.py:21-133 and
/root/reference/src/utils/dataloader.py:15-418, restated on numpy arrays (no pandas):

* train batch  = LongTensor[3, B] on device: users, pos items, neg items (dataloader.py:226-250);
* eval batch   = [LongTensor[Bu] users, LongTensor[2, nnz] (batch-local row, train item id)]
  (dataloader.py:359-368); additionally `mask_csr()` exposes the same mask as a per-user CSR
  for the fused score+mask+top-K kernel;
* shuffling uses numpy's *global* RNG exactly like `DataFrame.sample(frac=1)`
  (dataset.py:98-101 -> np.random.choice(n, n, replace=False));
* negative sampling replays `random.sample(all_items, 1)[0]` with history rejection
  (dataloader.py:267-275, 307-309) on Python's global `random`, so a seeded run draws the same
  negatives as the reference.
"""
from __future__ import annotations

import math
import random

import numpy as np
import torch
from scipy.sparse import coo_matrix


def _unique_in_order(a: np.ndarray) -> np.ndarray:
    """pandas `Series.unique()` semantics: first-appearance order."""
    _, idx = np.unique(a, return_index=True)
    return a[np.sort(idx)]


class RecDataset:
    """Interactions as two int64 arrays. dataset.py:21-133."""

    def __init__(self, config, users=None, items=None, labels=None, user_num=None, item_num=None,
                 path=None):
        self.config = config
        self.dataset_name = config["dataset"]
        self.uid_field = config["USER_ID_FIELD"]
        self.iid_field = config["ITEM_ID_FIELD"]
        self.splitting_label = config["inter_splitting_label"]
        if path is not None:
            users, items, labels = self._load_tsv(path)
        self.users = np.asarray(users, dtype=np.int64)
        self.items = np.asarray(items, dtype=np.int64)
        self.labels = None if labels is None else np.asarray(labels, dtype=np.int64)
        # dataset.py:47-48: num = max id + 1
        self.item_num = int(self.items.max()) + 1 if item_num is None else item_num
        self.user_num = int(self.users.max()) + 1 if user_num is None else user_num
        self.inter_num = len(self.users)

    def _load_tsv(self, path):
        """dataset.py:50-55: TSV with a header naming uid / iid / x_label columns."""
        sep = self.config["field_separator"]
        with open(path) as f:
            header = f.readline().rstrip("\n").split(sep)
        cols = [header.index(c) for c in (self.uid_field, self.iid_field, self.splitting_label)]
        arr = np.loadtxt(path, dtype=np.int64, delimiter=sep, skiprows=1, usecols=cols, ndmin=2)
        return arr[:, 0], arr[:, 1], arr[:, 2]

    def split(self):
        """dataset.py:57-74: by x_label, then drop val/test users unseen in train."""
        parts = []
        for lab in range(3):
            m = self.labels == lab
            parts.append((self.users[m], self.items[m]))
        if self.config["filter_out_cod_start_users"]:
            train_u = np.unique(parts[0][0])
            for i in (1, 2):
                keep = np.isin(parts[i][0], train_u)
                parts[i] = (parts[i][0][keep], parts[i][1][keep])
        return [self.copy(u, i) for u, i in parts]

    def copy(self, users, items):
        return RecDataset(self.config, users.copy(), items.copy(), None, self.user_num,
                          self.item_num)

    def get_user_num(self):
        return self.user_num

    def get_item_num(self):
        return self.item_num

    def shuffle(self):
        """dataset.py:98-101. pandas `sample(frac=1, replace=False)` with random_state=None
        draws `np.random.choice(n, size=n, replace=False)` from the global numpy state."""
        n = len(self.users)
        perm = np.random.choice(n, size=n, replace=False)
        self.users, self.items = self.users[perm], self.items[perm]

    def __len__(self):
        return len(self.users)


class AbstractDataLoader:
    def __init__(self, config, dataset, additional_dataset=None, batch_size=1, shuffle=False):
        self.config = config
        self.dataset = dataset
        self.dataset_bk = dataset.copy(dataset.users, dataset.items)
        self.additional_dataset = additional_dataset
        self.batch_size = self.step = batch_size
        self.shuffle = shuffle
        self.device = config["device"]
        self.pr = 0
        self.inter_pr = 0

    def __len__(self):
        return math.ceil(self.pr_end / self.step)

    def __iter__(self):
        if self.shuffle and not self.__dict__.pop("_preshuffled", False):
            self._shuffle()
        return self

    def prefetch_shuffle(self):
        """Draw the NEXT epoch's shuffle now (Trainer calls this while the device still runs the last
        steps of the current epoch, so the ~4 ms permutation of the interactions is off the critical
        path). The next `iter()` then skips its shuffle: same draws from numpy's global state in the
        same order -- nothing else in the training loop consumes that generator."""
        if self.shuffle and self.pr == 0 and not self.__dict__.get("_preshuffled", False):   # between epochs only
            self._shuffle()
            self._preshuffled = True

    def __next__(self):
        if self.pr >= self.pr_end:
            self.pr = 0
            self.inter_pr = 0
            raise StopIteration()
        return self._next_batch_data()


class TrainDataLoader(AbstractDataLoader):
    """dataloader.py:108-318 (pairwise negative-sampling path only)."""

    def __init__(self, config, dataset, batch_size=1, shuffle=False):
        super().__init__(config, dataset, batch_size=batch_size, shuffle=shuffle)
        self.all_items = _unique_in_order(dataset.items).tolist()
        self.all_item_len = len(self.all_items)
        # dataloader.py:311-318
        order = np.argsort(dataset.users, kind="stable")
        su, si = dataset.users[order], dataset.items[order]
        bounds = np.flatnonzero(np.diff(su)) + 1
        self.history_items_per_u = {
            int(g[0]): set(h.tolist())
            for g, h in zip(np.split(su, bounds), np.split(si, bounds))}
        # the same history as a per-user CSR (ascending inside a user) for the native sampler
        o2 = np.lexsort((dataset.items, dataset.users))
        self._hist_cols = np.ascontiguousarray(dataset.items[o2], dtype=np.int64)
        self._hist_rowptr = np.zeros(dataset.user_num + 1, dtype=np.int64)
        np.cumsum(np.bincount(dataset.users, minlength=dataset.user_num), out=self._hist_rowptr[1:])
        self._items_arr = None
        self.native_sampler = bool(config.get("native_sampler", True))

    def pretrain_setup(self):
        """dataloader.py:140-151: restore file order, sort items, then random.shuffle them."""
        if self.shuffle:
            self.dataset = self.dataset_bk.copy(self.dataset_bk.users, self.dataset_bk.items)
        self.all_items.sort()
        random.shuffle(self.all_items)
        self._items_arr = None

    def inter_matrix(self, form="coo", value_field=None):
        """dataloader.py:155-210: scipy COO U x I with float64 ones."""
        ds = self.dataset
        mat = coo_matrix((np.ones(len(ds)), (ds.users, ds.items)),
                         shape=(ds.user_num, ds.item_num))
        if form == "coo":
            return mat
        if form == "csr":
            return mat.tocsr()
        raise NotImplementedError(f"sparse matrix format [{form}] has not been implemented.")

    @property
    def pr_end(self):
        return len(self.dataset)

    def _shuffle(self):
        self.dataset.shuffle()

    def _sample_neg_ids_native(self, u):
        """Same draws as `_sample_neg_ids`, replayed in C on CPython's Mersenne Twister state
        (mmrec_neg_sample_mt19937_host); the advanced state is written back to `random`."""
        from . import lib
        if self._items_arr is None or len(self._items_arr) != len(self.all_items):
            self._items_arr = np.asarray(self.all_items, dtype=np.int64)
        ver, mt, gauss = random.getstate()
        st = np.array(mt, dtype=np.uint32)
        u = np.ascontiguousarray(u, dtype=np.int64)
        neg = np.empty(len(u), dtype=np.int64)
        lib.call("mmrec_neg_sample_mt19937_host", st.ctypes.data, self._items_arr.ctypes.data,
                 len(self._items_arr), self._hist_rowptr.ctypes.data, self._hist_cols.ctypes.data,
                 len(self._hist_rowptr) - 1, u.ctypes.data, len(u), neg.ctypes.data)
        random.setstate((ver, tuple(st.tolist()), gauss))
        return neg

    def _sample_neg_ids(self, u_ids):
        """dataloader.py:267-275 + 307-309, same `random` call per draw."""
        neg = []
        items, hist, sample = self.all_items, self.history_items_per_u, random.sample
        for u in u_ids:
            h = hist[u]
            iid = sample(items, 1)[0]
            while iid in h:
                iid = sample(items, 1)[0]
            neg.append(iid)
        return neg

    def _next_batch_data(self):
        """dataloader.py:226-250 -> LongTensor[3, B]; one H2D copy per batch."""
        u = self.dataset.users[self.pr: self.pr + self.step]
        i = self.dataset.items[self.pr: self.pr + self.step]
        self.pr += self.step
        if self.native_sampler:
            neg = self._sample_neg_ids_native(u)
        else:
            neg = np.asarray(self._sample_neg_ids(u.tolist()), dtype=np.int64)
        batch = torch.from_numpy(np.stack([u, i, neg]))
        if self.device.type == "cuda":
            batch = batch.pin_memory().to(self.device, non_blocking=True)
        return batch


class DeviceTrainLoader:
    """Training batches produced entirely on the device (config 5: hundreds of millions of
    interactions per epoch, where the reference's Python loop -- one `random.sample` per
    interaction, dataloader.py:267-275 -- cannot run at all). Same batch format as
    TrainDataLoader (`LongTensor[3, B]` = users, positive items, negative items on the device),
    same sampling rule (uniform item, rejected while in the user's training history) on the
    stateless counter stream of mmrec_neg_sample_counter, so every rank of a sharded run can
    regenerate exactly the same batch from (seed, epoch, batch index) without a broadcast.
    `users` / `items`: the training interactions on the device (int64).

    Per-rank batches (`rank` given; for a user-sharded model such as parallel.ShardedLightGCN):
    `users` / `items` are this rank's interactions only, its users [user_lo, user_lo + n_users);
    batches carry LOCAL user ids (global - user_lo) and negatives come from a history CSR over the
    local users, on the counter stream of seed `rank_seed(seed, rank)`. One all-gather of the ranks'
    interaction counts at set-up (the world size is the process group's) fixes the number of steps S = ceil(E_total / batch_size) on every
    rank; a rank's shuffled interactions are cut into exactly S slices of near-equal size (they
    differ by at most one, some are empty when the rank holds fewer than S interactions), so every
    rank runs the same collectives. The global batch of a step is the union of the ranks' slices.
    `pr` counts steps in this mode. `sampler` replaces the CUDA sampler with a callable of
    oracle.sampler.neg_sample_counter's arguments (users, all_items=None, n_items, hist_rowptr,
    hist_cols, seed, step, max_draws) -> negatives; then host tensors are accepted."""

    def __init__(self, users, items, n_users, n_items, batch_size, seed=999, shuffle=True, max_draws=64,
                 rank=None, world=None, user_lo=0, group=None, sampler=None):
        from . import lib
        if sampler is None:
            lib.require_cuda(users, items)
        self.sampler = sampler
        self.users, self.items = users.to(torch.int64).contiguous(), items.to(torch.int64).contiguous()
        self.n_users, self.n_items, self.step = int(n_users), int(n_items), int(batch_size)
        self.seed, self.shuffle, self.max_draws = int(seed), bool(shuffle), int(max_draws)
        self.device = users.device
        self.rank = rank
        if rank is not None:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                # S must come from every rank's count: a world size that disagrees with the group
                # would give ranks different step counts and hang the collectives of the last steps
                pg_world = dist.get_world_size(group)
                if world is not None and int(world) != pg_world:
                    raise ValueError(f"DeviceTrainLoader: world={world} but the process group has {pg_world} ranks")
                world = pg_world
            elif world not in (None, 1):
                raise ValueError("DeviceTrainLoader: world > 1 needs an initialised process group")
            world = 1 if world is None else int(world)
            self.users = self.users - int(user_lo)
            self.seed = rank_seed(seed, rank)
            self.nnz_per_rank = [int(self.users.numel())]
            if world > 1:
                self.nnz_per_rank = [None] * world
                dist.all_gather_object(self.nnz_per_rank, int(self.users.numel()), group=group)
            self.n_steps = -(-sum(self.nnz_per_rank) // self.step)
        # per-user history CSR, ascending item ids (the rejection test is a binary search)
        key = torch.sort(self.users * self.n_items + self.items)[0]
        self.hist_cols = (key % self.n_items).to(torch.int32).contiguous()
        counts = torch.bincount(key // self.n_items, minlength=self.n_users)
        self.hist_rowptr = torch.zeros(self.n_users + 1, dtype=torch.int64, device=self.device)
        self.hist_rowptr[1:] = torch.cumsum(counts, 0)
        self.epoch = -1
        self.pr = 0
        self.order = None

    def __len__(self):
        if self.rank is not None:
            return self.n_steps
        return -(-self.users.numel() // self.step)

    def __iter__(self):
        self.epoch += 1
        self.pr = 0
        if self.shuffle:
            g = torch.Generator(device=self.device).manual_seed((self.seed + self.epoch) & 0xFFFFFFFFFFFFFFFF)
            self.order = torch.randperm(self.users.numel(), generator=g, device=self.device)
        return self

    def sample_negatives(self, u, step_id):
        from . import lib
        if u.numel() == 0:             # an empty per-rank slice: nothing to draw (the C ABI rejects NULL operands)
            return torch.empty_like(u)
        if self.sampler is not None:
            neg = self.sampler(u.cpu().numpy(), None, self.n_items, self.hist_rowptr.cpu().numpy(),
                               self.hist_cols.cpu().numpy(), self.seed, int(step_id), self.max_draws)
            return torch.as_tensor(neg, dtype=torch.int64).to(u.device)
        neg = torch.empty_like(u)
        lib.call("mmrec_neg_sample_counter", lib.ptr(u), u.numel(), None, self.n_items, lib.ptr(self.hist_rowptr),
                 lib.ptr(self.hist_cols), self.seed, int(step_id), self.max_draws, lib.ptr(neg), lib.stream())
        return neg

    def __next__(self):
        if self.rank is not None:
            return self._next_rank_slice()
        if self.pr >= self.users.numel():
            raise StopIteration
        sl = slice(self.pr, self.pr + self.step)
        idx = self.order[sl] if self.order is not None else torch.arange(sl.start, min(sl.stop, self.users.numel()),
                                                                         device=self.device)
        u, i = self.users[idx].contiguous(), self.items[idx]
        step_id = self.epoch * len(self) + self.pr // self.step
        self.pr += self.step
        return torch.stack([u, i, self.sample_negatives(u, step_id)])

    def _next_rank_slice(self):
        s, S, n = self.pr, self.n_steps, self.users.numel()
        if s >= S:
            raise StopIteration
        a, b = s * n // S, (s + 1) * n // S
        idx = self.order[a:b] if self.order is not None else torch.arange(a, b, device=self.device)
        u, i = self.users[idx].contiguous(), self.items[idx]
        self.pr += 1
        return torch.stack([u, i, self.sample_negatives(u, self.epoch * S + s)])


def rank_seed(seed, rank):
    """Sampler / shuffle seed of rank `rank` in per-rank batching (rank 0 keeps `seed`)."""
    return (int(seed) ^ (int(rank) * 0x9E3779B97F4A7C15)) & 0xFFFFFFFFFFFFFFFF


class EvalDataLoader(AbstractDataLoader):
    """dataloader.py:321-418."""

    def __init__(self, config, dataset, additional_dataset=None, batch_size=1, shuffle=False):
        super().__init__(config, dataset, additional_dataset=additional_dataset,
                         batch_size=batch_size, shuffle=shuffle)
        if additional_dataset is None:
            raise ValueError("Training datasets is nan")
        eval_u = _unique_in_order(dataset.users)
        tr = additional_dataset
        # train items of every eval user, in training-file order (dataloader.py:370-391)
        order = np.argsort(tr.users, kind="stable")
        tu, ti = tr.users[order], tr.items[order]
        starts = np.searchsorted(tu, eval_u, side="left")
        ends = np.searchsorted(tu, eval_u, side="right")
        lens = ends - starts
        if (lens == 0).any():
            raise KeyError("eval user without training interactions")  # get_group would raise
        self.train_pos_len_list = lens.tolist()
        self.mask_rowptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
        flat = np.concatenate([ti[s:e] for s, e in zip(starts, ends)]) if len(eval_u) else \
            np.zeros(0, np.int64)
        rows = np.repeat(np.arange(len(eval_u), dtype=np.int64), lens)
        self.pos_items_per_u = torch.from_numpy(np.stack([rows, flat])).to(self.device)
        # ground truth per eval user (dataloader.py:393-406)
        order = np.argsort(dataset.users, kind="stable")
        eu, ei = dataset.users[order], dataset.items[order]
        s = np.searchsorted(eu, eval_u, side="left")
        e = np.searchsorted(eu, eval_u, side="right")
        self.eval_items_per_u = [ei[a:b] for a, b in zip(s, e)]
        self.eval_len_list = (e - s).astype(np.int64)
        self.eval_u = torch.from_numpy(eval_u).to(self.device)
        # device copies for the fused kernel: int32 CSR of the same mask
        self._mask_rowptr_dev = torch.from_numpy(self.mask_rowptr.astype(np.int32)).to(self.device)
        # ascending item ids inside each user (the kernel walks the list with a cursor)
        o = np.lexsort((flat, rows))
        self._mask_cols_dev = torch.from_numpy(flat[o].astype(np.int32)).to(self.device)

    @property
    def pr_end(self):
        return self.eval_u.shape[0]

    def _shuffle(self):
        self.dataset.shuffle()

    def _next_batch_data(self):
        inter_cnt = int(self.mask_rowptr[min(self.pr + self.step, self.pr_end)]
                        - self.mask_rowptr[self.pr])
        batch_users = self.eval_u[self.pr: self.pr + self.step]
        m = self.pos_items_per_u[:, self.inter_pr: self.inter_pr + inter_cnt].clone()
        m[0] -= self.pr
        self.inter_pr += inter_cnt
        self.pr += self.step
        return [batch_users, m]

    def mask_csr(self, start, stop):
        """Same mask as `_next_batch_data` for eval users [start, stop): (rowptr int32 with a
        global base, cols int32). The kernel subtracts rowptr[0]."""
        return self._mask_rowptr_dev[start: stop + 1], self._mask_cols_dev

    def gt_csr(self):
        """Ground-truth items per eval user as a device CSR (int32 row pointers, ascending int32
        item ids) for the metrics kernel; built once."""
        if getattr(self, "_gt_csr", None) is None:
            lens = np.asarray(self.eval_len_list, dtype=np.int64)
            rowptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
            flat = np.concatenate([np.sort(p) for p in self.eval_items_per_u]) if len(lens) else \
                np.zeros(0, np.int64)
            self._gt_csr = (torch.from_numpy(rowptr).to(self.device),
                            torch.from_numpy(flat.astype(np.int32)).to(self.device))
        return self._gt_csr

    def get_eval_items(self):
        return self.eval_items_per_u

    def get_eval_len_list(self):
        return self.eval_len_list

    def get_eval_users(self):
        return self.eval_u.cpu()
