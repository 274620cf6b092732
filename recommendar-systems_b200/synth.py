"""Deterministic synthetic datasets shaped like the reference's benchmarks.

The reference reads `<data_path>/<dataset>/<dataset>.inter` (TSV: userID, itemID, x_label;
/root/reference/src/utils/dataset.py:50-55) and `image_feat.npy` / `text_feat.npy`
(/root/reference/src/common/abstract_recommender.py:89-101). No dataset is available offline,
so every benchmark and parity test runs on graphs generated here (SURVEY.md section 8d):

* exactly (U, I, E_all) users / items / unique interactions, ids U-1 and I-1 present
  (`user_num = max id + 1`, dataset.py:47-48);
* user degree = 5 + power-law tail (Amazon 5-core shape), item popularity ~ Zipf(0.8) under a
  random permutation;
* x_label in {0,1,2} w.p. 0.8/0.1/0.1, each user's first row forced to 0 so every evaluated
  user has training rows (dataloader.py:386 `get_group`).

Config 5's scaled graph is generated on the device (`make_scaled_edges`), and its held-out split
(`scaled_edge_labels`) follows the same rules with a hash per edge instead of a sequential draw.
"""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np

SHAPES = {
    # name: (users, items, interactions)
    "tiny": (240, 96, 2400),
    "small": (1500, 640, 14000),
    "baby": (19445, 7050, 160792),
    "sports": (35598, 18357, 296337),
    "clothing": (39387, 23033, 278677),
}


@dataclass
class SynthData:
    name: str
    n_users: int
    n_items: int
    users: np.ndarray      # int64 [E_all]
    items: np.ndarray      # int64 [E_all]
    labels: np.ndarray     # int64 [E_all] in {0,1,2}
    image_feat: np.ndarray | None = None   # float32 [I, Fv]
    text_feat: np.ndarray | None = None    # float32 [I, Ft]

    def split(self, label: int):
        m = self.labels == label
        return self.users[m], self.items[m]


def _degrees(rng, n_users, n_items, n_inter):
    """User degrees: 5-core floor plus a Pareto tail, summing exactly to n_inter."""
    base = min(5, max(1, n_inter // n_users))
    extra = n_inter - base * n_users
    if extra < 0:
        raise ValueError("n_inter too small for the 5-core floor")
    w = rng.pareto(1.6, size=n_users) + 1e-3
    tail = np.floor(w / w.sum() * extra).astype(np.int64)
    rem = extra - int(tail.sum())
    if rem > 0:
        tail[rng.choice(n_users, size=rem, replace=False if rem <= n_users else True)] += 1
    deg = base + tail
    cap = max(base, n_items // 2)
    over = int(np.maximum(deg - cap, 0).sum())
    deg = np.minimum(deg, cap)
    while over > 0:                      # redistribute anything clipped by the cap
        room = np.flatnonzero(deg < cap)
        take = min(over, len(room))
        deg[rng.choice(room, size=take, replace=False)] += 1
        over -= take
    assert int(deg.sum()) == n_inter
    return deg


def make_interactions(n_users, n_items, n_inter, seed=2024):
    rng = np.random.default_rng(seed)
    deg = _degrees(rng, n_users, n_items, n_inter)
    pop = 1.0 / np.power(np.arange(1, n_items + 1, dtype=np.float64), 0.8)
    pop = pop[rng.permutation(n_items)]
    cdf = np.cumsum(pop / pop.sum())
    users = np.repeat(np.arange(n_users, dtype=np.int64), deg)
    items = np.minimum(np.searchsorted(cdf, rng.random(n_inter)), n_items - 1).astype(np.int64)
    # resolve duplicate (u, i) pairs by redrawing; a handful of rounds suffices
    for _ in range(200):
        key = users * n_items + items
        order = np.argsort(key, kind="stable")
        dup = np.zeros(n_inter, dtype=bool)
        dup[order[1:]] = key[order[1:]] == key[order[:-1]]
        n_dup = int(dup.sum())
        if n_dup == 0:
            break
        items[dup] = np.minimum(np.searchsorted(cdf, rng.random(n_dup)), n_items - 1)
    else:  # pragma: no cover - only for absurdly dense requests
        raise RuntimeError("could not make interactions unique")
    # make sure the last item id exists (user ids all exist: degree >= 1)
    if not (items == n_items - 1).any():
        cand = np.flatnonzero(users == n_users - 1)
        items[cand[0]] = n_items - 1
        key = users * n_items + items
        assert len(np.unique(key)) == n_inter
    labels = rng.choice(3, size=n_inter, p=[0.8, 0.1, 0.1]).astype(np.int64)
    first = np.concatenate(([0], np.cumsum(deg)[:-1]))
    labels[first] = 0
    return users, items, labels


def make_features(n_items, dim, seed, n_centroids=64):
    """Clustered features (centroid + 0.5 noise) so that kNN item graphs are not degenerate."""
    rng = np.random.default_rng(seed)
    cent = rng.standard_normal((n_centroids, dim)).astype(np.float32)
    assign = rng.integers(0, n_centroids, size=n_items)
    noise = rng.standard_normal((n_items, dim)).astype(np.float32)
    return (cent[assign] + np.float32(0.5) * noise).astype(np.float32)


def make_dataset(name="baby", image_dim=4096, text_dim=384, seed=2024, features=True,
                 shape=None) -> SynthData:
    n_users, n_items, n_inter = shape or SHAPES[name]
    users, items, labels = make_interactions(n_users, n_items, n_inter, seed)
    img = txt = None
    if features:
        img = make_features(n_items, image_dim, seed=7)
        txt = make_features(n_items, text_dim, seed=8)
    return SynthData(name, n_users, n_items, users, items, labels, img, txt)


def write_reference_layout(data: SynthData, root: str, uid="userID", iid="itemID",
                           label="x_label"):
    """Write the on-disk layout the reference loads (dataset.py:50-55,
    abstract_recommender.py:89-101). Returns the dataset directory."""
    d = os.path.join(root, data.name)
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, f"{data.name}.inter"), "w") as f:
        f.write(f"{uid}\t{iid}\t{label}\n")
        for u, i, l in zip(data.users.tolist(), data.items.tolist(), data.labels.tolist()):
            f.write(f"{u}\t{i}\t{l}\n")
    if data.image_feat is not None:
        np.save(os.path.join(d, "image_feat.npy"), data.image_feat)
    if data.text_feat is not None:
        np.save(os.path.join(d, "text_feat.npy"), data.text_feat)
    return d


def scaled_degrees(device, n_users, n_edges, seed=2024):
    """Planned user degrees of the scaled power-law graph (int64 [n_users]): 5 + Pareto tail."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    w = torch.rand(n_users, generator=g, device=device).clamp_min(1e-6).pow(-1.0 / 1.6)
    extra = max(0, n_edges - 5 * n_users)
    return 5 + torch.floor(w / w.sum() * extra).to(torch.int64)


def make_scaled_edges(device, n_users, n_items, n_edges, seed=2024, user_range=None, block=1 << 20):
    """Config 5 (scaled power-law graph): edges generated directly on the device -- user degrees
    ~ 5 + Pareto tail, item popularity ~ Zipf(0.8). Duplicate (u, i) pairs are removed, so the
    result has slightly fewer than `n_edges` edges. Returns int64 (users, items), sorted by
    (user, item).

    Users are generated in fixed blocks of `block` users, every block from its own seeded stream:
    `user_range = (lo, hi)` returns exactly the edges of those users that the full call would --
    a rank of the sharded benchmark builds its share without ever materialising the whole graph."""
    import torch
    deg = scaled_degrees(device, n_users, n_edges, seed)
    g = torch.Generator(device=device).manual_seed(seed + 1)
    pop = torch.arange(1, n_items + 1, device=device, dtype=torch.float64).pow(-0.8)
    pop = pop[torch.randperm(n_items, generator=g, device=device)]
    cdf = torch.cumsum(pop / pop.sum(), 0).to(torch.float32)
    lo, hi = (0, n_users) if user_range is None else (int(user_range[0]), int(user_range[1]))
    us, its = [], []
    for b0 in range(lo // block * block, hi, block):
        b1 = min(n_users, b0 + block)
        gb = torch.Generator(device=device).manual_seed(seed + 1000 + b0 // block)
        users = torch.repeat_interleave(torch.arange(b0, b1, device=device), deg[b0:b1])
        items = torch.searchsorted(cdf, torch.rand(users.numel(), generator=gb, device=device)).clamp_max(n_items - 1)
        key = torch.unique(users * n_items + items)
        u, i = key // n_items, key % n_items
        if b0 < lo or b1 > hi:
            m = (u >= lo) & (u < hi)
            u, i = u[m], i[m]
        us.append(u)
        its.append(i)
    if not us:
        z = torch.zeros(0, dtype=torch.int64, device=device)
        return z, z
    return torch.cat(us), torch.cat(its)


def _s64(c):
    """A 64-bit constant as the int64 with the same bits."""
    return c - (1 << 64) if c >= 1 << 63 else c


def _mix64(x):
    """splitmix64's finaliser on an int64 tensor: wrapping products, logical right shifts."""
    x = x ^ ((x >> 30) & ((1 << 34) - 1))
    x = x * _s64(0xBF58476D1CE4E5B9)
    x = x ^ ((x >> 27) & ((1 << 37) - 1))
    x = x * _s64(0x94D049BB133111EB)
    return x ^ ((x >> 31) & ((1 << 33) - 1))


def _mix64_int(x):
    """_mix64 on one Python int (the seed's salt)."""
    m = (1 << 64) - 1
    x &= m
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & m
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & m
    return _s64(x ^ (x >> 31))


SPLIT_P = (0.8, 0.1, 0.1)


def scaled_edge_labels(users, items, seed=2024):
    """Held-out split of make_scaled_edges' edges: int64 labels 0 / 1 / 2 (train / valid / test)
    with probabilities 0.8 / 0.1 / 0.1, as make_interactions draws them for the small shapes; each
    user's first edge (its lowest item id) is train, so every evaluated user has training rows.

    An edge's label is a counter-based hash of (seed, user, item) (splitmix64's finaliser), not a
    draw from a sequential stream: a rank that labels only its own users' edges gets exactly the
    labels the one-rank call gives them, at any world size. `users` / `items` must be sorted by
    (user, item), as make_scaled_edges returns them, and hold whole users (a user range)."""
    import torch
    u, i = users.to(torch.int64), items.to(torch.int64)
    salt = _mix64_int(int(seed) ^ 0x5851F42D4C957F2D)
    r = (_mix64((u << 32) + i + salt) >> 40) & ((1 << 24) - 1)          # top 24 bits: uniform in [0, 2^24)
    t1, t2 = round(SPLIT_P[0] * (1 << 24)), round((SPLIT_P[0] + SPLIT_P[1]) * (1 << 24))
    labels = (r >= t1).to(torch.int64) + (r >= t2).to(torch.int64)
    if u.numel():
        first = torch.ones_like(u, dtype=torch.bool)
        first[1:] = u[1:] != u[:-1]
        labels[first] = 0
    return labels
