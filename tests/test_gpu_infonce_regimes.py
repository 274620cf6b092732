"""InfoNCE (mmrec_infonce_*) in every split regime against float64, on buffers the test owns.

Two implementations: the tcgen05 kernel of infonce_tc.cu (d = 64, the only path behind the pair
entry) and the mma.sync tile kernels of loss.cu (d = 32 / 128). The host code cuts the "other"
dimension of the B x B score matrix into splits from the batch size alone -- infonce_splits for
mma.sync, infonce_tc_splits (capped by it, and by one wave of 128-row CTAs per problem) for
tcgen05 -- and the forward workspace query has to cover the layout of both. That policy is restated
below in plain Python; every case names the regime it pins, and the host-only part (no `gpu` mark)
checks the restatement against the library for every batch size the API accepts. No case sets an
environment switch: each regime is reached through its batch size and width.

The GPU cases call the C ABI with every written buffer carved out of a larger tensor: a 64-float
front guard and a back guard at least as long as the buffer, holding random bits that must come back
unchanged. Buffers start as NaN (tables of gradients as zeros), so the extent the kernels wrote can be
compared with the restated footprint exactly. The loss, ttl and both table gradients are compared
with oracle.ops.infonce in float64 (torch autograd through F.normalize and the row gather).
"""
import ctypes
import sys

import pytest
import torch
import torch.nn.functional as F

from conftest import pkg
from oracle import ops as oops

DEV = "cuda:0"

# ------------------------------------------------------------------ the host policy, restated
SMS = 148                          # kNumSMs
TILE, MAX_SPLITS, MAX_TILES = 64, 32, 1023   # kTile, kMaxInfoSplits, kMaxInfoTiles of loss.cu
TC_M, TC_N = 128, 64               # kTM (own rows per CTA), kTN (other rows per tile) of infonce_tc.cu
B_MAX = MAX_TILES * TILE           # 65472, the largest batch the forward entries accept
E_BADARG = -1


def cdiv(a, b):
    return -(-a // b)


def infonce_splits(B):
    """infonce_splits (loss.cu): column splits of the mma.sync kernels, ~4 co-resident CTAs per SM."""
    nt = cdiv(B, TILE)
    s = max(1, min(nt, MAX_SPLITS, cdiv(4 * SMS, nt)))
    return cdiv(nt, cdiv(nt, s))


def fwd_workspace_floats(B):
    """mmrec_infonce_fwd_workspace_floats."""
    return (1 + max(2, infonce_splits(B))) * B + cdiv(B, TILE)


def tc_splits(B, cap, n_prob):
    """infonce_tc_splits (infonce_tc.cu) with the caller's cap."""
    n_ot = cdiv(B, TC_N)
    s = max(1, min(n_ot, cap // 2, SMS // (cdiv(B, TC_M) * n_prob)))
    return cdiv(n_ot, cdiv(n_ot, s))


def regime(path, B, n_prob=1, n_splits=None):
    """What the host code launches for a batch of B rows: path "tc" (tcgen05) or "mma" (mma.sync).
    `n_splits`: the split count the caller passes to the backward (default mmrec_infonce_splits)."""
    cap = infonce_splits(B)
    if path == "tc":
        tiles = cdiv(B, TC_N)
        bounds = {"tiles": tiles, "cap/2": cap // 2, "wave": SMS // (cdiv(B, TC_M) * n_prob)}
    else:
        tiles = cdiv(B, TILE)
        bounds = {"tiles": tiles, "cap": MAX_SPLITS, "4/SM": cdiv(4 * SMS, tiles)}
    low = min(bounds.values())
    tps = cdiv(tiles, max(1, low))
    splits = cdiv(tiles, tps)
    bwd_splits = n_splits if n_splits is not None else cap
    if path == "tc":
        fwd_floats = B + 2 * splits * B          # pos[B] | ttl_part[2 * splits][B] (two epilogue halves)
        bwd_slabs = bwd_live = tc_splits(B, bwd_splits, n_prob)
    else:
        fwd_floats = (1 + splits) * B + tiles    # pos[B] | ttl_part[splits][B] | tile_loss[tiles]
        bwd_slabs = bwd_splits                   # splits past the last tile write zero slabs
        bwd_live = cdiv(tiles, cdiv(tiles, bwd_splits))
    return dict(path=path, cap=cap, tiles=tiles, splits=splits, tps=tps,
                per_split=[min(tps, tiles - k * tps) for k in range(splits)],
                limiter=tuple(k for k, v in bounds.items() if v == low),
                fwd_floats=fwd_floats, bwd_slabs=bwd_slabs, bwd_live_slabs=bwd_live)


def _ranges(values):
    out = []
    for v in values:
        if out and v == out[-1][1] + 1:
            out[-1][1] = v
        else:
            out.append([v, v])
    return ", ".join(f"[{a}, {b}]" for a, b in out)


# ------------------------------------------------------------------ the cases
class Case:
    def __init__(self, path, B, d, expect, temp=0.2, idx=("rep", "perm"), coef=(0.3, -1.7), n_splits=None):
        self.path, self.B, self.d, self.expect, self.temp = path, B, d, expect, temp
        self.n_prob = 2 if path == "pair" else 1
        self.idx, self.coef, self.n_splits = idx[:self.n_prob], coef[:self.n_prob], n_splits
        self.kernel = "tc" if d == 64 else "mma"
        extra = "" if temp == 0.2 else f"-t{temp}"
        extra += "" if n_splits is None else f"-nsplits{n_splits}"
        extra += "-coef0" if 0 in self.coef else ""
        self.name = f"{path}-d{d}-B{B}{extra}-" + "+".join(self.idx)

    def regime(self):
        return regime(self.kernel, self.B, self.n_prob, self.n_splits)


def _r(**kw):
    return kw


# idx patterns: "rep" random with repeats (scatter-add), "perm" no repeats, "same" one index B times
# (all scores equal), "zeros" some referenced rows are zero (normalize eps), "scaled" rows x 1e-3 / x 1e3
CASES = [
    # pair entry, tcgen05, two problems per launch
    Case("pair", 1, 64, _r(tiles=1, splits=1, cap=1), idx=("rep", "perm")),
    Case("pair", 2, 64, _r(cap=1, splits=1, fwd_floats=6), idx=("same", "rep")),
    Case("pair", 43, 64, _r(cap=1, splits=1, fwd_floats=129), idx=("perm", "zeros")),
    Case("pair", 63, 64, _r(cap=1, splits=1, fwd_floats=189), idx=("scaled", "rep")),
    Case("pair", 64, 64, _r(cap=1, splits=1, fwd_floats=192), idx=("rep", "same")),
    Case("pair", 65, 64, _r(tiles=2, cap=2, splits=1, limiter=("cap/2",)), idx=("zeros", "perm"), coef=(0.0, -1.7)),
    Case("pair", 127, 64, _r(tiles=2, cap=2, splits=1, limiter=("cap/2",)), idx=("perm", "scaled")),
    Case("pair", 128, 64, _r(tiles=2, cap=2, splits=1, limiter=("cap/2",)), idx=("rep", "perm"), temp=0.05),
    Case("pair", 129, 64, _r(tiles=3, cap=3, splits=1, limiter=("cap/2",)), idx=("scaled", "zeros")),
    Case("pair", 300, 64, _r(tiles=5, splits=2, per_split=[3, 2]), idx=("rep", "perm")),
    Case("pair", 300, 64, _r(tiles=5, splits=2, per_split=[3, 2]), idx=("scaled", "same"), temp=0.05),
    Case("pair", 1900, 64, _r(splits=4, per_split=[8, 8, 8, 6], limiter=("wave",)), idx=("zeros", "rep")),
    Case("pair", 2048, 64, _r(splits=4, per_split=[8, 8, 8, 8], limiter=("wave",)), idx=("rep", "perm")),
    Case("pair", 2048, 64, _r(splits=4, per_split=[8, 8, 8, 8]), idx=("perm", "scaled"), temp=1.0),
    Case("pair", 37824, 64, _r(cap=2, splits=1, tiles=591), idx=("rep", "perm")),
    Case("pair", 37825, 64, _r(cap=1, splits=1, tiles=592), idx=("perm", "rep")),
    Case("pair", B_MAX, 64, _r(cap=1, splits=1, tiles=1023), idx=("rep", "scaled")),
    # single-problem entry, tcgen05 (n_prob = 1: a wave holds twice the splits)
    Case("single", 2, 64, _r(cap=1, splits=1, fwd_floats=6), idx=("rep",)),
    Case("single", 64, 64, _r(cap=1, splits=1, fwd_floats=192), idx=("perm",), coef=(0.0,)),
    Case("single", 300, 64, _r(splits=2, per_split=[3, 2]), idx=("scaled",)),
    Case("single", 2048, 64, _r(splits=8, per_split=[4] * 8, limiter=("cap/2",)), idx=("perm",)),
    Case("single", 9000, 64, _r(splits=2, per_split=[71, 70], limiter=("cap/2", "wave")), idx=("zeros",), temp=1.0),
    Case("single", B_MAX, 64, _r(cap=1, splits=1, tiles=1023), idx=("perm",)),
    # single-problem entry, mma.sync (d = 32 / 128): splits limited by the tile count up to 300 rows, by
    # four CTAs per SM from 2048 (the cap of 32 never binds)
    *[Case("single", B, d, e, idx=(p,), temp=t) for d in (32, 128) for B, e, p, t in [
        (1, _r(splits=1, tiles=1, limiter=("tiles",)), "rep", 0.2),
        (65, _r(splits=2, per_split=[1, 1], limiter=("tiles",)), "scaled", 0.2),
        (300, _r(splits=5, per_split=[1] * 5, limiter=("tiles",)), "rep", 0.05 if d == 32 else 1.0),
        (2048, _r(splits=16, per_split=[2] * 16, limiter=("4/SM",)), "perm", 0.2),
        (4096, _r(splits=10, per_split=[7] * 9 + [1], limiter=("4/SM",)), "zeros", 0.2),
        (9000, _r(splits=5, per_split=[29] * 4 + [25], limiter=("4/SM",)), "same", 0.2),
    ]],
    Case("single", B_MAX, 128, _r(splits=1, tiles=1023, limiter=("4/SM",)), idx=("rep",)),
    # mma.sync backward with more splits than tiles: splits past the end write zero slabs
    Case("single", 300, 128, _r(tiles=5, bwd_slabs=64, bwd_live_slabs=5), idx=("rep",), n_splits=64),
    Case("single", 300, 32, _r(tiles=5, bwd_slabs=64, bwd_live_slabs=5), idx=("perm",), n_splits=64,
         coef=(0.0,)),
]
CASE_IDS = [c.name for c in CASES]


# ------------------------------------------------------------------ host-only checks
def test_splits_restatement_matches_library_at_every_batch():
    L = pkg("lib").load()
    bad = [B for B in range(1, B_MAX + 1) if infonce_splits(B) != L.mmrec_infonce_splits(B)]
    assert not bad, f"infonce_splits restatement differs at B in {_ranges(bad)}"


def test_workspace_query_restatement_matches_library():
    L = pkg("lib").load()
    bad = [B for B in range(1, B_MAX + 1) if fwd_workspace_floats(B) != L.mmrec_infonce_fwd_workspace_floats(B)]
    assert not bad, f"mmrec_infonce_fwd_workspace_floats differs from the restatement at B in {_ranges(bad)}"


def test_workspace_query_covers_every_footprint():
    """For every batch the API accepts: the forward workspace query holds the mma.sync layout and the
    tcgen05 layout of both entries, and the tcgen05 backward (which takes the caller's split count as
    its cap) never needs more slabs than the mmrec_infonce_splits the caller sized dV*_ws for."""
    L = pkg("lib").load()
    short = {"mma.sync forward": [], "tcgen05 forward, n_prob 1": [], "tcgen05 forward, n_prob 2": [],
             "tcgen05 backward slabs": []}
    for B in range(1, B_MAX + 1):
        q, S = L.mmrec_infonce_fwd_workspace_floats(B), L.mmrec_infonce_splits(B)
        if (1 + S) * B + cdiv(B, TILE) > q:
            short["mma.sync forward"].append(B)
        for p in (1, 2):
            s = tc_splits(B, S, p)
            if B + 2 * s * B > q:
                short[f"tcgen05 forward, n_prob {p}"].append(B)
            if s > S:
                short["tcgen05 backward slabs"].append(B)
    msg = "; ".join(f"{k} exceeds its workspace at B in {_ranges(v)}" for k, v in short.items() if v)
    assert not msg, msg


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_policy_pins_regime(case):
    """The case is still in the regime it names, and the restated split count is the library's."""
    reg = case.regime()
    assert reg["cap"] == pkg("lib").load().mmrec_infonce_splits(case.B)
    got = {k: reg[k] for k in case.expect}
    assert got == case.expect, f"{case.name}: {reg}"


def test_entries_refuse_bad_sizes_and_widths():
    """Refused before any launch (the pointers are never dereferenced): batches outside [1, 65472],
    widths the kernels do not instantiate, and any width but 64 at the pair entries."""
    L = pkg("lib").load()
    P = [ctypes.c_void_p(256 * (i + 1)) for i in range(14)]          # non-null, 16-byte aligned

    def pa():
        return (ctypes.c_void_p * 2)(256, 512)

    assert L.mmrec_infonce_pair_supported(64) == 1
    for d in (32, 96, 128):
        assert L.mmrec_infonce_pair_supported(d) == 0
    for B in (0, B_MAX + 1):
        assert L.mmrec_infonce_fwd_f32(P[0], P[1], 64, P[2], B, 5.0, *P[3:10], None) == E_BADARG
        assert b"batch must be in [1, 65472]" in L.mmrec_last_error()
        assert L.mmrec_infonce_pair_fwd_f32(pa(), pa(), 64, pa(), B, 5.0, *[pa() for _ in range(6)], None) \
            == E_BADARG
        assert b"batch must be in [1, 65472]" in L.mmrec_last_error()
    for d in (32, 96, 128):
        assert L.mmrec_infonce_pair_fwd_f32(pa(), pa(), d, pa(), 64, 5.0, *[pa() for _ in range(6)], None) \
            == E_BADARG
        assert b"not on the batched path" in L.mmrec_last_error()
        assert L.mmrec_infonce_pair_bwd_f32(pa(), pa(), pa(), pa(), d, pa(), 64, 5.0, pa(), 1,
                                            *[pa() for _ in range(4)], None) == E_BADARG
        assert b"not on the batched path" in L.mmrec_last_error()
    assert L.mmrec_infonce_bwd_f32(*P[0:4], 96, P[4], 64, 5.0, P[5], 1, *P[6:10], None) == E_BADARG
    assert b"unsupported d=96" in L.mmrec_last_error()
    for n in (0, 65):
        assert L.mmrec_infonce_bwd_f32(*P[0:4], 64, P[4], 64, 5.0, P[5], n, *P[6:10], None) == E_BADARG


# ------------------------------------------------------------------ float64 reference
CHUNK_FROM, CHUNK = 16384, 2048        # B x B float64 at 65472 rows is 34 GB: rows in chunks from here on


def _no_tf32(fn):
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        return fn()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def reference(T1, T2, idx, temp, coef, dtype):
    """coef * InfoNCE(T1[idx], T2[idx]) in `dtype`: loss, ttl, the diagonal scores and the gradients of
    both tables (autograd through the gather and F.normalize). oracle.ops.infonce below CHUNK_FROM rows,
    the same formula over row chunks above."""
    def run():
        t1 = T1.detach().to(dtype).requires_grad_(True)
        t2 = T2.detach().to(dtype).requires_grad_(True)
        B = idx.numel()
        v1, v2 = F.normalize(t1[idx], dim=1), F.normalize(t2[idx], dim=1)
        if B < CHUNK_FROM:
            loss = oops.infonce(t1[idx], t2[idx], temp)
            (coef * loss).backward()
            with torch.no_grad():
                ttl = torch.exp(v1 @ v2.t() / temp).sum(dim=1)
        else:
            a1, a2 = v1.detach(), v2.detach().requires_grad_(True)
            g1, ttl, loss = torch.empty_like(a1), torch.empty(B, dtype=dtype, device=a1.device), 0.0
            for r0 in range(0, B, CHUNK):
                x1 = a1[r0:r0 + CHUNK].clone().requires_grad_(True)
                tt = torch.exp(x1 @ a2.t() / temp).sum(dim=1)
                lc = (torch.log(tt) - (x1 * a2[r0:r0 + CHUNK]).sum(dim=1) / temp).sum() / B
                gx, gy = torch.autograd.grad(lc, (x1, a2))
                g1[r0:r0 + CHUNK] = gx
                g2 = gy if r0 == 0 else g2 + gy
                ttl[r0:r0 + CHUNK] = tt.detach()
                loss = loss + lc.detach()
            torch.autograd.backward((v1, v2), (coef * g1, coef * g2))
        with torch.no_grad():
            pos = (v1 * v2).sum(dim=1)
        return dict(loss=loss.detach(), ttl=ttl, pos=pos.detach(), dT1=t1.grad, dT2=t2.grad)
    return _no_tf32(run)


def grad_view(dT, T):
    """dT scaled row-wise by the row norm (clamped at F.normalize's eps): the gradient in the units of
    the normalized rows, so that rows scaled by 1e-3, 1e3 or zero (x 1e12) weigh the same."""
    return dT.double() * T.double().norm(dim=1, keepdim=True).clamp_min(1e-12)


def errors(got, r64, T1, T2, temp, coef):
    """Kernel (or float32 reference) against float64, each relative to the magnitude of its quantity:
    the loss to mean |log ttl| + mean |s_ii| / t (the size of the terms it sums), ttl to its max, the
    gradients (see grad_view) to their max but at least |coef| / (B t), the size of one diagonal term."""
    B = r64["ttl"].numel()
    scale = r64["ttl"].log().abs().mean() + r64["pos"].abs().mean() / temp
    e = dict(loss=float((got["loss"].double() - r64["loss"]).abs() / scale),
             ttl=float((got["ttl"].double() - r64["ttl"]).abs().max() / r64["ttl"].abs().max()))
    floor = abs(coef) / (B * temp)
    for k, T in (("dT1", T1), ("dT2", T2)):
        want = grad_view(r64[k], T)
        den = max(float(want.abs().max()), floor) if coef else 1.0
        e[k] = float((grad_view(got[k], T) - want).abs().max() / den)
    return e


TOL = dict(loss=1e-5, ttl=1e-5, dT1=2e-5, dT2=2e-5)


def tc_bwd_chain_tol(reg):
    """Gradient bound of the tcgen05 backward beyond TOL. Its GEMM 2 (dOwn += G Other) keeps the whole
    tile range of a split in one TMEM accumulator, which the tensor core truncates after every
    instruction (<= 1 ulp, as in gemm_tau): 3 passes x 8 k-steps = 24 instructions per 64-row tile,
    on a running sum bounded by ~2 max |dV| (the diagonal term and the off-diagonal mass). Measured on
    a B200 (1000 W power limit): 1.6e-4 to 2.4e-4 of the max at 1023 tiles per split (bound 5.9e-3),
    5e-6 at 8 tiles per split (the 2048-row training batch, bound 4.6e-5)."""
    return 2 * 24 * reg["tps"] * 2.0 ** -23 if reg["path"] == "tc" else 0.0


def assert_close(got, T1, T2, idx, temp, coef, what, grad_tol=0.0):
    r64 = reference(T1, T2, idx, temp, coef, torch.float64)
    r32 = reference(T1, T2, idx, temp, coef, torch.float32)
    e = errors(got, r64, T1, T2, temp, coef)
    e32 = errors(r32, r64, T1, T2, temp, coef)
    bound = {k: max(TOL[k], 4 * e32[k], grad_tol if k.startswith("dT") else 0.0) for k in TOL}
    bad = {k: (e[k], bound[k]) for k in TOL if not e[k] <= bound[k]}     # NaN fails
    assert not bad, f"{what}: error / bound {bad} (float32 torch: {e32})"
    return e, e32


# ------------------------------------------------------------------ the tolerance against kernel mutants
def _tf32(x):
    """Round float32 to tf32 (10 mantissa bits), nearest even."""
    b = x.float().contiguous().view(torch.int32)
    b = (b + 0xFFF + ((b >> 13) & 1)) & ~0x1FFF
    return b.view(torch.float32)


def _mutant(T1, T2, idx, temp, coef, kind):
    """The float64 formula with one defect a kernel could have: "1xtf32" products of tf32-rounded
    operands only (the lo * hi passes dropped), "pad" a padded column counted in every row sum
    (exp(0) = 1), "slab" the last 64-column tile's partial sums lost."""
    t1 = T1.double().requires_grad_(True)
    t2 = T2.double().requires_grad_(True)
    v1, v2 = F.normalize(t1[idx], dim=1), F.normalize(t2[idx], dim=1)
    B = idx.numel()
    if kind == "1xtf32":                                   # straight-through rounding of both operands
        v1 = v1 + (_tf32(v1.detach()).double() - v1.detach())
        v2 = v2 + (_tf32(v2.detach()).double() - v2.detach())
    S = v1 @ v2.t() / temp
    E = torch.exp(S)
    if kind == "slab":
        E = E[:, :TILE * (cdiv(B, TILE) - 1)]
    ttl = E.sum(dim=1) + (1.0 if kind == "pad" else 0.0)
    loss = (torch.log(ttl) - torch.diagonal(S)).mean()
    (coef * loss).backward()
    return dict(loss=loss.detach(), ttl=ttl.detach(), dT1=t1.grad, dT2=t2.grad)


@pytest.mark.parametrize("kind", ["1xtf32", "pad", "slab"])
def test_tolerance_rejects_kernel_mutants(kind):
    """The bound the GPU cases apply is tight enough to fail a kernel with one of these defects
    (restated on the CPU in float64, B = 300: five tiles, the last one ragged)."""
    gen = torch.Generator().manual_seed(5)
    B, d, temp, coef = 300, 64, 0.2, -1.7
    T1, T2 = torch.randn(B + 37, d, generator=gen), torch.randn(B + 37, d, generator=gen)
    idx = torch.randint(0, B + 37, (B,), generator=gen)
    got = _mutant(T1, T2, idx, temp, coef, kind)
    with pytest.raises(AssertionError, match="error / bound"):
        assert_close(got, T1, T2, idx, temp, coef, kind)
    # ... while the exact formula passes
    ok = _mutant(T1, T2, idx, temp, coef, None)
    assert_close(ok, T1, T2, idx, temp, coef, "exact")


def test_chunked_reference_equals_oracle(monkeypatch):
    """The row-chunked float64 reference of the large batches is oracle.ops.infonce (ragged last chunk)."""
    gen = torch.Generator().manual_seed(6)
    B, d, temp, coef = 300, 64, 0.05, 0.3
    T1, T2 = torch.randn(B + 5, d, generator=gen), torch.randn(B + 5, d, generator=gen)
    idx = torch.randint(0, B + 5, (B,), generator=gen)
    want = reference(T1, T2, idx, temp, coef, torch.float64)
    monkeypatch.setattr(sys.modules[__name__], "CHUNK_FROM", 100)
    monkeypatch.setattr(sys.modules[__name__], "CHUNK", 64)
    got = reference(T1, T2, idx, temp, coef, torch.float64)
    e = errors(got, want, T1, T2, temp, coef)
    assert max(e.values()) < 1e-13, e


# ------------------------------------------------------------------ GPU harness
FRONT = 64                                     # floats of front guard (keeps 16-byte alignment)


class Guarded:
    """n floats (NaN, or `fill`) inside [FRONT guard | n | back guard of max(n, FRONT)] of random bits."""

    def __init__(self, n, gen, fill=float("nan")):
        self.n = n
        self.buf = torch.randint(-2 ** 31, 2 ** 31, (FRONT + n + max(n, FRONT),), dtype=torch.int64,
                                 generator=gen, device=DEV).to(torch.int32).view(torch.float32)
        self.ref = self.buf.clone()
        self.t = self.buf[FRONT:FRONT + n]
        self.t.fill_(fill)

    def check(self, what):
        bits, ref = self.buf.view(torch.int32), self.ref.view(torch.int32)
        assert torch.equal(bits[:FRONT], ref[:FRONT]), f"{what}: write before the buffer"
        after = (bits[FRONT + self.n:] != ref[FRONT + self.n:]).nonzero()
        assert after.numel() == 0, f"{what}: write after the buffer, {after.numel()} floats from offset " \
                                   f"{int(after[0])} past its end ({self.n} floats)"

    def written(self):
        """Number of leading non-NaN floats; every later one must still be NaN."""
        live = ~self.t.isnan()
        n = int(live.sum())
        assert bool(live[:n].all()), "the written floats are not a prefix of the buffer"
        return n


def _problems(case, gen):
    """side / content tables [n_users + n_items, d] (n_users odd) and, per problem, (row0, n, idx):
    problem 0 = the item rows (side[n_users:]), problem 1 = the user rows, as ops.infonce_pair orders them."""
    B, d = case.B, case.d
    nu, ni = B + 37 + B % 2, B + 20                        # odd n_users, as in the datasets
    side = torch.randn(nu + ni, d, generator=gen, device=DEV)
    content = torch.randn(nu + ni, d, generator=gen, device=DEV)
    out = []
    for p, pattern in enumerate(case.idx):
        row0, n = (nu, ni) if p == 0 else (0, nu)
        if pattern == "perm":
            idx = torch.randperm(n, generator=gen, device=DEV)[:B]
        elif pattern == "same":
            idx = torch.randint(0, n, (1,), generator=gen, device=DEV).expand(B).contiguous()
        else:
            idx = torch.randint(0, n, (B,), generator=gen, device=DEV)
        sec1, sec2 = side[row0:row0 + n], content[row0:row0 + n]
        if pattern == "zeros":                             # a sixteenth of the rows zero, in one table or both
            z = idx[torch.randperm(B, generator=gen, device=DEV)[:max(1, B // 16)]]
            sec1[z[0::2]] = 0.0
            sec2[z[len(z) // 3:]] = 0.0
        elif pattern == "scaled":
            r = torch.rand(n, 1, generator=gen, device=DEV)
            f = torch.where(r < 1 / 3, 1e-3, torch.where(r < 2 / 3, 1e3, 1.0))
            sec1.mul_(f)
            sec2.mul_(f.flip(0))
        out.append((row0, n, idx))
    return side, content, out


def _ptrs(ts):
    return pkg("lib").ptr_array(ts)


def _forward(case, side, content, probs, gen):
    """One forward on fresh guarded buffers; returns (buffers per problem, partial floats the query gave)."""
    lib = pkg("lib")
    L = lib.load()
    B, d, inv_t = case.B, case.d, 1.0 / case.temp
    n_ws = L.mmrec_infonce_fwd_workspace_floats(B)
    bufs = [dict(loss=Guarded(1, gen), V1n=Guarded(B * d, gen), V2n=Guarded(B * d, gen),
                 inv_norm=Guarded(2 * B, gen), ttl=Guarded(B, gen), partial=Guarded(n_ws, gen))
            for _ in probs]
    T1 = [side[row0:] for row0, _, _ in probs]
    T2 = [content[row0:] for row0, _, _ in probs]
    idx = [i for _, _, i in probs]
    if case.path == "pair":
        lib.call("mmrec_infonce_pair_fwd_f32", _ptrs(T1), _ptrs(T2), d, _ptrs(idx), B, inv_t,
                 *[_ptrs([b[k].t for b in bufs]) for k in ("loss", "V1n", "V2n", "inv_norm", "ttl", "partial")],
                 lib.stream())
    else:
        counter = torch.zeros(1 + cdiv(B, TILE) + 64, dtype=torch.int32, device=DEV)
        b = bufs[0]
        lib.call("mmrec_infonce_fwd_f32", lib.ptr(T1[0]), lib.ptr(T2[0]), d, lib.ptr(idx[0]), B, inv_t,
                 *[lib.ptr(b[k].t) for k in ("loss", "V1n", "V2n", "inv_norm", "ttl", "partial")],
                 lib.ptr(counter), lib.stream())
        torch.cuda.synchronize()
        assert not counter.any(), "arrival counters not reset"
    torch.cuda.synchronize()
    return bufs, n_ws


def _backward(case, n_rows, probs, fw, coefs, gen):
    """One backward into fresh zero tables [n_rows, d] (guarded); returns (dside, dcontent, ws per problem)."""
    lib = pkg("lib")
    L = lib.load()
    B, d, inv_t = case.B, case.d, 1.0 / case.temp
    n_splits = case.n_splits if case.n_splits is not None else L.mmrec_infonce_splits(B)
    dside, dcont = Guarded(n_rows * d, gen, fill=0.0), Guarded(n_rows * d, gen, fill=0.0)
    ws = [(Guarded(n_splits * B * d, gen), Guarded(n_splits * B * d, gen)) for _ in probs]
    coef_t = [torch.tensor([c], dtype=torch.float32, device=DEV) for c in coefs]
    dT1 = [dside.t[row0 * d:] for row0, _, _ in probs]
    dT2 = [dcont.t[row0 * d:] for row0, _, _ in probs]
    idx = [i for _, _, i in probs]
    if case.path == "pair":
        lib.call("mmrec_infonce_pair_bwd_f32", *[_ptrs([b[k].t for b in fw]) for k in ("V1n", "V2n", "inv_norm", "ttl")],
                 d, _ptrs(idx), B, inv_t, _ptrs(coef_t), n_splits, _ptrs([w[0].t for w in ws]),
                 _ptrs([w[1].t for w in ws]), _ptrs(dT1), _ptrs(dT2), lib.stream())
    else:
        b = fw[0]
        lib.call("mmrec_infonce_bwd_f32", *[lib.ptr(b[k].t) for k in ("V1n", "V2n", "inv_norm", "ttl")], d,
                 lib.ptr(idx[0]), B, inv_t, lib.ptr(coef_t[0]), n_splits, lib.ptr(ws[0][0].t), lib.ptr(ws[0][1].t),
                 lib.ptr(dT1[0]), lib.ptr(dT2[0]), lib.stream())
    torch.cuda.synchronize()
    return dside, dcont, ws


# ------------------------------------------------------------------ GPU: every regime against float64
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_infonce_regime_against_float64(case):
    reg = case.regime()
    assert {k: reg[k] for k in case.expect} == case.expect, f"{case.name} left its regime: {reg}"
    gen = torch.Generator(device=DEV).manual_seed(1000 + CASE_IDS.index(case.name))
    side, content, probs = _problems(case, gen)
    B, d = case.B, case.d
    n_rows = side.shape[0]

    fw, n_ws = _forward(case, side, content, probs, gen)
    for p, b in enumerate(fw):
        for k, g in b.items():
            g.check(f"problem {p} {k}")
        assert b["partial"].written() == reg["fwd_floats"], \
            f"problem {p}: the forward wrote {b['partial'].written()} floats of partial, the restated " \
            f"footprint is {reg['fwd_floats']} (query {n_ws})"
        for k in ("loss", "V1n", "V2n", "inv_norm", "ttl"):
            assert b[k].written() == b[k].n, f"problem {p} {k} not fully written"
    fw2, _ = _forward(case, side, content, probs, gen)
    for p in range(len(probs)):
        for k in ("loss", "ttl"):
            assert torch.equal(fw[p][k].t.view(torch.int32), fw2[p][k].t.view(torch.int32)), \
                f"problem {p} {k} differs between two forward calls"

    dside, dcont, ws = _backward(case, n_rows, probs, fw, case.coef, gen)
    dside.check("dT1")
    dcont.check("dT2")
    slab = B * d
    for p, (w1, w2) in enumerate(ws):
        for name, w in (("dV1_ws", w1), ("dV2_ws", w2)):
            w.check(f"problem {p} {name}")
            assert w.written() == reg["bwd_slabs"] * slab, \
                f"problem {p} {name}: {w.written() / slab} slabs written, restated {reg['bwd_slabs']}"
            if reg["bwd_live_slabs"] < reg["bwd_slabs"]:            # splits past the last tile
                assert not w.t[reg["bwd_live_slabs"] * slab:reg["bwd_slabs"] * slab].any()
    referenced = torch.zeros(n_rows, dtype=torch.bool, device=DEV)
    for row0, _, idx in probs:
        referenced[row0 + idx] = True
    for name, g in (("dT1", dside), ("dT2", dcont)):
        rows = g.t.view(n_rows, d)
        assert not rows[~referenced].any(), f"{name}: a row no index references was written"

    dside2, dcont2, _ = _backward(case, n_rows, probs, fw, case.coef, gen)
    for p, (row0, n, idx) in enumerate(probs):
        if idx.unique().numel() == B:                              # no repeats: no atomics on one row
            for a, b in ((dside, dside2), (dcont, dcont2)):
                sec = slice(row0 * d, (row0 + n) * d)
                assert torch.equal(a.t[sec].view(torch.int32), b.t[sec].view(torch.int32)), \
                    f"problem {p}: backward not bit-identical without repeated indices"

    for p, (row0, n, idx) in enumerate(probs):
        T1, T2 = side[row0:row0 + n], content[row0:row0 + n]
        coef = case.coef[p]
        got = dict(loss=fw[p]["loss"].t[0], ttl=fw[p]["ttl"].t,
                   dT1=dside.t.view(n_rows, d)[row0:row0 + n], dT2=dcont.t.view(n_rows, d)[row0:row0 + n])
        v64 = F.normalize(T1[idx].double(), dim=1)
        assert float((fw[p]["V1n"].t.view(B, d).double() - v64).abs().max()) < 1e-6
        if coef == 0:
            assert not got["dT1"].any() and not got["dT2"].any(), "coefficient 0: gradients not exactly zero"
        e, e32 = assert_close(got, T1, T2, idx, case.temp, coef, f"{case.name} problem {p}", tc_bwd_chain_tol(reg))
        print(f"{case.name} p{p} [{reg['path']} splits={reg['splits']} {reg['per_split'][:4]} "
              f"lim={reg['limiter']}]: " + " ".join(f"{k}={e[k]:.1e}/{e32[k]:.1e}" for k in TOL))


@pytest.mark.gpu
def test_single_forward_refuses_d96():
    """d = 96 is neither the tcgen05 width nor an mma.sync instantiation: an error, nothing computed."""
    lib = pkg("lib")
    L = lib.load()
    B, d = 100, 96
    gen = torch.Generator(device=DEV).manual_seed(3)
    T = torch.randn(B, d, generator=gen, device=DEV)
    idx = torch.arange(B, device=DEV)
    loss, partial = Guarded(1, gen), Guarded(L.mmrec_infonce_fwd_workspace_floats(B), gen)
    V1, V2 = torch.empty(B, d, device=DEV), torch.empty(B, d, device=DEV)
    inv, ttl = torch.empty(2 * B, device=DEV), torch.empty(B, device=DEV)
    counter = torch.zeros(64, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match="unsupported d=96"):
        lib.call("mmrec_infonce_fwd_f32", lib.ptr(T), lib.ptr(T), d, lib.ptr(idx), B, 5.0, lib.ptr(loss.t),
                 lib.ptr(V1), lib.ptr(V2), lib.ptr(inv), lib.ptr(ttl), lib.ptr(partial.t), lib.ptr(counter),
                 lib.stream())
    torch.cuda.synchronize()
    assert loss.written() == 0 and partial.written() == 0
    loss.check("loss")
    partial.check("partial")


# ------------------------------------------------------------------ GPU: the autograd wiring
@pytest.mark.gpu
@pytest.mark.parametrize("B,n_pos,d", [(43, 43, 64), (300, 300, 64), (300, 257, 64), (513, 513, 128)],
                         ids=["pair-B43", "pair-B300", "single-tc-unequal", "mma-d128"])
def test_ops_infonce_pair_reduce_false(B, n_pos, d):
    """ops.infonce_pair(reduce=False) with a different upstream coefficient per problem (a swap of the
    items / users problems fails) on tables whose item rows start at an odd n_users; the pair entry when
    both index counts match and d = 64, otherwise one single-problem call per problem."""
    ops = pkg("ops")
    gen = torch.Generator(device=DEV).manual_seed(B + n_pos + d)
    nu, ni = 151, 120
    side = torch.randn(nu + ni, d, generator=gen, device=DEV)
    content = torch.randn(nu + ni, d, generator=gen, device=DEV)
    users = torch.randint(0, nu, (B,), generator=gen, device=DEV)
    pos = torch.randint(0, ni, (n_pos,), generator=gen, device=DEV)
    s, c = side.clone().requires_grad_(True), content.clone().requires_grad_(True)
    losses = ops.infonce_pair(s, c, nu, users, pos, 0.2, reduce=False)
    assert losses.shape == (2,)
    coef = torch.tensor([0.3, -1.7], device=DEV)
    (losses * coef).sum().backward()
    so, co = side.double().requires_grad_(True), content.double().requires_grad_(True)
    lo = torch.stack([oops.infonce(so[nu:][pos], co[nu:][pos], 0.2), oops.infonce(so[:nu][users], co[:nu][users], 0.2)])
    (lo * coef.double()).sum().backward()
    assert float(((losses.detach().double() - lo.detach()).abs() / lo.detach().abs()).max()) < 1e-5
    for got, want in ((s.grad, so.grad), (c.grad, co.grad)):
        assert float((got.double() - want).abs().max() / want.abs().max()) < 2e-5
