"""The 3xTF32 GEMM (mmrec_gemm_tf32x3_f32) in every dispatch regime against float64, elementwise.

The host code picks the kernel and its partition from the shape alone: the tcgen05 kind (1 forward,
2 dW stored transposed, 3 dx), the N tile, the split-K count, the row tiles per CTA and the N tiles
per CTA -- or one of the eight mma.sync tile kernels. The policy is restated below in plain Python;
every case names the regime it pins, and the host-only part (no `gpu` mark) checks the restatement
against the library's own split count and activation support, so a policy change that moves a shape
off its regime fails here instead of silently testing something else. No case sets an environment
switch: each regime is reached through its shape.

The GPU cases call the C ABI with buffers they own: the output and the split-K workspace start as
NaN (an element the kernel never writes fails), and sentinel rows around them must come back
bit-unchanged. Every element must satisfy |C - C64| <= tau * (|A| |B| + |bias|), with tau derived
from the regime (see `gemm_tau`).
"""
import math

import pytest
import torch

from conftest import pkg

DEV = "cuda:0"
U = 2.0 ** -24                       # fp32 unit roundoff (round to nearest)

# ------------------------------------------------------------------ the host policy, restated
SMS, BM, KB, CHUNK_KB = 148, 128, 32, 2      # kNumSMs, kBM, kKB, kChunkKB of gemm_tc05.cu
FB_BK = 32                                   # BK of gemm_tf32x3.cu


def cdiv(a, b):
    return -(-a // b)


def tc05_kind(M, N, K, a_k, b_k):
    """gemm_tc05_kind: 1 forward, 2 dW, 3 dx, 0 = not covered (mma.sync fallback)."""
    if a_k and b_k:
        return 1 if (((M >= 1024 and K >= 256) or (M >= 8192 and K == 128 and N == 128))
                     and N in (32, 64, 128) and K % 4 == 0) else 0
    if not a_k and not b_k:
        return 2 if (((N >= 1024 and K >= 256) or (K >= 8192 and M == 128 and N == 128))
                     and M in (32, 64, 128) and N % 4 == 0) else 0
    if a_k and not b_k:
        wide_dense = K == 128 or N == 128
        return 3 if (((M >= 1024 and N >= 1024) or (M >= 8192 and N == 128 and wide_dense))
                     and N % 128 == 0 and K % 4 == 0 and K <= 256) else 0
    return 0


def best_parts(row_tiles, units, max_parts, fill):
    best, best_cost = 1, -1
    for p in range(1, max_parts + 1):
        per = cdiv(units, p)
        if cdiv(units, per) != p:
            continue
        cost = cdiv(row_tiles * p, SMS) * (per + fill)
        if best_cost < 0 or cost < best_cost:
            best, best_cost = p, cost
    return best


def parts_cost(row_tiles, units, p, mt, fill):
    per = cdiv(units, p)
    if cdiv(units, per) != p:
        return -1
    return cdiv(cdiv(row_tiles, mt) * p, SMS) * (per * mt + fill)


def best_mt(row_tiles, units, p, fill):
    best, best_cost = 1, parts_cost(row_tiles, units, p, 1, fill)
    if best_cost < 0:
        return 1
    for mt in range(2, min(4, row_tiles) + 1):
        c = parts_cost(row_tiles, units, p, mt, fill)
        if 0 <= c < best_cost:
            best, best_cost = mt, c
    return best


def best_parts_mt(row_tiles, units, max_parts, fill):
    best, best_cost = 1, -1
    for p in range(1, max_parts + 1):
        c = parts_cost(row_tiles, units, p, best_mt(row_tiles, units, p, fill), fill)
        if c < 0:
            continue
        c = 2 * c + p                     # every split writes a slab and the reduce reads it
        if best_cost < 0 or c < best_cost:
            best, best_cost = p, c
    return best


def tc05_splits(M, N, K, kind):
    if kind == 3:
        return 1
    row_tiles = cdiv(N if kind == 2 else M, BM)
    units = cdiv(cdiv(K, KB), CHUNK_KB)
    if row_tiles == 1:
        return best_parts(row_tiles, units, 128, 3)
    return best_parts_mt(row_tiles, units, 32, 3)


def fallback_tile(M, N, a_k, b_k):
    """(BM, BN) of the mma.sync instantiation mmrec_gemm_tf32x3_f32 launches."""
    big_m, big_n = a_k and M > 64, (not b_k) and N > 64
    return (128 if big_m else 64), (128 if big_n else 64)


def fallback_splits(M, N, K, a_k, b_k):
    bm, bn = fallback_tile(M, N, a_k, b_k)
    tiles = cdiv(M, bm) * cdiv(N, bn)
    s = min(cdiv(2 * SMS, tiles), cdiv(K, 4 * FB_BK), 64)
    return max(s, 1)


def gemm_splits(M, N, K, a_k, b_k):
    """mmrec_gemm_splits."""
    kind = tc05_kind(M, N, K, a_k, b_k)
    return tc05_splits(M, N, K, kind) if kind else fallback_splits(M, N, K, a_k, b_k)


def linear_act_tc_supported(M, K, N):
    """mmrec_linear_act_tc_supported: kind 1 without split-K (the activation rides in the store)."""
    return int(tc05_kind(M, N, K, 1, 1) == 1 and tc05_splits(M, N, K, 1) == 1)


def regime(M, N, K, a_k, b_k, splits, bias=False):
    """What gemm_tc05_dispatch / the fallback launch do for this call (`splits` as passed)."""
    kind = tc05_kind(M, N, K, a_k, b_k)
    n_kb = cdiv(K, KB)
    units = cdiv(n_kb, CHUNK_KB)
    refused = None
    if kind in (1, 2):
        kb_per_split = cdiv(units, splits) * CHUNK_KB
        k_splits = cdiv(n_kb, kb_per_split)
        if k_splits != splits:
            refused = "split count"
        elif kind == 2 and bias and splits == 1:
            refused = "bias axis"
        else:
            rows = M if kind == 1 else N                  # UMMA M: kind 2 computes C^T
            row_tiles = cdiv(rows, BM)
            if k_splits > 1:
                mt = best_mt(row_tiles, units, k_splits, 3)
            elif kind == 1 and row_tiles > SMS:
                mt = cdiv(row_tiles, SMS)                 # tiles_per_cta
            else:
                mt = 1
            last_kb = n_kb - (k_splits - 1) * kb_per_split
            return dict(path="tc05", kind=kind, nt=(N if kind == 1 else M), splits=k_splits, mt=mt,
                        row_tiles=row_tiles, ragged=row_tiles % mt != 0,
                        last_cta_tiles=row_tiles - (cdiv(row_tiles, mt) - 1) * mt, row_rem=rows % BM,
                        n_kb=n_kb, k_tail=K % KB, last_split_kb=last_kb,
                        chunks_per_split=cdiv(kb_per_split, CHUNK_KB))
    elif kind == 3:
        if splits != 1:
            refused = "split count"
        else:
            row_tiles, n_tiles = cdiv(M, BM), N // 64
            chunks = best_parts(row_tiles, n_tiles, n_tiles, 1)
            per = cdiv(n_tiles, chunks)
            chunks = cdiv(n_tiles, per)
            mt = cdiv(row_tiles, SMS) if chunks == 1 and row_tiles > SMS else 1
            return dict(path="tc05", kind=3, nt=64, splits=1, n_chunks=chunks, nt_per_cta=per, mt=mt,
                        row_tiles=row_tiles, ragged=row_tiles % mt != 0, row_rem=M % BM, n_kb=n_kb,
                        k_tail=K % KB, chunks_per_split=cdiv(n_kb, CHUNK_KB))
    bm, bn = fallback_tile(M, N, a_k, b_k)
    k_per_split = cdiv(cdiv(K, splits), FB_BK) * FB_BK
    return dict(path="mma.sync", kind=0, refused=refused, tile=(a_k, b_k, bm, bn),
                splits=cdiv(K, k_per_split), m_rem=M % bm, n_rem=N % bn, k_tail=K % FB_BK,
                kb_per_split=cdiv(k_per_split, FB_BK))


def gemm_tau(reg):
    """Elementwise relative bound of one call: |C - C64| <= tau * (|A| |B| + |bias|)_ij.

    * Split: hi = tf32(x) rounded to nearest (|lo| <= 2^-11 |x|); the tensor core reads lo as tf32,
      dropping its 13 low bits (<= 2^-10 |lo|, i.e. 2^-21 |x|) in each of lo*hi and hi*lo, and
      lo*lo (<= 2^-22 |a||b|) is never formed: 2 * 2^-21 + 2^-22 per product.
    * Chains: the tensor core truncates its fp32 accumulator after every instruction (<= 1 ulp,
      2^-23 of a running sum bounded by the chain's sum of |a||b|). A tcgen05 chain is 2 K blocks x
      4 k-steps x 3 products = 24 instructions (gemm_tc05.cu, epilogue comment); an mma.sync chain
      is one 32-wide K block, 12 instructions. Over all chains of a row: n_instr * 2^-23.
    * The chains of a split, the split-K slabs and the bias are added in round-to-nearest fp32:
      each addition <= 2^-24 of a partial sum bounded by the row's sum of |a||b| + |bias|.
    For the 7050 x 64 x 4096 forward (5 splits of 13 chains) this is 1.2e-6 + 2.9e-6 + 19 * 6e-8
    = 5.2e-6; the largest, the 122-split dW over 62420 rows, is 1.2e-5. A lost product costs
    ~1e-4 of |a||b| per term, a skipped 32-float K block ~1 / n_kb of the row, a missing bias the
    whole bias in the rows scaled by 1e-3: all far above tau.
    """
    split = 2 * 2.0 ** -21 + 2.0 ** -22
    if reg["path"] == "tc05":
        chain = 24 * 2.0 ** -23
        adds = reg["chunks_per_split"] + reg["splits"] + 1
    else:
        chain = 12 * 2.0 ** -23
        adds = reg["kb_per_split"] + reg["splits"] + 1
    return split + chain + adds * U


# ------------------------------------------------------------------ the cases
class Case:
    def __init__(self, name, M, N, K, a_k, b_k, expect, bias=False, splits=None, act=False):
        self.name, self.M, self.N, self.K, self.a_k, self.b_k = name, M, N, K, a_k, b_k
        self.expect, self.bias, self.splits, self.act = expect, bias, splits, act

    def shape(self):
        return self.M, self.N, self.K, self.a_k, self.b_k

    def call_splits(self):
        return gemm_splits(*self.shape()) if self.splits is None else self.splits

    def regime(self):
        return regime(*self.shape(), self.call_splits(), self.bias)


def _tc(kind, **kw):
    return dict(path="tc05", kind=kind, **kw)


def _fb(a_k, b_k, bm, bn, **kw):
    return dict(path="mma.sync", tile=(a_k, b_k, bm, bn), **kw)


CASES = [
    # kind 1 (forward y = x W^T), A [M, K], B [N, K]
    Case("fwd-d32", 7050, 32, 4096, 1, 1, _tc(1, nt=32, splits=5, mt=2, ragged=False, row_rem=10)),
    Case("fwd-d64-bias-in-reduce", 7050, 64, 4096, 1, 1, _tc(1, nt=64, splits=5, mt=2, ragged=False), bias=True),
    Case("fwd-d128", 7050, 128, 4096, 1, 1, _tc(1, nt=128, splits=5, mt=2, ragged=False)),
    Case("fwd-mt2-ragged", 6919, 64, 4096, 1, 1, _tc(1, splits=5, mt=2, ragged=True, last_cta_tiles=1)),
    Case("fwd-mt3-ragged-8splits", 6395, 64, 4096, 1, 1, _tc(1, splits=8, mt=3, ragged=True, last_cta_tiles=2)),
    Case("fwd-d32-mt3-ragged-2splits", 20000, 32, 512, 1, 1, _tc(1, nt=32, splits=2, mt=3, ragged=True)),
    Case("fwd-mt4-ragged", 14386, 64, 4096, 1, 1, _tc(1, splits=5, mt=4, ragged=True, last_cta_tiles=1)),
    Case("fwd-ktail4", 1030, 64, 388, 1, 1, _tc(1, splits=4, mt=1, n_kb=13, k_tail=4, last_split_kb=1)),
    Case("fwd-odd-kblocks", 7050, 64, 4128, 1, 1, _tc(1, splits=5, n_kb=129, last_split_kb=25)),
    Case("fwd-threshold-tc05", 1024, 32, 256, 1, 1, _tc(1, nt=32, splits=2, mt=1, row_rem=0)),
    Case("fwd-threshold-m1023", 1023, 64, 256, 1, 1, _fb(1, 1, 128, 64)),
    Case("fwd-threshold-k252", 2000, 64, 252, 1, 1, _fb(1, 1, 128, 64)),
    Case("dense-nosplit-bias-in-store", 28422, 128, 128, 1, 1,
         _tc(1, nt=128, splits=1, mt=2, ragged=True, last_cta_tiles=1), bias=True, act=True),
    Case("dense-nosplit-mt4", 62420, 128, 128, 1, 1, _tc(1, nt=128, splits=1, mt=4, ragged=False), act=True),
    Case("dense-split2-no-act", 23033, 128, 128, 1, 1, _tc(1, nt=128, splits=2, mt=3), act=True),
    # kind 2 (dW = dy^T x, stored transposed), A [K, M], B [K, N]
    Case("dW-d32", 32, 4096, 7050, 0, 0, _tc(2, nt=32, splits=4, mt=1, k_tail=10, row_tiles=32)),
    Case("dW-d64-bias-in-reduce", 64, 4096, 7050, 0, 0, _tc(2, nt=64, splits=4, k_tail=10), bias=True),
    Case("dW-d128", 128, 4096, 7050, 0, 0, _tc(2, nt=128, splits=4, k_tail=10)),
    Case("dW-ragged-n", 64, 1028, 300, 0, 0, _tc(2, splits=3, row_rem=4, k_tail=12)),
    Case("dW-single-row-tile", 128, 128, 62420, 0, 0, _tc(2, nt=128, splits=122, row_tiles=1, k_tail=20)),
    Case("dW-single-row-tile-last-split-1kb", 128, 128, 28422, 0, 0, _tc(2, splits=112, last_split_kb=1)),
    # the caller's split count: 1 runs the whole 7050-long K in one CTA per row tile; 1 with a bias,
    # or a count the K blocks cannot be cut into, is refused by the tcgen05 dispatch (mma.sync instead)
    Case("dW-forced-1split", 64, 4096, 7050, 0, 0, _tc(2, splits=1, mt=1, chunks_per_split=111), splits=1),
    Case("dW-forced-1split-bias-refused", 64, 4096, 7050, 0, 0,
         _fb(0, 0, 64, 128, refused="bias axis", splits=1), bias=True, splits=1),
    Case("dW-split-count-refused", 64, 4096, 7050, 0, 0, _fb(0, 0, 64, 128, refused="split count", splits=111),
         bias=True, splits=112),
    Case("dW-nosplit-bias-refused", 64, 40000, 256, 0, 0, _fb(0, 0, 64, 128, refused="bias axis", splits=1),
         bias=True),
    Case("dW-nosplit", 64, 40000, 256, 0, 0, _tc(2, splits=1, mt=1, row_tiles=313, row_rem=64)),
    # kind 3 (dx = dy W), A [M, K], B [K, N]
    Case("dx-d64-bias", 7050, 4096, 64, 1, 0, _tc(3, n_chunks=5, nt_per_cta=13, mt=1), bias=True),
    Case("dx-d128", 7050, 4096, 128, 1, 0, _tc(3, n_chunks=5, nt_per_cta=13, mt=1)),
    Case("dx-mt2-ragged", 19000, 128, 128, 1, 0, _tc(3, n_chunks=1, nt_per_cta=2, mt=2, ragged=True)),
    Case("dx-threshold-tc05", 1030, 1024, 256, 1, 0, _tc(3, n_chunks=16, nt_per_cta=1)),
    Case("dx-threshold-k260", 7050, 4096, 260, 1, 0, _fb(1, 0, 128, 128)),
    # the eight mma.sync instantiations, split-K > 1, M and N not multiples of the tile, K tail of 8
    Case("mma-kk-128x64", 300, 100, 1000, 1, 1, _fb(1, 1, 128, 64, splits=8, k_tail=8)),
    Case("mma-kk-64x64", 50, 68, 1000, 1, 1, _fb(1, 1, 64, 64, splits=8)),
    Case("mma-kn-128x128", 300, 200, 1000, 1, 0, _fb(1, 0, 128, 128, splits=8)),
    Case("mma-kn-128x64", 300, 60, 1000, 1, 0, _fb(1, 0, 128, 64, splits=8)),
    Case("mma-kn-64x128", 50, 200, 1000, 1, 0, _fb(1, 0, 64, 128, splits=8)),
    Case("mma-kn-64x64", 50, 60, 1000, 1, 0, _fb(1, 0, 64, 64, splits=8)),
    Case("mma-nn-64x128", 100, 200, 1000, 0, 0, _fb(0, 0, 64, 128, splits=8)),
    Case("mma-nn-64x64", 100, 60, 1000, 0, 0, _fb(0, 0, 64, 64, splits=8), bias=True),
]
CASE_IDS = [c.name for c in CASES]


def describe(reg):
    if reg["path"] == "mma.sync":
        a_k, b_k, bm, bn = reg["tile"]
        return f"mma.sync {'K' if a_k else 'M'}{'K' if b_k else 'N'} {bm}x{bn} splits={reg['splits']}"
    s = f"kind={reg['kind']} NT={reg['nt']} splits={reg['splits']} mt={reg['mt']}"
    return s + (" ragged" if reg["ragged"] else "")


# ------------------------------------------------------------------ host-only checks
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_policy_restatement_pins_regime(case):
    """The restated policy agrees with the library, and the case is still in the regime it names."""
    L = pkg("lib").load()
    assert gemm_splits(*case.shape()) == L.mmrec_gemm_splits(*case.shape()), case.name
    if case.act:
        M, N, K = case.M, case.N, case.K
        assert linear_act_tc_supported(M, K, N) == L.mmrec_linear_act_tc_supported(M, K, N)
    reg = case.regime()
    got = {k: reg.get(k) for k in case.expect}
    assert got == case.expect, f"{case.name}: {describe(reg)} {reg}"


def test_policy_activation_support():
    L = pkg("lib").load()
    want = {28422: 1, 62420: 1, 10001: 1, 16384: 1, 23033: 0, 8192: 0, 8191: 0}
    for M, w in want.items():
        assert linear_act_tc_supported(M, 128, 128) == w == L.mmrec_linear_act_tc_supported(M, 128, 128), M
    assert L.mmrec_linear_act_tc_supported(28422, 64, 64) == 0          # the dense 128 x 128 rule only


def test_fallback_instantiations_all_named():
    tiles = {c.regime()["tile"] for c in CASES if c.name.startswith("mma-")}
    assert tiles == {(1, 1, 128, 64), (1, 1, 64, 64), (1, 0, 128, 128), (1, 0, 128, 64), (1, 0, 64, 128),
                     (1, 0, 64, 64), (0, 0, 64, 128), (0, 0, 64, 64)}
    for c in CASES:
        r = c.regime()
        if c.name.startswith("mma-"):
            assert r["splits"] > 1 and r["m_rem"] and r["n_rem"] and r["k_tail"], c.name


# ------------------------------------------------------------------ GPU helpers
def _pow10(n, lo, hi, gen):
    """Per-row scales 10^e, e uniform in [lo, hi]: the elementwise bound sees small rows too."""
    e = torch.randint(lo, hi + 1, (n, 1), generator=gen, device=DEV)
    return torch.pow(10.0, e.double()).float()


def _operands(M, N, K, seed, lo=-3, hi=3):
    """Logical a [M, K] and b [N, K] (C = a b^T) with rows of a and of b scaled by powers of 10."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    a = torch.randn(M, K, generator=gen, device=DEV) * _pow10(M, lo, hi, gen)
    b = torch.randn(N, K, generator=gen, device=DEV) * _pow10(N, lo, hi, gen)
    bias = torch.randn(N, generator=gen, device=DEV) * _pow10(N, lo, hi, gen).view(-1)
    return a, b, bias


def _sentinel_buffer(n_lead, n_rows, n_tail, n_cols, seed):
    """[n_lead + n_rows + n_tail, n_cols]: NaN in the middle, random bits around it."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    buf = torch.randn(n_lead + n_rows + n_tail, n_cols, generator=gen, device=DEV)
    buf[n_lead:n_lead + n_rows] = float("nan")
    return buf


def _check_sentinels(buf, n_lead, n_rows, ref):
    assert torch.equal(buf[:n_lead].view(torch.int32), ref[:n_lead].view(torch.int32)), "write before the output"
    assert torch.equal(buf[n_lead + n_rows:].view(torch.int32), ref[n_lead + n_rows:].view(torch.int32)), \
        "write after the output"


def _assert_within(out, want64, bound64, what):
    err = (out.detach().double() - want64).abs()
    ok = err <= bound64                                 # NaN (unwritten) compares False
    n_bad = int((~ok).sum())
    if n_bad:
        idx = int((~ok).flatten().nonzero()[0])
        ratio = float((err / bound64.clamp_min(1e-300)).nan_to_num(float("inf")).max())
        raise AssertionError(f"{what}: {n_bad} of {ok.numel()} elements outside the bound; first at flat "
                             f"index {idx} (got {float(out.flatten()[idx])}, want {float(want64.flatten()[idx])}, "
                             f"bound {float(bound64.flatten()[idx]):.3e}); worst err / bound {ratio:.3g}")
    return float((err / bound64.clamp_min(1e-300)).max())


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _cublas(fn):
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False          # plain fp32 SGEMM
    try:
        return fn()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


LEAD, TAIL = 2, 3                      # sentinel rows before / after every output


def _run_gemm_abi(case, seed):
    """One mmrec_gemm_tf32x3_f32 call on NaN-filled buffers; returns (C, a, b, bias)."""
    lib = pkg("lib")
    M, N, K, a_k, b_k = case.shape()
    a, b, bias = _operands(M, N, K, seed)
    bias = bias if case.bias else None
    A = a if a_k else a.t().contiguous()
    B = b if b_k else b.t().contiguous()
    splits = case.call_splits()
    cbuf = _sentinel_buffer(LEAD, M, TAIL, N, seed + 1)
    cref = cbuf.clone()
    C = cbuf[LEAD:LEAD + M]
    ws = wref = None
    if splits > 1:
        ws = _sentinel_buffer(0, splits * M, TAIL, N, seed + 2)
        wref = ws.clone()
    lib.call("mmrec_gemm_tf32x3_f32", lib.ptr(A), a_k, lib.ptr(B), b_k, lib.ptr(bias), C.data_ptr(), M, N, K,
             splits, lib.ptr(ws), lib.stream())
    torch.cuda.synchronize()
    _check_sentinels(cbuf, LEAD, M, cref)
    if ws is not None:
        _check_sentinels(ws, 0, splits * M, wref)
    return C, a, b, bias


def _reference(a, b, bias):
    a64, b64 = a.double(), b.double()
    want = a64 @ b64.t()
    mag = a64.abs() @ b64.abs().t()
    if bias is not None:
        want += bias.double()
        mag += bias.double().abs()
    return want, mag


# ------------------------------------------------------------------ GPU: the GEMM in every regime
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_gemm_regime_against_float64(case):
    reg = case.regime()
    got = {k: reg.get(k) for k in case.expect}
    assert got == case.expect, f"{case.name} left its regime: {describe(reg)}"
    C, a, b, bias = _run_gemm_abi(case, seed=1000 + 10 * CASE_IDS.index(case.name))
    want, mag = _reference(a, b, bias)
    tau = gemm_tau(reg)
    worst = _assert_within(C, want, tau * mag, f"{case.name} [{describe(reg)}] tau={tau:.2e}")
    print(f"{case.name}: {describe(reg)} tau={tau:.2e} worst err/bound={worst:.3f}")
    # second guard: within 4x of cuBLAS SGEMM's own (normwise) distance to float64
    yc = _cublas(lambda: a @ b.t() + (bias if bias is not None else 0.0))
    assert _rel(C, want) < 4 * max(_rel(yc, want), 1e-7)


@pytest.mark.gpu
def test_gemm_refuses_mn_contiguous_a_with_k_contiguous_b():
    lib = pkg("lib")
    A = torch.zeros(256, 64, device=DEV)            # [K, M]
    B = torch.zeros(64, 256, device=DEV)            # [N, K]
    C = torch.full((64, 64), float("nan"), device=DEV)
    L = lib.load()
    rc = L.mmrec_gemm_tf32x3_f32(lib.ptr(A), 0, lib.ptr(B), 1, None, lib.ptr(C), 64, 64, 256, 1, None, lib.stream())
    assert rc == -1 and b"not instantiated" in L.mmrec_last_error()
    with pytest.raises(RuntimeError, match="not instantiated"):
        lib.call("mmrec_gemm_tf32x3_f32", lib.ptr(A), 0, lib.ptr(B), 1, None, lib.ptr(C), 64, 64, 256, 1, None,
                 lib.stream())
    torch.cuda.synchronize()
    assert bool(C.isnan().all())                    # nothing launched


# ------------------------------------------------------------------ GPU: the activation epilogue
ACT_BOUND = {1: (4e-7, 0.0), 2: (1e-6, 1.5e-7)}     # fast_tanh / fast_sigmoid: rel, abs (test_fast_activations)


def _act64(z, act):
    return z if act == 0 else (torch.tanh(z) if act == 1 else torch.sigmoid(z))


def _act_bound(y64, bound_z, act):
    """Bound on |y - act(z64)| given |z - z64| <= bound_z: the derivative at z64, the second-order
    term (|act''| <= 1), and the error of the fast activation itself."""
    if act == 0:
        return bound_z
    d = 1 - y64 * y64 if act == 1 else y64 * (1 - y64)
    rel, ab = ACT_BOUND[act]
    return d * bound_z + bound_z * bound_z + rel * y64.abs() + ab


@pytest.mark.gpu
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("act", [0, 1, 2])
@pytest.mark.parametrize("M", [28422, 62420])
def test_linear_act_tc_against_float64(M, act, bias):
    """mmrec_linear_act_tc_f32 (bias and tanh / sigmoid in the tcgen05 store epilogue) at the
    ragged tiles_per_cta shape and at 62420 rows; then the backward as ops.dense_act runs it:
    mmrec_act_bwd_f32, dx on kind 3, dW on kind 2, db by colsum."""
    lib, ops = pkg("lib"), pkg("ops")
    d = 128
    reg = regime(M, d, d, 1, 1, 1, bias)
    assert reg["kind"] == 1 and reg["splits"] == 1 and linear_act_tc_supported(M, d, d)
    gen = torch.Generator(device=DEV).manual_seed(M + 10 * act + bias)
    x = torch.randn(M, d, generator=gen, device=DEV) * _pow10(M, -3, 0, gen)
    W = torch.randn(d, d, generator=gen, device=DEV) * 0.1 * _pow10(d, -2, 0, gen)
    b = (torch.randn(d, generator=gen, device=DEV) * 0.5) if bias else None
    ybuf = _sentinel_buffer(LEAD, M, TAIL, d, M + 1)
    yref = ybuf.clone()
    y = ybuf[LEAD:LEAD + M]
    lib.call("mmrec_linear_act_tc_f32", lib.ptr(x), lib.ptr(W), lib.ptr(b), y.data_ptr(), M, d, d, act, lib.stream())
    torch.cuda.synchronize()
    _check_sentinels(ybuf, LEAD, M, yref)
    z64, mag = _reference(x, W, b)
    y64 = _act64(z64, act)
    bound_y = _act_bound(y64, gemm_tau(reg) * mag, act)
    worst = _assert_within(y, y64, bound_y, f"linear_act M={M} act={act} bias={bias}")
    print(f"linear_act M={M} act={act} bias={bias}: worst err/bound={worst:.3f}")

    # backward through the Python wiring, against float64 autograd
    name = {0: None, 1: "tanh", 2: "sigmoid"}[act]
    xg, Wg = x.clone().requires_grad_(True), W.clone().requires_grad_(True)
    bg = b.clone().requires_grad_(True) if bias else None
    yo = ops.dense_act(xg, Wg, bg, name)
    assert torch.equal(yo.detach(), y)
    dy = torch.randn(M, d, generator=gen, device=DEV)
    yo.backward(dy)
    x64, W64 = x.double().requires_grad_(True), W.double().requires_grad_(True)
    b64 = b.double().requires_grad_(True) if bias else None
    out64 = _act64(torch.nn.functional.linear(x64, W64, b64), act)
    out64.backward(dy.double())
    # dz = dy * act'(y) from the kernel's y: its error, then the two GEMMs (their own tau)
    dy64 = dy.double()
    if act == 0:
        e_dz = torch.zeros_like(dy64)
    elif act == 1:
        e_dz = dy64.abs() * (2 * y64.abs() * bound_y + bound_y * bound_y) + 3 * U * dy64.abs()
    else:
        e_dz = dy64.abs() * ((1 - 2 * y64).abs() * bound_y + bound_y * bound_y) + 3 * U * dy64.abs()
    dz64 = dy64 * (1 - y64 * y64) if act == 1 else (dy64 * y64 * (1 - y64) if act == 2 else dy64)
    rdx = regime(M, d, d, 1, 0, gemm_splits(M, d, d, 1, 0))
    rdw = regime(d, d, M, 0, 0, gemm_splits(d, d, M, 0, 0))
    assert rdx["kind"] == 3 and rdw["kind"] == 2
    dzm = dz64.abs() + e_dz
    bound_dx = e_dz @ W64.detach().abs() + gemm_tau(rdx) * (dzm @ W64.detach().abs())
    bound_dw = e_dz.t() @ x64.detach().abs() + gemm_tau(rdw) * (dzm.t() @ x64.detach().abs())
    _assert_within(xg.grad, x64.grad, bound_dx, f"dx ({describe(rdx)})")
    _assert_within(Wg.grad, W64.grad, bound_dw, f"dW ({describe(rdw)})")
    if bias:
        assert _rel(bg.grad, b64.grad) < 1e-5


# ------------------------------------------------------------------ GPU: Python wiring
@pytest.mark.gpu
def test_linear_and_table_project_wiring():
    """ops.linear and ops.table_project (forward kind 1 + reduce with bias, backward dx kind 3 /
    dW kind 2 / db colsum) against float64 autograd, elementwise."""
    ops = pkg("ops")
    I, F, d = 7050, 4096, 64
    gen = torch.Generator(device=DEV).manual_seed(71)
    x = torch.randn(I, F, generator=gen, device=DEV) * _pow10(I, -2, 2, gen)
    W = torch.randn(d, F, generator=gen, device=DEV) * 0.05 * _pow10(d, -2, 2, gen)
    b = torch.randn(d, generator=gen, device=DEV)
    dy = torch.randn(I, d, generator=gen, device=DEV) * _pow10(I, -2, 2, gen)
    rf, rx, rw = (regime(*s, gemm_splits(*s), True) for s in
                  ((I, d, F, 1, 1), (I, F, d, 1, 0), (d, F, I, 0, 0)))
    assert (rf["kind"], rx["kind"], rw["kind"]) == (1, 3, 2)
    xg, Wg, bg = (t.clone().requires_grad_(True) for t in (x, W, b))
    y = ops.linear(xg, Wg, bg)
    y.backward(dy)
    x64, W64, b64 = (t.double().requires_grad_(True) for t in (x, W, b))
    y64 = torch.nn.functional.linear(x64, W64, b64)
    y64.backward(dy.double())
    ax, aw, ady = x64.detach().abs(), W64.detach().abs(), dy.double().abs()
    _assert_within(y, y64.detach(), gemm_tau(rf) * (ax @ aw.t() + b64.detach().abs()), "linear y")
    _assert_within(xg.grad, x64.grad, gemm_tau(rx) * (ady @ aw), "linear dx")
    _assert_within(Wg.grad, W64.grad, gemm_tau(rw) * (ady.t() @ ax), "linear dW")
    assert _rel(bg.grad, b64.grad) < 1e-5

    emb = torch.nn.Embedding.from_pretrained(x.clone(), freeze=False)
    W2, b2 = W.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y2 = ops.table_project(emb, W2, b2)
    assert torch.equal(y2, y)
    y2.backward(dy)
    assert torch.equal(W2.grad, Wg.grad) and torch.equal(b2.grad, bg.grad) and emb.weight.grad is None
    lr = emb.weight._mmrec_lowrank
    assert torch.equal(lr.dY, dy) and torch.equal(lr.W, W)
    _assert_within(lr.dense(), x64.grad, gemm_tau(rx) * (ady @ aw), "LowRankGrad.dense")
    emb.weight._mmrec_lowrank = None


# ------------------------------------------------------------------ GPU: the fused table Adam
TA_SENT = 40                 # sentinel rows after the table and its moments (more than a TMA box)
BETA1, BETA2, EPS, LR = 0.9, 0.999, 1e-8, 1e-2
TA_SCALES = (1.0, 1.0, -0.2)                        # grad_scale of the three steps


def _ta_tau(d):
    """gemm_tau of the product tile the table-Adam epilogue consumes: K = d <= 128 is one split of
    at most two chains (kind 3 layout: A = dY K-major, B = W MN-major)."""
    n_kb = cdiv(d, KB)
    return gemm_tau(dict(path="tc05", chunks_per_split=cdiv(n_kb, CHUNK_KB), splits=1))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,d,wd,nonneg", [
    (7050, 4096, 64, 0.0, False),          # flat partition: 56 x 128 tiles of 32 columns over 148 CTAs
    (7050, 4096, 32, 1e-2, False),
    (7050, 64, 128, 1e-2, False),          # 112 tiles: fewer than the SMs
    (129, 4096, 128, 0.0, False),          # one row in the last tile
    (129, 64, 64, 1e-2, False),
    (31, 4096, 32, 1e-2, False),           # a single, partial row tile
    (31, 64, 128, 0.0, False),
    (7050, 4096, 64, 1e-2, True),          # dY, W >= 0: no cancellation, compared everywhere
])
def test_table_adam_lowrank_against_float64(rows, cols, d, wd, nonneg):
    """mmrec_table_adam_lowrank_f32 (G = dY W on tcgen05, Adam in the epilogue, table and moments
    moved by TMA) for three steps against Adam restated in float64 on G64 = dY64 @ W64, with
    elementwise error bounds carried through the recursion. exp_avg / exp_avg_sq are compared
    everywhere; the table where Adam's division is well conditioned (|G64| far above the GEMM bound
    at every step), elsewhere no step may move a parameter by more than 2 lr."""
    lib = pkg("lib")
    L = lib.load()
    assert L.mmrec_table_lowrank_supported(rows, cols, d)
    gen = torch.Generator(device=DEV).manual_seed(rows * 7 + cols + d)
    bufs = []
    # moments of an optimizer five steps in, with exp_avg^2 <= exp_avg_sq as Adam keeps them, so that
    # no step moves a parameter by more than ~lr
    m0 = torch.randn(rows, cols, generator=gen, device=DEV) * 1e-3
    v0 = m0 * m0 + torch.rand(rows, cols, generator=gen, device=DEV) * 1e-6
    for init in (torch.randn(rows, cols, generator=gen, device=DEV), m0, v0):
        buf = torch.randn(rows + TA_SENT, cols, generator=gen, device=DEV)
        buf[:rows] = init
        bufs.append(buf)
    refs = [buf.clone() for buf in bufs]
    P, Mo, V = (buf[:rows] for buf in bufs)
    p64, m64, v64 = P.double(), Mo.double(), V.double()
    Ep, Em, Ev = (torch.zeros_like(p64) for _ in range(3))
    W = torch.randn(d, cols, generator=gen, device=DEV) * 0.05
    if nonneg:
        W = W.abs()
    W64 = W.double()
    count0 = 5.0
    hyper = torch.tensor([LR, count0], dtype=torch.float64, device=DEV)
    ws = torch.empty(L.mmrec_table_lowrank_workspace_bytes(rows, cols) // 8, dtype=torch.float64, device=DEV)
    sumsq = torch.zeros(1, dtype=torch.float64, device=DEV)
    g2 = torch.zeros(1, dtype=torch.float64, device=DEV)
    tau = _ta_tau(d)
    checked = 0
    for it, scale in enumerate(TA_SCALES):
        dY = torch.randn(rows, d, generator=gen, device=DEV) * (10.0 ** (it - 1))
        if nonneg:
            dY = dY.abs()
        dY64 = dY.double()
        G64 = dY64 @ W64
        EG = tau * (dY64.abs() @ W64.abs())
        # ||dY W||_F^2 and the updated table's sum of squares
        lib.call("mmrec_table_lowrank_sumsq_f64", lib.ptr(dY), lib.ptr(W), rows, cols, d, lib.ptr(ws), lib.ptr(g2),
                 lib.stream())
        want_g2 = float(G64.pow(2).sum())
        assert abs(float(g2) - want_g2) / want_g2 < 1e-6
        p_before = P.clone()
        lib.call("mmrec_table_adam_lowrank_f32", lib.ptr(P), lib.ptr(Mo), lib.ptr(V), lib.ptr(dY), lib.ptr(W), rows,
                 cols, d, lib.ptr(hyper), BETA1, BETA2, EPS, wd, scale, 1, lib.ptr(sumsq), lib.ptr(ws), lib.stream())
        torch.cuda.synchronize()
        for buf, ref in zip(bufs, refs):
            assert torch.equal(buf[rows:].view(torch.int32), ref[rows:].view(torch.int32)), "write beyond rows"
        want_p2 = float(P.double().pow(2).sum())
        assert abs(float(sumsq) - want_p2) / want_p2 < 1e-6
        # float64 Adam step and first-order error bounds of the kernel's fp32 sequence
        step = count0 + it + 1
        step_size = LR / (1 - BETA1 ** step)
        bc2s = math.sqrt(1 - BETA2 ** step)
        g64 = scale * G64 + wd * p64
        Eg = abs(scale) * EG + wd * Ep + 2 * U * (abs(scale) * G64.abs() + wd * p64.abs())
        m_new = m64 + (1 - BETA1) * (g64 - m64)
        Em = BETA1 * Em + (1 - BETA1) * Eg + 3 * U * (m64.abs() + g64.abs())
        v_new = BETA2 * v64 + (1 - BETA2) * g64 * g64
        Ev = BETA2 * Ev + (1 - BETA2) * (2 * g64.abs() * Eg + Eg * Eg) + 4 * U * (BETA2 * v64 + (1 - BETA2) * g64 * g64)
        m64, v64 = m_new, v_new
        sq = v64.sqrt()
        den = sq / bc2s + EPS
        # sqrt.approx / rcp.approx: <= 2 ulp each with their roundings
        Eden = (Ev / (2 * sq) + 2 * U * sq) / bc2s + 2 * U * den
        upd = step_size * m64 / den
        Eupd = step_size * (Em / den + m64.abs() * Eden / (den * den) + 5 * U * m64.abs() / den)
        well = (Eden <= 1e-2 * den) & (G64.abs() >= 100 * EG)
        p64 = p64 - upd
        Ep = torch.where(well, Ep + Eupd, Ep + 2 * LR) + U * p64.abs()
        wellp = well if it == 0 else (wellp & well)
        _assert_within(Mo, m64, 1.05 * Em, f"exp_avg step {it}")
        _assert_within(V, v64, 1.05 * Ev, f"exp_avg_sq step {it}")
        moved = (P - p_before).abs()
        assert float(moved.max()) <= 2 * LR + 4 * U * float(P.abs().max()), f"step {it} moved a parameter by > 2 lr"
        _assert_within(P[wellp], p64[wellp], 1.05 * Ep[wellp], f"table step {it}")
        checked = int(wellp.sum())
    assert float(hyper[1]) == count0 + len(TA_SCALES)
    assert checked >= (rows * cols if nonneg else 0.8 * rows * cols), (checked, rows * cols)
