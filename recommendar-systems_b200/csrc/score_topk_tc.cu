// Full-rank scoring on the 5th-generation tensor cores, fused with train-item masking and a
// per-user top-K (K8/K9/K10): the tcgen05 path behind mmrec_score_mask_topk_f32 and
// mmrec_score_mask_topk_rows_f32 for d = 32 / 64 / 128.
//
// One CTA owns 128 users (the M = 128 rows of the MMA = the 128 TMEM lanes) and walks its item
// range in tiles of 64 items. Warp roles:
//   warps 4-7  producers : two independent groups stream item rows from HBM/L2 (coalesced float4,
//                          one tile in flight per group), split every value into tf32 hi/lo and
//                          store both halves into 128-byte-swizzled K-major shared-memory tiles;
//   warp  8    MMA       : one elected thread issues tcgen05.mma kind::tf32, 3 x (d/8) per tile
//                          (lo*hi + hi*lo + hi*hi -> fp32-accurate scores), accumulating in one of
//                          four 64-column TMEM buffers; tcgen05.commit frees the smem stage and
//                          publishes the accumulator. For d >= 64 the user tile (A operand, hi and
//                          lo halves) sits in TMEM columns [256, 256 + 2d), written once with
//                          tcgen05.st, and the MMA is issued in its A-from-TMEM form;
//   warps 0-3  epilogue  : tcgen05.ld -- TMEM lane i is user i, so every thread reads the scores
//                          of its own user, 32 items at a time, appends those above its running
//                          K-th best to a pending list in shared memory; warp-synchronous flushes
//                          apply the train-item mask (ascending cursor) and push the survivors
//                          into a K-entry 8-ary heap ordered by (score, -id).
// Scores never reach HBM. Stages hand over through mbarriers (smem full/empty, TMEM full/empty).
// Output: per item-split partial lists, descending score, ties -> lower id, merged by
// topk_merge_kernel (score_topk.cu).
#include <math_constants.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc05.cuh"

namespace mmrec {
namespace {

using namespace tc05;

constexpr int kTileM = 128;     // users per CTA
constexpr int kTileN = 64;      // items per MMA tile
constexpr int kAcc = 4;         // TMEM accumulator buffers (64 columns each)
constexpr int kThreadsTC = 288; // 4 epilogue + 4 producer + 1 MMA warp
constexpr int kChunk = 32;      // scores handled per tcgen05.ld

// A_TMEM: the user tile (hi and lo halves) lives in tensor memory next to the accumulators
// (columns [256, 256 + 2D)) instead of shared memory and the MMAs are issued in the A-from-TMEM
// form. That is what makes d = 128 fit: 128 KB of A tiles + 2 x 64 KB item stages + the heaps
// would be 330 KB of shared memory; with A in TMEM it is 200 KB.
template <int D, bool A_TMEM>
struct Cfg {
  static constexpr int KB = D / 32;                         // 128-byte K atoms per row
  static constexpr int STAGES = D <= 32 ? 4 : (D <= 64 && A_TMEM ? 3 : 2);
  static constexpr uint32_t A_HALF = KB * kTileM * 128;     // bytes of the hi (or lo) user tile
  static constexpr uint32_t B_HALF = KB * kTileN * 128;     // bytes of the hi (or lo) item tile
  static constexpr uint32_t STAGE = 2 * B_HALF;
  static constexpr uint32_t OFF_B = A_TMEM ? 0 : 2 * A_HALF;
  static constexpr uint32_t TMEM_COLS = A_TMEM ? 512 : kAcc * kTileN;   // power of two >= 256 + 2D
  static constexpr uint32_t A_COL = kAcc * kTileN;          // first TMEM column of the hi user tile
  static constexpr uint32_t OFF_HEAP = OFF_B + STAGES * STAGE;
  static constexpr int VEC = kTileN * (D / 4) / 128;        // float4 per producer thread per tile
};

struct Better {   // strict total order on (score, id): a ranks before b
  __device__ static bool worse(float av, int ai, float bv, int bi) { return av < bv || (av == bv && ai > bi); }
};

// The K best of a user live in an 8-ary heap in shared memory, column `tid` of [k][128] arrays
// (bank = lane: conflict-free), root = the worst kept entry. K <= 73 gives depth 2: replacing the
// root is two rounds of eight independent shared-memory loads instead of the six dependent
// rounds of a binary heap -- the epilogue is a chain of dependent smem latencies, not throughput.
constexpr int kAry = 8;

// Place (sc, gid) at `pos` of the heap prefix [0, lim) and sift it down.
__device__ __forceinline__ void heap_sift_down(float *hv, int32_t *hi_, int pos, int lim, float sc, int gid) {
  for (;;) {
    const int c0 = kAry * pos + 1;
    if (c0 >= lim) break;
    float v[kAry];
    int id[kAry];
#pragma unroll
    for (int j = 0; j < kAry; ++j) {
      const bool in = c0 + j < lim;
      v[j] = in ? hv[(c0 + j) * kTileM] : CUDART_INF_F;      // +inf never wins "worst"
      id[j] = in ? hi_[(c0 + j) * kTileM] : 0;
    }
    // worst child = lowest score, ties -> highest id. Shallow trees instead of a 7-step scan: the
    // epilogue is one warp per scheduler, so the DEPTH of the dependent chain is what costs (loading
    // the id of the chosen child only, after the min, was slower: one more dependent load per level).
    const float wv = fminf(fminf(fminf(v[0], v[1]), fminf(v[2], v[3])), fminf(fminf(v[4], v[5]), fminf(v[6], v[7])));
    int t[kAry];
#pragma unroll
    for (int j = 0; j < kAry; ++j) t[j] = v[j] == wv ? id[j] : -1;
    const int wi = max(max(max(t[0], t[1]), max(t[2], t[3])), max(max(t[4], t[5]), max(t[6], t[7])));
    int w = 0;
#pragma unroll
    for (int j = 1; j < kAry; ++j) w = t[j] == wi ? j : w;
    w = t[0] == wi ? 0 : w;
    if (!Better::worse(wv, wi, sc, gid)) break;
    hv[pos * kTileM] = wv;
    hi_[pos * kTileM] = wi;
    pos = c0 + w;
  }
  hv[pos * kTileM] = sc;
  hi_[pos * kTileM] = gid;
}

// Append (sc, gid) at `pos` (= current size) and sift it up.
__device__ __forceinline__ void heap_sift_up(float *hv, int32_t *hi_, int pos, float sc, int gid) {
  while (pos > 0) {
    const int par = (pos - 1) / kAry;
    const float pv = hv[par * kTileM];
    const int pi = hi_[par * kTileM];
    if (!Better::worse(sc, gid, pv, pi)) break;
    hv[pos * kTileM] = pv;
    hi_[pos * kTileM] = pi;
    pos = par;
  }
  hv[pos * kTileM] = sc;
  hi_[pos * kTileM] = gid;
}

template <int D, bool A_TMEM>
__global__ void __launch_bounds__(kThreadsTC, 1)
score_topk_tc_kernel(const float *__restrict__ user_emb, const int64_t *__restrict__ users, int n_users,
                     const float *__restrict__ item_emb, int n_items, int item_offset,
                     const int32_t *__restrict__ mask_rowptr, const int32_t *__restrict__ mask_cols,
                     int mask_by_user, int k, int items_per_split, float *__restrict__ ws_val,
                     int32_t *__restrict__ ws_idx, int pend_cap,
                     int dbg) {
  using C = Cfg<D, A_TMEM>;
  static_assert(!A_TMEM || kAcc * kTileN + 2 * D <= 512, "user tile does not fit beside the accumulators");
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment (SW128 atoms) by an offset on the __shared__ array itself: pointers derived
  // through an integer cast would lose their address space and compile to generic LD/ST
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float *h_val = reinterpret_cast<float *>(smem + C::OFF_HEAP);              // [k][128]
  int32_t *h_idx = reinterpret_cast<int32_t *>(h_val + (size_t)k * kTileM);  // [k][128]
  float *p_val = reinterpret_cast<float *>(h_idx + (size_t)k * kTileM);      // [pend_cap][128] pending
  int32_t *p_idx = reinterpret_cast<int32_t *>(p_val + (size_t)pend_cap * kTileM);   // candidates
  uint64_t *bars = reinterpret_cast<uint64_t *>(p_idx + (size_t)pend_cap * kTileM);
  uint64_t *full = bars, *empty = bars + C::STAGES, *tfull = bars + 2 * C::STAGES, *tempty = tfull + kAcc;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + kAcc);

  // warp index through a broadcast: provably warp-uniform, so role branches and the MMA issue
  // loop (descriptor arithmetic included) compile to the uniform datapath
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int j_begin = blockIdx.y * items_per_split;
  const int j_end = min(n_items, j_begin + items_per_split);
  const int n_tiles = (j_end - j_begin + kTileN - 1) / kTileN;
  const uint32_t smem_base = smem_u32(smem);

  if (tid == 0) {
    for (int s = 0; s < C::STAGES; ++s) { mbar_init(full + s, 64); mbar_init(empty + s, 1); }
    for (int b = 0; b < kAcc; ++b) { mbar_init(tfull + b, 1); mbar_init(tempty + b, 128); }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, C::TMEM_COLS);

  // ---- user tile -> hi/lo A operand (thread = user row = TMEM lane) ------------------------
  const int b_user = blockIdx.x * kTileM + tid;
  const bool live = tid < kTileM && b_user < n_users;
  if constexpr (A_TMEM) {
    fence_before_sync();
    __syncthreads();                 // barriers initialised, TMEM base address published
    fence_after_sync();
    if (tid < kTileM) {
      const uint32_t a_row = *tmem_slot + ((uint32_t)(warp * 32) << 16) + C::A_COL;
      const float *src = live ? user_emb + (size_t)users[b_user] * D : nullptr;
#pragma unroll
      for (int c32 = 0; c32 < D / 32; ++c32) {
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          float4 v = live ? ldg4(src + c32 * 32 + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f), h, l;
          split_tf32x4(v, h, l);
          hi[c4 * 4 + 0] = __float_as_uint(h.x); hi[c4 * 4 + 1] = __float_as_uint(h.y);
          hi[c4 * 4 + 2] = __float_as_uint(h.z); hi[c4 * 4 + 3] = __float_as_uint(h.w);
          lo[c4 * 4 + 0] = __float_as_uint(l.x); lo[c4 * 4 + 1] = __float_as_uint(l.y);
          lo[c4 * 4 + 2] = __float_as_uint(l.z); lo[c4 * 4 + 3] = __float_as_uint(l.w);
        }
        tmem_st_32x32b_x32(a_row + c32 * 32, hi);          // warp-collective: dead rows store zeros
        tmem_st_32x32b_x32(a_row + D + c32 * 32, lo);
      }
      tmem_st_wait();
    }
  } else if (tid < kTileM) {
    const float *src = live ? user_emb + (size_t)users[b_user] * D : nullptr;
#pragma unroll
    for (int c4 = 0; c4 < D / 4; ++c4) {
      float4 v = live ? ldg4(src + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f), hi, lo;
      split_tf32x4(v, hi, lo);
      const uint32_t off = (c4 / 8) * (kTileM * 128) + sw128_off(tid, c4 % 8);
      *reinterpret_cast<float4 *>(smem + off) = hi;
      *reinterpret_cast<float4 *>(smem + C::A_HALF + off) = lo;
    }
    fence_proxy_async_smem();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp >= 4 && warp < 8) {
    // =============================== producers ===============================================
    // Two independent groups of two warps; group g owns tiles g, g + 2, ... and keeps ONE batch of
    // loads in flight (load -> wait -> split -> store). Prefetching the next tile into a second
    // register set of the same threads ran at one tile per L2 round trip: the loads of both tiles
    // share scoreboards, so waiting for the older one waited for the newer one too (same finding
    // as gemm_tc05.cu). STAGES >= 2 = number of groups, so the parity waits cannot alias.
    constexpr int GT = 64;                                   // threads per group
    constexpr int VB = (kTileN * (D / 4) / GT) > 16 ? 16 : (kTileN * (D / 4) / GT);   // float4 per batch
    constexpr int NB = kTileN * (D / 4) / GT / VB;           // batches per tile (2 for d = 128)
    const int grp = (tid - 128) / GT, ptid = (tid - 128) % GT;
    for (int t = grp; t < n_tiles; t += 2) {
      const int j0 = j_begin + t * kTileN;
      const int s = t % C::STAGES;
      uint8_t *stage = smem + C::OFF_B + s * C::STAGE;
#pragma unroll
      for (int nb = 0; nb < NB; ++nb) {
        float4 v[VB];
#pragma unroll
        for (int i = 0; i < VB; ++i) {
          const int idx = ptid + GT * (nb * VB + i), row = idx / (D / 4), c4 = idx % (D / 4);
          v[i] = (j0 + row < j_end) ? ldg4(item_emb + (size_t)(j0 + row) * D + c4 * 4)
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (nb == 0) mbar_wait(empty + s, ((t / C::STAGES) & 1) ^ 1);
#pragma unroll
        for (int i = 0; i < VB; ++i) {
          const int idx = ptid + GT * (nb * VB + i), row = idx / (D / 4), c4 = idx % (D / 4);
          float4 hi, lo;
          split_tf32x4(v[i], hi, lo);
          const uint32_t off = (c4 / 8) * (kTileN * 128) + sw128_off(row, c4 % 8);
          *reinterpret_cast<float4 *>(stage + off) = hi;
          *reinterpret_cast<float4 *>(stage + C::B_HALF + off) = lo;
        }
      }
      fence_proxy_async_smem();
      mbar_arrive(full + s);
    }
  } else if (warp == 8) {
    // =============================== MMA issuer ==============================================
    constexpr uint32_t idesc = idesc_tf32(kTileM, kTileN, false, false);
    const uint64_t a_hi = smem_desc_sw128(smem_base, 16, 1024);
    const uint64_t a_lo = smem_desc_sw128(smem_base + C::A_HALF, 16, 1024);
    const uint32_t at_hi = tmem_base + C::A_COL, at_lo = at_hi + D;   // A_TMEM: one column per K element
    for (int t = 0; t < n_tiles; ++t) {
      const int s = t % C::STAGES, b = t % kAcc;
      mbar_wait(full + s, (t / C::STAGES) & 1);
      mbar_wait(tempty + b, ((t / kAcc) & 1) ^ 1);
      fence_after_sync();
      const uint32_t d_tmem = tmem_base + b * kTileN;
      const uint64_t b_hi = smem_desc_sw128(smem_base + C::OFF_B + s * C::STAGE, 16, 1024);
      const uint64_t b_lo = b_hi + (C::B_HALF >> 4);
      // small cross terms first, the dominant hi*hi product last; a K step inside the swizzle atom
      // (and the next atom) is a plain offset in the descriptor's 16-byte-unit address field
#pragma unroll
      for (int pass = 0; pass < 3; ++pass) {
        const uint64_t a0 = pass == 0 ? a_lo : a_hi;
        const uint64_t b0 = pass == 1 ? b_lo : b_hi;
#pragma unroll
        for (int kb = 0; kb < C::KB; ++kb)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t bd = b0 + ((kb * (kTileN * 128) + ks * 32) >> 4);
            if constexpr (A_TMEM) {
              const uint32_t at = (pass == 0 ? at_lo : at_hi) + kb * 32 + ks * 8;
              if (elect_one()) umma_tf32_ts(d_tmem, at, bd, idesc, (pass | kb | ks) != 0);
            } else {
              const uint64_t ad = a0 + ((kb * (kTileM * 128) + ks * 32) >> 4);
              if (elect_one()) umma_tf32_ss(d_tmem, ad, bd, idesc, (pass | kb | ks) != 0);
            }
          }
      }
      if (elect_one()) {
        umma_commit(empty + s);     // smem stage reusable once these MMAs have read it
        umma_commit(tfull + b);     // accumulator ready for the epilogue
      }
      __syncwarp();
    }
  } else {
    // =============================== epilogue: mask + top-K ==================================
    int mp = 0, mend = 0, next_masked = INT_MAX;
    if (live && mask_rowptr != nullptr) {
      const int mrow = mask_by_user ? (int)users[b_user] : b_user;   // batch entry, or the user's own row
      int lo = mask_rowptr[mrow];
      mend = mask_rowptr[mrow + 1];
      int hi = mend;
      const int target = item_offset + j_begin;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (mask_cols[mid] < target) lo = mid + 1; else hi = mid;
      }
      mp = lo;
      if (mp < mend) next_masked = mask_cols[mp];
    }
    // Candidates (scores above the user's K-th best as of the last flush) are only APPENDED to a
    // per-user pending list while tiles stream by; the heap work happens in warp-synchronous
    // flushes, when some lane could not take another full chunk. Inserting on arrival made every
    // lane's insert a separate divergent excursion (~190 cycles each, 32 lanes x K ln(N/K) of
    // them per warp: 1.35 of the 2.5 ms on 16k x 100k); in a flush all 32 lanes walk their lists
    // together. A stale threshold only admits extra candidates, which the flush rejects with one
    // compare against the fresh one. thr = -inf until the heap holds K entries.
    int cnt = 0, pend = 0;
    float thr = -CUDART_INF_F;
    float *hv = h_val + tid;
    int32_t *hi_ = h_idx + tid;
    float *pv = p_val + tid;
    int32_t *pi = p_idx + tid;

    auto flush = [&]() {
      // (letting every lane skip ahead to its next live entry before each heap update was slower:
      // 304 vs 275 us at Baby size -- the per-iteration latency chain, not lane utilisation, binds)
      for (int i = 0; i < pend; ++i) {
        float sc = pv[i * kTileM];
        if (!(sc > thr)) continue;
        const int gid = pi[i * kTileM];
        while (next_masked < gid) {                               // ascending ids: a cursor is enough
          ++mp;
          next_masked = mp < mend ? mask_cols[mp] : INT_MAX;
        }
        if (gid == next_masked) sc = -1e10f;                      // trainer.py:524
        if (cnt < k) {
          heap_sift_up(hv, hi_, cnt++, sc, gid);
          if (cnt == k) thr = hv[0];
        } else if (sc > thr) {
          heap_sift_down(hv, hi_, 0, k, sc, gid);                 // replace the worst kept entry
          thr = hv[0];
        }
      }
      pend = 0;
      __syncwarp();
    };

    for (int t = 0; t < n_tiles; ++t) {
      const int b = t % kAcc;
      mbar_wait(tfull + b, (t / kAcc) & 1);
      fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + b * kTileN;
#pragma unroll
      for (int half = 0; half < kTileN / kChunk; ++half) {
        uint32_t r[kChunk];
        tmem_ld_32x32b_x32(taddr + half * kChunk, r);
        tmem_ld_wait();
        if (half == kTileN / kChunk - 1) {
          fence_before_sync();
          mbar_arrive(tempty + b);       // all columns of this buffer are in registers
        }
        if (__any_sync(0xffffffffu, pend > pend_cap - kChunk)) flush();
        const int j0 = j_begin + t * kTileN + half * kChunk;
        const int valid = min(kChunk, j_end - j0);
        if (valid < kChunk) {            // ragged last tile (warp-uniform)
#pragma unroll
          for (int c = 0; c < kChunk; ++c)
            if (c >= valid) r[c] = __float_as_uint(-CUDART_INF_F);
        }
        // cheap reject: nothing in this chunk beats any lane's K-th best
        float m = -CUDART_INF_F;
#pragma unroll
        for (int c = 0; c < kChunk; ++c) m = fmaxf(m, __uint_as_float(r[c]));
        if (dbg == 1) m = -CUDART_INF_F;
        if (__any_sync(0xffffffffu, live && m > thr) && dbg != 2) {
          const float lim = live ? thr : CUDART_INF_F;            // dead rows take nothing
          const int g0 = item_offset + j0;
          int off = pend * kTileM;
#pragma unroll
          for (int c = 0; c < kChunk; ++c) {
            const float sc = __uint_as_float(r[c]);
            if (sc > lim) {
              pv[off] = sc;
              pi[off] = g0 + c;
              off += kTileM;
            }
          }
          pend = off / kTileM;
        }
        __syncwarp();       // tcgen05.ld / mbarrier waits are warp-collective
      }
    }
    flush();
    // heap -> descending list (in-place heap sort: the worst entry moves to the end each round)
    if (live) {
      for (int size = cnt; size > 1; --size) {
        const float lv = hv[(size - 1) * kTileM];
        const int li = hi_[(size - 1) * kTileM];
        hv[(size - 1) * kTileM] = hv[0];
        hi_[(size - 1) * kTileM] = hi_[0];
        heap_sift_down(hv, hi_, 0, size - 1, lv, li);
      }
      float *ov = ws_val + ((size_t)blockIdx.y * n_users + b_user) * k;
      int32_t *oi = ws_idx + ((size_t)blockIdx.y * n_users + b_user) * k;
      for (int t = 0; t < k; ++t) {
        ov[t] = t < cnt ? hv[t * kTileM] : -CUDART_INF_F;        // index 0 = best after the sort
        oi[t] = t < cnt ? hi_[t * kTileM] : INT_MAX;
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 8) {
    fence_after_sync();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

inline int dbg_mode() {
  static int m = getenv("MMREC_TOPK_DEBUG") ? atoi(getenv("MMREC_TOPK_DEBUG")) : 0;
  return m;
}

inline bool a_tmem_64() {   // A/B switch for d <= 64 (d = 128 always keeps its user tile in TMEM)
  static int m = getenv("MMREC_TOPK_ATMEM") ? atoi(getenv("MMREC_TOPK_ATMEM")) : 0;
  return m != 0;
}

template <int D, bool A_TMEM>
int launch_tc(const float *user_emb, const int64_t *users, int n_users, const float *item_emb, int n_items,
              int item_offset, const int32_t *mask_rowptr, const int32_t *mask_cols, int mask_by_user, int k,
              int n_splits, float *ws_val, int32_t *ws_idx, cudaStream_t stream) {
  using C = Cfg<D, A_TMEM>;
  const size_t fixed = 1024 + C::OFF_HEAP + (size_t)k * kTileM * 8 + (2 * C::STAGES + 2 * kAcc) * 8 + 16;
  const size_t cap = 227 * 1024;
  if (fixed + (size_t)(kChunk + 8) * kTileM * 8 > cap) return 1;     // K too large for this tiling: SIMT path
  const int pend_cap = (int)min((size_t)64, (cap - fixed) / (kTileM * 8));
  const size_t smem = fixed + (size_t)pend_cap * kTileM * 8;
  MMREC_CUDA(cudaFuncSetAttribute(score_topk_tc_kernel<D, A_TMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int items_per_split = ((n_items + n_splits - 1) / n_splits + kTileN - 1) / kTileN * kTileN;
  dim3 grid((n_users + kTileM - 1) / kTileM, n_splits);
  score_topk_tc_kernel<D, A_TMEM><<<grid, kThreadsTC, smem, stream>>>(user_emb, users, n_users, item_emb, n_items,
                                                              item_offset, mask_rowptr, mask_cols, mask_by_user, k,
                                                              items_per_split, ws_val, ws_idx, pend_cap,
                                                              dbg_mode());
  MMREC_CHECK_LAUNCH("score_topk_tc_kernel");
  return MMREC_OK;
}

}  // namespace

// Called by mmrec_score_mask_topk_f32 / _rows_f32 (score_topk.cu). Returns 1 if d is not covered here.
int score_topk_tc_dispatch(const float *user_emb, const int64_t *users, int n_users, const float *item_emb,
                           int n_items, int item_offset, int d, const int32_t *mask_rowptr,
                           const int32_t *mask_cols, int mask_by_user, int k, int n_splits, float *ws_val,
                           int32_t *ws_idx, cudaStream_t stream) {
#define MMREC_TC(D_, T_) launch_tc<D_, T_>(user_emb, users, n_users, item_emb, n_items, item_offset, mask_rowptr, \
                                            mask_cols, mask_by_user, k, n_splits, ws_val, ws_idx, stream)
  switch (d) {
    case 32: return MMREC_TC(32, false);
    case 64: return a_tmem_64() ? MMREC_TC(64, true) : MMREC_TC(64, false);
    case 128: return MMREC_TC(128, true);
    default: return 1;
  }
#undef MMREC_TC
}

}  // namespace mmrec
