// Full-rank scoring fused with train-item masking and per-user top-K (K8/K9/K10).
//
// One thread owns one user: its embedding row lives in registers, item rows stream through shared
// memory in tiles (every lane reads the same address -> broadcast, conflict-free), each score is
// masked against the user's ascending train-item list and offered to a per-thread sorted top-K
// list held in shared memory ([k][thread] layout: lane-contiguous, conflict-free). Scores never
// reach HBM. The item range is split over blockIdx.y so that small user batches still fill the
// 148 SMs; a merge kernel combines the per-split lists (also used for the cross-rank merge of
// item-sharded evaluation). Order: descending score, ties -> lower item id, which is what a
// stable descending sort of the masked score row gives.
#include <math_constants.h>

#include "common.cuh"

namespace mmrec {
namespace {

constexpr int kUsers = 128;   // threads (= users) per CTA
constexpr int kItemTile = 32;

template <int D>
__global__ void __launch_bounds__(kUsers)
score_topk_kernel(const float *__restrict__ user_emb, const int64_t *__restrict__ users, int n_users,
                  const float *__restrict__ item_emb, int n_items, int item_offset,
                  const int32_t *__restrict__ mask_rowptr, const int32_t *__restrict__ mask_cols, int mask_by_user,
                  int k, int items_per_split, float *__restrict__ ws_val, int32_t *__restrict__ ws_idx) {
  extern __shared__ __align__(16) float smem[];
  float *sV = smem;                                   // [kItemTile][D]
  float *l_val = smem + kItemTile * D;                // [k][kUsers]
  int32_t *l_idx = reinterpret_cast<int32_t *>(l_val + (size_t)k * kUsers);
  const int tid = threadIdx.x;
  const int b = blockIdx.x * kUsers + tid;
  const bool live = b < n_users;
  const int j_begin = blockIdx.y * items_per_split;
  const int j_end = min(n_items, j_begin + items_per_split);

  float u[D];
  if (live) {
    const float *src = user_emb + (size_t)users[b] * D;
#pragma unroll
    for (int c = 0; c < D; c += 4) {
      const float4 v = ldg4(src + c);
      u[c] = v.x; u[c + 1] = v.y; u[c + 2] = v.z; u[c + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int c = 0; c < D; ++c) u[c] = 0.f;
  }
  // mask cursor: first train item of this user with global id >= item_offset + j_begin; the mask
  // row is the batch entry b, or the user id itself (mask_by_user: a CSR over the user table)
  int mp = 0, mend = 0, next_masked = INT_MAX;
  if (live && mask_rowptr != nullptr) {
    const int mrow = mask_by_user ? (int)users[b] : b;
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
  int cnt = 0;
  float thr = -CUDART_INF_F;

  for (int j0 = j_begin; j0 < j_end; j0 += kItemTile) {
    __syncthreads();
    const int tile = min(kItemTile, j_end - j0);
    for (int t = tid; t < tile * (D / 4); t += kUsers)
      reinterpret_cast<float4 *>(sV)[t] = ldg4(item_emb + (size_t)j0 * D + (size_t)t * 4);
    __syncthreads();
    if (!live) continue;
    for (int jj = 0; jj < tile; jj += 4) {
      float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < D; c += 4) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          // rows past `tile` hold stale but finite data from earlier tiles; discarded below
          const float4 v = *reinterpret_cast<const float4 *>(sV + (jj + q) * D + c);
          s[q] = fmaf(u[c], v.x, s[q]);
          s[q] = fmaf(u[c + 1], v.y, s[q]);
          s[q] = fmaf(u[c + 2], v.z, s[q]);
          s[q] = fmaf(u[c + 3], v.w, s[q]);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (jj + q >= tile) break;
        const int gid = item_offset + j0 + jj + q;
        float sc = s[q];
        if (gid == next_masked) {
          sc = -1e10f;                                   // trainer.py:524
          ++mp;
          next_masked = mp < mend ? mask_cols[mp] : INT_MAX;
        }
        if (cnt < k || sc > thr) {
          int pos = cnt < k ? cnt : k - 1;
          while (pos > 0 && l_val[(pos - 1) * kUsers + tid] < sc) {
            l_val[pos * kUsers + tid] = l_val[(pos - 1) * kUsers + tid];
            l_idx[pos * kUsers + tid] = l_idx[(pos - 1) * kUsers + tid];
            --pos;
          }
          l_val[pos * kUsers + tid] = sc;
          l_idx[pos * kUsers + tid] = gid;
          if (cnt < k) ++cnt;
          if (cnt == k) thr = l_val[(k - 1) * kUsers + tid];
        }
      }
    }
  }
  if (live) {
    float *ov = ws_val + ((size_t)blockIdx.y * n_users + b) * k;
    int32_t *oi = ws_idx + ((size_t)blockIdx.y * n_users + b) * k;
    for (int t = 0; t < k; ++t) {
      ov[t] = t < cnt ? l_val[t * kUsers + tid] : -CUDART_INF_F;
      oi[t] = t < cnt ? l_idx[t * kUsers + tid] : INT_MAX;
    }
  }
}

constexpr int kMaxLists = 64;

// K-way merge by ranking: one warp per user. The n_lists * k candidates of the user are staged in
// shared memory; every candidate computes its final rank directly -- its position in its own
// (sorted) list plus, for every other list, the number of entries that beat it (binary search:
// the lists are sorted by (score desc, id asc), padding (-inf, INT_MAX) last; list index breaks
// exact ties so the order is total) -- and the k best write themselves to their slot. No serial
// k-step selection loop, no per-thread local arrays, coalesced traffic.
constexpr int kMergeWarps = 4;

__global__ void __launch_bounds__(kMergeWarps * 32)
topk_merge_kernel(const float *__restrict__ vals, const int32_t *__restrict__ idx, int n_lists,
                  int n_users, int k, float *__restrict__ out_val, int64_t *__restrict__ out_idx) {
  extern __shared__ float merge_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kMergeWarps + warp;
  if (b >= n_users) return;
  const int n = n_lists * k;
  float *sv = merge_smem + (size_t)warp * 2 * n;
  int32_t *si = reinterpret_cast<int32_t *>(sv + n);
  for (int c = lane; c < n; c += 32) {
    const int l = c / k, j = c % k;
    const size_t o = ((size_t)l * n_users + b) * k + j;
    sv[c] = vals[o];
    si[c] = idx[o];
  }
  __syncwarp();
  for (int c = lane; c < n; c += 32) {
    const int l = c / k, j = c % k;
    const float v = sv[c];
    const int id = si[c];
    int rank = j;
    for (int l2 = 0; l2 < n_lists && rank < k; ++l2) {
      if (l2 == l) continue;
      const float *lv = sv + l2 * k;
      const int32_t *li = si + l2 * k;
      int lo = 0, hi = k;                       // first position whose entry does NOT beat (v, id)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const float ev = lv[mid];
        const int ei = li[mid];
        const bool beats = ev > v || (ev == v && (ei < id || (ei == id && l2 < l)));
        if (beats) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) {
      if (out_val) out_val[(size_t)b * k + rank] = v;
      out_idx[(size_t)b * k + rank] = (int64_t)id;
    }
  }
}

template <int D>
int launch_score(const float *user_emb, const int64_t *users, int n_users, const float *item_emb, int n_items,
                 int item_offset, const int32_t *mask_rowptr, const int32_t *mask_cols, int mask_by_user, int k,
                 int n_splits, float *ws_val, int32_t *ws_idx, cudaStream_t stream) {
  const size_t smem = (size_t)kItemTile * D * sizeof(float) + (size_t)k * kUsers * 8;
  MMREC_REQUIRE(smem <= 227 * 1024, MMREC_E_BADARG, "score_mask_topk: k=%d needs %zu B of shared memory", k, smem);
  MMREC_CUDA(cudaFuncSetAttribute(score_topk_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int items_per_split = ((n_items + n_splits - 1) / n_splits + kItemTile - 1) / kItemTile * kItemTile;
  dim3 grid((n_users + kUsers - 1) / kUsers, n_splits);
  score_topk_kernel<D><<<grid, kUsers, smem, stream>>>(user_emb, users, n_users, item_emb, n_items, item_offset,
                                                      mask_rowptr, mask_cols, mask_by_user, k, items_per_split,
                                                      ws_val, ws_idx);
  MMREC_CHECK_LAUNCH("score_topk_kernel");
  return MMREC_OK;
}

}  // namespace

int score_topk_tc_dispatch(const float *user_emb, const int64_t *users, int n_users, const float *item_emb,
                           int n_items, int item_offset, int d, const int32_t *mask_rowptr,
                           const int32_t *mask_cols, int mask_by_user, int k, int n_splits, float *ws_val,
                           int32_t *ws_idx, cudaStream_t stream);   // score_topk_tc.cu
}  // namespace mmrec

using namespace mmrec;

extern "C" int mmrec_topk_merge(const float *vals, const int32_t *idx, int32_t n_lists, int32_t n_users,
                                int32_t k, float *out_val, int64_t *out_idx, void *stream) {
  MMREC_REQUIRE(vals && idx && out_idx, MMREC_E_BADARG, "topk_merge: null pointer");
  MMREC_REQUIRE(n_lists >= 1 && n_lists <= kMaxLists && n_users > 0 && k > 0 && k <= 255, MMREC_E_BADARG,
                "topk_merge: need 1 <= n_lists <= %d, n_users > 0, 0 < k <= 255", kMaxLists);
  const size_t smem = (size_t)kMergeWarps * 2 * n_lists * k * sizeof(float);
  MMREC_REQUIRE(smem <= 200 * 1024, MMREC_E_BADARG, "topk_merge: n_lists * k = %d is too large", n_lists * k);
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    MMREC_CUDA(cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  topk_merge_kernel<<<(n_users + kMergeWarps - 1) / kMergeWarps, kMergeWarps * 32, smem, (cudaStream_t)stream>>>(
      vals, idx, n_lists, n_users, k, out_val, out_idx);
  MMREC_CHECK_LAUNCH("topk_merge_kernel");
  return MMREC_OK;
}

static int score_mask_topk(bool allow_tc, bool mask_by_user, const float *user_emb, const int64_t *users,
                           int32_t n_users, const float *item_emb, int32_t n_items, int32_t item_offset, int32_t d,
                           const int32_t *mask_rowptr, const int32_t *mask_cols, int32_t k,
                           int32_t n_splits, float *ws_val, int32_t *ws_idx, float *out_val,
                           int64_t *out_idx, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMREC_REQUIRE(user_emb && users && item_emb && ws_val && ws_idx && out_idx, MMREC_E_BADARG,
                "score_mask_topk: null pointer");
  MMREC_REQUIRE((mask_rowptr == nullptr) == (mask_cols == nullptr), MMREC_E_BADARG,
                "score_mask_topk: mask_rowptr and mask_cols must be given together");
  MMREC_REQUIRE(n_users > 0 && n_items > 0 && k > 0 && k <= 255, MMREC_E_BADARG, "score_mask_topk: bad sizes");
  MMREC_REQUIRE(n_splits >= 1 && n_splits <= kMaxLists, MMREC_E_BADARG, "score_mask_topk: bad n_splits");
  MMREC_REQUIRE(aligned16(user_emb) && aligned16(item_emb), MMREC_E_ALIGN,
                "score_mask_topk: tables must be 16-byte aligned");
  int rc = 1;
  if (allow_tc)      // tcgen05 path (d = 32 / 64); 1 = not covered -> SIMT kernel below
    rc = score_topk_tc_dispatch(user_emb, users, n_users, item_emb, n_items, item_offset, d, mask_rowptr, mask_cols,
                                mask_by_user, k, n_splits, ws_val, ws_idx, stream);
  if (rc < 0) return rc;
  if (rc == 1) switch (d) {
    case 32: rc = launch_score<32>(user_emb, users, n_users, item_emb, n_items, item_offset, mask_rowptr, mask_cols,
                                   mask_by_user, k, n_splits, ws_val, ws_idx, stream); break;
    case 64: rc = launch_score<64>(user_emb, users, n_users, item_emb, n_items, item_offset, mask_rowptr, mask_cols,
                                   mask_by_user, k, n_splits, ws_val, ws_idx, stream); break;
    case 128: rc = launch_score<128>(user_emb, users, n_users, item_emb, n_items, item_offset, mask_rowptr,
                                     mask_cols, mask_by_user, k, n_splits, ws_val, ws_idx, stream); break;
    default:
      set_error("score_mask_topk: unsupported d=%d (32, 64, 128)", d);
      return MMREC_E_BADARG;
  }
  if (rc != MMREC_OK) return rc;
  return mmrec_topk_merge(ws_val, ws_idx, n_splits, n_users, k, out_val, out_idx, stream);
}

extern "C" int mmrec_score_mask_topk_f32(const float *user_emb, const int64_t *users, int32_t n_users,
                                         const float *item_emb, int32_t n_items, int32_t item_offset, int32_t d,
                                         const int32_t *mask_rowptr, const int32_t *mask_cols, int32_t k,
                                         int32_t n_splits, float *ws_val, int32_t *ws_idx, float *out_val,
                                         int64_t *out_idx, void *stream) {
  return score_mask_topk(true, false, user_emb, users, n_users, item_emb, n_items, item_offset, d, mask_rowptr,
                         mask_cols, k, n_splits, ws_val, ws_idx, out_val, out_idx, stream);
}

extern "C" int mmrec_score_mask_topk_rows_f32(const float *user_emb, const int64_t *users, int32_t n_users,
                                              const float *item_emb, int32_t n_items, int32_t item_offset,
                                              int32_t d, const int32_t *mask_rowptr, const int32_t *mask_cols,
                                              int32_t k, int32_t n_splits, float *ws_val, int32_t *ws_idx,
                                              float *out_val, int64_t *out_idx, void *stream) {
  return score_mask_topk(true, true, user_emb, users, n_users, item_emb, n_items, item_offset, d, mask_rowptr,
                         mask_cols, k, n_splits, ws_val, ws_idx, out_val, out_idx, stream);
}

extern "C" int mmrec_score_mask_topk_simt_f32(const float *user_emb, const int64_t *users, int32_t n_users,
                                              const float *item_emb, int32_t n_items, int32_t item_offset,
                                              int32_t d, const int32_t *mask_rowptr, const int32_t *mask_cols,
                                              int32_t k, int32_t n_splits, float *ws_val, int32_t *ws_idx,
                                              float *out_val, int64_t *out_idx, void *stream) {
  return score_mask_topk(false, false, user_emb, users, n_users, item_emb, n_items, item_offset, d, mask_rowptr,
                         mask_cols, k, n_splits, ws_val, ws_idx, out_val, out_idx, stream);
}
