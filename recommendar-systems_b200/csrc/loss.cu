// BPR gather-dot loss (K6) and streaming InfoNCE (K7) -- see include/mmrec_b200.h.
//
// BPR: one warp per (user, pos, neg) triple; the three embedding rows are gathered with 16-byte
// loads, the two dots, -logsigmoid and the L2 term are formed in registers; per-sample results go
// to a small buffer and the last CTA to finish reduces it in a fixed order (deterministic scalar).
// Backward: sigma(-x) saved by the forward scales the rows, gradients are scatter-added with
// vector atomics (red.global.add.v4.f32) because users/items repeat inside a batch: the order of
// those float additions is not fixed, so rows that repeat in a batch are reproducible to rounding
// (~1e-7), not bit for bit, from run to run -- unlike the SpMM / dense / optimizer kernels, which
// use no floating-point atomics. The ids are trusted (see ops.CHECK_IDS for the checked mode).
//
// InfoNCE: rows are gathered + L2-normalised once, then a 64x64-tile kernel streams V1 V2^T
// through shared memory (tile products on the tensor cores: mma.sync, 3xTF32 split = fp32-class
// scores), applies exp(s/t) and keeps only row sums -- the B x B matrix never reaches HBM.
// Backward recomputes the tiles (flash-style) for the row pass (dV1) and the column pass (dV2);
// the gradient tile G goes straight back into a second tensor-core product G * V. All scalars
// are reduced in a fixed order.
#include "common.cuh"
#include "dense_tile.cuh"

namespace mmrec {
namespace {

constexpr int kThreads = 256;
static_assert(kThreads == dense::kT, "the tensor-core tile helpers assume 256-thread CTAs");

__device__ __forceinline__ float softplus_neg(float x) {  // -logsigmoid(x)
  return fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float sigmoid_neg(float x) {  // sigmoid(-x)
  if (x >= 0.f) {
    const float e = expf(-x);
    return e / (1.f + e);
  }
  return 1.f / (1.f + expf(x));
}

// Returns true in every thread of the last CTA to arrive; resets the counter for the next call.
__device__ __forceinline__ bool last_block_arrives(uint32_t *counter) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t total = gridDim.x * gridDim.y;
    const uint32_t prev = atomicAdd(counter, 1u);
    is_last = (prev == total - 1);
    if (is_last) *counter = 0u;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// ------------------------------------------------------------------------------------------ BPR
__global__ void __launch_bounds__(kThreads)
bpr_fwd_kernel(const float *__restrict__ ue, const float *__restrict__ ie, int d,
               const int64_t *__restrict__ users, const int64_t *__restrict__ pos,
               const int64_t *__restrict__ neg, int batch, float *__restrict__ out2,
               float *__restrict__ sig, float *__restrict__ partial, uint32_t *counter) {
  __shared__ float red[kThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * (kThreads / 32) + warp;
  if (b < batch) {
    const float *u = ue + (size_t)users[b] * d;
    const float *p = ie + (size_t)pos[b] * d;
    const float *n = ie + (size_t)neg[b] * d;
    float sp = 0.f, sn = 0.f, sq = 0.f;
    for (int c = lane * 4; c < d; c += 128) {
      const float4 a = ldg4(u + c), x = ldg4(p + c), y = ldg4(n + c);
      sp += dot4(a, x);
      sn += dot4(a, y);
      sq += dot4(a, a) + dot4(x, x) + dot4(y, y);
    }
    sp = warp_sum(sp);
    sn = warp_sum(sn);
    sq = warp_sum(sq);
    if (lane == 0) {
      const float x = sp - sn;
      partial[b] = softplus_neg(x);
      partial[batch + b] = 0.5f * sq;
      sig[b] = sigmoid_neg(x);
    }
  }
  if (last_block_arrives(counter)) {
    float l = 0.f, r = 0.f;
    for (int i = threadIdx.x; i < batch; i += kThreads) {
      l += __ldcg(partial + i);
      r += __ldcg(partial + batch + i);
    }
    l = block_sum<kThreads>(l, red);
    r = block_sum<kThreads>(r, red);
    if (threadIdx.x == 0) {
      out2[0] = l;
      out2[1] = r;
    }
  }
}

__device__ __forceinline__ void red_add4(float *addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

__global__ void __launch_bounds__(kThreads)
bpr_bwd_kernel(const float *__restrict__ ue, const float *__restrict__ ie, int d,
               const int64_t *__restrict__ users, const int64_t *__restrict__ pos,
               const int64_t *__restrict__ neg, int batch, const float *__restrict__ sig,
               const float *__restrict__ coef2, float *__restrict__ d_ue, float *__restrict__ d_ie) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * (kThreads / 32) + warp;
  if (b >= batch) return;
  const float c0 = coef2[0], c1 = coef2[1];
  const float s = -c0 * sig[b];  // d(-logsigmoid(x))/dx = -sigmoid(-x)
  const size_t ou = (size_t)users[b] * d, op = (size_t)pos[b] * d, on = (size_t)neg[b] * d;
  for (int c = lane * 4; c < d; c += 128) {
    const float4 a = ldg4(ue + ou + c), x = ldg4(ie + op + c), y = ldg4(ie + on + c);
    float4 gu, gp, gn;
    gu.x = s * (x.x - y.x) + c1 * a.x; gu.y = s * (x.y - y.y) + c1 * a.y;
    gu.z = s * (x.z - y.z) + c1 * a.z; gu.w = s * (x.w - y.w) + c1 * a.w;
    gp.x = s * a.x + c1 * x.x; gp.y = s * a.y + c1 * x.y; gp.z = s * a.z + c1 * x.z; gp.w = s * a.w + c1 * x.w;
    gn.x = -s * a.x + c1 * y.x; gn.y = -s * a.y + c1 * y.y; gn.z = -s * a.z + c1 * y.z; gn.w = -s * a.w + c1 * y.w;
    red_add4(d_ue + ou + c, gu);
    red_add4(d_ie + op + c, gp);
    red_add4(d_ie + on + c, gn);
  }
}

// -------------------------------------------------------------------------------------- InfoNCE
// Up to two problems of the same batch size per launch (blockIdx.y): the item-row and user-row calls
// of a batch (mgcn.py:250-251, smore.py:406-407).
constexpr int kMaxInfoProb = 2;
struct NormArgs {
  const float *T1[kMaxInfoProb], *T2[kMaxInfoProb];
  const int64_t *idx[kMaxInfoProb];
  float *V1n[kMaxInfoProb], *V2n[kMaxInfoProb], *inv_norm[kMaxInfoProb];
};
struct ScatterArgs {
  const float *V1n[kMaxInfoProb], *V2n[kMaxInfoProb], *inv_norm[kMaxInfoProb], *dV1[kMaxInfoProb], *dV2[kMaxInfoProb];
  const int64_t *idx[kMaxInfoProb];
  float *dT1[kMaxInfoProb], *dT2[kMaxInfoProb];
};

__global__ void __launch_bounds__(kThreads)
infonce_normalize_kernel(const __grid_constant__ NormArgs A, int d, int batch) {
  const float *__restrict__ T1 = A.T1[blockIdx.y], *__restrict__ T2 = A.T2[blockIdx.y];
  const int64_t *__restrict__ idx = A.idx[blockIdx.y];
  float *__restrict__ V1n = A.V1n[blockIdx.y], *__restrict__ V2n = A.V2n[blockIdx.y],
                     *__restrict__ inv_norm = A.inv_norm[blockIdx.y];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * (kThreads / 32) + warp;
  if (b >= batch) return;
  const size_t src = (size_t)idx[b] * d, dst = (size_t)b * d;
  float n1 = 0.f, n2 = 0.f;
  for (int c = lane * 4; c < d; c += 128) {
    const float4 a = ldg4(T1 + src + c), x = ldg4(T2 + src + c);
    n1 += dot4(a, a);
    n2 += dot4(x, x);
  }
  const float i1 = 1.f / fmaxf(sqrtf(warp_sum(n1)), 1e-12f);
  const float i2 = 1.f / fmaxf(sqrtf(warp_sum(n2)), 1e-12f);
  for (int c = lane * 4; c < d; c += 128) {
    float4 a = ldg4(T1 + src + c), x = ldg4(T2 + src + c);
    a.x *= i1; a.y *= i1; a.z *= i1; a.w *= i1;
    x.x *= i2; x.y *= i2; x.z *= i2; x.w *= i2;
    *reinterpret_cast<float4 *>(V1n + dst + c) = a;
    *reinterpret_cast<float4 *>(V2n + dst + c) = x;
  }
  if (lane == 0) {
    inv_norm[b] = i1;
    inv_norm[batch + b] = i2;
  }
}

constexpr int kTile = 64;  // 64 x 64 score tile, 16 x 16 threads, 4 x 4 scores per thread

// Load `kTile` rows (row0..) of M [batch, D] into smem [kTile][D + 4]; rows past `batch` -> 0.
// Every load of the thread is in flight before the first store: one L2 round trip per tile.
template <int D>
__device__ __forceinline__ void load_tile(float *s, const float *__restrict__ M, int row0, int batch) {
  constexpr int LD = D + 4, V = D / 4, PER = kTile * V / kThreads;
  static_assert(kTile * V % kThreads == 0, "tile must be a multiple of the CTA");
  float4 v[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int t = threadIdx.x + i * kThreads, r = t / V, c = (t % V) * 4;
    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row0 + r < batch) v[i] = ldg4(M + (size_t)(row0 + r) * D + c);
  }
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int t = threadIdx.x + i * kThreads, r = t / V, c = (t % V) * 4;
    *reinterpret_cast<float4 *>(s + r * LD + c) = v[i];
  }
}

// acc[i][j] = <A[ty + 16 i], B[tx + 16 j]> over D: the 64 x 64 x D product runs on the tensor cores
// (mma.sync, 3xTF32: fp32-class scores), passes through the shared tile sS [kTile][kTile + 4] and is
// picked up in the (tx, ty) ownership the exp / row-sum / gradient code uses. Callers synchronise
// before (operand tiles staged) -- this function synchronises after the product.
template <int D>
__device__ __forceinline__ void tile_dots(float (&acc)[4][4], float *sS, const float *sA, const float *sB, int tx,
                                          int ty) {
  constexpr int LD = D + 4, GL = kTile + 4;
  dense::tile_mma_tc<D, kTile, kTile, LD, LD, false, dense::EpiIdentity, true>(sS, GL, kTile, sA, sB);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = sS[(ty + 16 * i) * GL + tx + 16 * j];
}

// grid = (row tiles, column splits). ttl_part[split][row] = sum over the split's columns of
// exp(s/t); pos[row] = s_ii. The last CTA of every row tile adds the splits in order (ttl, and the
// 64 per-row losses -> tile_loss); the last row tile adds the tile losses in order: the scalar is
// bit-reproducible and no single CTA walks the whole batch.
// counters: [0] = row tiles done, [1 + row tile] = splits done (zero on entry, self-resetting).
template <int D>
__global__ void __launch_bounds__(kThreads)
infonce_fwd_kernel(const float *__restrict__ V1n, const float *__restrict__ V2n, int batch,
                   float inv_temp, int tiles_per_split, float *__restrict__ ttl_part,
                   float *__restrict__ pos, float *__restrict__ tile_loss, float *__restrict__ ttl,
                   float *__restrict__ loss_out, uint32_t *counters) {
  extern __shared__ __align__(16) float smem[];
  constexpr int LD = D + 4;
  float *sA = smem, *sB = smem + kTile * LD, *sS = smem + 2 * kTile * LD;
  __shared__ float red[kThreads / 32];
  __shared__ bool is_last;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int row0 = blockIdx.x * kTile;
  const int n_tiles = (batch + kTile - 1) / kTile;
  const int t_begin = blockIdx.y * tiles_per_split, t_end = min(n_tiles, t_begin + tiles_per_split);
  load_tile<D>(sA, V1n, row0, batch);
  float rowsum[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t = t_begin; t < t_end; ++t) {
    __syncthreads();
    load_tile<D>(sB, V2n, t * kTile, batch);
    __syncthreads();
    float acc[4][4];
    tile_dots<D>(acc, sS, sA, sB, tx, ty);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = row0 + ty + 16 * i;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = t * kTile + tx + 16 * j;
        if (c < batch) rowsum[i] += expf(acc[i][j] * inv_temp);
        if (c == r && r < batch) pos[r] = acc[i][j];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float s = group_sum<16>(rowsum[i]);
    const int r = row0 + ty + 16 * i;
    if (tx == 0 && r < batch) ttl_part[(size_t)blockIdx.y * batch + r] = s;
  }
  // ---- last split of this row tile: ttl + per-row loss ----
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t prev = atomicAdd(counters + 1 + blockIdx.x, 1u);
    is_last = prev == gridDim.y - 1;
    if (is_last) counters[1 + blockIdx.x] = 0u;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  float l = 0.f;
  if (threadIdx.x < kTile && row0 + threadIdx.x < batch) {
    const int r = row0 + threadIdx.x;
    float s = 0.f;
#pragma unroll 4
    for (int sp = 0; sp < (int)gridDim.y; ++sp) s += __ldcg(ttl_part + (size_t)sp * batch + r);
    ttl[r] = s;
    l = logf(s) - __ldcg(pos + r) * inv_temp;      // -log(exp(s_ii/t) / ttl)
  }
  l = block_sum<kThreads>(l, red);
  if (threadIdx.x == 0) tile_loss[blockIdx.x] = l;
  // ---- last row tile: the scalar ----
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t prev = atomicAdd(counters, 1u);
    is_last = prev == gridDim.x - 1;
    if (is_last) counters[0] = 0u;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  float tot = 0.f;
  for (int t = threadIdx.x; t < n_tiles; t += kThreads) tot += __ldcg(tile_loss + t);
  tot = block_sum<kThreads>(tot, red);
  if (threadIdx.x == 0) loss_out[0] = tot / (float)batch;
}

// Backward tile pass. ROWPASS: CTA owns 64 rows i of V1 and loops over column tiles j, producing
// dV1n[i] = sum_j g_ij V2n[j]. Otherwise the CTA owns 64 columns j and loops over row tiles i,
// producing dV2n[j] = sum_i g_ij V1n[i]. g_ij = coef/B/t * (exp(s_ij/t)/ttl_i - delta_ij).
template <int D, bool ROWPASS>
__global__ void __launch_bounds__(kThreads)
infonce_bwd_kernel(const float *__restrict__ V1n, const float *__restrict__ V2n,
                   const float *__restrict__ ttl, int batch, float inv_temp, int tiles_per_split,
                   const float *__restrict__ coef, float *__restrict__ dOutAll) {
  extern __shared__ __align__(16) float smem[];
  constexpr int LD = D + 4, GL = kTile + 4;
  float *sOwn = smem, *sOther = smem + kTile * LD, *sG = smem + 2 * kTile * LD;  // sG[own][other]
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int own0 = blockIdx.x * kTile;
  const int n_tiles = (batch + kTile - 1) / kTile;
  const float scale = coef[0] / (float)batch * inv_temp;
  const float *Own = ROWPASS ? V1n : V2n, *Other = ROWPASS ? V2n : V1n;
  // blockIdx.y owns a contiguous range of "other" tiles; partial sums go to its own slab
  const int t_begin = blockIdx.y * tiles_per_split, t_end = min(n_tiles, t_begin + tiles_per_split);
  float *dOut = dOutAll + (size_t)blockIdx.y * batch * D;
  load_tile<D>(sOwn, Own, own0, batch);
  // Both products of a tile pair run on the tensor cores: S = Own Other^T (through sG, which then
  // holds G in place), and dOut (+)= G Other, accumulated across the CTA's tiles in its output slab.
  bool first = true;
  for (int t = t_begin; t < t_end; ++t) {
    __syncthreads();
    load_tile<D>(sOther, Other, t * kTile, batch);
    __syncthreads();
    float acc[4][4];
    tile_dots<D>(acc, sG, sOwn, sOther, tx, ty);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int o = own0 + ty + 16 * i;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int x = t * kTile + tx + 16 * j;
        const int row = ROWPASS ? o : x, col = ROWPASS ? x : o;
        float g = 0.f;
        if (o < batch && x < batch) {
          g = expf(acc[i][j] * inv_temp) / __ldg(ttl + row);
          if (row == col) g -= 1.f;
          g *= scale;
        }
        sG[(ty + 16 * i) * GL + tx + 16 * j] = g;     // same element this thread just read
      }
    }
    __syncthreads();
    // dOut[own][:] (+)= sum_x G[own][x] * Other[x][:]
    dense::tile_mma_tc<kTile, D, kTile, GL, LD, false>(dOut + (size_t)own0 * D, D, batch - own0, sG, sOther, !first);
    first = false;
  }
  if (first) {                                          // a split past the last tile: zero slab
    for (int i = threadIdx.x; i < kTile * D; i += kThreads)
      if (own0 + i / D < batch) dOut[(size_t)own0 * D + i] = 0.f;
  }
}

// Chain through F.normalize and scatter-add into the table-shaped gradients.
__global__ void __launch_bounds__(kThreads)
infonce_scatter_kernel(const __grid_constant__ ScatterArgs A, int n_splits, int d, int batch) {
  const float *__restrict__ V1n = A.V1n[blockIdx.y], *__restrict__ V2n = A.V2n[blockIdx.y],
                           *__restrict__ inv_norm = A.inv_norm[blockIdx.y], *__restrict__ dV1 = A.dV1[blockIdx.y],
                           *__restrict__ dV2 = A.dV2[blockIdx.y];
  const int64_t *__restrict__ idx = A.idx[blockIdx.y];
  float *__restrict__ dT1 = A.dT1[blockIdx.y], *__restrict__ dT2 = A.dT2[blockIdx.y];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * (kThreads / 32) + warp;
  if (b >= batch) return;
  const size_t src = (size_t)b * d, dst = (size_t)idx[b] * d;
  const size_t slab = (size_t)batch * d;
  // sum the per-split partial gradients in split order (deterministic)
  auto sum_splits = [&](const float *p, int c) {
    float4 s = ldg4(p + src + c);
#pragma unroll 8
    for (int k = 1; k < n_splits; ++k) {
      const float4 v = ldg4(p + k * slab + src + c);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    return s;
  };
  float p1 = 0.f, p2 = 0.f;
  for (int c = lane * 4; c < d; c += 128) {
    p1 += dot4(ldg4(V1n + src + c), sum_splits(dV1, c));
    p2 += dot4(ldg4(V2n + src + c), sum_splits(dV2, c));
  }
  p1 = warp_sum(p1);
  p2 = warp_sum(p2);
  const float i1 = inv_norm[b], i2 = inv_norm[batch + b];
  // norm clamped at eps: v = x / eps is linear in x, no projection term
  const float k1 = i1 < 1e12f ? p1 : 0.f, k2 = i2 < 1e12f ? p2 : 0.f;
  for (int c = lane * 4; c < d; c += 128) {
    const float4 v1 = ldg4(V1n + src + c), g1 = sum_splits(dV1, c);
    const float4 v2 = ldg4(V2n + src + c), g2 = sum_splits(dV2, c);
    float4 a, x;
    a.x = i1 * (g1.x - k1 * v1.x); a.y = i1 * (g1.y - k1 * v1.y);
    a.z = i1 * (g1.z - k1 * v1.z); a.w = i1 * (g1.w - k1 * v1.w);
    x.x = i2 * (g2.x - k2 * v2.x); x.y = i2 * (g2.y - k2 * v2.y);
    x.z = i2 * (g2.z - k2 * v2.z); x.w = i2 * (g2.w - k2 * v2.w);
    red_add4(dT1 + dst + c, a);
    red_add4(dT2 + dst + c, x);
  }
}

constexpr int kMaxInfoSplits = 32;
constexpr int kMaxInfoTiles = 1023;   // arrival counters: 1 + row tiles (ops.py keeps 1024)

// column splits so that the grid is ~4 CTAs per SM (35 KB of smem each: they are co-resident)
inline int infonce_splits(int batch) {
  const int n_tiles = (batch + kTile - 1) / kTile;
  int splits = max(1, min(min(n_tiles, kMaxInfoSplits), (4 * kNumSMs + n_tiles - 1) / n_tiles));
  const int tps = (n_tiles + splits - 1) / splits;
  return (n_tiles + tps - 1) / tps;
}

template <int D>
int infonce_fwd_launch(const float *V1n, const float *V2n, int batch, float inv_temp, float *partial,
                       float *ttl, float *loss_out, uint32_t *counters, cudaStream_t stream) {
  const int n_tiles = (batch + kTile - 1) / kTile;
  const int splits = infonce_splits(batch);
  const int tps = (n_tiles + splits - 1) / splits;
  // partial layout: pos[batch], ttl_part[splits][batch], tile_loss[n_tiles]
  const size_t smem = (2 * kTile * (D + 4) + kTile * (kTile + 4)) * sizeof(float);
  static bool attr = false;
  if (!attr) {
    MMREC_CUDA(cudaFuncSetAttribute(infonce_fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  infonce_fwd_kernel<D><<<dim3(n_tiles, splits), kThreads, smem, stream>>>(
      V1n, V2n, batch, inv_temp, tps, partial + batch, partial, partial + (size_t)(1 + splits) * batch, ttl,
      loss_out, counters);
  MMREC_CHECK_LAUNCH("infonce_fwd_kernel");
  return MMREC_OK;
}

template <int D>
int infonce_bwd_launch(const float *V1n, const float *V2n, const float *ttl, int batch, float inv_temp,
                       int n_splits, const float *coef, float *dV1, float *dV2, cudaStream_t stream) {
  const int n_tiles = (batch + kTile - 1) / kTile;
  const int tps = (n_tiles + n_splits - 1) / n_splits;   // splits past the end write zeros
  const dim3 grid(n_tiles, n_splits);
  const size_t smem = (2 * kTile * (D + 4) + kTile * (kTile + 4)) * sizeof(float);
  static bool attr = false;
  if (!attr) {
    MMREC_CUDA(cudaFuncSetAttribute(infonce_bwd_kernel<D, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MMREC_CUDA(cudaFuncSetAttribute(infonce_bwd_kernel<D, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  infonce_bwd_kernel<D, true><<<grid, kThreads, smem, stream>>>(V1n, V2n, ttl, batch, inv_temp, tps, coef, dV1);
  MMREC_CHECK_LAUNCH("infonce_bwd_kernel<row>");
  infonce_bwd_kernel<D, false><<<grid, kThreads, smem, stream>>>(V1n, V2n, ttl, batch, inv_temp, tps, coef, dV2);
  MMREC_CHECK_LAUNCH("infonce_bwd_kernel<col>");
  return MMREC_OK;
}

}  // namespace

// tcgen05 path for d = 64 (infonce_tc.cu)
bool infonce_tc_enabled(int d);
int infonce_fwd_tc(int n_prob, const float *const *V1n, const float *const *V2n, int batch, float inv_temp,
                   int cap_splits, float *const *partial, float *const *ttl, float *const *loss_out,
                   cudaStream_t stream);
int infonce_bwd_tc(int n_prob, const float *const *V1n, const float *const *V2n, const float *const *ttl, int batch,
                   float inv_temp, int cap_splits, const float *const *coef, float *const *dV1, float *const *dV2,
                   int *splits_out, cudaStream_t stream);
}  // namespace mmrec

using namespace mmrec;

extern "C" int mmrec_bpr_fwd_f32(const float *user_emb, const float *item_emb, int32_t d,
                                 const int64_t *users, const int64_t *pos, const int64_t *neg, int32_t batch,
                                 float *out2, float *sig, float *partial, uint32_t *counter, void *stream) {
  MMREC_REQUIRE(user_emb && item_emb && users && pos && neg && out2 && sig && partial && counter,
                MMREC_E_BADARG, "bpr_fwd: null pointer");
  MMREC_REQUIRE(batch > 0 && d > 0 && d % 4 == 0, MMREC_E_BADARG, "bpr_fwd: need batch > 0 and d %% 4 == 0");
  MMREC_REQUIRE(aligned16(user_emb) && aligned16(item_emb), MMREC_E_ALIGN, "bpr_fwd: tables must be 16-byte aligned");
  const int wpb = kThreads / 32;
  bpr_fwd_kernel<<<(batch + wpb - 1) / wpb, kThreads, 0, (cudaStream_t)stream>>>(
      user_emb, item_emb, d, users, pos, neg, batch, out2, sig, partial, counter);
  MMREC_CHECK_LAUNCH("bpr_fwd_kernel");
  return MMREC_OK;
}

extern "C" int mmrec_bpr_bwd_f32(const float *user_emb, const float *item_emb, int32_t d,
                                 const int64_t *users, const int64_t *pos, const int64_t *neg, int32_t batch,
                                 const float *sig, const float *coef2, float *d_user_emb, float *d_item_emb,
                                 void *stream) {
  MMREC_REQUIRE(user_emb && item_emb && users && pos && neg && sig && coef2 && d_user_emb && d_item_emb,
                MMREC_E_BADARG, "bpr_bwd: null pointer");
  MMREC_REQUIRE(batch > 0 && d > 0 && d % 4 == 0, MMREC_E_BADARG, "bpr_bwd: need batch > 0 and d %% 4 == 0");
  MMREC_REQUIRE(aligned16(user_emb) && aligned16(item_emb) && aligned16(d_user_emb) && aligned16(d_item_emb),
                MMREC_E_ALIGN, "bpr_bwd: tables must be 16-byte aligned");
  const int wpb = kThreads / 32;
  bpr_bwd_kernel<<<(batch + wpb - 1) / wpb, kThreads, 0, (cudaStream_t)stream>>>(
      user_emb, item_emb, d, users, pos, neg, batch, sig, coef2, d_user_emb, d_item_emb);
  MMREC_CHECK_LAUNCH("bpr_bwd_kernel");
  return MMREC_OK;
}

extern "C" int32_t mmrec_infonce_splits(int32_t batch) { return infonce_splits(batch); }
// Enough for both forward layouts: mma.sync pos | ttl_part[splits] | tile_loss, tcgen05 pos | ttl_part[2 * s]
// with s = infonce_tc_splits(batch, splits) <= max(1, splits / 2), so 2 * s <= max(2, splits).
extern "C" size_t mmrec_infonce_fwd_workspace_floats(int32_t batch) {
  return (size_t)(1 + max(2, infonce_splits(batch))) * batch + (batch + kTile - 1) / kTile;
}

extern "C" int mmrec_infonce_fwd_f32(const float *T1, const float *T2, int32_t d, const int64_t *idx,
                                     int32_t batch, float inv_temp, float *loss_out, float *V1n, float *V2n,
                                     float *inv_norm, float *ttl, float *partial, uint32_t *counter,
                                     void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMREC_REQUIRE(T1 && T2 && idx && loss_out && V1n && V2n && inv_norm && ttl && partial && counter,
                MMREC_E_BADARG, "infonce_fwd: null pointer");
  MMREC_REQUIRE(batch > 0 && (batch + kTile - 1) / kTile <= kMaxInfoTiles, MMREC_E_BADARG,
                "infonce_fwd: batch must be in [1, %d]", kMaxInfoTiles * kTile);
  MMREC_REQUIRE(aligned16(T1) && aligned16(T2) && aligned16(V1n) && aligned16(V2n), MMREC_E_ALIGN,
                "infonce_fwd: operands must be 16-byte aligned");
  const int wpb = kThreads / 32;
  NormArgs NA{};
  NA.T1[0] = T1; NA.T2[0] = T2; NA.idx[0] = idx; NA.V1n[0] = V1n; NA.V2n[0] = V2n; NA.inv_norm[0] = inv_norm;
  infonce_normalize_kernel<<<(batch + wpb - 1) / wpb, kThreads, 0, stream>>>(NA, d, batch);
  MMREC_CHECK_LAUNCH("infonce_normalize_kernel");
  if (infonce_tc_enabled(d)) {
    const float *v1[1] = {V1n}, *v2[1] = {V2n};
    float *pp[1] = {partial}, *tt[1] = {ttl}, *lo[1] = {loss_out};
    return infonce_fwd_tc(1, v1, v2, batch, inv_temp, infonce_splits(batch), pp, tt, lo, stream);
  }
  switch (d) {
    case 32: return infonce_fwd_launch<32>(V1n, V2n, batch, inv_temp, partial, ttl, loss_out, counter, stream);
    case 64: return infonce_fwd_launch<64>(V1n, V2n, batch, inv_temp, partial, ttl, loss_out, counter, stream);
    case 128: return infonce_fwd_launch<128>(V1n, V2n, batch, inv_temp, partial, ttl, loss_out, counter, stream);
    default:
      set_error("infonce_fwd: unsupported d=%d (32, 64, 128)", d);
      return MMREC_E_BADARG;
  }
}

extern "C" int mmrec_infonce_bwd_f32(const float *V1n, const float *V2n, const float *inv_norm, const float *ttl,
                                     int32_t d, const int64_t *idx, int32_t batch, float inv_temp,
                                     const float *coef, int32_t n_splits, float *dV1_ws, float *dV2_ws,
                                     float *dT1, float *dT2, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMREC_REQUIRE(V1n && V2n && inv_norm && ttl && idx && coef && dV1_ws && dV2_ws && dT1 && dT2, MMREC_E_BADARG,
                "infonce_bwd: null pointer");
  MMREC_REQUIRE(batch > 0 && n_splits >= 1 && n_splits <= 64, MMREC_E_BADARG, "infonce_bwd: bad sizes");
  MMREC_REQUIRE(aligned16(V1n) && aligned16(V2n) && aligned16(dV1_ws) && aligned16(dV2_ws) && aligned16(dT1) &&
                    aligned16(dT2), MMREC_E_ALIGN, "infonce_bwd: operands must be 16-byte aligned");
  int rc;
  if (infonce_tc_enabled(d)) {
    int used = n_splits;
    const float *v1[1] = {V1n}, *v2[1] = {V2n}, *tt[1] = {ttl}, *cf[1] = {coef};
    float *d1[1] = {dV1_ws}, *d2[1] = {dV2_ws};
    rc = infonce_bwd_tc(1, v1, v2, tt, batch, inv_temp, n_splits, cf, d1, d2, &used, stream);
    n_splits = used;
  } else
  switch (d) {
    case 32: rc = infonce_bwd_launch<32>(V1n, V2n, ttl, batch, inv_temp, n_splits, coef, dV1_ws, dV2_ws, stream); break;
    case 64: rc = infonce_bwd_launch<64>(V1n, V2n, ttl, batch, inv_temp, n_splits, coef, dV1_ws, dV2_ws, stream); break;
    case 128: rc = infonce_bwd_launch<128>(V1n, V2n, ttl, batch, inv_temp, n_splits, coef, dV1_ws, dV2_ws, stream); break;
    default:
      set_error("infonce_bwd: unsupported d=%d (32, 64, 128)", d);
      return MMREC_E_BADARG;
  }
  if (rc != MMREC_OK) return rc;
  const int wpb = kThreads / 32;
  ScatterArgs SA{};
  SA.V1n[0] = V1n; SA.V2n[0] = V2n; SA.inv_norm[0] = inv_norm; SA.dV1[0] = dV1_ws; SA.dV2[0] = dV2_ws;
  SA.idx[0] = idx; SA.dT1[0] = dT1; SA.dT2[0] = dT2;
  infonce_scatter_kernel<<<(batch + wpb - 1) / wpb, kThreads, 0, stream>>>(SA, n_splits, d, batch);
  MMREC_CHECK_LAUNCH("infonce_scatter_kernel");
  return MMREC_OK;
}

// ---- both InfoNCE problems of a batch (item rows, user rows) in one launch per stage ----------
extern "C" int mmrec_infonce_pair_supported(int32_t d) { return infonce_tc_enabled(d) ? 1 : 0; }

extern "C" int mmrec_infonce_pair_fwd_f32(const float *const *T1_host, const float *const *T2_host, int32_t d,
                                          const int64_t *const *idx_host, int32_t batch, float inv_temp,
                                          float *const *loss_out_host, float *const *V1n_host, float *const *V2n_host,
                                          float *const *inv_norm_host, float *const *ttl_host,
                                          float *const *partial_host, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMREC_REQUIRE(T1_host && T2_host && idx_host && loss_out_host && V1n_host && V2n_host && inv_norm_host && ttl_host &&
                    partial_host, MMREC_E_BADARG, "infonce_pair_fwd: null pointer");
  MMREC_REQUIRE(infonce_tc_enabled(d), MMREC_E_BADARG, "infonce_pair_fwd: d=%d is not on the batched path", d);
  MMREC_REQUIRE(batch > 0 && (batch + kTile - 1) / kTile <= kMaxInfoTiles, MMREC_E_BADARG,
                "infonce_pair_fwd: batch must be in [1, %d]", kMaxInfoTiles * kTile);
  NormArgs NA{};
  for (int p = 0; p < kMaxInfoProb; ++p) {
    NA.T1[p] = T1_host[p]; NA.T2[p] = T2_host[p]; NA.idx[p] = idx_host[p];
    NA.V1n[p] = V1n_host[p]; NA.V2n[p] = V2n_host[p]; NA.inv_norm[p] = inv_norm_host[p];
    MMREC_REQUIRE(NA.T1[p] && NA.T2[p] && NA.idx[p] && NA.V1n[p] && NA.V2n[p] && NA.inv_norm[p] && ttl_host[p] &&
                      partial_host[p] && loss_out_host[p], MMREC_E_BADARG, "infonce_pair_fwd: null tensor %d", p);
    MMREC_REQUIRE(aligned16(NA.T1[p]) && aligned16(NA.T2[p]) && aligned16(NA.V1n[p]) && aligned16(NA.V2n[p]),
                  MMREC_E_ALIGN, "infonce_pair_fwd: operands must be 16-byte aligned");
  }
  const int wpb = kThreads / 32;
  infonce_normalize_kernel<<<dim3((batch + wpb - 1) / wpb, kMaxInfoProb), kThreads, 0, stream>>>(NA, d, batch);
  MMREC_CHECK_LAUNCH("infonce_normalize_kernel");
  return infonce_fwd_tc(kMaxInfoProb, V1n_host, V2n_host, batch, inv_temp, infonce_splits(batch), partial_host,
                        ttl_host, loss_out_host, stream);
}

extern "C" int mmrec_infonce_pair_bwd_f32(const float *const *V1n_host, const float *const *V2n_host,
                                          const float *const *inv_norm_host, const float *const *ttl_host, int32_t d,
                                          const int64_t *const *idx_host, int32_t batch, float inv_temp,
                                          const float *const *coef_host, int32_t n_splits, float *const *dV1_ws_host,
                                          float *const *dV2_ws_host, float *const *dT1_host, float *const *dT2_host,
                                          void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMREC_REQUIRE(V1n_host && V2n_host && inv_norm_host && ttl_host && idx_host && coef_host && dV1_ws_host &&
                    dV2_ws_host && dT1_host && dT2_host, MMREC_E_BADARG, "infonce_pair_bwd: null pointer");
  MMREC_REQUIRE(infonce_tc_enabled(d), MMREC_E_BADARG, "infonce_pair_bwd: d=%d is not on the batched path", d);
  MMREC_REQUIRE(batch > 0 && n_splits >= 1 && n_splits <= 64, MMREC_E_BADARG, "infonce_pair_bwd: bad sizes");
  ScatterArgs SA{};
  for (int p = 0; p < kMaxInfoProb; ++p) {
    SA.V1n[p] = V1n_host[p]; SA.V2n[p] = V2n_host[p]; SA.inv_norm[p] = inv_norm_host[p];
    SA.dV1[p] = dV1_ws_host[p]; SA.dV2[p] = dV2_ws_host[p]; SA.idx[p] = idx_host[p];
    SA.dT1[p] = dT1_host[p]; SA.dT2[p] = dT2_host[p];
    MMREC_REQUIRE(SA.V1n[p] && SA.V2n[p] && SA.inv_norm[p] && SA.dV1[p] && SA.dV2[p] && SA.idx[p] && SA.dT1[p] &&
                      SA.dT2[p] && ttl_host[p] && coef_host[p], MMREC_E_BADARG, "infonce_pair_bwd: null tensor %d", p);
    MMREC_REQUIRE(aligned16(SA.V1n[p]) && aligned16(SA.V2n[p]) && aligned16(SA.dV1[p]) && aligned16(SA.dV2[p]) &&
                      aligned16(SA.dT1[p]) && aligned16(SA.dT2[p]), MMREC_E_ALIGN,
                  "infonce_pair_bwd: operands must be 16-byte aligned");
  }
  int used = n_splits;
  const int rc = infonce_bwd_tc(kMaxInfoProb, V1n_host, V2n_host, ttl_host, batch, inv_temp, n_splits, coef_host,
                                dV1_ws_host, dV2_ws_host, &used, stream);
  if (rc != MMREC_OK) return rc;
  const int wpb = kThreads / 32;
  infonce_scatter_kernel<<<dim3((batch + wpb - 1) / wpb, kMaxInfoProb), kThreads, 0, stream>>>(SA, used, d, batch);
  MMREC_CHECK_LAUNCH("infonce_scatter_kernel");
  return MMREC_OK;
}
