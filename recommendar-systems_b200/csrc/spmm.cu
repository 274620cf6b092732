// CSR row-split SpMM with fused layer combination (K1/K2/K3) -- see include/mmrec_b200.h.
//
// Layout: CSR (int32 row_ptr / col_idx, float32 vals), X and Y row-major [n, d].
// Work split: the graph carries a task list built once per graph (graph.py): every task is one
// sub-warp of LANES = d/4 threads (16 lanes x float4 for d = 64, a full warp for d = 128) and at
// most SEG = 64 non-zeros, so the longest dependent chain of gathers in the whole launch is a
// handful of rounds whatever the degree distribution (power-law item rows would otherwise
// serialise thousands of DRAM round trips in one sub-warp). Light rows (deg <= SEG) are one task;
// a heavy row is cut into ceil(deg/SEG) tasks whose partial sums go to a scratch buffer, and
// the last task to arrive (per-row counter, self-resetting) adds them in part order and runs
// the fused epilogue -- no floating-point atomics, results are bit-reproducible run to run.
// Each gathered embedding row is one coalesced 16-byte-per-lane request; the column indices and
// values of a whole task are loaded in one round and broadcast with shuffles; eight gathers are
// kept in flight per lane. The kernel is a chain of dependent L2/DRAM round trips: on the small
// graphs (Baby: 27k tasks = 1.4 waves) the length of that chain IS the kernel time, on graphs
// larger than L2 the bytes in flight per SM (4 CTAs x 16 tasks x 8 rows x 256 B) saturate HBM.
#include "common.cuh"

namespace mmrec {
namespace {

constexpr int kThreads = 256;

template <int LANES>
__device__ __forceinline__ unsigned group_mask() {
  if constexpr (LANES == 32) {
    return 0xffffffffu;
  } else {
    const unsigned lane = threadIdx.x & 31u;
    return ((1u << LANES) - 1u) << (LANES * (lane / LANES));
  }
}

__device__ __forceinline__ int ld_stream_i32(const int32_t *p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// L2 eviction policies for operands that do not fit the cache (flags & MMREC_SPMM_STREAM). The
// gathered X rows are the only data with reuse: they are loaded evict_last; everything that is
// touched exactly once per launch (CSR arrays, the task list, the epilogue operand and the output
// rows) goes through evict_first, so that ~10 GB of streamed bytes per launch do not push the hot
// rows of a power-law graph out of the 126 MB L2 (ncu, 10M x 2M graph, default policy: 34 % sector
// hit rate on the item table although the hottest 25 % of the items carry 75 % of the edges).
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float4 ldg4_hint(const float *ptr, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(ptr), "l"(pol));
  return v;
}
__device__ __forceinline__ void stg4_hint(float *ptr, const float4 &v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(ptr), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w), "l"(pol)
               : "memory");
}
__device__ __forceinline__ int ld_stream_i32_hint(const int32_t *p, uint64_t pol) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float ld_stream_f32_hint(const float *p, uint64_t pol) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}

constexpr int kSeg = 64;   // non-zeros per task; must match graph.py SEG
constexpr int kDepth = 8;  // embedding-row gathers in flight per lane

// Accumulate the (at most kSeg) non-zeros [begin, end) of one task. A task is a chain of dependent
// memory round trips (task -> indices -> rows), so the chain is kept as short as it can be: every
// column index / value of the task is fetched in ONE round (kSeg / LANES per lane), then the rows
// are gathered kDepth at a time (16 bytes per lane each); partial groups are predicated off, not
// padded. The sum runs in CSR order whatever the grouping.
// `after_indices()` runs between the index round and the first gather: the kernels put pdl_wait() there
// (the CSR arrays and the task list are never written by a kernel of the step, X is).
template <int LANES, int CHUNKS, bool STREAM = false, typename Hook>
__device__ __forceinline__ void gather_rows(float4 (&acc)[CHUNKS], const int32_t *__restrict__ col_idx,
                                            const float *__restrict__ vals, int begin, int end, int lane,
                                            const float *__restrict__ X, int d, int col_offset, Hook &&after_indices) {
  uint64_t pol_first = 0, pol_last = 0;
  if constexpr (STREAM) { pol_first = policy_evict_first(); pol_last = policy_evict_last(); }
  constexpr int NIDX = kSeg / LANES;
  constexpr int DEPTH = CHUNKS == 1 ? kDepth : kDepth / 2;
  const unsigned mask = group_mask<LANES>();
  const int n = end - begin;
  int c[NIDX];
  float v[NIDX];
#pragma unroll
  for (int i = 0; i < NIDX; ++i) {
    const int k = begin + i * LANES + lane;
    c[i] = 0;
    v[i] = 0.f;
    if (k < end) {
      if constexpr (STREAM) {
        c[i] = ld_stream_i32_hint(col_idx + k, pol_first) - col_offset;
        v[i] = ld_stream_f32_hint(vals + k, pol_first);
      } else {
        c[i] = ld_stream_i32(col_idx + k) - col_offset;
        v[i] = ld_stream_f32(vals + k);
      }
    }
  }
  {
    // ptxas is free to sink loads below griddepcontrol.wait (an acquire): the hook gets a value that
    // depends on every index load and makes its wait conditional on it (never false), which pins the
    // loads in front of the wait.
    int probe = 0;
#pragma unroll
    for (int i = 0; i < NIDX; ++i) probe |= c[i] | (int)__float_as_uint(v[i]);
    after_indices(probe);
  }
#pragma unroll
  for (int i = 0; i < NIDX; ++i) {
#pragma unroll
    for (int j = 0; j < LANES; j += DEPTH) {
      const int base = i * LANES + j;
      if (base < n) {
        int cc[DEPTH];
        float vv[DEPTH];
        float4 x[DEPTH][CHUNKS];
#pragma unroll
        for (int t = 0; t < DEPTH; ++t) {
          cc[t] = __shfl_sync(mask, c[i], j + t, LANES);
          vv[t] = __shfl_sync(mask, v[i], j + t, LANES);
        }
#pragma unroll
        for (int t = 0; t < DEPTH; ++t)
#pragma unroll
          for (int q = 0; q < CHUNKS; ++q)
            x[t][q] = base + t < n ? (STREAM ? ldg4_hint(X + (size_t)cc[t] * d + (q * LANES + lane) * 4, pol_last)
                                             : ldg4(X + (size_t)cc[t] * d + (q * LANES + lane) * 4))
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int t = 0; t < DEPTH; ++t)
#pragma unroll
          for (int q = 0; q < CHUNKS; ++q) fma4(acc[q], vv[t], x[t][q]);
      }
    }
  }
}

struct Epilogue {
  float *Y;
  const float *acc_in;
  float *acc_out;
  float acc_scale;
  const float *cos_ref;
  float *cos_w;
  float *Y_pre;
};

template <int LANES, int CHUNKS, bool STREAM = false>
__device__ __forceinline__ void finish_row(float4 (&acc)[CHUNKS], int row, int lane, int d,
                                           const Epilogue &ep) {
  const size_t off = (size_t)row * d;
  uint64_t pol_first = 0;
  if constexpr (STREAM) pol_first = policy_evict_first();
  if (ep.cos_ref != nullptr) {
    float4 e0[CHUNKS];
    float dot = 0.f, ny = 0.f, n0 = 0.f;
#pragma unroll
    for (int q = 0; q < CHUNKS; ++q) {
      e0[q] = ldg4(ep.cos_ref + off + (q * LANES + lane) * 4);
      if (ep.Y_pre) *reinterpret_cast<float4 *>(ep.Y_pre + off + (q * LANES + lane) * 4) = acc[q];
      ny += dot4(acc[q], acc[q]);
      n0 += dot4(e0[q], e0[q]);
    }
    ny = group_sum<LANES>(ny);
    n0 = group_sum<LANES>(n0);
    const float iy = 1.f / fmaxf(sqrtf(ny), 1e-8f), i0 = 1.f / fmaxf(sqrtf(n0), 1e-8f);
#pragma unroll
    for (int q = 0; q < CHUNKS; ++q) {
      float4 a = acc[q], b = e0[q];
      a.x *= iy; a.y *= iy; a.z *= iy; a.w *= iy;
      b.x *= i0; b.y *= i0; b.z *= i0; b.w *= i0;
      dot += dot4(a, b);
    }
    const float w = group_sum<LANES>(dot);
    if (lane == 0 && ep.cos_w) ep.cos_w[row] = w;
#pragma unroll
    for (int q = 0; q < CHUNKS; ++q) {
      acc[q].x *= w; acc[q].y *= w; acc[q].z *= w; acc[q].w *= w;
    }
  }
#pragma unroll
  for (int q = 0; q < CHUNKS; ++q) {
    const size_t o = off + (q * LANES + lane) * 4;
    if (ep.Y) {
      if constexpr (STREAM) stg4_hint(ep.Y + o, acc[q], pol_first);
      else *reinterpret_cast<float4 *>(ep.Y + o) = acc[q];
    }
    if (ep.acc_out) {
      float4 r = acc[q];
      if (ep.acc_in) {
        float4 a;
        if constexpr (STREAM) a = ldg4_hint(ep.acc_in + o, pol_first);   // read once (in place: before the store below)
        else a = *reinterpret_cast<const float4 *>(ep.acc_in + o);
        r.x += a.x; r.y += a.y; r.z += a.z; r.w += a.w;
      }
      r.x *= ep.acc_scale; r.y *= ep.acc_scale; r.z *= ep.acc_scale; r.w *= ep.acc_scale;
      if constexpr (STREAM) stg4_hint(ep.acc_out + o, r, pol_first);
      else *reinterpret_cast<float4 *>(ep.acc_out + o) = r;
    }
  }
}

struct Problem {
  const int32_t *row_ptr, *col_idx;
  const float *vals;
  const int4 *tasks;
  int n_tasks;
  const int32_t *slot_base;
  int32_t *counters;
  float *scratch;
  int col_offset;
  const float *X;
  Epilogue ep;
};

// One task (<= kSeg non-zeros of one row) by one sub-warp of LANES threads.
template <int LANES, int CHUNKS, bool STREAM = false>
__device__ __forceinline__ void run_task(const Problem &P, int t, int lane, int d) {
  const int4 task = __ldg(P.tasks + t);          // {row, begin, end, slot}
  const int row = task.x;
  const Epilogue &ep = P.ep;
  float4 acc[CHUNKS];
#pragma unroll
  for (int q = 0; q < CHUNKS; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  gather_rows<LANES, CHUNKS, STREAM>(acc, P.col_idx, P.vals, task.y, task.z, lane, P.X, d, P.col_offset, [&](int probe) {
    // Everything above read graph constants only (task, column indices, values): under programmatic
    // dependent launch it ran while the previous layer's launch was still finishing. From here on the
    // kernel touches what that launch wrote.
    if (probe != 0x7fc00001) pdl_wait();      // (a NaN payload no adjacency value carries, OR-ed with indices >= 0)
    if (task.w < 0) {
      // start fetching the epilogue operands of this row while the gathers are in flight
      const size_t o = (size_t)row * d + lane * 4;
      if (ep.acc_in) asm volatile("prefetch.global.L2 [%0];" ::"l"(ep.acc_in + o));
      if (ep.cos_ref) asm volatile("prefetch.global.L2 [%0];" ::"l"(ep.cos_ref + o));
    }
  });
  if (task.w >= 0) {
    // heavy row: publish this part, the last arriver reduces all parts in order
    const unsigned mask = group_mask<LANES>();
    const int r0 = P.row_ptr[row];
    const int n_parts = (P.row_ptr[row + 1] - r0 + kSeg - 1) / kSeg;
    const int part = (task.y - r0) / kSeg;
    float *base = P.scratch + (size_t)P.slot_base[task.w] * d;
#pragma unroll
    for (int q = 0; q < CHUNKS; ++q)
      __stcg(reinterpret_cast<float4 *>(base + (size_t)part * d + (q * LANES + lane) * 4), acc[q]);
    __threadfence();
    __syncwarp(mask);
    int last = 0;
    if (lane == 0) {
      last = atomicAdd(P.counters + task.w, 1) == n_parts - 1;
      if (last) P.counters[task.w] = 0;
    }
    last = __shfl_sync(mask, last, 0, LANES);
    if (!last) return;
    __threadfence();
#pragma unroll
    for (int q = 0; q < CHUNKS; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = 0; p < n_parts; p += 4) {
      float4 v[4][CHUNKS];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int q = 0; q < CHUNKS; ++q)
          v[u][q] = p + u < n_parts
                        ? __ldcg(reinterpret_cast<const float4 *>(base + (size_t)(p + u) * d + (q * LANES + lane) * 4))
                        : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int q = 0; q < CHUNKS; ++q) {
          acc[q].x += v[u][q].x; acc[q].y += v[u][q].y; acc[q].z += v[u][q].z; acc[q].w += v[u][q].w;
        }
    }
  }
  finish_row<LANES, CHUNKS, STREAM>(acc, row, lane, d, ep);
}

template <int LANES, int CHUNKS, bool STREAM = false>
__global__ void __launch_bounds__(kThreads, CHUNKS == 1 || LANES <= 16 ? 4 : 3)
spmm_csr_kernel(const Problem P, int d) {
  constexpr int GROUPS = kThreads / LANES;
  pdl_trigger();     // the next launch may park its CTAs (and read its task list) behind this one's last wave
  const int lane = threadIdx.x % LANES;
  const int t = blockIdx.x * GROUPS + threadIdx.x / LANES;
  if (t >= P.n_tasks) return;
  run_task<LANES, CHUNKS, STREAM>(P, t, lane, d);
}

// Several independent SpMMs in one launch (the three modality views of SMORE/MGCN: small graphs
// that each fill a fraction of the GPU). block_end[p] = first block after problem p.
constexpr int kMaxProblems = 4;
struct MultiArgs {
  Problem p[kMaxProblems];
  int block_end[kMaxProblems];
  int n;
};

template <int LANES, int CHUNKS>
__global__ void __launch_bounds__(kThreads, CHUNKS == 1 ? 4 : 3)
spmm_csr_multi_kernel(const MultiArgs A, int d) {
  constexpr int GROUPS = kThreads / LANES;
  pdl_trigger();
  int pi = 0;
  while (pi + 1 < A.n && (int)blockIdx.x >= A.block_end[pi]) ++pi;
  const int b0 = pi == 0 ? 0 : A.block_end[pi - 1];
  const Problem &P = A.p[pi];
  const int lane = threadIdx.x % LANES;
  const int t = (blockIdx.x - b0) * GROUPS + threadIdx.x / LANES;
  if (t >= P.n_tasks) return;
  run_task<LANES, CHUNKS>(P, t, lane, d);
}

// ---- LayerGCN cosine refinement, backward row operator --------------------------------------
template <int LANES, int CHUNKS>
__global__ void __launch_bounds__(kThreads)
layergcn_cos_bwd_kernel(const float *__restrict__ dE, const float *__restrict__ P,
                        const float *__restrict__ E0, const float *__restrict__ W, int n_rows,
                        int d, float *__restrict__ dP, float *__restrict__ dE0) {
  constexpr int GROUPS = kThreads / LANES;
  const int lane = threadIdx.x % LANES;
  const int row = blockIdx.x * GROUPS + threadIdx.x / LANES;
  if (row >= n_rows) return;
  const size_t off = (size_t)row * d;
  float4 g[CHUNKS], p[CHUNKS], e0[CHUNKS];
  float gp = 0.f, ny = 0.f, n0 = 0.f;
#pragma unroll
  for (int q = 0; q < CHUNKS; ++q) {
    const size_t o = off + (q * LANES + lane) * 4;
    g[q] = ldg4(dE + o);
    p[q] = ldg4(P + o);
    e0[q] = ldg4(E0 + o);
    gp += dot4(g[q], p[q]);
    ny += dot4(p[q], p[q]);
    n0 += dot4(e0[q], e0[q]);
  }
  gp = group_sum<LANES>(gp);
  ny = sqrtf(group_sum<LANES>(ny));
  n0 = sqrtf(group_sum<LANES>(n0));
  const float w = W[row];
  const float cy = fmaxf(ny, 1e-8f), c0 = fmaxf(n0, 1e-8f);
  const float iy = 1.f / cy, i0 = 1.f / c0;
  // d cos / dp = (e0n - [ny > eps] * w * pn) / max(ny, eps); same for e0 with roles swapped
  const float sy = ny > 1e-8f ? w : 0.f, s0 = n0 > 1e-8f ? w : 0.f;
#pragma unroll
  for (int q = 0; q < CHUNKS; ++q) {
    const size_t o = off + (q * LANES + lane) * 4;
    const float4 a = p[q], b = e0[q], gg = g[q];
    float4 dp, de;
    dp.x = w * gg.x + gp * (b.x * i0 - sy * a.x * iy) * iy;
    dp.y = w * gg.y + gp * (b.y * i0 - sy * a.y * iy) * iy;
    dp.z = w * gg.z + gp * (b.z * i0 - sy * a.z * iy) * iy;
    dp.w = w * gg.w + gp * (b.w * i0 - sy * a.w * iy) * iy;
    *reinterpret_cast<float4 *>(dP + o) = dp;
    float4 acc = *reinterpret_cast<const float4 *>(dE0 + o);
    de.x = gp * (a.x * iy - s0 * b.x * i0) * i0;
    de.y = gp * (a.y * iy - s0 * b.y * i0) * i0;
    de.z = gp * (a.z * iy - s0 * b.z * i0) * i0;
    de.w = gp * (a.w * iy - s0 * b.w * i0) * i0;
    acc.x += de.x; acc.y += de.y; acc.z += de.z; acc.w += de.w;
    *reinterpret_cast<float4 *>(dE0 + o) = acc;
  }
}

// ---- bf16 operand, fp32 accumulation (mmrec_spmm_csr_bf16_f32) ------------------------------
// The task walk of run_task with X stored as bf16: one 16-byte gather is 8 values, so a sub-warp
// has LANES = d / 8 lanes (CHUNKS 16-byte pieces per lane in the narrow tiling) and lane `lane`
// owns the elements (q * LANES + lane) * 8 + [0, 8) of a row. The values are widened in registers
// (exactly: a bf16 is the top half of a float32) and every product and sum is the fp32 arithmetic
// of the fp32 kernel in the same order (CSR order inside a task, parts in order for a split row,
// the same epilogue), so the output equals mmrec_spmm_csr_f32's on the widened operand bit for bit.
struct ProblemBf16 {
  const int32_t *row_ptr, *col_idx;
  const float *vals;
  const int4 *tasks;
  int n_tasks;
  const int32_t *slot_base;
  int32_t *counters;
  float *scratch;
  int col_offset;
  const uint16_t *X;
  float *Y;
  uint16_t *Y16;
  const float *acc_in;
  float *acc_out;
  float acc_scale;
};

__device__ __forceinline__ void fma8_bf16(float4 &lo, float4 &hi, float s, const uint4 &x) {
  fma4(lo, s, make_float4(__uint_as_float(x.x << 16), __uint_as_float(x.x & 0xffff0000u),
                          __uint_as_float(x.y << 16), __uint_as_float(x.y & 0xffff0000u)));
  fma4(hi, s, make_float4(__uint_as_float(x.z << 16), __uint_as_float(x.z & 0xffff0000u),
                          __uint_as_float(x.w << 16), __uint_as_float(x.w & 0xffff0000u)));
}

// round to nearest even, two floats -> one word (low half first, the memory order of a bf16 row)
__device__ __forceinline__ unsigned pack_bf16x2(float a, float b) {
  unsigned r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

template <int LANES, int CHUNKS>
__device__ __forceinline__ void run_task_bf16(const ProblemBf16 &P, int t, int lane, int d) {
  constexpr int NIDX = kSeg / LANES;
  constexpr int DEPTH0 = CHUNKS == 1 ? kDepth : kDepth / 2;
  constexpr int DEPTH = DEPTH0 < LANES ? DEPTH0 : LANES;   // shuffle sources stay inside the sub-warp
  const int4 task = __ldg(P.tasks + t);                    // {row, begin, end, slot}
  const int row = task.x, begin = task.y, end = task.z, n = end - begin;
  const unsigned mask = group_mask<LANES>();
  float4 acc[2 * CHUNKS];
#pragma unroll
  for (int q = 0; q < 2 * CHUNKS; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  int c[NIDX];
  float v[NIDX];
#pragma unroll
  for (int i = 0; i < NIDX; ++i) {
    const int k = begin + i * LANES + lane;
    c[i] = 0;
    v[i] = 0.f;
    if (k < end) {
      c[i] = ld_stream_i32(P.col_idx + k) - P.col_offset;
      v[i] = ld_stream_f32(P.vals + k);
    }
  }
  {
    // graph constants above, the previous launch's outputs below (see gather_rows / run_task)
    int probe = 0;
#pragma unroll
    for (int i = 0; i < NIDX; ++i) probe |= c[i] | (int)__float_as_uint(v[i]);
    if (probe != 0x7fc00001) pdl_wait();
    if (task.w < 0 && P.acc_in) {
      const size_t o = (size_t)row * d + lane * 8;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(P.acc_in + o));
    }
  }
#pragma unroll
  for (int i = 0; i < NIDX; ++i) {
#pragma unroll
    for (int j = 0; j < LANES; j += DEPTH) {
      const int base = i * LANES + j;
      if (base < n) {
        int cc[DEPTH];
        float vv[DEPTH];
        uint4 x[DEPTH][CHUNKS];
#pragma unroll
        for (int s = 0; s < DEPTH; ++s) {
          cc[s] = __shfl_sync(mask, c[i], j + s, LANES);
          vv[s] = __shfl_sync(mask, v[i], j + s, LANES);
        }
#pragma unroll
        for (int s = 0; s < DEPTH; ++s)
#pragma unroll
          for (int q = 0; q < CHUNKS; ++q)
            x[s][q] = base + s < n
                          ? __ldg(reinterpret_cast<const uint4 *>(P.X + (size_t)cc[s] * d + (q * LANES + lane) * 8))
                          : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int s = 0; s < DEPTH; ++s)
#pragma unroll
          for (int q = 0; q < CHUNKS; ++q) fma8_bf16(acc[2 * q], acc[2 * q + 1], vv[s], x[s][q]);
      }
    }
  }
  if (task.w >= 0) {
    // heavy row: publish this part, the last arriver reduces all parts in order
    const int r0 = P.row_ptr[row];
    const int n_parts = (P.row_ptr[row + 1] - r0 + kSeg - 1) / kSeg;
    const int part = (begin - r0) / kSeg;
    float *base = P.scratch + (size_t)P.slot_base[task.w] * d;
#pragma unroll
    for (int q = 0; q < CHUNKS; ++q) {
      float4 *p = reinterpret_cast<float4 *>(base + (size_t)part * d + (q * LANES + lane) * 8);
      __stcg(p, acc[2 * q]);
      __stcg(p + 1, acc[2 * q + 1]);
    }
    __threadfence();
    __syncwarp(mask);
    int last = 0;
    if (lane == 0) {
      last = atomicAdd(P.counters + task.w, 1) == n_parts - 1;
      if (last) P.counters[task.w] = 0;
    }
    last = __shfl_sync(mask, last, 0, LANES);
    if (!last) return;
    __threadfence();
#pragma unroll
    for (int q = 0; q < 2 * CHUNKS; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int U = CHUNKS == 1 ? 4 : 2;
    for (int p = 0; p < n_parts; p += U) {
      float4 w[U][2 * CHUNKS];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int q = 0; q < 2 * CHUNKS; ++q)
          w[u][q] = p + u < n_parts ? __ldcg(reinterpret_cast<const float4 *>(
                                          base + (size_t)(p + u) * d + (q / 2 * LANES + lane) * 8 + (q % 2) * 4))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int q = 0; q < 2 * CHUNKS; ++q) {
          acc[q].x += w[u][q].x; acc[q].y += w[u][q].y; acc[q].z += w[u][q].z; acc[q].w += w[u][q].w;
        }
    }
  }
  // epilogue of finish_row (no cosine mode), plus the rounded copy of y
  const size_t off = (size_t)row * d;
#pragma unroll
  for (int q = 0; q < CHUNKS; ++q) {
    const size_t o = off + (q * LANES + lane) * 8;
    if (P.Y) {
      *reinterpret_cast<float4 *>(P.Y + o) = acc[2 * q];
      *reinterpret_cast<float4 *>(P.Y + o + 4) = acc[2 * q + 1];
    }
    if (P.Y16) {
      const float4 a = acc[2 * q], b = acc[2 * q + 1];
      *reinterpret_cast<uint4 *>(P.Y16 + o) =
          make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
    }
    if (P.acc_out) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float4 r = acc[2 * q + h];
        if (P.acc_in) {
          const float4 a = *reinterpret_cast<const float4 *>(P.acc_in + o + 4 * h);
          r.x += a.x; r.y += a.y; r.z += a.z; r.w += a.w;
        }
        r.x *= P.acc_scale; r.y *= P.acc_scale; r.z *= P.acc_scale; r.w *= P.acc_scale;
        *reinterpret_cast<float4 *>(P.acc_out + o + 4 * h) = r;
      }
    }
  }
}

// 4-lane and two-chunk tilings hold 16 indices or 16 accumulators per lane: 3 CTAs (80 registers) keep
// them from spilling
template <int LANES, int CHUNKS>
__global__ void __launch_bounds__(kThreads, CHUNKS == 1 && LANES >= 8 ? 4 : 3)
spmm_csr_bf16_kernel(const ProblemBf16 P, int d) {
  constexpr int GROUPS = kThreads / LANES;
  pdl_trigger();
  const int lane = threadIdx.x % LANES;
  const int t = blockIdx.x * GROUPS + threadIdx.x / LANES;
  if (t >= P.n_tasks) return;
  run_task_bf16<LANES, CHUNKS>(P, t, lane, d);
}

// Narrow tiling for graphs of very short rows (the column blocks of graph.ColumnBlockedCSR: a
// handful of non-zeros per task): half the lanes per task, two float4 per lane -- twice as many
// tasks in flight per SM for a kernel whose time is the number of dependent round trips per task
// divided by the tasks in flight.
template <typename F>
int dispatch_width_narrow(int d, F &&f) {
  switch (d) {
    case 32: return f(std::integral_constant<int, 8>{}, std::integral_constant<int, 1>{});
    case 64: return f(std::integral_constant<int, 8>{}, std::integral_constant<int, 2>{});
    case 128: return f(std::integral_constant<int, 16>{}, std::integral_constant<int, 2>{});
    case 256: return f(std::integral_constant<int, 32>{}, std::integral_constant<int, 2>{});
    default:
      set_error("unsupported embedding width d=%d (supported: 32, 64, 128, 256)", d);
      return MMREC_E_BADARG;
  }
}

template <typename F>
int dispatch_width(int d, F &&f) {
  switch (d) {
    case 32: return f(std::integral_constant<int, 8>{}, std::integral_constant<int, 1>{});
    case 64: return f(std::integral_constant<int, 16>{}, std::integral_constant<int, 1>{});
    case 128: return f(std::integral_constant<int, 32>{}, std::integral_constant<int, 1>{});
    case 256: return f(std::integral_constant<int, 32>{}, std::integral_constant<int, 2>{});
    default:
      set_error("unsupported embedding width d=%d (supported: 32, 64, 128, 256)", d);
      return MMREC_E_BADARG;
  }
}

// (LANES, CHUNKS) of the bf16 kernel: LANES * CHUNKS * 8 = d; the narrow tiling halves the lanes.
template <typename F>
int dispatch_width_bf16(int d, bool narrow, F &&f) {
  using std::integral_constant;
  switch (d) {
    case 32: return f(integral_constant<int, 4>{}, integral_constant<int, 1>{});
    case 64: return narrow ? f(integral_constant<int, 4>{}, integral_constant<int, 2>{})
                           : f(integral_constant<int, 8>{}, integral_constant<int, 1>{});
    case 128: return narrow ? f(integral_constant<int, 8>{}, integral_constant<int, 2>{})
                            : f(integral_constant<int, 16>{}, integral_constant<int, 1>{});
    default:
      set_error("spmm_bf16: unsupported embedding width d=%d (supported: 32, 64, 128)", d);
      return MMREC_E_BADARG;
  }
}

}  // namespace
}  // namespace mmrec

using namespace mmrec;

static int spmm_csr_impl(int flags, const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                         const int32_t *tasks, int32_t n_tasks, const int32_t *slot_base,
                         int32_t *counters, float *scratch, int32_t col_offset, const float *X,
                         int32_t d, float *Y, const float *acc_in, float *acc_out, float acc_scale,
                         const float *cos_ref, float *cos_w, float *Y_pre, void *stream) {
  MMREC_REQUIRE(row_ptr && col_idx && vals && tasks && X, MMREC_E_BADARG, "spmm: null input");
  MMREC_REQUIRE(Y || acc_out, MMREC_E_BADARG, "spmm: no output requested");
  MMREC_REQUIRE(n_tasks >= 0, MMREC_E_BADARG, "spmm: bad sizes");
  MMREC_REQUIRE(aligned16(X) && aligned16(Y) && aligned16(acc_in) && aligned16(acc_out) &&
                    aligned16(cos_ref) && aligned16(Y_pre) && aligned16(tasks) && aligned16(scratch),
                MMREC_E_ALIGN, "spmm: dense operands and the task list must be 16-byte aligned");
  MMREC_REQUIRE(X != Y && X != acc_out, MMREC_E_BADARG, "spmm: X must not alias an output");
  if (n_tasks == 0) return MMREC_OK;
  Problem P{row_ptr, col_idx, vals, reinterpret_cast<const int4 *>(tasks), n_tasks, slot_base, counters, scratch,
            col_offset, X, Epilogue{Y, acc_in, acc_out, acc_scale, cos_ref, cos_w, Y_pre}};
  const bool narrow = flags & MMREC_SPMM_NARROW, streaming = flags & MMREC_SPMM_STREAM;
  MMREC_REQUIRE(!(streaming && cos_ref), MMREC_E_BADARG, "spmm: the streaming cache policy has no cosine epilogue");
  auto launch = [&](auto lanes, auto chunks) {
    constexpr int L = decltype(lanes)::value, C = decltype(chunks)::value;
    constexpr int GROUPS = kThreads / L;
    const int blocks = (n_tasks + GROUPS - 1) / GROUPS;
    if (streaming) MMREC_CUDA(launch_pdl(spmm_csr_kernel<L, C, true>, blocks, kThreads, 0, (cudaStream_t)stream, P, d));
    else MMREC_CUDA(launch_pdl(spmm_csr_kernel<L, C, false>, blocks, kThreads, 0, (cudaStream_t)stream, P, d));
    MMREC_CHECK_LAUNCH("spmm_csr_kernel");
    return MMREC_OK;
  };
  return narrow ? dispatch_width_narrow(d, launch) : dispatch_width(d, launch);
}

extern "C" int mmrec_spmm_csr_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                                  const int32_t *tasks, int32_t n_tasks, const int32_t *slot_base,
                                  int32_t *counters, float *scratch, int32_t col_offset, const float *X,
                                  int32_t d, float *Y, const float *acc_in, float *acc_out, float acc_scale,
                                  const float *cos_ref, float *cos_w, float *Y_pre, void *stream) {
  return spmm_csr_impl(0, row_ptr, col_idx, vals, tasks, n_tasks, slot_base, counters, scratch, col_offset, X, d,
                       Y, acc_in, acc_out, acc_scale, cos_ref, cos_w, Y_pre, stream);
}

extern "C" int mmrec_spmm_csr_ex_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                                     const int32_t *tasks, int32_t n_tasks, const int32_t *slot_base,
                                     int32_t *counters, float *scratch, int32_t col_offset, const float *X,
                                     int32_t d, float *Y, const float *acc_in, float *acc_out, float acc_scale,
                                     const float *cos_ref, float *cos_w, float *Y_pre, int32_t flags, void *stream) {
  return spmm_csr_impl(flags, row_ptr, col_idx, vals, tasks, n_tasks, slot_base, counters, scratch, col_offset, X, d,
                       Y, acc_in, acc_out, acc_scale, cos_ref, cos_w, Y_pre, stream);
}

extern "C" int mmrec_spmm_csr_bf16_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                                       const int32_t *tasks, int32_t n_tasks, const int32_t *slot_base,
                                       int32_t *counters, float *scratch, int32_t col_offset, const uint16_t *X,
                                       int32_t d, float *Y, uint16_t *Y16, const float *acc_in, float *acc_out,
                                       float acc_scale, const float *cos_ref, float *cos_w, float *Y_pre,
                                       int32_t flags, void *stream) {
  MMREC_REQUIRE(row_ptr && col_idx && vals && tasks && X, MMREC_E_BADARG, "spmm_bf16: null input");
  MMREC_REQUIRE(Y || Y16 || acc_out, MMREC_E_BADARG, "spmm_bf16: no output requested");
  MMREC_REQUIRE(n_tasks >= 0, MMREC_E_BADARG, "spmm_bf16: bad sizes");
  MMREC_REQUIRE(!cos_ref && !cos_w && !Y_pre, MMREC_E_BADARG, "spmm_bf16: the cosine epilogue has no bf16 variant");
  MMREC_REQUIRE(!(flags & ~MMREC_SPMM_NARROW), MMREC_E_BADARG,
                "spmm_bf16: flags 0x%x not supported (MMREC_SPMM_NARROW only)", flags);
  MMREC_REQUIRE(aligned16(X) && aligned16(Y) && aligned16(Y16) && aligned16(acc_in) && aligned16(acc_out) &&
                    aligned16(tasks) && aligned16(scratch),
                MMREC_E_ALIGN, "spmm_bf16: dense operands and the task list must be 16-byte aligned");
  const void *x = X;
  MMREC_REQUIRE(x != Y && x != Y16 && x != acc_out, MMREC_E_BADARG, "spmm_bf16: X must not alias an output");
  const bool narrow = flags & MMREC_SPMM_NARROW;
  // the width is checked before the n_tasks == 0 exit, so that a bad d never passes unnoticed
  return dispatch_width_bf16(d, narrow, [&](auto lanes, auto chunks) {
    constexpr int L = decltype(lanes)::value, C = decltype(chunks)::value;
    constexpr int GROUPS = kThreads / L;
    if (n_tasks == 0) return MMREC_OK;
    const ProblemBf16 P{row_ptr, col_idx, vals, reinterpret_cast<const int4 *>(tasks), n_tasks, slot_base, counters,
                        scratch, col_offset, X, Y, Y16, acc_in,
                        acc_out, acc_scale};
    const int blocks = (n_tasks + GROUPS - 1) / GROUPS;
    MMREC_CUDA(launch_pdl(spmm_csr_bf16_kernel<L, C>, blocks, kThreads, 0, (cudaStream_t)stream, P, d));
    MMREC_CHECK_LAUNCH("spmm_csr_bf16_kernel");
    return MMREC_OK;
  });
}

extern "C" int mmrec_spmm_csr_multi_f32(const MmrecSpmmProblem *problems_host, int32_t n_problems, int32_t d,
                                        void *stream) {
  MMREC_REQUIRE(problems_host && n_problems >= 1 && n_problems <= kMaxProblems, MMREC_E_BADARG,
                "spmm_multi: 1..%d problems", kMaxProblems);
  MultiArgs A{};
  A.n = 0;
  for (int i = 0; i < n_problems; ++i) {
    const MmrecSpmmProblem &q = problems_host[i];
    MMREC_REQUIRE(q.row_ptr && q.col_idx && q.vals && q.tasks && q.X, MMREC_E_BADARG, "spmm_multi: null input (%d)", i);
    MMREC_REQUIRE(q.Y || q.acc_out, MMREC_E_BADARG, "spmm_multi: no output requested (%d)", i);
    MMREC_REQUIRE(aligned16(q.X) && aligned16(q.Y) && aligned16(q.acc_in) && aligned16(q.acc_out) &&
                      aligned16(q.tasks) && aligned16(q.scratch), MMREC_E_ALIGN,
                  "spmm_multi: dense operands and the task list must be 16-byte aligned (%d)", i);
    MMREC_REQUIRE(q.X != q.Y && q.X != q.acc_out, MMREC_E_BADARG, "spmm_multi: X must not alias an output (%d)", i);
    if (q.n_tasks <= 0) continue;
    A.p[A.n] = Problem{q.row_ptr, q.col_idx, q.vals, reinterpret_cast<const int4 *>(q.tasks), q.n_tasks, q.slot_base,
                       q.counters, q.scratch, q.col_offset, q.X,
                       Epilogue{q.Y, q.acc_in, q.acc_out, q.acc_scale, nullptr, nullptr, nullptr}};
    ++A.n;
  }
  if (A.n == 0) return MMREC_OK;
  return dispatch_width(d, [&](auto lanes, auto chunks) {
    constexpr int L = decltype(lanes)::value, C = decltype(chunks)::value;
    constexpr int GROUPS = kThreads / L;
    int blocks = 0;
    for (int i = 0; i < A.n; ++i) {
      blocks += (A.p[i].n_tasks + GROUPS - 1) / GROUPS;
      A.block_end[i] = blocks;
    }
    MMREC_CUDA(launch_pdl(spmm_csr_multi_kernel<L, C>, blocks, kThreads, 0, (cudaStream_t)stream, A, d));
    MMREC_CHECK_LAUNCH("spmm_csr_multi_kernel");
    return MMREC_OK;
  });
}

extern "C" int mmrec_layergcn_cos_bwd_f32(const float *dE, const float *P, const float *E0,
                                          const float *W, int32_t n_rows, int32_t d, float *dP,
                                          float *dE0_accum, void *stream) {
  MMREC_REQUIRE(dE && P && E0 && W && dP && dE0_accum, MMREC_E_BADARG, "layergcn_cos_bwd: null");
  MMREC_REQUIRE(aligned16(dE) && aligned16(P) && aligned16(E0) && aligned16(dP) && aligned16(dE0_accum),
                MMREC_E_ALIGN, "layergcn_cos_bwd: operands must be 16-byte aligned");
  if (n_rows == 0) return MMREC_OK;
  return dispatch_width(d, [&](auto lanes, auto chunks) {
    constexpr int L = decltype(lanes)::value, C = decltype(chunks)::value;
    constexpr int GROUPS = kThreads / L;
    layergcn_cos_bwd_kernel<L, C><<<(n_rows + GROUPS - 1) / GROUPS, kThreads, 0, (cudaStream_t)stream>>>(
        dE, P, E0, W, n_rows, d, dP, dE0_accum);
    MMREC_CHECK_LAUNCH("layergcn_cos_bwd_kernel");
    return MMREC_OK;
  });
}
