// LightGCN's training loss (lightgcn.py:133-159: BPRLoss with gamma + EmbLoss) on any subset of a
// batch's triples -- see include/mmrec_b200.h.
//
// Forward: one warp per (user, pos, neg) triple, a fixed number of triples per warp (grid-stride
// over a grid whose size depends on the batch alone), so every partial sum is formed in the same
// order on every run and every GPU; per-CTA sums go to a small buffer that the last CTA to finish
// reduces in a fixed order. Backward: the saved per-triple derivative scales the rows, gradients
// are scatter-added with vector atomics (users / items repeat inside a batch). The four outputs are
// per-call partials: a sharded run all-reduces them, and the replicated tables never see these
// atomics after that all-reduce.
#include "common.cuh"

namespace mmrec {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxBlocks = 1024;  // fixed cap: the reduction order depends on `batch` only

__device__ __forceinline__ bool last_block_arrives(uint32_t *counter) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t prev = atomicAdd(counter, 1u);
    is_last = (prev == gridDim.x - 1);
    if (is_last) *counter = 0u;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

__device__ __forceinline__ void red_add4(float *addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

__device__ __forceinline__ float4 axpby4(float a, float4 x, float b, float4 y) {
  return make_float4(a * x.x + b * y.x, a * x.y + b * y.y, a * x.z + b * y.z, a * x.w + b * y.w);
}

// out4 = (sum -log(gamma + sigmoid(x_b)), sum |u0_b|^2, sum |p0_b|^2, sum |n0_b|^2),
// x_b = <u_b, p_b> - <u_b, n_b> on the final tables; dx[b] = d(-log(gamma + sigmoid(x)))/dx.
__global__ void __launch_bounds__(kThreads)
lightgcn_loss_fwd_kernel(const float *__restrict__ uo, const float *__restrict__ io, const float *__restrict__ ue,
                         const float *__restrict__ ie, int d, const int64_t *__restrict__ users,
                         const int64_t *__restrict__ pos, const int64_t *__restrict__ neg, int batch, float gamma,
                         float *__restrict__ out4, float *__restrict__ dx, float *__restrict__ partial,
                         uint32_t *counter) {
  __shared__ float red[4][kWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int b = blockIdx.x * kWarps + warp; b < batch; b += gridDim.x * kWarps) {
    const size_t ou = (size_t)users[b] * d, op = (size_t)pos[b] * d, on = (size_t)neg[b] * d;
    float sp = 0.f, sn = 0.f, qu = 0.f, qp = 0.f, qn = 0.f;
    for (int c = lane * 4; c < d; c += 128) {
      const float4 a = ldg4(uo + ou + c), x = ldg4(io + op + c), y = ldg4(io + on + c);
      const float4 a0 = ldg4(ue + ou + c), x0 = ldg4(ie + op + c), y0 = ldg4(ie + on + c);
      sp += dot4(a, x);
      sn += dot4(a, y);
      qu += dot4(a0, a0);
      qp += dot4(x0, x0);
      qn += dot4(y0, y0);
    }
    sp = warp_sum(sp);
    sn = warp_sum(sn);
    qu = warp_sum(qu);
    qp = warp_sum(qp);
    qn = warp_sum(qn);
    const float x = sp - sn;
    // sigmoid(x) and 1 - sigmoid(x) without cancellation
    const float e = expf(-fabsf(x));
    const float big = 1.f / (1.f + e), small = e / (1.f + e);
    const float s = x >= 0.f ? big : small, s1 = x >= 0.f ? small : big;
    const float t = gamma + s;
    if (lane == 0) dx[b] = -s * s1 / t;
    acc[0] += -logf(t);
    acc[1] += qu;
    acc[2] += qp;
    acc[3] += qn;
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 4; ++k) red[k][warp] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    for (int w = 0; w < kWarps; ++w) s += red[threadIdx.x][w];
    partial[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = s;
  }
  if (last_block_arrives(counter)) {
    // thread k sums partial k over the CTAs, in CTA order
    if (threadIdx.x < 4) {
      float s = 0.f;
      for (int i = 0; i < (int)gridDim.x; ++i) s += __ldcg(partial + (size_t)threadIdx.x * gridDim.x + i);
      out4[threadIdx.x] = s;
    }
  }
}

// coef4 = (c_bpr, c_u, c_p, c_n): dL/d(loss sum) and dL/d|U|^2-style reg coefficients (device scalars).
__global__ void __launch_bounds__(kThreads)
lightgcn_loss_bwd_kernel(const float *__restrict__ uo, const float *__restrict__ io, const float *__restrict__ ue,
                         const float *__restrict__ ie, int d, const int64_t *__restrict__ users,
                         const int64_t *__restrict__ pos, const int64_t *__restrict__ neg, int batch,
                         const float *__restrict__ dx, const float *__restrict__ coef4, float *__restrict__ d_uo,
                         float *__restrict__ d_io, float *__restrict__ d_ue, float *__restrict__ d_ie) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kWarps + warp;
  if (b >= batch) return;
  const float s = coef4[0] * dx[b], cu = coef4[1], cp = coef4[2], cn = coef4[3];
  const size_t ou = (size_t)users[b] * d, op = (size_t)pos[b] * d, on = (size_t)neg[b] * d;
  for (int c = lane * 4; c < d; c += 128) {
    const float4 a = ldg4(uo + ou + c), x = ldg4(io + op + c), y = ldg4(io + on + c);
    red_add4(d_uo + ou + c, axpby4(s, x, -s, y));
    red_add4(d_io + op + c, axpby4(s, a, 0.f, a));
    red_add4(d_io + on + c, axpby4(-s, a, 0.f, a));
    const float4 a0 = ldg4(ue + ou + c), x0 = ldg4(ie + op + c), y0 = ldg4(ie + on + c);
    red_add4(d_ue + ou + c, axpby4(cu, a0, 0.f, a0));
    red_add4(d_ie + op + c, axpby4(cp, x0, 0.f, x0));
    red_add4(d_ie + on + c, axpby4(cn, y0, 0.f, y0));
  }
}

int fwd_blocks(int batch) { return batch <= 0 ? 1 : std::min(kMaxBlocks, (batch + kWarps - 1) / kWarps); }

}  // namespace
}  // namespace mmrec

using namespace mmrec;

extern "C" size_t mmrec_lightgcn_loss_fwd_workspace_floats(int32_t batch) { return 4 * (size_t)fwd_blocks(batch); }

extern "C" int mmrec_lightgcn_loss_fwd_f32(const float *user_out, const float *item_out, const float *user_ego,
                                           const float *item_ego, int32_t d, const int64_t *users, const int64_t *pos,
                                           const int64_t *neg, int32_t batch, float gamma, float *out4, float *dx,
                                           float *partial, uint32_t *counter, void *stream) {
  MMREC_REQUIRE(out4 && partial && counter, MMREC_E_BADARG, "lightgcn_loss_fwd: null pointer");
  MMREC_REQUIRE(batch >= 0 && d > 0 && d % 4 == 0, MMREC_E_BADARG,
                "lightgcn_loss_fwd: need batch >= 0 and d %% 4 == 0 (batch=%d, d=%d)", batch, d);
  if (batch > 0) {
    MMREC_REQUIRE(user_out && item_out && user_ego && item_ego && users && pos && neg && dx, MMREC_E_BADARG,
                  "lightgcn_loss_fwd: null pointer");
    MMREC_REQUIRE(aligned16(user_out) && aligned16(item_out) && aligned16(user_ego) && aligned16(item_ego),
                  MMREC_E_ALIGN, "lightgcn_loss_fwd: tables must be 16-byte aligned");
  }
  // batch 0: one CTA writes four zeros (the call still contributes to a cross-rank reduction)
  lightgcn_loss_fwd_kernel<<<fwd_blocks(batch), kThreads, 0, (cudaStream_t)stream>>>(
      user_out, item_out, user_ego, item_ego, d, users, pos, neg, batch, gamma, out4, dx, partial, counter);
  MMREC_CHECK_LAUNCH("lightgcn_loss_fwd_kernel");
  return MMREC_OK;
}

extern "C" int mmrec_lightgcn_loss_bwd_f32(const float *user_out, const float *item_out, const float *user_ego,
                                           const float *item_ego, int32_t d, const int64_t *users, const int64_t *pos,
                                           const int64_t *neg, int32_t batch, const float *dx, const float *coef4,
                                           float *d_user_out, float *d_item_out, float *d_user_ego, float *d_item_ego,
                                           void *stream) {
  MMREC_REQUIRE(batch >= 0 && d > 0 && d % 4 == 0, MMREC_E_BADARG,
                "lightgcn_loss_bwd: need batch >= 0 and d %% 4 == 0 (batch=%d, d=%d)", batch, d);
  if (batch == 0) return MMREC_OK;
  MMREC_REQUIRE(user_out && item_out && user_ego && item_ego && users && pos && neg && dx && coef4 && d_user_out &&
                    d_item_out && d_user_ego && d_item_ego,
                MMREC_E_BADARG, "lightgcn_loss_bwd: null pointer");
  MMREC_REQUIRE(aligned16(user_out) && aligned16(item_out) && aligned16(user_ego) && aligned16(item_ego) &&
                    aligned16(d_user_out) && aligned16(d_item_out) && aligned16(d_user_ego) && aligned16(d_item_ego),
                MMREC_E_ALIGN, "lightgcn_loss_bwd: tables must be 16-byte aligned");
  lightgcn_loss_bwd_kernel<<<(batch + kWarps - 1) / kWarps, kThreads, 0, (cudaStream_t)stream>>>(
      user_out, item_out, user_ego, item_ego, d, users, pos, neg, batch, dx, coef4, d_user_out, d_item_out,
      d_user_ego, d_item_ego);
  MMREC_CHECK_LAUNCH("lightgcn_loss_bwd_kernel");
  return MMREC_OK;
}
