/*
 * mmrec_b200 -- C ABI of the B200-native graph-propagation hot path.
 *
 * The reference (EXLYSHA/Recommendar-Systems, an MMRec fork) has no FFI layer: its operator
 * boundary is the set of torch call sites inside the model files. Every entry point below
 * replaces one family of those call sites (cited as path:line under /root/reference/src).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - Every pointer is a DEVICE pointer unless its name ends in _host.
 *   - Matrices are dense row-major float32 with leading dimension == number of columns.
 *   - `stream` is a cudaStream_t passed as void*. No entry point synchronises, allocates or
 *     frees device memory, so all of them can be captured in a CUDA graph.
 *   - Return value: 0 on success, a negative MMREC_E_* code otherwise; mmrec_last_error()
 *     returns a thread-local human-readable message for the last failure.
 *   - Index widths: node / item / user ids int32 on the device side of a CSR, int64 where the
 *     reference hands over LongTensors (batches, COO indices). Row pointers are int32 unless
 *     the function takes a `rowptr64` flag.
 */
#ifndef MMREC_B200_H
#define MMREC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMREC_OK 0
#define MMREC_E_BADARG (-1)     /* null pointer, negative size, unsupported embedding width */
#define MMREC_E_ALIGN (-2)      /* pointer not 16-byte aligned */
#define MMREC_E_OVERFLOW (-3)   /* index does not fit the kernel's index type */
#define MMREC_E_CUDA (-4)       /* CUDA runtime error, see mmrec_last_error() */
#define MMREC_E_WORKSPACE (-5)  /* workspace too small */

int mmrec_abi_version(void);
const char *mmrec_last_error(void);
/* Number of kernels launched by this library since load (bench.py's gpu_launches claim). */
int64_t mmrec_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Adjacency construction (K11/K12).
 * Replaces LayerGCN/FREEDOM/LightGCN.get_norm_adj_mat (models/layergcn.py:91-117,
 * models/freedom.py:102-128, models/lightgcn.py:65-103), MGCN/SMORE.get_adj_mat
 * (models/mgcn.py:109-136, models/smore.py:176-199) and the per-epoch re-normalisation in
 * pre_epoch_processing/_normalize_adj_m (models/layergcn.py:51-81, models/freedom.py:130-156).
 *
 * Builds the CSR of A_hat = D^-1/2 [[0,R],[R^T,0]] D^-1/2 (N = U + I rows, 2E non-zeros, columns
 * sorted inside each row) from E unique training edges. deg^-1/2 comes from a caller-supplied
 * look-up table indexed by degree (the caller evaluates the reference's own pow() on the host so
 * the result is bit-exact): lut_is_f64 = 1 -> value = (float)(lut[deg_r] * lut[deg_c]) with the
 * product in double (layergcn.py recipe); 0 -> float product (mgcn.py / _normalize_adj_m recipe).
 * deg_out (int32[N], optional) receives the degrees.
 * ---------------------------------------------------------------------------------------- */
size_t mmrec_ui_adj_workspace_bytes(int64_t n_edges, int32_t n_users, int32_t n_items);
int mmrec_ui_adj_build(const int64_t *users, const int64_t *items, int64_t n_edges,
                       int32_t n_users, int32_t n_items, const void *lut, int32_t lut_len,
                       int32_t lut_is_f64, int32_t *row_ptr, int32_t *col_idx, float *vals,
                       int32_t *deg_out, void *workspace, size_t workspace_bytes, void *stream);

/* Generic COO (int64 indices, possibly unsorted, duplicates kept) -> CSR with sorted columns.
 * Replaces the per-call coalesce()+COO->CSR conversion torch.sparse.mm performs on the
 * reference's uncoalesced tensors (every call site listed under mmrec_spmm_csr_f32). If
 * `transpose` is non-zero the CSR of A^T is produced (needed for the backward of the
 * non-symmetric item-item graphs, utils/utils.py:171-184). perm_out (int64[nnz], optional)
 * receives, for every CSR slot, the index of the COO entry it came from. */
size_t mmrec_csr_from_coo_workspace_bytes(int64_t nnz);
int mmrec_csr_from_coo(const int64_t *rows, const int64_t *cols, const float *vals, int64_t nnz,
                       int32_t n_rows, int32_t n_cols, int32_t transpose, int32_t *row_ptr,
                       int32_t *col_idx, float *out_vals, int64_t *perm_out, void *workspace,
                       size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * SpMM with fused layer combination (K1/K2/K3).
 * Replaces torch.sparse.mm at models/layergcn.py:133, models/freedom.py:169,174,
 * models/mgcn.py:162,172,176,180,184, models/smore.py:282,293,297,303,307,313,317,
 * models/lightgcn.py:122, the stack+mean at freedom.py:177-178 / mgcn.py:165-166 /
 * smore.py:285-286 / lightgcn.py:124-125 and the cosine refinement at layergcn.py:134-138.
 *
 *   y[r]  = sum_k vals[k] * X[col_idx[k] - col_offset]      for k in row r
 *   LayerGCN mode (cos_ref != NULL): Y_pre[r] = y (optional), w = cos(y, cos_ref[r]) with
 *       torch-2 semantics (each vector / max(norm, 1e-8)), cos_w[r] = w, y *= w
 *   Y[r]       = y                                   (optional)
 *   acc_out[r] = (acc_in[r] + y) * acc_scale  or  y * acc_scale if acc_in == NULL   (optional)
 *
 * Work list (built once per graph, see graph.py): `tasks` is int32[n_tasks][4] =
 * {row, begin, end, slot}; one sub-warp of d/4 lanes runs one task of at most 64 non-zeros.
 * slot < 0: the task covers a whole row. slot >= 0: the row is cut into ceil(deg/64) tasks;
 * partial sums go to scratch[(slot_base[slot] + part) * d ...] and the last task to arrive on
 * counters[slot] (zero-initialised, self-resetting) reduces them in part order and runs the
 * epilogue. d must be 32, 64, 128 or 256. The same entry point runs the backward (A_hat is
 * symmetric; otherwise pass the CSR of A^T).
 * ---------------------------------------------------------------------------------------- */
int mmrec_spmm_csr_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                       const int32_t *tasks, int32_t n_tasks, const int32_t *slot_base,
                       int32_t *counters, float *scratch, int32_t col_offset, const float *X,
                       int32_t d, float *Y, const float *acc_in, float *acc_out, float acc_scale,
                       const float *cos_ref, float *cos_w, float *Y_pre, void *stream);
/* The same operator with tuning flags for graphs whose operand X does not fit the 126 MB L2:
 *   MMREC_SPMM_NARROW  half the lanes per task, two 16-byte chunks per lane: twice the tasks in
 *                      flight for graphs of very short rows (the column blocks of an operand cut
 *                      into L2-sized slices);
 *   MMREC_SPMM_STREAM  L2 eviction policies: gathered X rows evict_last, everything touched once
 *                      (CSR arrays, epilogue operand, output rows) evict_first. Not with cos_ref. */
#define MMREC_SPMM_NARROW 1
#define MMREC_SPMM_STREAM 2
int mmrec_spmm_csr_ex_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                       const int32_t *tasks, int32_t n_tasks, const int32_t *slot_base,
                       int32_t *counters, float *scratch, int32_t col_offset, const float *X,
                       int32_t d, float *Y, const float *acc_in, float *acc_out, float acc_scale,
                       const float *cos_ref, float *cos_w, float *Y_pre, int32_t flags, void *stream);

/* Several independent SpMMs of the same width d in ONE launch (at most 4): the item-item and R
 * propagation of the three modality views (smore.py:291-317, mgcn.py:170-184), which are
 * independent of one another and each too small to fill the GPU. Fields as the arguments of
 * mmrec_spmm_csr_f32 (no cosine epilogue). Problems that share a graph need their own `counters`
 * and `scratch`. `problems_host` is a HOST array. */
typedef struct MmrecSpmmProblem {
  const int32_t *row_ptr, *col_idx;
  const float *vals;
  const int32_t *tasks;
  int32_t n_tasks;
  const int32_t *slot_base;
  int32_t *counters;
  float *scratch;
  int32_t col_offset;
  const float *X;
  float *Y;
  const float *acc_in;
  float *acc_out;
  float acc_scale;
} MmrecSpmmProblem;
int mmrec_spmm_csr_multi_f32(const MmrecSpmmProblem *problems_host, int32_t n_problems, int32_t d,
                             void *stream);

/* Backward row-operator of one LayerGCN layer (layergcn.py:134-135 differentiated):
 * given dE = dL/d(w*p), p = Y_pre, w = cos_w, e0 = cos_ref:
 *   dP[r]   = w*dE + <dE,p> * d cos(p,e0)/dp ;  dE0[r] += <dE,p> * d cos(p,e0)/de0        */
int mmrec_layergcn_cos_bwd_f32(const float *dE, const float *P, const float *E0, const float *W,
                               int32_t n_rows, int32_t d, float *dP, float *dE0_accum,
                               void *stream);

/* ------------------------------------------------------------------------------------------
 * BPR gather-dot loss (K6). Replaces LayerGCN.bpr_loss + emb_loss (layergcn.py:142-163),
 * FREEDOM.bpr_loss (freedom.py:182-189), MGCN/SMORE.bpr_loss (mgcn.py:210-222,
 * smore.py:366-378).
 *   x_b = <u_b, p_b> - <u_b, n_b>;   out[0] = sum_b -logsigmoid(x_b);
 *   out[1] = sum_b 0.5*(|u_b|^2 + |p_b|^2 + |n_b|^2);   sig[b] = sigmoid(-x_b)  (saved)
 * Backward: with coef[0] = dL/d out[0], coef[1] = dL/d out[1] (device scalars),
 *   d_user[u_b] += coef0*(-sig_b)*(p_b - n_b) + coef1*u_b, etc. (atomic scatter-add,
 *   duplicates allowed). partial must hold 2*B floats; counter one zero-initialised uint32.
 * ---------------------------------------------------------------------------------------- */
int mmrec_bpr_fwd_f32(const float *user_emb, const float *item_emb, int32_t d,
                      const int64_t *users, const int64_t *pos, const int64_t *neg, int32_t batch,
                      float *out2, float *sig, float *partial, uint32_t *counter, void *stream);
int mmrec_bpr_bwd_f32(const float *user_emb, const float *item_emb, int32_t d,
                      const int64_t *users, const int64_t *pos, const int64_t *neg, int32_t batch,
                      const float *sig, const float *coef2, float *d_user_emb, float *d_item_emb,
                      void *stream);

/* ------------------------------------------------------------------------------------------
 * LightGCN loss (lightgcn.py:133-159: BPRLoss with gamma + EmbLoss) on any subset of a batch's
 * triples, e.g. the triples one rank of a user-sharded run owns. `users` index the user tables
 * (shard-local rows), `pos` / `neg` the item tables; batch may be 0.
 *   x_b = <uo_b, po_b> - <uo_b, no_b>   (final tables user_out / item_out)
 *   out4 = (sum_b -log(gamma + sigmoid(x_b)), sum_b |u0_b|^2, sum_b |p0_b|^2, sum_b |n0_b|^2)
 *          (u0 / p0 / n0: rows of the ego tables user_ego / item_ego), reduced in a fixed order;
 *   dx[b] = d(-log(gamma + sigmoid(x)))/dx at x_b  (saved for the backward).
 * The caller reduces out4 (across ranks), forms the loss and the coefficients
 *   coef4 = (1/B, reg/(B |U|), reg/(B |P|), reg/(B |N|))  (device scalars; B and the norms global)
 * and the backward scatter-adds (atomics, duplicates allowed) into four zeroed outputs:
 *   d_user_out[u_b] += c0 dx_b (po_b - no_b); d_item_out[p_b] += c0 dx_b uo_b; d_item_out[n_b] -= c0 dx_b uo_b;
 *   d_user_ego[u_b] += c1 u0_b; d_item_ego[p_b] += c2 p0_b; d_item_ego[n_b] += c3 n0_b.
 * d % 4 == 0, tables 16-byte aligned; partial holds
 * mmrec_lightgcn_loss_fwd_workspace_floats(batch) floats; counter one zero-initialised uint32.
 * ---------------------------------------------------------------------------------------- */
size_t mmrec_lightgcn_loss_fwd_workspace_floats(int32_t batch);
int mmrec_lightgcn_loss_fwd_f32(const float *user_out, const float *item_out, const float *user_ego,
                                const float *item_ego, int32_t d, const int64_t *users, const int64_t *pos,
                                const int64_t *neg, int32_t batch, float gamma, float *out4, float *dx,
                                float *partial, uint32_t *counter, void *stream);
int mmrec_lightgcn_loss_bwd_f32(const float *user_out, const float *item_out, const float *user_ego,
                                const float *item_ego, int32_t d, const int64_t *users, const int64_t *pos,
                                const int64_t *neg, int32_t batch, const float *dx, const float *coef4,
                                float *d_user_out, float *d_item_out, float *d_user_ego, float *d_item_ego,
                                void *stream);

/* ------------------------------------------------------------------------------------------
 * InfoNCE (K7). Replaces MGCN/SMORE.InfoNCE (mgcn.py:224-231, smore.py:380-387).
 *   v1 = normalize(T1[idx]), v2 = normalize(T2[idx]) (F.normalize, eps 1e-12)
 *   loss = mean_i( -log( exp(<v1_i,v2_i>/t) / sum_j exp(<v1_i,v2_j>/t) ) )
 * The B x B score matrix never reaches HBM. fwd saves V1n,V2n [B,d], inv norms [2B], ttl [B].
 * bwd scatter-adds into dT1/dT2 (table-shaped, atomics). coef = dL/dloss (device scalar).
 * The "other" dimension of each backward pass is cut into n_splits ranges (grid.y) so that a
 * 2048-row batch fills 148 SMs; dV1_ws/dV2_ws hold n_splits*batch*d floats of partial sums that
 * the scatter kernel adds in split order; mmrec_infonce_splits(batch) is the count that fills
 * the GPU (4 co-resident CTAs per SM). partial (fwd) must hold
 * mmrec_infonce_fwd_workspace_floats(batch) floats; counter is an array of 1 + ceil(batch/64)
 * zero-initialised uint32 (self-resetting); batch <= 65472.
 * ---------------------------------------------------------------------------------------- */
int32_t mmrec_infonce_splits(int32_t batch);
size_t mmrec_infonce_fwd_workspace_floats(int32_t batch);
int mmrec_infonce_fwd_f32(const float *T1, const float *T2, int32_t d, const int64_t *idx,
                          int32_t batch, float inv_temp, float *loss_out, float *V1n, float *V2n,
                          float *inv_norm, float *ttl, float *partial, uint32_t *counter,
                          void *stream);
int mmrec_infonce_bwd_f32(const float *V1n, const float *V2n, const float *inv_norm,
                          const float *ttl, int32_t d, const int64_t *idx, int32_t batch,
                          float inv_temp, const float *coef, int32_t n_splits, float *dV1_ws,
                          float *dV2_ws, float *dT1, float *dT2, void *stream);
/* The item-row and user-row InfoNCE problems of a batch (mgcn.py:250-251, smore.py:406-407: same
 * batch size, same d) in ONE launch per stage. Every pointer argument is a HOST array of two device
 * pointers; partial / workspaces are sized per problem exactly as for the single-problem calls.
 * Available where mmrec_infonce_pair_supported(d) != 0 (d = 64: the tcgen05 kernels). */
int mmrec_infonce_pair_supported(int32_t d);
int mmrec_infonce_pair_fwd_f32(const float *const *T1_host, const float *const *T2_host, int32_t d,
                               const int64_t *const *idx_host, int32_t batch, float inv_temp,
                               float *const *loss_out_host, float *const *V1n_host, float *const *V2n_host,
                               float *const *inv_norm_host, float *const *ttl_host, float *const *partial_host,
                               void *stream);
int mmrec_infonce_pair_bwd_f32(const float *const *V1n_host, const float *const *V2n_host,
                               const float *const *inv_norm_host, const float *const *ttl_host, int32_t d,
                               const int64_t *const *idx_host, int32_t batch, float inv_temp,
                               const float *const *coef_host, int32_t n_splits, float *const *dV1_ws_host,
                               float *const *dV2_ws_host, float *const *dT1_host, float *const *dT2_host,
                               void *stream);

/* ------------------------------------------------------------------------------------------
 * Spectrum-based modality fusion (K5). Replaces SMORE.spectrum_convolution
 * (models/smore.py:209-238): rfft -> complex filter (unit-magnitude normalised when
 * weight_norm) -> irfft for image and text, and irfft(rfft(t)*rfft(v)*w_f) for the fusion
 * view, norm='ortho'. Implemented as the equivalent real circulant operators (SURVEY K5).
 * w_* are the raw parameters [d/2+1, 2]. d in {32, 64, 128}. taps_ws: 3*d floats, receives the
 * real impulse responses h = irfft(w_hat) of the three filters (reused by the backward).
 * Backward produces dImg, dTxt and the gradients of the three raw weights ([d/2+1,2] each,
 * overwritten). dh_ws: 3*d floats, zero-initialised by the caller (tap gradients are
 * accumulated there with atomics, then chained through irfft and the unit-magnitude map).
 * ---------------------------------------------------------------------------------------- */
int mmrec_spectral_fwd_f32(const float *img, const float *txt, int32_t n_rows, int32_t d,
                           const float *w_img, const float *w_txt, const float *w_fus,
                           int32_t weight_norm, float *taps_ws, float *img_conv, float *txt_conv,
                           float *fus_conv, void *stream);
int mmrec_spectral_bwd_f32(const float *img, const float *txt, int32_t n_rows, int32_t d,
                           const float *w_img, const float *w_txt, const float *w_fus,
                           int32_t weight_norm, const float *taps_ws, const float *g_img_conv,
                           const float *g_txt_conv, const float *g_fus_conv, float *d_img,
                           float *d_txt, float *dh_ws, float *d_w_img, float *d_w_txt,
                           float *d_w_fus, void *stream);

/* ------------------------------------------------------------------------------------------
 * Dense projections (K4): fp32-accurate tensor-core GEMM (3xTF32 split, fp32 accumulate).
 * Replaces nn.Linear / F.linear over whole tables and its two backward GEMMs:
 * image_trs / text_trs (smore.py:257-259, mgcn.py:148-150, freedom.py:207-210) and the d x d
 * gate / query layers (smore.py:265-272, 321-330; mgcn.py:153-154, 188-203).
 *   C[M,N] = op(A) * op(B) (+ bias[N])
 *   a_kcontig = 1: A is [M,K] row-major;  0: A is stored [K,M] row-major (A^T of a [K,M] array)
 *   b_kcontig = 1: B is [N,K] row-major;  0: B is stored [K,N] row-major
 * forward  y = x W^T + b : (A=x, 1), (B=W, 1);  dW = dy^T x : (A=dy, 0), (B=x, 0);
 * dx = dy W : (A=dy, 1), (B=W, 0). (A M-contiguous with B K-contiguous is not provided.)
 * splits > 1 cuts K over grid.z; ws must then hold splits*M*N floats (summed in split order).
 * N and the contiguous dimensions must be multiples of 4. mmrec_gemm_splits suggests `splits`.
 * ---------------------------------------------------------------------------------------- */
int mmrec_gemm_splits(int32_t M, int32_t N, int32_t K, int32_t a_kcontig, int32_t b_kcontig);
int mmrec_gemm_tf32x3_f32(const float *A, int32_t a_kcontig, const float *B, int32_t b_kcontig,
                          const float *bias, float *C, int32_t M, int32_t N, int32_t K,
                          int32_t splits, float *ws, void *stream);

/* ------------------------------------------------------------------------------------------
 * d x d dense layers of the modality side networks with fused bias + activation (K4b):
 * gate_v/gate_t/gate_f, query_v/query_t, gate_*_prefer (smore.py:265-272, 321-330) and the MGCN
 * gates / query_common (mgcn.py:153-154, 188-203), i.e. nn.Sequential(nn.Linear(d, d), nn.Tanh() |
 * nn.Sigmoid()) and bare nn.Linear(d, d). X [M,K], W [N,K] row-major, K = N in {32, 64, 128}.
 *   act: 0 = identity, 1 = tanh, 2 = sigmoid
 *   fwd: Y = act(X W^T + bias)                         (bias may be NULL)
 *   bwd: dZ = dY * act'(Y); dX = dZ W (skipped if dX NULL); dW = dZ^T X; db = sum_rows dZ (if db)
 * Tile products on mma.sync tensor cores with the 3xTF32 split (fp32-class accuracy, ~1e-7).
 * The backward needs mmrec_dense_act_bwd_workspace_bytes of scratch; per-CTA partial sums of
 * dW/db are added in a fixed order (bit-reproducible).
 * ---------------------------------------------------------------------------------------- */
/* act(x W^T + b) for x [M, K] with MANY rows on the tcgen05 GEMM (bias and tanh / sigmoid in its
 * store epilogue): the 128 x 128 layers of the side network and gates at d = 128 (SMORE on the
 * Clothing-shaped data: 62k node rows; smore.py:265-272, 321-330), where the mma.sync tile kernels
 * behind mmrec_dense_act_* run at a tenth of it. act: 0 none, 1 tanh, 2 sigmoid.
 * Backward: dz = mmrec_act_bwd_f32(dy, y) (dy * act'(y)), then dx = dz W, dW = dz^T x on
 * mmrec_gemm_tf32x3_f32 (tcgen05 for these shapes) and db = mmrec_colsum_f32(dz). */
int mmrec_linear_act_tc_supported(int32_t M, int32_t K, int32_t N);
int mmrec_linear_act_tc_f32(const float *x, const float *W, const float *b, float *y, int32_t M, int32_t K, int32_t N,
                            int32_t act, void *stream);
int mmrec_act_bwd_f32(const float *dy, const float *y, int64_t numel, int32_t act, float *dz, void *stream);
/* The activation forms every fused kernel uses (nn.Tanh / nn.Sigmoid / the exp of nn.Softmax on the
 * special-function unit, csrc/common.cuh), elementwise, for the accuracy tests:
 * act 1 tanh, 2 sigmoid, 3 exp. */
int mmrec_activation_f32(const float *x, int64_t numel, int32_t act, float *y, void *stream);
int mmrec_dense_act_supported(int32_t K, int32_t N);
size_t mmrec_dense_act_bwd_workspace_bytes(int32_t K, int32_t N);
int mmrec_dense_act_fwd_f32(const float *X, const float *W, const float *bias, float *Y, int32_t M,
                            int32_t K, int32_t N, int32_t act, void *stream);
int mmrec_dense_act_bwd_f32(const float *dY, const float *Y, const float *X, const float *W,
                            float *dX, float *dW, float *db, float *ws, int32_t M, int32_t K,
                            int32_t N, int32_t act, void *stream);
/* The same two operations for n_batch <= 4 independent layers of one shape and activation in one
 * launch each (SMORE's gate_v / gate_t / gate_f, smore.py:269-272; MGCN's gates mgcn.py:153-154).
 * Pointer arrays are HOST arrays of n_batch device pointers (bias / dX / db entries may be NULL);
 * ws holds n_batch * mmrec_dense_act_bwd_workspace_bytes(K, N) bytes. */
int mmrec_dense_act_batch_fwd_f32(const float *const *X_host, const float *const *W_host,
                                  const float *const *bias_host, float *const *Y_host, int32_t n_batch,
                                  int32_t M, int32_t K, int32_t N, int32_t act, void *stream);
int mmrec_dense_act_batch_bwd_f32(const float *const *dY_host, const float *const *Y_host,
                                  const float *const *X_host, const float *const *W_host,
                                  float *const *dX_host, float *const *dW_host, float *const *db_host,
                                  float *ws, int32_t n_batch, int32_t M, int32_t K, int32_t N, int32_t act,
                                  void *stream);

/* ------------------------------------------------------------------------------------------
 * SMORE modality-aware preference module, fused (K14). Replaces smore.py:321-341 -- query_v /
 * query_t (Linear, Tanh, Linear), nn.Softmax(dim=-1), the three gate_*_prefer (Linear, Sigmoid),
 * nn.Dropout on each gate, the products, torch.stack + torch.mean and `content + side` -- and the
 * whole autograd graph under it, by one forward and one backward launch (+ a partial-sum reduce).
 *   F = fusion_embeds, V = image_embeds, T = text_embeds, C = content_embeds: [n, d], d in {32, 64, 128}
 *   W_host / b_host: HOST arrays of 7 device pointers, order
 *       query_v.0, query_v.2, query_t.0, query_t.2, gate_image_prefer.0, gate_text_prefer.0,
 *       gate_fusion_prefer.0   (each [d, d] row-major as nn.Linear stores it; b NULL = no bias)
 *   masks: [3, n, d] dropout multipliers (0 or 1/(1-p)) for the image / text / fusion gate, or
 *          NULL (eval, p = 0)
 *   saved: [7, n, d] written by fwd, read by bwd (tanh outputs, softmax outputs, gate sigmoids);
 *          NULL in fwd = inference (full_sort_predict under no_grad): nothing is kept
 *   fwd -> side [n, d] (smore.py:339-340) and all = C + side (smore.py:341)
 *   bwd <- d_all, d_side (either may be NULL) -> dF, dV, dT, dC (dC includes d_all), dW[7], db[7]
 *          (db entries may be NULL); ws = mmrec_smore_side_bwd_workspace_bytes(n, d) of scratch.
 * Tile products on mma.sync tensor cores with the 3xTF32 split (fp32-class accuracy); gradients are
 * bit-reproducible (partials added in a fixed order).
 * ---------------------------------------------------------------------------------------- */
/* In-kernel nn.Dropout (smore.py:331-333) for the *_drop_* entry points: no mask tensor exists.
 * The multiplier of element (plane g of 3, row, column) is 0 or 1/(1-p), a pure function of
 * (seed, *counter, g, row, column): forward and backward regenerate the same mask, and a step
 * captured in a CUDA graph draws fresh masks on every replay because `counter` is read on the
 * device (FusedAdam's update count; NULL = 0). p is applied in steps of 2^-16.
 * mmrec_dropout_mask_f32 materialises the multipliers a *_drop_* call uses (tests, diagnostics);
 * oracle/dropout.py restates the generator in numpy. */
typedef struct MmrecDropout {
  float p;                /* drop probability in [0, 1) */
  uint64_t seed;          /* host constant of this call site / call */
  const double *counter;  /* device pointer to one double holding an integer count, or NULL */
  /* Batch-row calls (the module evaluated on rows gathered by mmrec_gather_batch_rows_f32): row m of the
   * call draws the multipliers of row row_ids[m] (device, int64) of a dense [n_total, d] call, so the
   * compact and the dense evaluation drop the same elements. NULL / 0 = identity. */
  const int64_t *row_ids;
  int32_t n_total;
} MmrecDropout;
int mmrec_dropout_mask_f32(float *out, int32_t planes, int32_t n, int32_t d, const MmrecDropout *drop, void *stream);

/* Batch rows of node tables around a row-local module (the preference module above; smore.py:395-407
 * consumes only ua[users], ia[pos], ia[neg], side / content [users], [pos] of it). Row m of the compact
 * tables is users[m] (m < B), n_users + pos[m - B], n_users + neg[m - 2 B]: gather copies those rows of
 * up to 4 tables [*, d] into [3 B, d] tables and writes the row ids (int64 [3 B]: the `row_ids` of
 * MmrecDropout and the index of the scatter); scatter_add adds [n_rows, d] gradient tables into dense,
 * ZEROED tables at those ids (rows repeat in a batch: vector reductions, order not fixed -- like the BPR
 * scatter). A NULL source table is skipped. Replaces nothing in the reference: it computes all rows. */
int mmrec_gather_batch_rows_f32(const float *const *src_host, int32_t n_tables, const int64_t *users,
                                const int64_t *pos, const int64_t *neg, int32_t batch, int32_t n_users, int32_t d,
                                float *const *dst_host, int64_t *idx_out, void *stream);
int mmrec_scatter_batch_rows_add_f32(const float *const *dsrc_host, int32_t n_tables, const int64_t *idx,
                                     int32_t n_rows, int32_t d, float *const *ddst_host, void *stream);

/* The same for the modality views cat([R x', x']) of smore.py:289-317 / mgcn.py:170-184: compact row m < B
 * is row users[m] of R (CSR of the users x items block; col_idx - col_offset = item) times the item tables
 * x'_v [I, d] (1..3 views in one pass over the row), rows B .. 3 B - 1 are the item rows pos / neg of x'_v; the
 * content table [U + I, d] (may be NULL) is gathered alongside. This replaces the user-side SpMM of the views
 * (torch.sparse.mm(self.R, x)) and its R^T backward in TRAINING, where only the batch rows are consumed.
 * scatter_add: the gradients of the compact views / content added into ZEROED dense item tables [I, d] /
 * [U + I, d] along the same non-zeros (vector reductions). d in {32, 64, 128}. */
int mmrec_gather_batch_views_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals, int32_t col_offset,
                                 const float *const *item_tables_host, int32_t n_views, const float *content,
                                 const int64_t *users, const int64_t *pos, const int64_t *neg, int32_t batch,
                                 int32_t n_users, int32_t d, float *const *views_out_host, float *content_out,
                                 int64_t *idx_out, void *stream);
int mmrec_scatter_batch_views_add_f32(const int32_t *row_ptr, const int32_t *col_idx, const float *vals,
                                      int32_t col_offset, const float *const *d_views_host, int32_t n_views,
                                      const float *d_content, const int64_t *users, const int64_t *pos,
                                      const int64_t *neg, int32_t batch, int32_t n_users, int32_t d,
                                      float *const *d_item_tables_host, float *d_content_out, void *stream);

int mmrec_smore_side_supported(int32_t d);
size_t mmrec_smore_side_bwd_workspace_bytes(int32_t n, int32_t d);
int mmrec_smore_side_fwd_drop_f32(const float *F, const float *V, const float *T, const float *C,
                                  const float *const *W_host, const float *const *b_host,
                                  const MmrecDropout *drop, float *saved, float *side, float *all, int32_t n,
                                  int32_t d, void *stream);
/* The forward on the 5th-generation tensor cores (tcgen05 + TMEM, d = 64, no mask tensor: in-kernel
 * dropout or none): same outputs as mmrec_smore_side_fwd_drop_f32 to fp32 rounding. `ws` = scratch of
 * mmrec_smore_side_fwd_tc_workspace_bytes(n, d) bytes, 1024-byte aligned (the pre-split weight images);
 * that function returns 0 when this path does not cover d (or under MMREC_SIDE_TC=0, which keeps the
 * mma.sync forward: the A/B switch of the tests and of profiles/r02_side_tc.txt). */
size_t mmrec_smore_side_fwd_tc_workspace_bytes(int32_t n, int32_t d);
int mmrec_smore_side_fwd_tc_f32(const float *F, const float *V, const float *T, const float *C,
                                const float *const *W_host, const float *const *b_host,
                                const MmrecDropout *drop, float *saved, float *side, float *all, int32_t n,
                                int32_t d, void *ws, void *stream);
int mmrec_smore_side_bwd_drop_f32(const float *d_all, const float *d_side, const float *F, const float *V,
                                  const float *T, const float *C, const float *const *W_host,
                                  const float *const *b_host, const MmrecDropout *drop, const float *saved,
                                  float *dF, float *dV, float *dT, float *dC, float *const *dW_host,
                                  float *const *db_host, float *ws, int32_t n, int32_t d, void *stream);
int mmrec_smore_side_fwd_f32(const float *F, const float *V, const float *T, const float *C,
                             const float *const *W_host, const float *const *b_host,
                             const float *masks, float *saved, float *side, float *all, int32_t n,
                             int32_t d, void *stream);
int mmrec_smore_side_bwd_f32(const float *d_all, const float *d_side, const float *F, const float *V,
                             const float *T, const float *C, const float *const *W_host,
                             const float *const *b_host, const float *masks, const float *saved,
                             float *dF, float *dV, float *dT, float *dC, float *const *dW_host,
                             float *const *db_host, float *ws, int32_t n, int32_t d, void *stream);

/* ------------------------------------------------------------------------------------------
 * Fused multi-tensor Adam (K13). Replaces optim.Adam.step (common/trainer.py:126-143, 255, 331)
 * with one pass: 28 bytes per parameter. The four pointer arrays and numel are HOST arrays of
 * n_tensors device pointers / element counts (they travel as kernel arguments). hyper is a
 * DEVICE array of two doubles: hyper[0] = learning rate, hyper[1] = update count; the call
 * increments hyper[1] and uses it for the bias corrections, so a captured CUDA graph replays
 * with the right step and a host-updated learning rate. Same formulas as torch's Adam.
 * grad_scale multiplies every gradient as it is read (fp32; pass 1.0): the mirror-gradient step
 * uses -mg_beta (trainer.py:325-331) instead of a separate pass over all gradients.
 * ---------------------------------------------------------------------------------------- */
int mmrec_adam_step_f32(float *const *params_host, const float *const *grads_host,
                        float *const *exp_avg_host, float *const *exp_avg_sq_host,
                        const int64_t *numel_host, int32_t n_tensors, double *hyper, double beta1,
                        double beta2, double eps, double weight_decay, double grad_scale,
                        const float *const *undo_host, const float *undo_coef, int32_t tick, void *stream);
/* tick = 1: increment the update count hyper[1] first (the normal case); 0 when another entry point
 * of the same optimizer step (mmrec_table_adam_lowrank_f32, mmrec_adam_tick) already has. */
int mmrec_adam_tick(double *hyper, void *stream);
/* undo_host / undo_coef (both NULL, or n_tensors device pointers + a device scalar): every
 * parameter is first moved by p += undo_coef[0] * undo_t, the return from the mirror point
 * theta - c*g to theta (trainer.py:322-329), in the same pass that applies the update.
 *
 * mmrec_mirror_coef_f32 -- the step size of the mirror-gradient perturbation (trainer.py:289-305):
 *   alpha_eff = clamp(target_rel_step * rms(theta) / (lr * rms(g) + 1e-12), alpha_base,
 *                     alpha_base * alpha_max_scale),  rms over all numel_total elements,
 *   coef_out[0] = alpha_eff * lr (device float, feeds mmrec_axpy_multi_f32 / undo_coef),
 *   coef_out[1] = alpha_eff. One pass over parameters and gradients + a fixed-order final sum. */
size_t mmrec_mirror_coef_workspace_bytes(const int64_t *numel_host, int32_t n_tensors);
int mmrec_mirror_coef_f32(const float *const *params_host, const float *const *grads_host,
                          const int64_t *numel_host, int32_t n_tensors, const double *hyper,
                          double numel_total, double alpha_base, double alpha_max_scale,
                          double target_rel_step, const double *extra, int32_t n_extra_p2,
                          int32_t n_extra_g2, void *workspace, float *coef_out, void *stream);
/* extra (device doubles, may be NULL with both counts 0): extra[0 .. n_extra_p2) are added to
 * sum theta^2 and extra[n_extra_p2 .. n_extra_p2 + n_extra_g2) to sum g^2 -- the contributions of
 * tensors whose gradient is a never-materialised low-rank product (below); numel_total counts
 * their elements too.
 *
 * ------------------------------------------------------------------------------------------
 * Feature tables with a rank-d gradient. The trainable image / text tables X [I, F] (F = 4096 /
 * 384; smore.py:76-77, mgcn.py:62-72, freedom.py:48-55) enter the model only through
 * Y = X W^T + b (smore.py:257-259), so their gradient is G = dY W with dY [I, d], W [d, F]: a
 * 115 MB tensor that torch writes in the backward and re-reads in every optimizer / mirror-gradient
 * pass (trainer.py:268-335). It is never materialised here: tcgen05 computes each 128 x 64 tile of
 * G (3xTF32, the products of the dX GEMM of mmrec_gemm_tf32x3_f32) into TMEM and the epilogue
 * consumes it on the spot.
 *   mmrec_table_adam_lowrank_f32: optim.Adam.step on X with g = grad_scale * (dY W): reads and
 *     writes X / exp_avg / exp_avg_sq once (24 B per element instead of 28 + the 4 of writing G).
 *     Must be enqueued BEFORE the Adam update of W itself. tick as in mmrec_adam_step_f32.
 *     sumsq_out (device double or NULL) receives sum X'^2 of the updated table.
 *   mmrec_table_lowrank_sumsq_f64: out = ||dY W||_F^2 (for mmrec_mirror_coef_f32's `extra`).
 * cols % 64 == 0, d in {32, 64, 128}, 16-byte aligned rows; workspace of
 * mmrec_table_lowrank_workspace_bytes(rows, cols) bytes.
 * ---------------------------------------------------------------------------------------- */
int mmrec_table_lowrank_supported(int32_t rows, int32_t cols, int32_t d);
size_t mmrec_table_lowrank_workspace_bytes(int32_t rows, int32_t cols);
int mmrec_table_adam_lowrank_f32(float *table, float *exp_avg, float *exp_avg_sq, const float *dY,
                                 const float *W, int32_t rows, int32_t cols, int32_t d, double *hyper,
                                 double beta1, double beta2, double eps, double weight_decay,
                                 double grad_scale, int32_t tick, double *sumsq_out, void *workspace,
                                 void *stream);
int mmrec_table_lowrank_sumsq_f64(const float *dY, const float *W, int32_t rows, int32_t cols, int32_t d,
                                  void *workspace, double *out, void *stream);
/* y_t += sign * coef[0] * x_t for n_tensors tensors in one launch; coef is a device scalar
 * (the mirror-gradient perturbation theta -/+ alpha_eff*lr*g of trainer.py:307-329 without a
 * host round trip for alpha_eff). */
int mmrec_axpy_multi_f32(float *const *y_host, const float *const *x_host, const int64_t *numel_host,
                         int32_t n_tensors, const float *coef, float sign, void *stream);

/* ------------------------------------------------------------------------------------------
 * Full-rank scoring fused with train-item masking and per-user top-K (K8/K9/K10).
 * Replaces `scores = u @ item_e.T` (layergcn.py:187, freedom.py:221, mgcn.py:262,
 * smore.py:421), `scores[mask] = -1e10` (common/trainer.py:522-524) and
 * torch.topk(scores, max(topk)) (trainer.py:526). Scores never reach HBM.
 *   users[b] selects the row of user_emb; items are item_emb[0..n_items) with global ids
 *   item_offset + j (item-sharded evaluation); mask_rowptr[b]..mask_rowptr[b+1] index
 *   mask_cols (global item ids, ascending inside each user). Tie rule: lower id first.
 * Produces `n_splits` partial lists per user (item range split across CTAs) in ws_val/ws_idx
 * ([n_splits, n_users, k]) and merges them into out_val/out_idx ([n_users, k], ids int64).
 * ---------------------------------------------------------------------------------------- */
int mmrec_score_mask_topk_f32(const float *user_emb, const int64_t *users, int32_t n_users,
                              const float *item_emb, int32_t n_items, int32_t item_offset,
                              int32_t d, const int32_t *mask_rowptr, const int32_t *mask_cols,
                              int32_t k, int32_t n_splits, float *ws_val, int32_t *ws_idx,
                              float *out_val, int64_t *out_idx, void *stream);
/* The same contract on the CUDA-core (fp32 FMA) kernel: K too large for the shared-memory heaps of
 * the tensor-core tiling, and the A/B baseline. mmrec_score_mask_topk_f32 runs the tcgen05 kernel
 * (3xTF32 split, fp32-accurate; d = 128 with the user tile in TMEM) for d = 32 / 64 / 128 and this
 * one otherwise. */
int mmrec_score_mask_topk_simt_f32(const float *user_emb, const int64_t *users, int32_t n_users,
                                   const float *item_emb, int32_t n_items, int32_t item_offset,
                                   int32_t d, const int32_t *mask_rowptr, const int32_t *mask_cols,
                                   int32_t k, int32_t n_splits, float *ws_val, int32_t *ws_idx,
                                   float *out_val, int64_t *out_idx, void *stream);
/* mmrec_score_mask_topk_f32 with the mask row of entry b looked up by user id: mask_rowptr[users[b]]
 * ..mask_rowptr[users[b] + 1] index mask_cols, i.e. the mask is a CSR over the rows of user_emb
 * (for instance a rank's training CSR in user-sharded evaluation) instead of a per-batch CSR.
 * Same kernels (tcgen05 for d = 32 / 64 / 128 where K fits, CUDA cores otherwise), same output. */
int mmrec_score_mask_topk_rows_f32(const float *user_emb, const int64_t *users, int32_t n_users,
                                   const float *item_emb, int32_t n_items, int32_t item_offset,
                                   int32_t d, const int32_t *mask_rowptr, const int32_t *mask_cols,
                                   int32_t k, int32_t n_splits, float *ws_val, int32_t *ws_idx,
                                   float *out_val, int64_t *out_idx, void *stream);
/* ----------------------------------------------------------------------------------------
 * a5 -- item-item kNN modality graphs: build_sim / build_knn_normalized_graph /
 * get_sparse_laplacian (utils/utils.py:134-137, 171-184, 139-152) and FREEDOM.get_knn_adj_mat /
 * compute_normalized_laplacian (freedom.py:79-100).
 *   mmrec_row_normalize_f32: out[r] = x[r] / ||x[r]||_2 (utils.py:135, freedom.py:80); the cosine
 *     matrix itself is mmrec_gemm_tf32x3_f32(out, out^T).
 *   mmrec_row_topk_f32: replaces torch.topk(sim, k, dim=-1) (utils.py:172, freedom.py:81) on a
 *     dense [n_rows, ld] matrix (first n_cols columns): values / int32 columns [n_rows, k],
 *     descending, ties -> lower column (torch's tie order is unspecified); NaNs are never picked.
 *   mmrec_knn_weights_f32: edge weights of the [n, k] neighbour lists.
 *     mode 0 (MGCN / SMORE, utils.py:139-152): deg[r] = sum_j w[r][j] (row sums on BOTH sides, so the
 *       result is not symmetric), out = deg[r]^-1/2 * w * deg[c]^-1/2 with inf -> 0; dis_ws [n].
 *     mode 1 (FREEDOM, freedom.py:87-100): binary edges, out = ((k + 1e-7)^-1/2)^2 in float32.
 * ---------------------------------------------------------------------------------------- */
int mmrec_row_normalize_f32(const float *x, int32_t n_rows, int32_t d, float *out, void *stream);
int mmrec_row_topk_f32(const float *mat, int32_t n_rows, int32_t n_cols, int64_t ld, int32_t k, float *out_val,
                       int32_t *out_idx, void *stream);
/* out[N] = column sums of the row-major [M, N] matrix x (N % 4 == 0): the bias gradient
 * `dy.sum(0)` of nn.Linear over a whole table (smore.py:257-259, mgcn.py:148-150 autograd);
 * fixed summation order, one launch. */
int mmrec_colsum_f32(const float *x, int32_t M, int32_t N, float *out, void *stream);
/* The same with a workspace of mmrec_colsum_workspace_bytes(M, N) bytes (0: not needed): tall
 * matrices (M >= 16384) are summed in two coalesced stages instead of one strided pass. */
size_t mmrec_colsum_workspace_bytes(int32_t M, int32_t N);
int mmrec_colsum_ws_f32(const float *x, int32_t M, int32_t N, float *out, float *workspace, void *stream);
/* SMORE residual modality injection (smore.py:269-272): o_m = item + scale * g_m for the image /
 * text / fusion gates in one launch, and its autograd in one launch:
 * d_item = d0 + d1 + d2, dg_m = scale * d_m. numel % 4 == 0, 16-byte aligned. */
int mmrec_inject3_fwd_f32(const float *item, const float *g0, const float *g1, const float *g2, float scale,
                          int64_t numel, float *o0, float *o1, float *o2, void *stream);
int mmrec_inject3_bwd_f32(const float *d0, const float *d1, const float *d2, float scale, int64_t numel,
                          float *d_item, float *dg0, float *dg1, float *dg2, void *stream);
/* Loss head of MGCN / SMORE (mgcn.py:241-253, smore.py:396-411):
 *   out[0] = o2[0] * inv_batch + reg_weight * (o2[1] * inv_train_batch_size) + cl_weight * (cl2[0] + cl2[1])
 * with o2 = mmrec_bpr_fwd_f32's two sums and cl2 = the two InfoNCE losses (device scalars), in the
 * float32 operation order of the reference's tensor expression; and its gradient for a device
 * scalar g: d_o2 = (g * inv_batch, g * reg_weight * inv_train_batch_size), d_cl2 = (g * cl_weight) x 2. */
int mmrec_loss_head_fwd_f32(const float *o2, const float *cl2, float inv_batch, float reg_weight,
                            float inv_train_batch_size, float cl_weight, float *out, void *stream);
int mmrec_loss_head_bwd_f32(const float *g, float inv_batch, float reg_weight, float inv_train_batch_size,
                            float cl_weight, float *d_o2, float *d_cl2, void *stream);
int mmrec_knn_weights_f32(const int32_t *idx, const float *val, int32_t n, int32_t k, int32_t mode, float *dis_ws,
                          float *out_vals, void *stream);

/* ------------------------------------------------------------------------------------------
 * Row part of SMORE's modality-aware preference module (models/smore.py:321-341) for widths whose
 * d x d layers run as separate tensor-core launches (d = 128): everything after the seven Linear
 * layers in one launch each way. zv / zt = query_v / query_t outputs (pre-softmax), gi / gt / gf =
 * sigmoid outputs of the three gate_*_prefer layers, masks = [3, n, d] nn.Dropout multipliers or
 * NULL:
 *   side = (gi m_i softmax(zv) V + gt m_t softmax(zt) T + gf m_f F) / 3,  all = C + side.
 * The backward recomputes the softmax; g_all / g_side may be NULL (not both). d in {32, 64, 128}.
 * ---------------------------------------------------------------------------------------- */
int mmrec_smore_combine_supported(int32_t d);
/* the same with the dropout multipliers generated in the kernel (MmrecDropout above) */
int mmrec_smore_combine_fwd_drop_f32(const float *zv, const float *zt, const float *V, const float *T, const float *F,
                                     const float *C, const float *gi, const float *gt, const float *gf,
                                     const MmrecDropout *drop, int32_t n, int32_t d, float *side, float *all,
                                     void *stream);
int mmrec_smore_combine_bwd_drop_f32(const float *g_all, const float *g_side, const float *zv, const float *zt,
                                     const float *V, const float *T, const float *F, const float *gi, const float *gt,
                                     const float *gf, const MmrecDropout *drop, int32_t n, int32_t d, float *dzv,
                                     float *dzt, float *dV, float *dT, float *dF, float *dC, float *dgi, float *dgt,
                                     float *dgf, void *stream);
int mmrec_smore_combine_fwd_f32(const float *zv, const float *zt, const float *V, const float *T, const float *F,
                                const float *C, const float *gi, const float *gt, const float *gf,
                                const float *masks, int32_t n, int32_t d, float *side, float *all, void *stream);
int mmrec_smore_combine_bwd_f32(const float *g_all, const float *g_side, const float *zv, const float *zt,
                                const float *V, const float *T, const float *F, const float *gi, const float *gt,
                                const float *gf, const float *masks, int32_t n, int32_t d, float *dzv, float *dzt,
                                float *dV, float *dT, float *dF, float *dC, float *dgi, float *dgt, float *dgf,
                                void *stream);

/* ------------------------------------------------------------------------------------------
 * MGCN's two-way attention fuser (models/mgcn.py:188-205), one launch each way. Replaces
 *   att = softmax(cat([query_common(image_embeds), query_common(text_embeds)], -1))   (the
 *         Linear(d, 1) of query_common is the row dot with w2 = query_common.2.weight [1, d])
 *   common = att[:, 0] * image_embeds + att[:, 1] * text_embeds
 *   sep_m  = gate_m_prefer(content) * (m_embeds - common);  side = (sep_i + sep_t + common) / 3
 *   all    = content + side
 * Hi / Ht = tanh(query_common.0(E_m)) and Pi / Pt = sigmoid(gate_*_prefer.0(content)) come from
 * mmrec_dense_act_batch_fwd_f32. All row tensors are [n_rows, d] float32 row-major, d in
 * {32, 64, 128}; att [n_rows, 2] is written forward and read backward.
 * Backward: g_all / g_side may be NULL (not both); dw2_partial is scratch of
 * mmrec_mgcn_fuse_bwd_blocks(n_rows, d) * d floats (per-CTA column sums in fixed order; the
 * final sum goes to dw2 [d] with mmrec_colsum_f32: no float atomics).
 * ---------------------------------------------------------------------------------------- */
int mmrec_mgcn_fuse_supported(int32_t d);
int32_t mmrec_mgcn_fuse_bwd_blocks(int32_t n_rows, int32_t d);
int mmrec_mgcn_fuse_fwd_f32(const float *Hi, const float *Ht, const float *w2, const float *Ei, const float *Et,
                            const float *Pi, const float *Pt, const float *content, int32_t n_rows, int32_t d,
                            float *att, float *side, float *all, void *stream);
int mmrec_mgcn_fuse_bwd_f32(const float *g_all, const float *g_side, const float *Hi, const float *Ht,
                            const float *w2, const float *Ei, const float *Et, const float *Pi, const float *Pt,
                            const float *att, int32_t n_rows, int32_t d, float *dHi, float *dHt, float *dEi,
                            float *dEt, float *dPi, float *dPt, float *dC, float *dw2_partial, float *dw2,
                            void *stream);

/* ------------------------------------------------------------------------------------------
 * Top-K metrics on the device (K15). Replaces TopKEvaluator.evaluate / _calculate_metrics
 * (utils/topk_evaluator.py:58-143) and recall_/recall2_/precision_/ndcg_/map_
 * (utils/metrics.py:12-109): the Python membership loop that builds the hit matrix and the numpy
 * float64 reductions.
 *   topk [n_users, k] int64 item ids (the evaluator's batch_matrix_list, concatenated), k <= 64
 *   gt_rowptr [n_users + 1] / gt_items: ground-truth items per eval user, ascending int32 CSR
 *   disc[k] = 1 / log2(r + 2), idcg_all[k] = cumsum(disc): float64, computed by the host in numpy
 *   hits_out [n_users, k] uint8 or NULL
 *   sums_out [5, k] float64: SUM over users of recall, cumulative hits (recall2 numerator),
 *            precision, ndcg, map at every rank; the caller divides by n_users (recall2: by the
 *            total number of positives) and rounds like topk_evaluator.py:101.
 * Per-user values are bit-identical to numpy's (same float64 operations in the same order).
 * ---------------------------------------------------------------------------------------- */
size_t mmrec_topk_metrics_workspace_bytes(int32_t n_users);
int mmrec_topk_metrics_f64(const int64_t *topk, int32_t n_users, int32_t k, const int32_t *gt_rowptr,
                           const int32_t *gt_items, const double *disc, const double *idcg_all,
                           uint8_t *hits_out, double *sums_out, void *workspace, void *stream);
/* K-way merge of `n_lists` descending lists per user (local top-K of every rank after the
 * all-gather, SURVEY 8e). Same tie rule. lists are [n_lists, n_users, k]. */
int mmrec_topk_merge(const float *vals, const int32_t *idx, int32_t n_lists, int32_t n_users,
                     int32_t k, float *out_val, int64_t *out_idx, void *stream);

/* ------------------------------------------------------------------------------------------
 * Negative sampling (host side of the [3, B] training batch, SURVEY 8 a16). Replaces the Python
 * loop of TrainDataLoader._sample_neg_ids / _random (utils/dataloader.py:267-275, 307-309):
 *   iid = random.sample(all_items, 1)[0]; while iid in history_items_per_u[u]: redraw
 * with a bit-exact replay of CPython's Mersenne Twister (random.sample(list, 1) ==
 * list[_randbelow(len)], _randbelow = getrandbits(n.bit_length()) with rejection).
 * ALL pointers are HOST pointers. mt_state_host holds random.getstate()[1] (624 words + the
 * position) and is advanced in place; the caller writes it back with random.setstate().
 * hist_rowptr/hist_cols: per-user CSR of training items, ascending inside a user.
 * ---------------------------------------------------------------------------------------- */
int mmrec_neg_sample_mt19937_host(uint32_t *mt_state_host, const int64_t *all_items_host,
                                  int64_t n_items, const int64_t *hist_rowptr_host,
                                  const int64_t *hist_cols_host, int64_t n_hist_users,
                                  const int64_t *users_host, int64_t n, int64_t *neg_out_host);

/* Counter-based negative sampler on the DEVICE (SURVEY 8(f)-3; config 5: 500 M draws per epoch).
 * Same rule as the reference (uniform item, re-drawn while it is in the user's training history,
 * utils/dataloader.py:267-275, 307-309) on a stateless splitmix64 stream keyed by (seed, step,
 * position, draw): any rank regenerates any batch without communication. All pointers are DEVICE
 * pointers; hist_rowptr int64 [n_users + 1] / hist_cols int32 ascending inside a user; all_items
 * maps the draw to an item id (NULL: identity). neg_out[b] = -1 if max_draws were all rejected. */
int mmrec_neg_sample_counter(const int64_t *users, int64_t n, const int64_t *all_items, int64_t n_items,
                             const int64_t *hist_rowptr, const int32_t *hist_cols, uint64_t seed, uint64_t step,
                             int32_t max_draws, int64_t *neg_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MMREC_B200_H */
