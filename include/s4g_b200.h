/*
 * s4g_b200 — C ABI of the B200-native PointNet++ hot path of S4G.
 *
 * This is the drop-in boundary: every entry point replaces one function of the reference's
 * `pn2_ext` torch extension (yzqin/s4g-release,
 * inference/grasp_proposal/network_models/models/pointnet2_utils/csrc/main.cpp:7-13) or one fused
 * stage of the module stack above it.  Plain pointers and sizes only; no torch types.
 *
 * Conventions
 *   - all pointers are DEVICE pointers on the current CUDA device unless a name ends in `_host`;
 *   - tensors use the reference's interface layout: fp32, channel-first (B, C, N), contiguous;
 *     indices are int64 (the `_i32` variants feed the fused path);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *     enqueued on it and nothing synchronises the host;
 *   - return value: 0 on success, otherwise a negative S4G_E_* code (argument errors, mirroring
 *     the reference's CHECK_* macros) or a positive cudaError_t; s4g_last_error() gives the text
 *     (thread-local).  Inputs are never modified; outputs are written completely (no need to
 *     pre-zero them).
 */
#ifndef S4G_B200_H_
#define S4G_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S4G_OK 0
#define S4G_E_ARG (-1)         /* a CHECK_* precondition of the reference failed            */
#define S4G_E_UNSUPPORTED (-2) /* valid for the reference, not (yet) supported by this build */

/* ABI version of this header (bumped on any signature change). */
int s4g_version(void);
/* Text of the last error raised on the calling thread ("" if none). */
const char* s4g_last_error(void);
/* number of CUDA kernels this library has launched in the process so far (bench.py reports the per-step delta) */
unsigned long long s4g_launch_count(void);

/* ---- pn2_ext replacements --------------------------------------------------------------- */

/* farthest_point_sample — csrc/sampling.h:7-9, sampling_kernel.cu:128-172.
 * points (B,3,N) -> index (B,M) int64.  index[:,0] = 0; reproduces the reference's tie-breaking
 * (block tree reduction, sampling_kernel.cu:100-113) exactly.  Requires N >= M > 0. */
int s4g_farthest_point_sample_f32(const float* points, int B, int N, int M, int64_t* index, void* stream);
int s4g_farthest_point_sample_f32_i32(const float* points, int B, int N, int M, int32_t* index, void* stream);
/* Experimental: route clouds of 4 096 .. 55 000 points through the exact bucket-pruned FPS kernel (same results; slower
 * than the default kernels on the measured workloads, see csrc/fps.cu).  Returns the previous setting. */
int s4g_fps_set_bucket_mode(int on);

/* gather_points — pointnet2_utils/functions.py:10-25.  out[b,c,m] = points[b,c,index[b,m]]. */
int s4g_gather_points_f32(const float* points, const int64_t* index, int B, int C, int N, int M, float* out,
                          void* stream);

/* ball_query — csrc/ball_query.h:7-11, ball_query_kernel.cu:89-133.
 * points (B,3,N), centroids (B,3,M) -> index (B,M,K) int64, count (B,M) int64 (count may be NULL).
 * First K points in index order with d2 < radius*radius (strict, fp32); the first hit pads every
 * unused slot; no hit -> zeros and count 0. */
int s4g_ball_query_f32(const float* points, const float* centroids, int B, int N, int M, float radius, int K,
                       int64_t* index, int64_t* count, void* stream);
int s4g_ball_query_f32_i32(const float* points, const float* centroids, int B, int N, int M, float radius, int K,
                           int32_t* index, int32_t* count, void* stream);
/* The same query in two calls (reference: ball_query_kernel.cu:20-97, one call there).  The spatial index only needs the
 * cloud, so it can be built on another stream while the centroids are still being sampled.  s4g_ball_query_uses_grid
 * tells whether the grid path serves this shape (else use the one-call form); the build returns NULL on failure;
 * the query's stream must be ordered after the build; the free is stream-ordered after the queries on `stream`. */
typedef struct s4g_ball_grid s4g_ball_grid;
int s4g_ball_query_uses_grid(int N, int K, float radius);
s4g_ball_grid* s4g_ball_grid_build_f32(const float* points, int B, int N, float radius, void* stream);
int s4g_ball_query_with_grid_f32_i32(const s4g_ball_grid* grid, const float* points, const float* centroids, int M, int K,
                                     int32_t* index, int32_t* count, void* stream);
int s4g_ball_grid_free(s4g_ball_grid* grid, void* stream);

/* group_points_forward / backward — csrc/grouping.h:7-14, grouping_kernel.cu:32-54,106-152.
 * fwd: input (B,C,N), index (B,M,K) -> out (B,C,M,K).   bwd: grad_out (B,C,M,K) -> grad_in (B,C,N). */
int s4g_group_points_forward_f32(const float* input, const int64_t* index, int B, int C, int N, int M, int K,
                                 float* out, void* stream);
/* A/B switch (measurements): 1 (default) = the forward stages channel planes in shared memory with bulk copies when they
 * fit (gathers from shared memory, all global traffic coalesced), 0 = always the plain gather.  Same results. */
int s4g_group_points_set_staged(int on);
int s4g_group_points_backward_f32(const float* grad_out, const int64_t* index, int B, int C, int N, int M, int K,
                                  float* grad_in, void* stream);

/* point_search (3-NN) — csrc/interpolate.h:8-11, interpolate_kernel.cu:92-132.
 * query (B,3,Nq), key (B,3,Nk) -> index (B,Nq,3) int64, distance (B,Nq,3) = SQUARED distances,
 * ascending, earlier key wins ties.  num_neighbours must be 3 and Nk >= 3.  A key counts only when its squared
 * distance is below 1e40 (+inf in fp32), so NaN and overflowing distances never do.  When c < 3 keys count (a NaN
 * query, NaN keys, |x| >~ 2e19 in fp32), the slots keep the reference's start values (interpolate_kernel.cu:53-54):
 * slot c is (distance 1e40, index -1) and the slots after it (0, index 0). */
int s4g_point_search_f32(const float* query, const float* key, int B, int Nq, int Nk, int num_neighbours,
                         int64_t* index, float* distance, void* stream);

/* interpolate_forward / backward — csrc/interpolate.h:13-22, interpolate_kernel.cu:191-236,296-341.
 * fwd: input (B,C,Nk), index (B,Nq,3), weight (B,Nq,3) -> out (B,C,Nq);  bwd scatters grad*w. */
int s4g_interpolate_forward_f32(const float* input, const int64_t* index, const float* weight, int B, int C, int Nk,
                                int Nq, float* out, void* stream);
int s4g_interpolate_backward_f32(const float* grad_out, const int64_t* index, const float* weight, int B, int C,
                                 int Nk, int Nq, float* grad_in, void* stream);

/* ---- fp64 instantiation of the same seven operators ---------------------------------------
 * The reference dispatches each kernel over float and double (AT_DISPATCH_FLOATING_TYPES:
 * sampling_kernel.cu:21, ball_query_kernel.cu:116, grouping_kernel.cu:137, interpolate_kernel.cu:118,222,327).
 * Same contracts as the _f32 entry points with double data; `radius` is the reference's float argument
 * converted to double by the caller (ball_query_kernel.cu:119).  farthest_point_sample_f64 keeps its running
 * minima in shared memory when a cloud fits and otherwise needs
 * s4g_farthest_point_sample_f64_workspace(B, N) bytes of device scratch (0 = none). */
size_t s4g_farthest_point_sample_f64_workspace(int B, int N);
int s4g_farthest_point_sample_f64(const double* points, int B, int N, int M, int64_t* index, void* workspace,
                                  size_t workspace_bytes, void* stream);
int s4g_ball_query_f64(const double* points, const double* centroids, int B, int N, int M, double radius, int K,
                       int64_t* index, int64_t* count, void* stream);
int s4g_group_points_forward_f64(const double* input, const int64_t* index, int B, int C, int N, int M, int K,
                                 double* out, void* stream);
int s4g_group_points_backward_f64(const double* grad_out, const int64_t* index, int B, int C, int N, int M, int K,
                                  double* grad_in, void* stream);
int s4g_point_search_f64(const double* query, const double* key, int B, int Nq, int Nk, int num_neighbours,
                         int64_t* index, double* distance, void* stream);
int s4g_interpolate_forward_f64(const double* input, const int64_t* index, const double* weight, int B, int C, int Nk,
                                int Nq, double* out, void* stream);
int s4g_interpolate_backward_f64(const double* grad_out, const int64_t* index, const double* weight, int B, int C,
                                 int Nk, int Nq, double* grad_in, void* stream);

/* ---- tight-parity layer (TF32 tensor cores) ------------------------------------------------ */

/* One shared-MLP block — Conv{1,2}d 1x1 (bias-free) + BatchNorm (eval, folded by the caller) + ReLU, reference
 * nn_utils/conv.py:30-36,70-76 — as Y[P][N] = act(X[P][K] W[N][K]^T + shift[N]) on tcgen05 kind::tf32 with fp32
 * accumulation: the arithmetic cuDNN's TF32 default gives the unmodified reference on this GPU.  X, W, Y fp32 row-major
 * (channel-last rows), ldx / ldw multiples of 4 floats and 16-byte aligned bases; relu: apply max(.,0); round_out: round
 * the result to the nearest TF32 value (for the next layer's operand).  Layer by layer, nothing fused: the tight-parity
 * mode of the fused path (its throughput path is the bf16 chain below). */
int s4g_linear_tf32(const float* x, long long ldx, const float* w, long long ldw, const float* shift, float* y,
                    long long ldy, long long P, int N, int K, int relu, int round_out, void* stream);

/* ---- training path (channel-last bf16 rows, fp32 accumulation) ------------------------------- */
/* A shared-MLP block of the reference in TRAINING mode — Conv{1,2}d 1x1 (bias-free) -> BatchNorm with batch statistics ->
 * ReLU (-> dropout), nn_utils/conv.py:30-36,70-76, nn_utils/mlp.py:99-101 — and its backward, decomposed into one
 * tcgen05 GEMM over channel-last bf16 rows and fused element-wise kernels.  All row matrices are [P][C] bf16 with
 * C % 8 == 0 and 16-byte aligned rows.  (Host side: s4g_release_b200/train_engine.py.) */

/* C[P][N] = A[P][K] · B[N][K]^T, bf16 in / bf16 out, fp32 accumulation in TMEM (persistent tcgen05 kernel).
 * Forward: A = layer input, B = conv weight [cout][cin].  Input gradient: A = dY, B = weight^T [cin][cout]. */
int s4g_gemm_bf16(const void* a, long long lda, const void* b, long long ldb, void* c, long long ldc, long long P, int N,
                  int K, void* stream);
/* A/B switch (measurements): 1 (default) = weight-stationary schedule where it applies (K <= 512 and enough row tiles: a
 * CTA keeps one 128-column slice of B in shared memory for all its row tiles), 0 = always stream B.  Returns the
 * previous setting.  Both schedules compute the same bits. */
int s4g_gemm_bf16_set_weight_stationary(int on);
/* A/B switch (measurements): number of epilogue warp groups, 1 or 2 (one group per TMEM accumulator / tile parity, a
 * staging tile each), 0 (default) = chosen per launch (2 when K <= 128).  Returns the previous setting.  Same bits. */
int s4g_gemm_bf16_set_epilogue_groups(int groups);
/* A/B switch (measurements): output columns per tile, 128 or 256 (one N = 256 MMA per K step, two epilogue groups splitting
 * the tile; streaming schedule), 0 (default) = chosen per launch.  Returns the previous setting.  Same bits. */
int s4g_gemm_bf16_set_tile_n(int bn);
/* The launch the three GEMM entry points (mode 0 = s4g_gemm_bf16, 1 = _stats, 2 = _bwd) would make for a shape on a GPU with
 * `sms` SMs (0 = the current device): out7 = {tile columns, epilogue groups, weight-stationary, ring stages, grid, threads,
 * dynamic shared memory bytes}.  Host arithmetic only (the CPU tests check the shared-memory budget with it). */
int s4g_gemm_bf16_plan(long long P, int N, int K, int mode, int sms, long long* out7);
/* Input-gradient GEMM whose RESULT is the upstream gradient of the block that produced y_prev (its rows [P][N] before
 * BatchNorm; scale / shift = its folded BatchNorm; relu / seed / drop_p = its activation and dropout):
 *   c = (a · b^T) * relu'(y_prev * scale + shift) * dropout mask     (stored MASKED, bf16)
 *   sums2n[0..N) = sum_r c[r][n],  sums2n[N..2N) = sum_r c[r][n] * y_prev[r][n]   (fp64, zeroed here)
 * i.e. s4g_train_bn_bwd_reduce_bf16 of that block done in this GEMM's epilogue (no pass over c and y_prev); hand c to
 * s4g_train_bn_bwd_apply_bf16 with relu = 0, drop_p = 0.  (reference: the autograd backward of conv.py:30-36,70-76.) */
int s4g_gemm_bf16_bwd(const void* a, long long lda, const void* b, long long ldb, void* c, long long ldc, long long P, int N,
                      int K, const void* y_prev, long long ldy, const float* scale, const float* shift, int relu,
                      unsigned seed, float drop_p, double* sums2n, void* stream);
/* the same GEMM with the BatchNorm batch statistics of its (bf16-rounded) result accumulated in the epilogue:
 * stats2n[0..N) = sum_r c[r][n], stats2n[N..2N) = sum_r c[r][n]^2 (fp64, zeroed here) — no extra pass over C. */
int s4g_gemm_bf16_stats(const void* a, long long lda, const void* b, long long ldb, void* c, long long ldc, long long P, int N,
                        int K, double* stats2n, void* stream);
/* BatchNorm's per-channel algebra in one launch.  Forward: out4c = [mean | rstd | scale = gamma * rstd | shift = beta -
 * mean * scale]; running_mean / running_var (may both be NULL) updated like torch.nn.BatchNorm{1,2}d (momentum, unbiased
 * variance).  Backward: dgamma += sum g * xhat, dbeta += sum g, out3c = [ka | kb | kc] of s4g_train_bn_bwd_apply_bf16. */
int s4g_train_bn_finalize(const double* sums2c, long long P, int C, const float* gamma, const float* beta, float eps,
                          float momentum, float* running_mean, float* running_var, float* out4c, void* stream);
int s4g_train_bn_bwd_finalize(const double* sums2c, long long P, int C, const float* gamma, const float* mean_rstd,
                              float* dgamma, float* dbeta, float* out3c, void* stream);
/* sums2c[0..C) = sum_r y[r][c], sums2c[C..2C) = sum_r y[r][c]^2 (fp64; zeroed here) -> the batch mean / variance of
 * BatchNorm's training mode (torch.nn.BatchNorm{1,2}d over the (B, M, K) positions of a channel). */
int s4g_train_colstats_bf16(const void* y, long long ld, long long P, int C, double* sums2c, void* stream);
/* z = dropout(relu(y * scale + shift)): BatchNorm's normalise + affine folded into (scale, shift) by the caller, ReLU
 * when relu != 0, dropout with probability drop_p from a counter-based hash of (seed, row, channel) (0 = off). */
int s4g_train_bn_act_bf16(const void* y, const float* scale, const float* shift, void* z, long long P, int C, int relu,
                          unsigned seed, float drop_p, void* stream);
/* the same followed by torch.max over each group of K consecutive rows (pointnet2_utils/modules.py:243):
 * out [G][C] bf16, arg [G][C] uint8 = the row of the (first) maximum inside its group, kept for the backward; ymax
 * (may be NULL) [G][C] bf16 = y at that row: the backward's reduce of a pooled block only needs these G rows (the
 * gradient is zero everywhere else) — s4g_train_bn_bwd_reduce_bf16(dz_pooled, NULL, 0, ymax, ..., G, ...). */
int s4g_train_bn_act_maxpool_bf16(const void* y, const float* scale, const float* shift, void* out, uint8_t* arg,
                                  void* ymax, long long G, int K, int C, int relu, void* stream);
/* BatchNorm backward, pass 1: sums2c[0..C) = sum_r g, sums2c[C..2C) = sum_r g * y, with g = dz * relu'(.) * dropout mask
 * (s4g_train_bn_bwd_finalize turns the second into sum g * xhat = rstd * (sum g y - mean * sum g) in fp64).  Upstream
 * gradient: dz [P][C] (K = 0), or the pooled gradient [P/K][C] routed to the arg-max row of each group (K > 0, arg from
 * s4g_train_bn_act_maxpool_bf16). */
int s4g_train_bn_bwd_reduce_bf16(const void* dz, const uint8_t* arg, int K, const void* y, const float* scale,
                                 const float* shift, long long P, int C, int relu, unsigned seed, float drop_p,
                                 double* sums2c, void* stream);
/* pass 2: dy = coef * (g - m1 - xhat * m2) with coef = gamma * rstd, m1 = mean(g), m2 = mean(g * xhat), handed in folded
 * per channel as dy = ka * g + kb * y + kc  (ka = coef, kb = -coef * rstd * m2, kc = coef * (rstd * m2 * mean - m1)). */
int s4g_train_bn_bwd_apply_bf16(const void* dz, const uint8_t* arg, int K, const void* y, const float* scale,
                                const float* shift, const float* ka, const float* kb, const float* kc, long long P, int C,
                                int relu, unsigned seed, float drop_p, void* dy, void* stream);
/* The max over a GLOBAL set-abstraction level's one group per scene (num_centroids = 0, modules.py:93-98 + the torch.max of
 * :106): z = relu(y * scale + shift) over the N rows of each of the B scenes (y [B*N][C], any N >= 1), reduced per scene
 * and channel: out [B][C] bf16, arg [B][C] int32 = the row inside the scene of the FIRST maximum (like torch.max), ymax
 * (may be NULL) [B][C] bf16 = y at that row.  work: B*C 64-bit words of scratch.  The partial maxima of the CTAs are
 * merged with 64-bit atomicMax on (value, first row) keys: the result does not depend on their order. */
int s4g_train_bn_act_segmax_bf16(const void* y, const float* scale, const float* shift, void* out, int* arg, void* ymax,
                                 unsigned long long* work, int B, long long N, int C, int relu, void* stream);
/* The two BatchNorm-backward passes of such a block: the pooled gradient dz [P/N][C] routed to row arg[b][c] (int32, from
 * s4g_train_bn_act_segmax_bf16) of scene b; otherwise as s4g_train_bn_bwd_reduce_bf16 / _apply_bf16 (no dropout). */
int s4g_train_bn_bwd_reduce_seg_bf16(const void* dz, const int* arg, long long N, const void* y, const float* scale,
                                     const float* shift, long long P, int C, int relu, double* sums2c, void* stream);
int s4g_train_bn_bwd_apply_seg_bf16(const void* dz, const int* arg, long long N, const void* y, const float* scale,
                                    const float* shift, const float* ka, const float* kb, const float* kc, long long P, int C,
                                    int relu, void* dy, void* stream);
/* Channel dropout (F.dropout2d, the evaluation head's SharedMLP(ndim=2), nn_utils/mlp.py:27) in place of element dropout:
 * rows [P][C] of P / scene_rows scenes (P < 2^31, whole scenes); each (scene, channel) is kept with probability
 * 1 - drop_p, deterministically from (seed, scene, channel): the element hash of s4g_train_bn_act_bf16 evaluated at
 * row = scene.  Kept channels are scaled by 1 / (1 - drop_p) on every row of their scene, dropped ones are zero.
 * The forward (z = chdrop(relu(y * scale + shift))) and the two BatchNorm-backward passes, which recompute the mask;
 * otherwise as s4g_train_bn_act_bf16 / s4g_train_bn_bwd_reduce_bf16 / s4g_train_bn_bwd_apply_bf16 with a dense dz.
 * Rows 16-byte aligned. */
int s4g_train_bn_act_chdrop_bf16(const void* y, const float* scale, const float* shift, void* z, long long P, int C, int relu,
                                 long long scene_rows, unsigned seed, float drop_p, void* stream);
int s4g_train_bn_bwd_reduce_chdrop_bf16(const void* dz, const void* y, const float* scale, const float* shift, long long P,
                                        int C, int relu, long long scene_rows, unsigned seed, float drop_p, double* sums2c,
                                        void* stream);
int s4g_train_bn_bwd_apply_chdrop_bf16(const void* dz, const void* y, const float* scale, const float* shift, const float* ka,
                                       const float* kb, const float* kc, long long P, int C, int relu, long long scene_rows,
                                       unsigned seed, float drop_p, void* dy, void* stream);
/* The backward of a broadcast propagation level (num_fp_neighbours = 0, modules.py:131-134 expand) for its global input:
 * out[b][c] += sum_n dz[b*Nq + n][c] for c < C2 (dz rows ld wide, bf16; out fp32 [B][C2]).  Fixed summation order, no
 * atomics: the same bits on every run. */
int s4g_train_rows_segment_sum_bf16(const void* dz, long long ld, int B, long long Nq, int C2, float* out, void* stream);
/* QueryGrouper.forward (pointnet2_utils/modules.py:37-54) in the row layout: out row (b, m, k) =
 * [feat[b*N + nbr[b][m][k]][0..Cf) | xyz[b][:, nbr] - ctr[b][:, m] | 0 x 5]  (width Cf + 8; the weight columns are
 * re-ordered to match by the caller).  feat may be NULL when Cf == 0. */
int s4g_train_group_rows_bf16(const void* feat, const float* xyz, const float* ctr, const int* nbr, int B, int N, int M, int K,
                              int Cf, void* out, void* stream);
/* GroupPointsBackward (grouping_kernel.cu:57-96) in the row layout: dfeat[b*N + nbr][c] += dx[(b,m,k)][c], c < Cf; fp32
 * vector atomics; dfeat is NOT zeroed here (it may already hold the skip connection's gradient). */
int s4g_train_group_rows_bwd(const void* dx, long long ld, const int* nbr, int B, int N, int M, int K, int Cf, float* dfeat,
                             void* stream);
/* InterpolateBackward (interpolate_kernel.cu:243-286) in the row layout: dsparse[b*Nk + idx_k][c] += w_k * dx[(b,q)][c]. */
int s4g_train_interp_rows_bwd(const void* dx, long long ld, const int* index, const float* weight, int B, int Nk, int Nq,
                              int C2, float* dsparse, void* stream);
/* The scatter-add gradients (InterpolateBackward, GroupPointsBackward) as a GATHER over the INVERSE of their index
 * tensor (geometry, fixed for the step).  index (B, E) with values in [0, T): the 3-NN index (E = Nq * 3, T = Nk) or the
 * neighbour index (E = M * K, T = N).  count -> (caller: inclusive scan `end`, start = end - count) -> fill -> every target
 * row sums its own list of entries e = b * E + i:  out[b*T + j][c] (+)= sum weight[e] * dx[e / div][c]  (div = 3 with the
 * interpolation weights; div = 1, weight NULL for the grouping).  No atomics on the gradient; written once as fp32
 * and / or bf16 (either may be NULL); accumulate != 0 adds into out_f32. */
int s4g_train_index_inverse_count(const int* index, int B, int T, long long E, int* count, void* stream);
int s4g_train_index_inverse_fill(const int* index, int B, int T, long long E, int* cursor, int* list, void* stream);
int s4g_train_rows_bwd_gather(const void* dx, long long ld, const int* list, const int* end, const int* count,
                              const float* weight, int div, long long targets, int C, int accumulate, float* out_f32,
                              void* out_bf16, void* stream);
/* out = dz where y * scale + shift > 0, else 0 (rows [P][C], contiguous): the pooled gradient of a max-pooled block masked
 * once on its G rows (y = ymax of s4g_train_bn_act_maxpool_bf16); the two BatchNorm-backward passes then run with relu = 0. */
int s4g_train_relu_mask_rows_bf16(const void* dz, const void* y, const float* scale, const float* shift, long long P, int C,
                                  void* out, void* stream);
int s4g_train_f32_to_bf16(const float* x, void* y, long long n, void* stream);
/* The final biased 1x1 conv of a head (reference PointNet2_tcls.py:84-95, nn.Conv1d(C, k, 1), k <= 16) from the bf16 rows
 * h [P][C] straight into the reference's fp32 channel-first logits (P / n_points, k, n_points), and its input gradient
 * dh [P][C] bf16 = dlogits · w.  (dw / dbias are a plain reduction over P: left to the caller's library GEMM.) */
int s4g_train_head_logits_fwd(const void* h, const float* w, const float* bias, float* out, long long P, int C, int k,
                              int n_points, void* stream);
int s4g_train_head_logits_bwd(const float* dlogits, const float* w, void* dh, long long P, int C, int k, int n_points,
                              void* stream);
/* ... and its parameter gradients: dw[j][c] += sum_rows dlogits[b][j][n] * h[row][c], dbias[j] += sum_rows dlogits[b][j][n]
 * (fp32 atomics INTO dw [k][C] / dbias [k]: the caller's param.grad buffers). */
int s4g_train_head_logits_dw(const float* dlogits, const void* h, float* dw, float* dbias, long long P, int C, int k,
                             int n_points, void* stream);
/* out = a + b (+ c) (+ d): bf16 vectors of n elements (n % 8 == 0) summed in fp32 and rounded once — the sum of the four
 * heads' gradients w.r.t. the shared per-point features (autograd's accumulation at PointNet2_tcls.py:131-141). */
int s4g_train_sum_bf16(const void* a, const void* b, const void* c, const void* d, void* out, long long n, void* stream);

/* ---- fused inference path (channel-last bf16 features, int32 indices) ---------------------- */

/* PointSearch (interpolate_kernel.cu:33-81) fused with the inverse-squared-distance weights of
 * FeatureInterpolator.forward (pointnet2_utils/modules.py:115-120).  index (B,Nq,3) int32,
 * weight (B,Nq,3) fp32 (normalised): v_k = 1/max(d_k, 1e-10), w_k = v_k / ((v_0 + v_1) + v_2), IEEE fp32, on the
 * distances s4g_point_search_f32 returns, so with fewer than three finite distances too (an all-NaN query gets
 * [0, 0.5, 0.5]).  Where point_search returns index -1 this writes 0; the weight there is 0, so every index is a valid
 * key row in [0, Nk). */
int s4g_three_nn_weights_f32_i32(const float* query, const float* key, int B, int Nq, int Nk, int* index,
                                 float* weight, void* stream);

/* InterpolateForward (interpolate_kernel.cu:139-181) + channel concat (modules.py:124-127).
 * sparse [B*Nk][C2] bf16, dense [B*Nq][C1] bf16 (NULL when C1 == 0) -> out [B*Nq][C2+C1] bf16. */
int s4g_interp_concat_bf16(const void* sparse, const int* index, const float* weight, const void* dense, int B, int Nk,
                           int Nq, int C2, int C1, void* out, void* stream);
/* The same with ReLU on the interpolated channels (relu != 0).  Interpolation is linear, so the first layer of a
 * feature-propagation MLP can run on the SPARSE points first — W (sum_k w_k f_k) = sum_k w_k (W f_k), 5x fewer rows at
 * the finest level — and this kernel then interpolates the pre-activations (shift already added: the weights sum to
 * one) and applies the ReLU: PointnetFPModule.forward (modules.py:498-507) with conv and interpolation commuted. */
int s4g_interp_concat_act_bf16(const void* sparse, const int* index, const float* weight, const void* dense, int B, int Nk,
                               int Nq, int C2, int C1, int relu, void* out, void* stream);

/* gather_points for xyz with int32 indices (functions.py:10-25): (B,3,N),(B,M) -> (B,3,M). */
int s4g_gather_xyz_f32_i32(const float* xyz, const int* index, int B, int N, int M, float* out, void* stream);

/* gather_points for channel-last bf16 features (EdgeSAModule.forward's centroid features, modules.py:280-282):
 * src [B*N][C] bf16, index (B,M) int32 in [0, N) -> out [B*M][C] bf16, out[b*M + m] = src[b*N + index[b][m]], bit-equal.
 * C % 8 == 0, rows 16-byte aligned; 64-bit offsets (tables over 2 GiB). */
int s4g_gather_rows_bf16(const void* src, const int* index, int B, int N, int M, int C, void* out, void* stream);

/* Edge feature propagation (EdgeFPModule, pointnet2_utils/modules.py:287-308, fed by EdgeFeatureInterpolator, :227-247):
 * per dense point q and each of its 3 nearest sparse points k the MLP's first layer sees [interp_q | n_k - interp_q | d_q]
 * (2 C2 + C1 channels).  With its BN-folded weight split by those column groups, W' = [W_i | W_n | W_d], and shift b',
 *   y0[q,k] = sum_j w_qj U[idx_qj] + V[idx_qk] + T_q + b',   U = (W_i - W_n) S,  V = W_n S,  T = W_d d,
 * whatever the weights sum to.  This writes out[(b*Nq + q)*3 + k][c] = relu(((sum_j w_qj U + V[idx_qk]) + T_q) + b') in
 * fp32, in that order, rounded to bf16 once; the sum over j is fma(U2,w2, fma(U1,w1, U0*w0)); the ReLU is fmaxf(y, 0), so a
 * NaN pre-activation gives 0.
 *   uv     [B*Nk][2C] bf16, rows [U | V] (C = cout of the first layer, C % 8 == 0);
 *   index, weight (B,Nq,3) from s4g_three_nn_weights_f32_i32: int32 in [0, Nk), which it writes for non-finite clouds too;
 *   exactly one skip: t_rows [B*Nq][C] bf16 (T computed), or the cloud itself xyz (B,3,Nq) fp32 with w_xyz [C][3] fp32
 *   (T = fma(W_d2, z, fma(W_d1, y, W_d0 x)) in fp32: coordinates are not rounded to bf16);
 *   shift [C] fp32 = b'.  Rows and shift 16-byte aligned; 64-bit offsets (outputs over 2 GiB), Nq * C / 8 < 2^31. */
int s4g_edge_interp_rows_bf16(const void* uv, const int* index, const float* weight, const void* t_rows, const float* xyz,
                              const float* w_xyz, const float* shift, int B, int Nk, int Nq, int C, void* out,
                              void* stream);

/* EdgeFPModule's torch.mean over the 3 neighbour rows (modules.py:308): in [3R][C] bf16 -> out [R][C] bf16,
 * out[r] = ((in[3r] + in[3r+1]) + in[3r+2]) / 3 in fp32 with IEEE division, rounded once.  C % 8 == 0, rows 16-byte
 * aligned, R * C / 8 < 2^31; 64-bit offsets. */
int s4g_rows_group_mean_bf16(const void* in, long long R, int C, void* out, void* stream);

/* The max over the neighbours of a GLOBAL set-abstraction level (num_centroids = 0: one group of all N points centred
 * at the origin, PointNetSAModule.forward, modules.py:93-98 + :106 torch.max(new_feature, 3)).  The fused path runs the
 * group through the gathered max-pool chain as P partial groups; this reduces the P partial rows of each scene:
 * in [B*P][C] bf16 -> out [B][C] bf16 (C % 8 == 0).  Exact: max ignores order and repeated rows. */
int s4g_rows_segment_max_bf16(const void* in, int B, int P, int C, void* out, void* stream);

/* Zero-neighbour feature propagation (PointnetFPModule.forward, modules.py:131-134: sparse_feature.expand + channel
 * concat, broadcast first): sparse [B][C2] bf16, dense [B*Nq][C1] bf16 (NULL when C1 == 0) -> out [B*Nq][C2+C1] bf16.
 * C2, C1 multiples of 8. */
int s4g_broadcast_concat_bf16(const void* sparse, const void* dense, int B, int Nq, int C2, int C1, void* out,
                              void* stream);

/* Input rows of PN2_LOCAL's grasp-evaluation head (PointNet2_local.py:131-147: the in-place translation update of :135,
 * then torch.cat([per_point, frames.repeat(1, 4, 1, 1)], 1) ahead of mlp_grasp_eval): feat [B*N][C] bf16 (C % 8 == 0)
 * -> out [B*F*S][C + 48] bf16, row (b, f, s) = feat row b*N + f, then the candidate's 12 values [R0..R8 t0..t2] x 4,
 * each rounded to bf16 to nearest-even.
 *   given (frames != NULL): frames (B, 12, F, S) fp32, points (B, 3, N) fp32, 1 <= F <= N, S >= 1; channels 9..11 become
 *     t - points[b, :, f] (one fp32 subtraction), written back to frames, and are what the row holds;
 *   self (frames == NULL): R (B, 9, N), t (B, 3, N) fp32 head outputs, F = N, S = 1. */
int s4g_local_eval_rows_bf16(const void* feat, int B, int N, int C, float* frames, const float* points, int F, int S,
                             const float* R, const float* t, void* out, void* stream);
/* Its transpose (csrc/train_ops.cu), for the training step: d rows [B*F*S][C + 48] bf16 ->
 *   dfeat [B*N][C] bf16: row b*N + f = the sum of the first C columns of rows (b, f, 0..S-1), accumulated in fp32 in
 *     that order and rounded once; rows f >= F are zero;
 *   self mode only (dR, dt != NULL; F = N, S = 1): dR (B, 9, N) and dt (B, 3, N) fp32 += the sum over the 4 repeats of
 *     columns C..C+47 (the leaf gradients of the R and t logits the rows were written from).
 * No float atomics, 64-bit offsets (row buffers over 2 GiB); rows 16-byte aligned. */
int s4g_local_eval_rows_bwd_bf16(const void* d, int B, int N, int C, int F, int S, void* dfeat, float* dR, float* dt,
                                 void* stream);

/* Fused shared-MLP chain on tcgen05 tensor cores (csrc/mlp_chain.cu): replaces
 * SharedMLP / Conv1d / Conv2d (nn_utils/mlp.py:95-106, nn_utils/conv.py:30-36,70-76) with eval-mode
 * BatchNorm folded in, and around it the grouping + max-pool of PointNetSAModule.forward
 * (pointnet2_utils/modules.py:208-244) or the final biased 1x1 conv (+sigmoid) of the heads
 * (models/PointNet2_tcls.py:126-148).
 *   in_mode : 0 = bf16 rows [P][stride];  1 = gathered set-abstraction input (feat_c feature channels
 *             + relative xyz; reference channel order [xyz | feat] is handled by the weight packer);
 *             6 = the same for an edge level, with a per-centroid term in layer 0 (s4g_chain_run_gather_term)
 *   out_mode: 2 = bf16 rows [P][out_c];  3 = max-pool over groups of `group` rows -> bf16 [P/group][out_c];
 *             4 = fp32 logits, channel-first (P/n_points, out_c, n_points), bias, optional sigmoid
 * Layer l computes relu?(W_l x + bias_l) with W_l (cout x cin, fp32, BN-folded) packed to bf16 by
 * s4g_chain_pack_weights into a host buffer of s4g_chain_weight_bytes(); copy it to the device and
 * register it together with the per-layer fp32 shift vectors (length s4g_chain_cout_pad, zero padded). */
typedef struct s4g_chain s4g_chain;
s4g_chain* s4g_chain_create(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode, int feat_c,
                            int out_mode, int out_c, int group, int sigmoid);
/* s4g_chain_create with the number of 32 KB activation slots pinned (0 = the planner's choice; the rest of shared
 * memory becomes weight stages).  NULL if no deadlock-free plan exists with that count.  For host-side autotuning. */
s4g_chain* s4g_chain_create_slots(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode, int feat_c,
                                  int out_mode, int out_c, int group, int sigmoid, int slots);
/* ... and with the accumulator pairing (pairs: -1 planner's choice, 0 off, 1 on) and the cooperative-epilogue policy
 * (coop: -1 default, 0 none, 1 all row epilogues, 2 the unpaired ones) pinned as well; subs = row blocks of 128 rows
 * per tile (1, or 2: two tiles interleaved layer by layer so one's MMAs overlap the other's epilogue — narrow chains). */
s4g_chain* s4g_chain_create_tuned(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode, int feat_c,
                                  int out_mode, int out_c, int group, int sigmoid, int slots, int pairs, int coop,
                                  int subs);
/* ... and with the input path chosen: tma_in = 1 (row input, cin[0] a multiple of 64, not the max-pool output mode) has
 * one thread fetch the input blocks with 2-D TMA tensor copies into a 128-byte-swizzled layout instead of 64 threads
 * issuing 16-byte cp.async; the tensor map is encoded per s4g_chain_run_rows call.  Gathered max-pool chains (>= 2
 * layers, feat_c a multiple of 64, group % 4 == 0) fetch the neighbours' feature rows with tile::gather4 copies, four
 * rows per instruction (s4g_chain_run_gather then needs K % 4 == 0 and 16-byte aligned indices). */
s4g_chain* s4g_chain_create_tuned_in(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode,
                                     int feat_c, int out_mode, int out_c, int group, int sigmoid, int slots, int pairs,
                                     int coop, int subs, int tma_in);
void s4g_chain_destroy(s4g_chain* chain);
size_t s4g_chain_weight_bytes(const s4g_chain* chain);
int s4g_chain_cout_pad(const s4g_chain* chain, int layer);
/* Plan of the chain: MMA jobs per 128-row tile, activation slots / weight-ring stages in shared memory,
 * input blocks each loader thread keeps in flight, dynamic shared memory, and the planner's estimate of SM
 * cycles per tile (total, and tensor-pipe busy).  Works without a GPU. */
int s4g_chain_info(const s4g_chain* chain, int* n_jobs, int* slots, int* stages, int* load_depth, int* smem_bytes,
                   int* sim_cycles, int* mma_cycles);
/* Optional per-CTA cycle counters (16 x int64 per CTA, for >= 148 CTAs, device memory; NULL switches them
 * off): [0] producer total, [1] producer waiting for a free stage; [2] MMA warp total, [3..5] waiting for
 * activations / TMEM / weights; [6] epilogue warps total, [7] waiting for an accumulator, [12] for a free
 * slot, [10] epilogue work; [11] loader total, [8] loader waiting for a free slot, [9] for cp.async.
 * Measurement aid for profiles/chain_prof.py. */
int s4g_chain_set_profile(s4g_chain* chain, void* counters_dev);
/* Human-readable dump of the job streams into buf (debugging); returns bytes written. */
int s4g_chain_describe(const s4g_chain* chain, char* buf, int cap);
int s4g_chain_pack_weights(const s4g_chain* chain, int layer, const float* w_host, int cout_real, int cin_real,
                           void* packed_host);
int s4g_chain_set_params(s4g_chain* chain, const void* weights_dev, const float* const* bias_dev);
/* Chains created with in_mode 5 (gathered input without features, e.g. the first set-abstraction level): their
 * cin[0] is the OUTPUT width (multiple of 16, <= 128) of a 3 -> cin[0] layer on the relative coordinates
 * (conv + BN + ReLU of SharedMLP block 0, nn_utils/mlp.py:95-106) that the kernel evaluates in fp32 on the CUDA
 * cores while it stages the tile, instead of as a K = 3 tensor-core layer.  w4_host: [cin[0]][4] fp32 table in HOST
 * memory (w_x, w_y, w_z, shift), BN folded; copied into the chain. */
int s4g_chain_set_xyz_layer(s4g_chain* chain, const float* w4_host, int relu);
int s4g_chain_run_rows(const s4g_chain* chain, const void* in_rows, int in_stride, long long P, void* out,
                       int n_points, void* stream);
/* Refuses chains created with in_mode 6 (edge chains, below). */
int s4g_chain_run_gather(const s4g_chain* chain, const void* feat, const float* xyz, const float* ctr, const int* nbr,
                         int B, int N, int M, int K, void* out, void* stream);
/* Edge set abstraction (EdgeSAModule, pointnet2_utils/modules.py:250-284, fed by EdgeQueryGrouper, :202-221): the MLP's
 * first layer sees [x_j - x_c | f_j | f_j - f_c] (3 + 2C channels).  With its BN-folded weight split by those column
 * groups, W' = [W_x | W_a | W_b], that layer is
 *   [W_x | W_a + W_b] [x_j - x_c ; f_j] + b' + u_c,   u_c = -W_b f_c,
 * i.e. a plain gathered layer over 3 + C channels plus a term of the centroid alone.  A chain created with in_mode 6
 * (gathered max-pool, >= 2 layers, feat_c > 0, layer 0 = the 3 + C -> cout[0] weights [W_x | W_a + W_b]) adds
 * term[b * M + m][c] (bf16 [B*M][cout[0]], 16-byte aligned) to layer 0's shift, in fp32, for every row of centroid m's
 * group, before the ReLU and the bf16 rounding.  Refuses every other chain. */
int s4g_chain_run_gather_term(const s4g_chain* chain, const void* feat, const float* xyz, const float* ctr, const int* nbr,
                              const void* term, int B, int N, int M, int K, void* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device-side cloud pre-processing (csrc/preprocess.cu) — GraspDetector._pre_processing / sample_single_cloud
 * (grasp_detector.py:82-105) over transform_numpy_points (utils/math_utils.py:20-24).  The reference's voxelize() and
 * remove_outliers() discard the clouds open3d returns, so what it observably does is the axis change _REAL2TRAIN
 * and a random sub-sample: s4g_cloud_transform_select_f32, for a batch, with caller-supplied indices.
 * ------------------------------------------------------------------------------------------------ */
/* out[b,:,i] = (mat44 [cloud[b,:,index[b,i]]; 1])[:3].  cloud (B,3,n), index (B,m) int64 or NULL (identity, m == n),
 * mat44: 16 floats in HOST memory, row-major -> out (B,3,m). */
int s4g_cloud_transform_select_f32(const float* cloud, int B, int n, const int64_t* index, int m, const float* mat44,
                                   float* out, void* stream);
/* The intended (but inert in the reference) voxel filter, OUR definition: cell keys ((cz*ny + cy)*nx + cx) of a
 * (3,n) cloud on a grid of side `voxel` anchored at origin3 (host), and the per-voxel means given the sorted keys,
 * the sort permutation and the exclusive scan of the segment-start flags.  The radius-outlier filter is
 * s4g_ball_query_f32 with K = nb_points + 1 (count > nb_points keeps the point). */
int s4g_voxel_keys_f32(const float* cloud_3n, int n, const float* origin3, float voxel, const int* dims3, int64_t* key,
                       void* stream);
int s4g_voxel_means_f32(const float* cloud_3n, int n, const int64_t* sorted_key, const int64_t* order, const int* seg_rank,
                        float* out_3cap, int cap, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device-side grasp post-processing (csrc/postprocess.cu) — replaces the numpy / python tail of
 * GraspDetector: post_processing + orthogonalization (grasp_detector.py:124-185), the per-pose collision loop
 * (:214-232 over cloud_processor/view_collision_checker.py:37-65), importance sampling (:235-251), and adds
 * the translation de-duplication sketched at utils/file_logger_cls.py:220-225 (the reference ships no NMS).
 * All pointers are device pointers unless said otherwise.
 * ------------------------------------------------------------------------------------------------ */
/* softmax over the C score classes (fp32) and expectation with np.linspace(0,1,C+1)[1:] (fp64): (B,C,N) -> (B,N). */
int s4g_grasp_scores_f32(const float* score_logits, int B, int C, int N, double* score, void* stream);
/* threshold -> descending-score ranks -> verticalness filter, with the reference's indexing (see the file
 * header).  approach_row (HOST, 3 x fp64) = third row of -(camera2base_R @ TRAIN2REAL_R).  workspace: 2*B*N
 * int32.  n_out[b] may exceed max_out (then only max_out entries were written: enlarge and call again). */
int s4g_grasp_select(const double* score, const float* frame_R, int B, int N, double score_threshold,
                     double vertical_threshold, const double* approach_row, int* workspace, int max_out, int* out_point,
                     int* out_rot, int* n_out, int* n_high, void* stream);
/* translation decode + Gram-Schmidt + TRAIN2REAL: poses [B][max_out][4][4] fp64, out_score [B][max_out] fp64.
 * n_high and workspace are the outputs of s4g_grasp_select (the rank table lives in the workspace);
 * train2real (16 x fp64, row-major) and t_score (T x fp64) are HOST pointers. */
int s4g_grasp_poses(const float* points, const float* frame_R, const float* frame_t, const double* score, int B, int N,
                    int T, const int* out_point, const int* out_rot, const int* n_out, const int* n_high,
                    const int* workspace, int max_out, const double* train2real, const double* t_score, double* poses,
                    double* out_score, void* stream);
/* view_non_collision for every pose against the (n_points,3) cloud; ok[p] = 1 if the grasp is collision free.
 * gripper (HOST, 8 floats): finger_length, bottom_length, half_hand_thickness, half_bottom_width,
 * half_bottom_space, back_margin, back_threshold, finger_threshold.  counts (optional): [n_poses][2]. */
int s4g_grasp_collision_f32(const double* poses, int n_poses, const float* cloud_n3, int n_points, const float* gripper,
                            unsigned char* ok, int* counts, void* stream);
/* greedy de-duplication in the given order: drop a pose whose translation is within L1 distance min_dist of a
 * kept one.  kept: [n] int32, n_kept: 1 int32. */
int s4g_grasp_nms(const double* poses, const int* order, int n, double min_dist, int* kept, int* n_kept, void* stream);
/* importance sampling: cum = cumsum(exp(5 * scores)); picked[i] = first index with cum >= sorted_uniform[i] * cum[-1]. */
int s4g_grasp_importance_sample(const double* scores, int n, const double* sorted_uniform, int m, double* cum, int* picked,
                                void* stream);
/* The tail of GraspDetector.detect (grasp_detector.py:212-251) for a whole batch with no host round trip
 * (BASELINE config 5): collision test of every candidate (cloud (B,3,n_points) fp32, NULL = skip), ordered
 * compaction, optional de-duplication (nms_min_dist <= 0 = off; result in descending score order), importance
 * sampling with per-scene ascending uniforms [B][m] (device, NULL = first m) when more than m candidates are left,
 * else all of them.  poses / scores / n_cand as written by s4g_grasp_poses / s4g_grasp_select with max_out = cap.
 * Outputs: out_index [B][m] candidate indices, out_n [B], out_poses [B][m][16], out_scores [B][m]. */
size_t s4g_grasp_finish_batch_workspace(int B, int cap);
int s4g_grasp_finish_batch(const double* poses, const double* scores, const int* n_cand, int B, int cap,
                           const float* cloud_b3n, int n_points, const float* gripper, double nms_min_dist,
                           const double* sorted_uniform, int m, void* workspace, size_t workspace_bytes, int* out_index,
                           int* out_n, double* out_poses, double* out_scores, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* S4G_B200_H_ */
