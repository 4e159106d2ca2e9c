/*
 * clipnce.h -- C-ABI of the B200-native fused CLIP / InfoNCE hot path.
 *
 * The reference (SrikarK-code/clip-dplm) has no FFI of its own: the boundary of this path is the
 * tail of its model forwards and its loss functions (Python).  The entry points below are exactly
 * what a binding for that tail needs; each one names the reference lines it replaces (paths are
 * relative to the reference checkout).  `INTEGRATION.md` shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (e.g. the PyTorch caching allocator);
 *     the library never allocates or frees user-visible memory and never synchronises the host:
 *     all work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default);
 *   - matrices are dense row-major; "hat" buffers hold L2-normalised rows in the compute type:
 *     CLIPNCE_BF16 (tensor-core path, sm_100a tcgen05) or CLIPNCE_F32 (exact check mode, CUDA cores);
 *   - functions return 0 on success or a negative CLIPNCE_E* code; clipnce_last_error() returns a
 *     thread-local message.  No C++ exception crosses this boundary;
 *   - re-entrant: no global mutable state besides a mutex-guarded cache of kernel attributes.
 *
 * Notation:  Ahat_i = A_i / max(|A_i|, 1e-12),  S = s * Ahat Bhat^T,
 *            r_i = logsumexp_j S_ij,  c_j = logsumexp_i S_ij.
 */
#ifndef CLIPNCE_H_
#define CLIPNCE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLIPNCE_VERSION 110

/* element types */
#define CLIPNCE_BF16 0
#define CLIPNCE_F32  1

/* flags */
#define CLIPNCE_FLAG_FORCE_EXACT 1   /* use the CUDA-core exact (online-max) kernels even for bf16 */
#define CLIPNCE_FLAG_UNBOUNDED   2   /* |S_ij| <= s does not hold (un-normalised extra columns, tong/utils/losses.py:10-14):
                                        tensor-core kernels with true running maxima instead of the fixed shift */

/* error codes */
#define CLIPNCE_OK            0
#define CLIPNCE_EINVAL       -1      /* bad argument (null pointer, bad dtype, bad shape/alignment) */
#define CLIPNCE_EWORKSPACE   -2      /* workspace too small */
#define CLIPNCE_ECUDA        -3      /* CUDA runtime / driver error (message has the detail) */
#define CLIPNCE_EUNSUPPORTED -4      /* device is not sm_100 or shape outside every kernel's range */

int         clipnce_version(void);
const char* clipnce_last_error(void);

/* Kernel family serving (dtype, d, scale, flags):
 *   0  exact CUDA-core kernels (dtype F32, d % 8 != 0, d > 768, CLIPNCE_FLAG_FORCE_EXACT);
 *   1  tcgen05 tensor-core kernels with the fixed shift exp(S - s)   (2 * scale <= 80 and |S| <= s);
 *   2  tcgen05 kernels with per-row / per-column shifts (two-exponential backward): larger scales -- exp().clamp(max=100),
 *      old/clip_opt.py:100 -- and CLIPNCE_FLAG_UNBOUNDED; d % 128 == 0.  With bounded logits (no CLIPNCE_FLAG_UNBOUNDED)
 *      clipnce_forward first runs ONE fixed-shift sweep with the shift lowered to s - 72 and returns its sums as exactly
 *      rescaled (shift, sum) pairs; a row or column whose every logit lies below s - 134 raises a device flag, and the
 *      exact online soft-max sweeps enqueued behind it (true running maxima, one launch for the rows, one for the columns)
 *      run only then: the results are the same in every case, the common one costs a single sweep, nothing reads the host. */
int clipnce_uses_tensor_cores(int dtype, int64_t d, float scale, int flags);

/* 1 if clipnce_backward needs the transposed copy y_t for these arguments.  The CTA-pair kernels (d % 128 == 0,
 * d <= 768) read the streamed rows directly as an MN-major MMA operand and take y_t = NULL; only the single-CTA
 * tensor-core kernels (other d % 8 == 0 up to 768) stream a transposed copy. */
int clipnce_needs_transposed(int dtype, int64_t d, float scale, int flags);

/* Bytes of scratch clipnce_forward / clipnce_backward need for these shapes (max of the two). */
int clipnce_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t d, int dtype, int flags, size_t* out);

/*
 * Row norms (and, optionally, the normalised rows).  Replaces F.normalize(x, dim=-1):
 *   old/clip.py:63-64,100-101  run1/full.py:47-48,73-74  old/clip_opt.py:93-94
 *   current/rna_clip_codes.ipynb:1948-1949  current/tf_clip_codes (1).ipynb:13146-13148
 *   tong/utils/losses.py:6-7
 * x      [n,d]  in_dtype (BF16 or F32)
 * rinv   [n]    f32   1 / max(|x_i|, 1e-12)
 * x_hat  [n,d]  hat_dtype or NULL: normalised rows (what the reference returns as "*_embeds").
 * The contraction kernels do NOT consume x_hat: they take the raw rows plus rinv and apply
 * rinv_x[i] * rinv_y[j] to the fp32 accumulator ("normalise fused into the GEMM"), so the
 * tensor cores see the caller's exact bf16 values and no second rounding enters the logits.
 */
int clipnce_normalize(const void* x, int in_dtype, int64_t n, int64_t d, float* rinv,
                      void* x_hat, int hat_dtype, void* stream);

/*
 * Operand staging for the contraction kernels: x_c = x converted to c_dtype ([n,d], or NULL when x
 * already has that type) and x_c_t = the same values transposed ([d,ld_t], ld_t >= n, ld_t % 8 == 0,
 * or NULL).  The tensor-core backward streams the transposed copy as its second MMA operand; it is
 * also what is built from the all-gathered embeddings (old/clip_opt.py:102-112, run1/full.py:77-84).
 */
int clipnce_stage_operand(const void* x, int in_dtype, int64_t n, int64_t d, void* x_c, void* x_c_t,
                          int64_t ld_t, int c_dtype, void* stream);

/*
 * Forward statistics of S_ij = s * rinv_x[i] rinv_y[j] <x_i, y_j> without materialising S.  Replaces
 *   torch.matmul(a, b.t()) * logit_scale            old/clip.py:67,104  run1/full.py:50,85
 *                                                   old/clip_opt.py:115-121  rna_clip_codes.ipynb:1951
 *                                                   tf_clip_codes (1).ipynb:13152-13154  tong/utils/losses.py:14
 *   F.cross_entropy(S, arange) / F.cross_entropy(S.t(), arange)   (the log-sum-exp halves of it)
 *                                                   rna_clip_codes.ipynb:1952-1953  old/clip_opt.py:148-149
 *                                                   run1/full.py:98-99,133  tong/utils/losses.py:17-19
 * x [n_rows,d], y [n_cols,d]   raw rows in `dtype`: the rows local to this rank / all (gathered) columns
 * rinv_x [n_rows], rinv_y [n_cols]   from clipnce_normalize
 * diag_offset   column of row 0's positive: the positive of local row i is column i + diag_offset
 *               (0 on one GPU, rank * n_rows under the row-sharded global batch)
 * scale         s = exp(logit_scale), already clamped by the caller (old/clip_opt.py:100)
 * scale_dev     optional DEVICE scalar (f32) holding s.  When non-NULL the kernels read s from it and `scale` is only
 *               the host's (possibly one step old) hint used to pick the kernel family: the step then needs no host
 *               read of the logit_scale parameter and can be captured in a CUDA graph.  NULL: `scale` is used.
 * Log-sum-exps are returned as (max-like shift m, sum l = sum exp(S - m)) PAIRS and never collapsed
 * to a single float inside the library: r_i = row_m_i + log(row_l_i).  Keeping the pair is what lets the
 * backward form soft-max probabilities as exp(S - m) / l with full fp32 relative accuracy (the way
 * ATen's log_softmax does) -- a rounded r_i ~ 14 would cost 1e-6 absolute, i.e. 1e-4 relative on
 * 1 - p_ii once the model separates the positives.
 * row_m, row_l [n_rows]  complete (every column is seen locally)
 * col_m, col_l [n_cols]  partial column statistics over the LOCAL rows; across ranks:
 *               M_j = max col_m_j,  L_j = sum col_l_j * exp(col_m_j - M_j)
 * diag [n_rows]     S_{i, i+diag_offset}
 */
int clipnce_forward(const void* x, const void* y, const float* rinv_x, const float* rinv_y,
                    int64_t n_rows, int64_t n_cols, int64_t d,
                    int64_t diag_offset, float scale, const float* scale_dev, int dtype, int flags,
                    float* row_m, float* row_l, float* col_m, float* col_l, float* diag,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * One side of the backward.  Replaces autograd through cross_entropy + matmul (loss.backward():
 * rna_clip_codes.ipynb:2074, run1/full.py:134, old/clip_opt.py:167, old/ablation.py:16-17).
 * The logit tiles are recomputed; with
 *     G_ij = exp(S_ij - row_m_i) row_w_i + exp(S_ij - col_m_j) col_w_j - diag_w * [j == i + diag_offset]
 * it returns  dx_hat = grad_out * s * G Yhat  ([n_rows,d] f32; Yhat_j = rinv_y[j] y_j)  and
 *             *d_scale_sum += grad_out * sum_ij G_ij S_ij   (= dL/dlogit_scale when s = exp(logit_scale)).
 * Symmetric InfoNCE over a global batch N:
 *     row_w_i = 1 / (2N row_l_i),  col_w_j = 1 / (2N col_l_j),  diag_w = 1/N      (clipnce_softmax_weights)
 * one-directional (run1/full.py:133, tong/utils/losses.py:19): row_w_i = 1 / (N row_l_i), col_m = col_w = NULL.
 * Columns without positives (hard-negative cache, old/clip_opt.py:118-121) carry col_w_j = 0.
 * Call it once as (A, B, B^T, rinv_a, rinv_b, row, col, +offset) for dAhat and once as
 * (B, A, A^T, rinv_b, rinv_a, col, row, -offset) for dBhat.
 * y_t [d,ld_t] (clipnce_stage_operand) is only read when clipnce_needs_transposed() says so (NULL otherwise).
 * col_m/col_w (together) and d_scale_sum may be NULL.
 */
int clipnce_backward(const void* x, const void* y, const void* y_t, int64_t ld_t,
                     const float* rinv_x, const float* rinv_y,
                     int64_t n_rows, int64_t n_cols, int64_t d, int64_t diag_offset, float scale,
                     const float* scale_dev,
                     const float* row_m, const float* row_w, const float* col_m, const float* col_w,
                     float diag_w, float grad_out,
                     int dtype, int flags, float* dx_hat, float* d_scale_sum,
                     void* workspace, size_t workspace_bytes, void* stream);

/*
 * clipnce_backward followed by clipnce_normalize_backward as ONE call: returns the gradient of the caller's rows,
 *     dx_i = rinv_i (g_i - xhat_i (xhat_i . g_i)) * grad_scale,   g = s * G Yhat  (grad_out = 1),
 * in out_dtype, and *d_scale_sum += sum_ij G_ij S_ij.  The fp32 gradient of the normalised rows never leaves the
 * workspace: the per-work-item partial gradients of the CTA-pair kernels (column sweep split over the SMs when there
 * are few row blocks -- the row-sharded step), the row dots <xhat_i, g_i> that give sum G.S, and the normalise backward
 * are finished by one pass (`aux::finish_rows`) instead of three.
 * x_orig [n_rows,d] in_dtype: the caller's rows (x itself when in_dtype == dtype; fp32 rows of a bf16 step otherwise).
 * grad_scale: optional DEVICE scalar, the upstream gradient of the loss (NULL = 1).
 * workspace: clipnce_workspace_bytes() for these shapes (it includes the [n_rows,d] fp32 slab this call uses).
 */
int clipnce_backward_dx(const void* x, const void* y, const void* y_t, int64_t ld_t,
                        const float* rinv_x, const float* rinv_y,
                        int64_t n_rows, int64_t n_cols, int64_t d, int64_t diag_offset, float scale,
                        const float* scale_dev,
                        const float* row_m, const float* row_w, const float* col_m, const float* col_w,
                        float diag_w, int dtype, int flags,
                        const void* x_orig, int in_dtype, const float* grad_scale, void* dx, int out_dtype,
                        float* d_scale_sum, void* workspace, size_t workspace_bytes, void* stream);

/*
 * BOTH backward sides of the single-GPU symmetric step in ONE sweep over the logits tiles (8 N^2 d executed per step
 * instead of the 10 N^2 d of two clipnce_backward_dx calls): `loss.backward()` of current/rna_clip_codes.ipynb:2074,
 * run1/full.py:134, old/clip_opt.py:167.  A persistent role-specialised kernel (csrc/kernels_pair2.cuh): producer CTA
 * pairs recompute S, form the bf16 gradient tile G once, accumulate dA_hat and hand G through an L2-resident ring to
 * consumer pairs that accumulate dB_hat = G^T A_hat.
 * x = A rows, y = B rows [n,d] bf16 (n_rows == n_cols == n, positives on the diagonal), statistics as for
 * clipnce_backward_dx (row_* of the rows of x, col_* of the rows of y).  dx / dy [n,d] out_dtype: gradients of the
 * caller's rows x_orig / y_orig (the normalise backward and grad_scale are applied as in clipnce_backward_dx);
 * d_scale_sum [1] += sum_ij G_ij S_ij (or NULL).
 * clipnce_backward_both_workspace_bytes() returns 0 bytes in *out when the shape is not served (then use two
 * clipnce_backward_dx calls): bf16, kernel family 1 or 2 without CLIPNCE_FLAG_UNBOUNDED, d in {128,...,768}, n_rows % 128 == 0,
 * n_cols % 256 == 0, n_rows * n_cols >= 12288^2, and a device on which all CTA pairs of the persistent grid are
 * co-resident.  world = 0: one GPU (n_rows == n_cols); world >= 2: the row-sharded step below.  CLIPNCE_NO_BWD2=1
 * disables the path.
 */
int clipnce_backward_both_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t d, int dtype, float scale, int flags,
                                          int world, size_t* out);
int clipnce_backward_both_dx(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n,
                             int64_t d, float scale, const float* scale_dev,
                             const float* row_m, const float* row_w, const float* col_m, const float* col_w,
                             float diag_w, int dtype, int flags,
                             const void* x_orig, const void* y_orig, int in_dtype, const float* grad_scale,
                             void* dx, void* dy, int out_dtype, float* d_scale_sum,
                             void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same sweep for the ROW-SHARDED global batch (SURVEY.md section 8e; replaces what autograd + DDP do behind the
 * reference's all_gather formulation, old/clip_opt.py:102-112, run1/full.py:77-84): x = this rank's A rows [n_rows,d],
 * y = ALL ranks' B rows [n_cols,d] (n_cols = world * n_rows, rank r owns columns [r n_rows, (r+1) n_rows)),
 * diag_offset = rank * n_rows, row_* for the local rows, col_* for all columns.  One kernel is the contraction AND the
 * reduce-scatter of the partial dB: the segment slabs of dA_hat stay in `workspace`; the partial dB_hat of the columns
 * owned by rank s is stored, as it completes, straight into rank s's buffer over NVLink peer memory at
 *   peer_base[s] + slots_offset + rank * n_rows * d * 4        ([world][n_rows, d] f32 slots per rank).
 * After a barrier (clipnce_link_barrier) every rank finishes both sides with clipnce_finish_sharded.  peer_base: see the
 * exchange section below.
 */
int clipnce_backward_both_sharded(const void* x, const void* y, const float* rinv_x, const float* rinv_y,
                                  int64_t n_rows, int64_t n_cols, int64_t d, int64_t diag_offset, float scale,
                                  const float* scale_dev,
                                  const float* row_m, const float* row_w, const float* col_m, const float* col_w,
                                  float diag_w, int dtype, int flags,
                                  void* const* peer_base, int world, int rank, int64_t slots_offset,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* Both tails of clipnce_backward_both_sharded, to be enqueued behind the barrier with the sweep's `workspace`:
 * dx = normalise-backward(sum of the dA_hat slabs), dy = normalise-backward(sum of the world slots, in rank order),
 * d_scale_sum += sum G.S (or NULL).  y_local / y_orig / rinv_y_local: this rank's B rows [n_rows,d].  x_orig and dx have
 * the types x_in_dtype and x_out_dtype, y_orig and dy the types y_in_dtype and y_out_dtype, with the rules of
 * clipnce_backward_dx.  Sides of the same types are finished in ONE launch, so that they share the GPU instead of
 * queueing behind each other; otherwise one launch per side. */
int clipnce_finish_sharded(const void* x, const void* x_orig, const float* rinv_x, void* dx, const void* y_local,
                           const void* y_orig, const float* rinv_y_local, void* dy, const float* slots, int64_t n_rows,
                           int64_t n_cols, int64_t d, int dtype, float scale, int flags, int world, int x_in_dtype,
                           int x_out_dtype, int y_in_dtype, int y_out_dtype, const float* grad_scale, float* d_scale_sum,
                           void* workspace, size_t workspace_bytes, void* stream);

/*
 * Several pair problems of equal shape as ONE launch per kernel: the tri-modal model, whose three symmetric InfoNCE losses
 * (cell, pert), (cell, protein), (pert, protein) share one logit_scale and whose every embedding is an operand of two pairs
 *   current/tf_clip_codes (1).ipynb:13146-13165      (three matmul * logit_scale, six cross_entropy, summed)
 * At the batch sizes that model runs at a single pair leaves most of the GPU idle (N = 4096: 16 of 74 CTA-pair slots);
 * here the problems are the diagonal blocks of one virtual sweep and the backward runs BOTH sides of ALL problems in one
 * launch, followed by one pass that sums each member's contributions, applies the normalise backward and emits the
 * squared norm of the embedding gradients (what clip_grad_norm_, rna_clip_codes.ipynb:2076, would otherwise re-read them for).
 *
 * stack      [n_members * n_pad, d] bf16: member m's rows at [m n_pad, m n_pad + n), n_pad = n rounded up to 256; the
 *            padding rows must hold finite values (zeros).  rinv [n_members * n_pad] from ONE clipnce_normalize call.
 * problem k  rows of member x_member[k] against the rows of member y_member[k] (HOST arrays), k < n_prob <= 4,
 *            n_members <= 4; positives on the diagonal.
 * stat_m, stat_l [2][n_prob * n_pad]: row statistics of problem k at [k n_pad + i], column statistics at
 *            [n_prob n_pad + k n_pad + j] -- (shift, sum) pairs as in clipnce_forward; diag [n_prob * n_pad].
 * loss       [n_prob + 1]: the mean symmetric loss of every problem and, last, their sum.
 * clipnce_group_workspace_bytes returns 0 in *out when the group is not served (then issue the problems one by one):
 * bf16, d % 128 == 0, d <= 768, kernel families 1 and 2, no CLIPNCE_FLAG_UNBOUNDED.
 */
int clipnce_group_workspace_bytes(int n_members, int n_prob, int64_t n, int64_t d, int dtype, float scale, int flags,
                                  size_t* out);
int clipnce_group_forward(const void* stack, const float* rinv, int n_members, int n_prob, const int* x_member,
                          const int* y_member, int64_t n, int64_t d, float scale, const float* scale_dev, int dtype,
                          int flags, float* stat_m, float* stat_l, float* diag, float* loss, void* workspace,
                          size_t workspace_bytes, void* stream);
/* grad_scale: optional DEVICE [n_prob] upstream gradients of the problems' losses (NULL = 1 each).
 * d_stack [n_members * n_pad, d] out_dtype: gradient of the caller's rows stack_orig (in_dtype; the stack itself for bf16
 * rows); rows of the padding are not written.  *d_scale_sum += sum_k grad_scale[k] sum_ij G_ij S_ij (or NULL).
 * grad_sumsq [n_members] (or NULL): sum over member m's rows of |d_stack row|^2. */
int clipnce_group_backward(const void* stack, const float* rinv, int n_members, int n_prob, const int* x_member,
                           const int* y_member, int64_t n, int64_t d, float scale, const float* scale_dev,
                           const float* stat_m, const float* stat_l, int dtype, int flags, const void* stack_orig,
                           int in_dtype, const float* grad_scale, void* d_stack, int out_dtype, float* d_scale_sum,
                           float* grad_sumsq, void* workspace, size_t workspace_bytes, void* stream);

/* w_i = coef / l_i  (l = +inf -> 0).  Builds row_w / col_w from the forward's sums. */
int clipnce_softmax_weights(const float* l, int64_t n, float coef, float* w, void* stream);

/* lse_i = m_i + log(l_i)  (reporting only; the kernels consume the pairs). */
int clipnce_combine_lse(const float* m, const float* l, int64_t n, float* lse, void* stream);

/* Backward of the normalise: dx_i = rinv_i * (g_i - xhat_i (xhat_i . g_i)), xhat_i = x_i * rinv_i
 * (rows clamped at eps get dx_i = g_i * rinv_i, like clamp_min's sub-gradient).
 * x [n,d] in_dtype, dx_hat [n,d] f32, dx [n,d] out_dtype.  grad_scale: optional DEVICE scalar (f32)
 * multiplied into dx -- the upstream gradient of the loss, read on the device so that autograd's
 * grad_output never forces a host synchronisation; NULL = 1. */
int clipnce_normalize_backward(const void* x, int in_dtype, const float* rinv, const float* dx_hat,
                               const float* grad_scale, int64_t n, int64_t d, void* dx, int out_dtype,
                               void* stream);

/* loss[0] = [ sum_i (r_i - diag_i) + (symmetric ? sum_i (c_{i+diag_offset} - diag_i) : 0) ]
 *           / (symmetric ? 2 n_global : n_global)   with r = row_m + log row_l, c = col_m + log col_l,
 * summed in fp64 in a fixed order (deterministic).  Mean reduction of F.cross_entropy
 * (rna_clip_codes.ipynb:1953); under row sharding every rank contributes its rows' part. */
int clipnce_loss(const float* row_m, const float* row_l, const float* col_m, const float* col_l,
                 const float* diag, int64_t n_rows, int64_t diag_offset, int64_t n_global, int symmetric,
                 float* loss, void* stream);

/*
 * Retrieval: for every query row the k library rows of highest cosine similarity, without materialising the
 * [n_q, n_lib] similarity matrix.  Replaces the evaluation tail of the reference
 *   preds = logits.argmax(dim=1)                                        run1/full.py:152 (k = 1), :138-139, :265
 *   F.cosine_similarity(a.unsqueeze(1), b.unsqueeze(0), dim=2)          run1/full.py:157 ([N,N,d] intermediate)
 * and serves BASELINE.json config 5 (1M-entry protein library x 16k TF queries, top-10): the library is sharded by
 * rows over the ranks, each rank calls this on its shard with col_offset = first global row of the shard and the
 * [n_q, k] candidates of the ranks are merged by score.
 * q [n_q,d], lib [n_lib,d] raw bf16 rows; rinv_* from clipnce_normalize; scores are rinv_q[i] rinv_lib[j] <q_i, lib_j>.
 * out_score [n_q,k] f32 descending, out_idx [n_q,k] i64 = col_offset + j (ties: lower index first; -1 / -inf pad when
 * n_lib < k).  Same tcgen05 CTA-pair sweep as clipnce_forward with a running top-k per row in the epilogue; served for
 * CLIPNCE_BF16, d in {128, 256, 384, 512}, 1 <= k <= 16 -- anything else returns CLIPNCE_EUNSUPPORTED.
 */
int clipnce_topk_workspace_bytes(int64_t n_q, int64_t n_lib, int64_t d, int k, int dtype, size_t* out);
int clipnce_topk(const void* q, const void* lib, const float* rinv_q, const float* rinv_lib,
                 int64_t n_q, int64_t n_lib, int64_t d, int64_t col_offset, int k, int dtype,
                 float* out_score, int64_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Projection-head tail fused in front of the loss (the last two layers of the reference's heads + the normalise):
 *   e = nn.LayerNorm(p)(nn.Linear(k, p)(h))     old/clip.py:26-33, old/clip_opt.py:16-44, rna_clip_codes.ipynb:1901-1909
 *   rinv = 1 / max(|e|, 1e-12)                  F.normalize, old/clip.py:63-64
 * One tcgen05 GEMM whose epilogue is the LayerNorm and the row norm (the output row of p <= 512 columns lives in one
 * CTA's TMEM, so both are thread-local).  h [n,k] bf16, w [p,k] bf16 (nn.Linear's layout), bias/gamma/beta [p] f32
 * (bias may be NULL); e [n,p] bf16 and rinv [n] feed clipnce_forward / clipnce_backward* directly; zhat [n,p] bf16 and
 * rstd [n] (both optional) are what clipnce_head_tail_backward needs.  Served for k % 64 == 0, p in {128,256,384,512}.
 */
int clipnce_head_tail(const void* h, const void* w, const float* bias, const float* gamma, const float* beta, int64_t n,
                      int64_t k, int64_t p, float ln_eps, void* e, void* zhat, float* rstd, float* rinv, void* stream);
/* LayerNorm backward of the tail: dz = rstd (g - mean(g) - z_hat mean(g z_hat)), g = de * gamma; de [n,p] de_dtype,
 * dz [n,p] bf16 -- the operand of the two GEMMs dW = dz^T h, dh = dz W (plain library GEMMs, left to the caller). */
int clipnce_head_tail_backward(const void* de, int de_dtype, const void* zhat, const float* rstd, const float* gamma,
                               int64_t n, int64_t p, void* dz, void* stream);

/*
 * Exchange steps of the row-sharded global batch over NVLink / NVSwitch peer memory.  Replaces the reference's
 *   dist.all_gather(...) x2 + torch.cat      old/clip_opt.py:102-112   run1/full.py:77-84
 * (which also cuts autograd: the gathered negatives carry no gradient there; here gradients stay exact).
 *
 * Every rank allocates ONE buffer of the same size and layout and maps all ranks' buffers into its address space
 * (CUDA VMM / IPC handles, exchanged once by the host -- torch symmetric memory in this repository's Python host).
 * peer_base is a HOST array of `world` DEVICE pointers: peer_base[r] = rank r's buffer as addressed from this GPU
 * (peer_base[rank] = the own buffer).  The first clipnce_link_control_bytes() bytes of every buffer are the control
 * block (arrival flags, device-side epoch counters, a status word, scalar slots): zero it once before the first call
 * and leave it alone.  Everything else is laid out by the caller and addressed by BYTE OFFSETS from the base.
 * All calls enqueue on `stream`, never synchronise the host, and keep their epochs on the device, so a step that
 * contains them can be captured once in a CUDA graph and replayed.  Ranks must issue the same sequence of calls.
 * A peer that does not arrive within CLIPNCE_LINK_TIMEOUT_MS (default 600000 = 10 minutes, the order of NCCL's
 * watchdog) is FATAL: the waiting kernel records 1 + phase in the status word (u32 at status_offset of the own buffer,
 * for the post-mortem) and traps, so the CUDA error surfaces at the caller's next synchronisation -- a step never
 * continues on peer buffers that were not synchronised.
 */
int clipnce_link_control_bytes(int64_t* control_bytes, int64_t* status_offset);

/* Barrier `phase` (0..7; use a different phase for every exchange point of a step): every store this GPU issued
 * before it -- into peer buffers too -- is visible to kernels the peers launch after THEIR barrier of the same phase. */
int clipnce_link_barrier(void* const* peer_base, int world, int rank, int phase, void* stream);

/* Fused F.normalize row norms + all-gather: x [n,d] (in_dtype) -> rinv_i = 1 / max(|x_i|, 1e-12) and the rows,
 * converted to c_dtype, are stored into EVERY rank's buffer: rows at rows_offset + (row0 + i) * d * sizeof(c_dtype),
 * rinv at rinv_offset + (row0 + i) * 4.  row0 = rank * n.  Publish with clipnce_link_barrier.
 * The push takes the whole GPU: issue it where nothing else runs (the columns, before the forward sweep); rows that
 * travel beside a contraction kernel go by clipnce_link_copy. */
int clipnce_link_push_rows(const void* x, int in_dtype, int64_t n, int64_t d, int c_dtype, void* const* peer_base,
                           int world, int rank, int64_t rows_offset, int64_t rinv_offset, int64_t row0, void* stream);

/* Copy `bytes` from src to byte offset dst_offset of every rank's buffer with the COPY ENGINES (cudaMemcpyAsync per
 * peer, no SM involved): the background gather of rows that travel beside a contraction kernel -- the A rows, read by
 * the backward only -- which keeps every SM.  Publish with a barrier on a stream that waited for this one. */
int clipnce_link_copy(const void* src, size_t bytes, void* const* peer_base, int world, int rank, int64_t dst_offset,
                      void* stream);

/*
 * The gather of the columns BESIDE the forward sweep (replaces clipnce_link_push_rows + clipnce_link_barrier before
 * clipnce_forward; the reference's dist.all_gather is a blocking call in front of its matmul, old/clip_opt.py:102-112):
 *   clipnce_link_epoch_advance   opens phase `phase` of a new step on this GPU (one tiny kernel on the step's stream);
 *   clipnce_link_send_blocks     on a SIDE stream that waited for it: the copy engines deliver this rank's rows
 *                                (row_bytes at rows_offset) and 1/norms (rinv_bytes at rinv_offset) to every peer, the peer
 *                                that sweeps this block first served first, each delivery followed by a flag for that peer.
 *                                The caller copies its own block into its own buffer itself (on the step's stream);
 *   clipnce_forward_gathered     clipnce_forward over x = the local rows and y = the gathered buffer [world * n_rows, d]
 *                                (rinv_y likewise), diag_offset = rank * n_rows, sweeping the column blocks in the order
 *                                rank, rank + 1, ... and waiting for a block's flag before its first load -- the sweep
 *                                starts on the local block at once and the transfers hide behind it.  Served where
 *                                clipnce_forward_gathered_ok() says so (the CTA-pair kernels with a fixed-shift sweep:
 *                                family 1, and family 2 with bounded logits -- a function of type, d and flags only,
 *                                so that every rank of a step answers alike); otherwise gather with push_rows + barrier.
 * All ranks must take the same route in a step.  The side stream must be joined before the step's next barrier.
 */
int clipnce_link_epoch_advance(void* const* peer_base, int world, int rank, int phase, void* stream);
int clipnce_link_send_blocks(const void* rows, size_t row_bytes, const float* rinv, size_t rinv_bytes, void* const* peer_base,
                             int world, int rank, int64_t rows_offset, int64_t rinv_offset, int phase, void* stream);
int clipnce_forward_gathered_ok(int dtype, int64_t d, float scale, int flags);
int clipnce_forward_gathered(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n_rows,
                             int64_t n_cols, int64_t d, float scale, const float* scale_dev, int dtype, int flags,
                             float* row_m, float* row_l, float* col_m, float* col_l, float* diag, void* const* peer_base,
                             int world, int rank, int phase, void* workspace, size_t workspace_bytes, void* stream);

/* Copy n_seg (<= 4) local f32 vectors src[k][0..n[k]) to byte offset dst_offset[k] of every rank's buffer
 * (the statistics exchange after the forward sweep).  src, n, dst_offset are HOST arrays.  Publish with a barrier. */
int clipnce_link_push_f32(const float* const* src, const int64_t* n, const int64_t* dst_offset, int n_seg,
                          void* const* peer_base, int world, int rank, void* stream);

/* out[c] = sum over ranks of vals[c], c < cnt <= 8, in ONE kernel (push + barrier `phase` + fixed-order sum: every
 * rank gets bit-identical results).  Used for the scalar loss and for d logit_scale; being a barrier it also closes
 * the step: no peer touches this rank's gathered rows after it. */
int clipnce_link_sum_scalars(const float* vals, int cnt, void* const* peer_base, int world, int rank, int phase,
                             float* out, void* stream);

/* Combine n_part partial (shift, sum) pairs per entry, part_*[p * ld + i], in fixed order:
 * M_i = max_p m, L_i = sum_p l * exp(m - M_i)   (the column statistics of the ranks' row blocks). */
int clipnce_combine_partials(const float* part_m, const float* part_l, int n_part, int64_t ld, int64_t n, float* out_m,
                             float* out_l, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLIPNCE_H_ */
