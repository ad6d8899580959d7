/* summarizer_b200 — C ABI of libsummarizer_b200.so (hand-written sm_100a kernels).
 *
 * The reference (sylvainma/Summarizer) is pure Python and has NO FFI/plugin interface
 * (SURVEY.md §8b); this header therefore *defines* the boundary that sits directly beneath
 * the reference's Python surface.  Each entry point names the reference function(s) it
 * replaces (paths relative to /root/reference/summarizer/).  INTEGRATION.md shows the ctypes
 * stub a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain C types only.  Every function returns int: 0 = ok,
 *     SMZ_ERR_ARG (-1) bad argument/shape, SMZ_ERR_CUDA (-2) CUDA error,
 *     SMZ_ERR_UNSUPPORTED (-3) configuration outside the kernels' plan,
 *     SMZ_ERR_DEVICE (-5) not an sm_100 device.  smz_last_error() gives the message
 *     (thread-local).  Nothing throws.
 *   - All data pointers are DEVICE pointers owned by the caller unless the name starts with
 *     h_.  The library never allocates or frees device memory and never synchronises the
 *     host: work is enqueued on `stream` (a cudaStream_t passed as void*).  Work buffers are
 *     caller-provided and sized by the matching *_workspace_bytes function.
 *   - Ragged batches ("video batches") are described by an array of smz_video_desc in
 *     device memory; all packed arrays are indexed through its element offsets.
 *   - There is no CPU fallback and no other backend.
 */
#ifndef SUMMARIZER_B200_H
#define SUMMARIZER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMZ_OK 0
#define SMZ_ERR_ARG (-1)
#define SMZ_ERR_CUDA (-2)
#define SMZ_ERR_UNSUPPORTED (-3)
#define SMZ_ERR_NCCL (-4)
#define SMZ_ERR_DEVICE (-5)

#define SMZ_METHOD_KNAPSACK 0 /* utils/eval.py:98-99  */
#define SMZ_METHOD_RANK 1     /* utils/eval.py:100-107 */

/* per-video status bits written by smz_select_shots */
#define SMZ_STATUS_VALUE_RANGE 1 /* |int(score*1000)| * n_segs exceeds 2^29 (the int32 DP and its sign-bit take test); value clipped */
#define SMZ_STATUS_INTERVALS 2   /* more upsample intervals than scores+1 (reference: IndexError) */
#define SMZ_STATUS_WEIGHT_RANGE 4 /* a segment is longer than the max_seg_frames the caller declared */

/* frames handled by one CTA of the F-score kernel */
#define SMZ_FSCORE_CHUNK 2048

/* One video of a ragged batch.  Offsets are ELEMENT offsets into the packed arrays. 104 bytes. */
typedef struct smz_video_desc {
    int64_t score_off;   /* scores[]        float32, n_scores entries  (model output, one per step)      */
    int64_t picks_off;   /* picks[]         int32,   n_picks entries   (dataset /picks, ascending)        */
    int64_t seg_off;     /* cps[2*(seg_off+s)+{0,1}], nfps[seg_off+s]; per-segment outputs use it too    */
    int64_t user_off;    /* user_summary[]  float32, row u at user_off + u*user_ld, n_frames per row      */
    int64_t user_ld;     /* row stride (elements).  user_off%4==0 && user_ld%4==0 enables 128-bit loads   */
    int64_t summ_off;    /* machine_summary[] float32 output, summ_len = sum(nfps) entries                */
    int64_t frame_off;   /* frame_scores[]  float32 output of smz_upsample, n_frames entries              */
    int64_t mask_off;    /* summary bit mask (uint32 words), ceil(n_frames/32) words                      */
    int64_t ucount_off;  /* per-user outputs (overlap, gsum, f): n_users entries                          */
    int32_t n_scores, n_picks, n_segs, n_users;
    int32_t n_frames;    /* dataset /n_frames                                                             */
    int32_t summ_len;    /* sum(nfps) (utils/eval.py:111-122 output length; may differ from n_frames)     */
    int32_t capacity;    /* int(floor(n_frames * proportion)) computed in float64 (utils/eval.py:96)      */
    int32_t reserved;    /* must be 0                                                                     */
} smz_video_desc;

/* ---- library ------------------------------------------------------------------------- */
const char *smz_version(void);
const char *smz_last_error(void);
/* 0 when the current CUDA device is compute capability 10.x; SMZ_ERR_DEVICE otherwise. */
int smz_device_check(void);
/* SMZ_PROFILE=1 (development aid): prints the per-step device times collected so far to stderr. */
void smz_profile_report(void);

/* ---- shot selection: replaces utils/eval.py:74-123 generate_summary (+ utils/eval.py:15-35
 *      upsample inlined, utils/knapsack.py:5-23 knapsack_ortools incl. the OR-tools DP) ------
 * For every video v < n_videos:  upsample scores -> float32 numpy-pairwise segment means ->
 * values = trunc(double(mean)*1000) -> 0/1 knapsack (OR-tools DP semantics) or rank greedy ->
 * summary vector (float32 0/1, summ_len entries), the same summary as a bit mask truncated/
 * padded to n_frames, and msum = popcount(mask).
 * Outputs (per-segment arrays indexed seg_off+s; any may be NULL except picked/mask/msum):
 *   seg_mean float32, values int32, picked uint8, summary float32, mask uint32, msum int32[n_videos],
 *   status int32[n_videos] (0 = ok, SMZ_STATUS_* bits otherwise).
 * max_* are maxima over the batch (host knowledge; they size shared memory / the work buffer);
 * max_seg_frames = max(nfps).  values (and seg_mean for method 'rank') are required: they carry
 * the pooled scores from the pooling kernel to the DP kernel.
 * ws/ws_bytes: work buffer of at least smz_select_workspace_bytes(...) bytes (may be NULL/0
 * when that function returns 0). */
int smz_select_workspace_bytes(int n_videos, int max_n_segs, int max_capacity, int max_n_frames,
                               int max_seg_frames, int64_t *bytes);
int smz_select_shots(const smz_video_desc *desc, int n_videos, const float *scores, const int32_t *picks,
                     const int32_t *cps, const int32_t *nfps, int method, int max_n_segs, int max_capacity,
                     int max_n_frames, int max_seg_frames, float *seg_mean, int32_t *values, uint8_t *picked,
                     float *summary, uint32_t *mask, int32_t *msum, int32_t *status, void *ws, int64_t ws_bytes,
                     void *stream);

/* Stand-alone 0/1 knapsack: replaces utils/knapsack.py:5-23 knapsack_ortools when the caller
 * already holds the quantised int values (values[seg_off+s]); weights are nfps, the capacity is
 * desc.capacity.  Only n_segs, seg_off, capacity, n_frames (mask length, may be 0), mask_off are
 * read from the descriptor.  mask/msum may be NULL (then only picked[] is produced). */
int smz_knapsack(const smz_video_desc *desc, int n_videos, const int32_t *values, const int32_t *nfps,
                 int max_n_segs, int max_capacity, int max_n_frames, int max_seg_frames, uint8_t *picked,
                 uint32_t *mask, int32_t *msum, int32_t *status, void *ws, int64_t ws_bytes, void *stream);

/* ---- F-score: replaces utils/eval.py:125-165 evaluate_summary -------------------------------
 * Streams user_summary once.  mask/msum come from smz_select_shots or smz_pack_summary.
 * max_n_frames = max over the batch (grid sizing); total_users = sum of n_users (the counts are
 * zeroed inside the call).  n_users <= 1024 per video.
 * Outputs: overlap int32[sum n_users], gsum int32[sum n_users] (exact counts),
 *          f float32[sum n_users] (float32 arithmetic of utils/eval.py:153-159 as numpy 2 runs it),
 *          avg_f / max_f float64[n_videos]: np.mean / np.max of the per-user list exactly as numpy
 *          evaluates it — a float32 pairwise mean (widened) normally, a float64 pairwise mean when
 *          some user has zero overlap (the reference then appends the Python float 0., which
 *          promotes the list, utils/eval.py:156-164). */
int smz_fscore(const smz_video_desc *desc, int n_videos, int max_n_frames, int total_users,
               const float *user_summary, const uint32_t *mask, const int32_t *msum, int32_t *overlap,
               int32_t *gsum, float *f, double *avg_f, double *max_f, void *stream);

/* ---- whole evaluation path in ONE call: smz_select_shots + smz_fscore (or smz_fscore_packed) ----------------------
 * Replaces the per-key loop of models/__init__.py:88-119 (Trainer._eval_summary: generate_summary + evaluate_summary
 * for every test video).  The knapsack DP of a video is shared-memory bound, its F-score HBM bound; here the SAME
 * persistent CTA that solved a video's knapsack builds its summary mask in shared memory and streams its annotator
 * rows against it, so across the CTAs of an SM the DP of some videos overlaps the streaming of others and the stage
 * costs about max(DP, streaming) instead of their sum; the mask never makes a round trip through global memory.
 * Annotator rows: exactly one of user_summary (float32 rows, see smz_fscore) and user_bits + bits_off (1 bit per
 * frame, see smz_fscore_packed).  All other arguments and outputs as in smz_select_shots / smz_fscore; results are
 * identical to calling those two (which is what happens for videos whose DP rows do not fit the fused plan). */
/* DEVICE: float32 annotator rows -> 1 bit per frame (x > 0), the layout of smz_host_pack_user_summary: pack once, then
 * evaluate any number of score sets with smz_fscore_packed / smz_eval_batch(user_bits) at 1/32 of the bytes. */
int smz_pack_user_bits(const smz_video_desc *desc, int n_videos, const float *user_summary, const int64_t *bits_off,
                       uint32_t *user_bits, void *stream);
int smz_eval_batch(const smz_video_desc *desc, int n_videos, int total_users, const float *scores,
                   const int32_t *picks, const int32_t *cps, const int32_t *nfps, int method, int max_n_segs,
                   int max_capacity, int max_n_frames, int max_seg_frames, const float *user_summary,
                   const uint32_t *user_bits, const int64_t *bits_off, float *seg_mean, int32_t *values,
                   uint8_t *picked, float *summary, uint32_t *mask, int32_t *msum, int32_t *status, int32_t *overlap,
                   int32_t *gsum, float *f, double *avg_f, double *max_f, void *ws, int64_t ws_bytes, void *stream);

/* Binarise (>0), truncate/zero-pad an explicit machine summary to n_frames and pack it to the
 * bit mask smz_fscore consumes (utils/eval.py:136-145).  machine[] is indexed by summ_off /
 * summ_len like the summary output above. */
int smz_pack_summary(const smz_video_desc *desc, int n_videos, int max_n_frames, const float *machine,
                     uint32_t *mask, int32_t *msum, void *stream);

/* ---- upsample: replaces utils/eval.py:15-35 upsample / :37-47 generate_scores --------------- */
int smz_upsample(const smz_video_desc *desc, int n_videos, int max_n_frames, const float *scores,
                 const int32_t *picks, float *frame_scores, int32_t *status, void *stream);

/* ---- rank correlation: replaces utils/eval.py:49-72 evaluate_scores -------------------------------
 * For every video: ranks = scipy.stats.rankdata(-x) (average ties) of the machine frame scores and of each
 * annotator row, then Spearman rho (Pearson of the ranks, float64) or Kendall tau-b per annotator, and the
 * np.mean over annotators.  machine[] holds n_frames float32 per video at m_off (e.g. the output of
 * smz_upsample), user[] the annotator rows at u_off + u*u_ld.  rank_ws: float32 work buffer, video v uses
 * (1 + n_users) * n_frames entries at rank_off.  corr: float64 per annotator at row0 + u; corr_avg: per video
 * (NaN for a constant row, as scipy).  n_frames <= 32768 (one shared-memory sort per row). */
#define SMZ_METRIC_SPEARMAN 0
#define SMZ_METRIC_KENDALL 1
typedef struct smz_corr_desc {
    int64_t m_off, u_off, u_ld, rank_off;
    int32_t n_frames, n_users, row0, reserved;
} smz_corr_desc;
int smz_rank_correlation(const smz_corr_desc *desc, int n_videos, int max_n_frames, int max_n_users,
                         const float *machine, const float *user, int metric, float *rank_ws, double *corr,
                         double *corr_avg, void *stream);

/* ---- optimizer step of the training loops ----------------------------------------------------------
 * torch.optim.Adam (L2 term in the gradient; models/vasnet.py:160-161,211-212, models/dsn.py:100,147-149,
 * models/sumgan.py:268-275) and torch.nn.utils.clip_grad_norm_ (dsn.py:147, sumgan.py:433-436) over a whole parameter
 * list in a few launches.  tensors: HOST array (pointers inside are device pointers, float32, n elements each; grad may
 * be NULL = parameter skipped); it is copied into the kernel parameters, nothing captured in a CUDA graph points at it.
 *   smz_grad_sqnorm: *sqnorm (device float) = sum of squares of all gradients, summed in a fixed order (bit-stable);
 *                    ws: device scratch of smz_grad_sqnorm_workspace_floats() floats.
 *   smz_clip_grads:  g *= min(1, max_norm / (sqrt(*sqnorm) + 1e-6)) in place (clip_grad_norm_'s coefficient).
 *   smz_adam_step:   one Adam update; every tensor's *step (device float, completed updates of that tensor, as torch
 *                    counts per parameter) is read by the update and incremented behind it on the stream, so graph
 *                    replays advance it. */
#define SMZ_OPTIM_MAX_TENSORS 64     /* tensors per kernel launch (longer lists take several launches) */
typedef struct smz_optim_tensor {
    float *param, *grad, *exp_avg, *exp_avg_sq, *step;
    int64_t n;
} smz_optim_tensor;
int smz_grad_sqnorm_workspace_floats(const smz_optim_tensor *tensors, int n_tensors, int64_t *floats);
int smz_grad_sqnorm(const smz_optim_tensor *tensors, int n_tensors, float *sqnorm, float *ws, int64_t ws_floats, void *stream);
int smz_clip_grads(const smz_optim_tensor *tensors, int n_tensors, const float *sqnorm, float max_norm, void *stream);
int smz_adam_step(const smz_optim_tensor *tensors, int n_tensors, double lr, double beta1, double beta2, double eps,
                  double weight_decay, void *stream);
/* torch.nn.MSELoss() (mean reduction; vasnet.py:199,208 and the supervised baselines): loss[0] = mean((scores - target)^2)
 * and, when dscores != NULL, dscores[i] = 2 (scores[i] - target[i]) / n in the same launch (float32, device). */
int smz_mse_loss(const float *scores, const float *target, int64_t n, float *loss, float *dscores, void *stream);

/* ---- dense building block ------------------------------------------------------------------------
 * C[M,N] = epilogue(alpha * A[M,K] * B[N,K]^T) on the tcgen05 tensor cores: A and B bfloat16, K
 * contiguous (lda/ldb in elements, multiples of 8, 16-byte aligned bases), fp32 accumulation.
 * Epilogue, in this order: * alpha, + bias (float32, per column n; per row m with SMZ_GEMM_BIAS_M),
 * + residual[m,n] (bfloat16, or float32 with SMZ_GEMM_RES_F32; leading dimension ldr), ReLU with
 * SMZ_GEMM_RELU; C is bfloat16 or float32 (SMZ_GEMM_OUT_F32).  This is what replaces the cuBLAS
 * calls behind nn.Linear / torch.bmm in models/vasnet.py:114-140 and models/dsn.py:45,215-228. */
#define SMZ_GEMM_OUT_F32 1
#define SMZ_GEMM_RELU 2
#define SMZ_GEMM_RES_F32 4
#define SMZ_GEMM_BIAS_M 8
#define SMZ_GEMM_OUT_F16 2048   /* C is float16 (IEEE half) instead of bfloat16 */
#define SMZ_GEMM_A_F16 4096     /* A holds float16 instead of bfloat16 (the formats of A and B are independent) */
#define SMZ_GEMM_B_F16 8192     /* B holds float16 */
int smz_gemm_bf16_tn(const void *A, int64_t lda, const void *B, int64_t ldb, void *C, int64_t ldc, int M, int N,
                     int K, float alpha, const float *bias, const void *residual, int64_t ldr, int flags,
                     void *stream);
/* float32 -> bfloat16 copies of up to 8 tensors in one launch (src / dst / n are HOST arrays of device pointers and
 * element counts; 16-byte aligned segments): the parameter copies a training step refreshes. */
int smz_cvt_bf16_multi(const float *const *src, void *const *dst, const int64_t *n, int count, void *stream);
/* General operand storage: a_mn != 0 means A is given as [K, M] (m contiguous, lda >= M) instead of
 * [M, K]; b_mn != 0 means B is given as [K, N].  With these the autograd GEMMs of vasnet.py:209-211
 * (dX = dY.W, dW = dY^T.X) read the row-major activations directly, no transposed copies. */
int smz_gemm_bf16(int a_mn, int b_mn, const void *A, int64_t lda, const void *B, int64_t ldb, void *C, int64_t ldc,
                  int M, int N, int K, float alpha, const float *bias, const void *residual, int64_t ldr, int flags,
                  void *stream);
/* Float32-accurate form (the reference's torch.matmul / nn.Linear compute in float32, vasnet.py:114-140): every
 * operand is a hi + lo pair of bfloat16 arrays of the same layout, hi = bf16(x), lo = bf16(x - hi)
 * (smz_split_bf16_multi makes them from float32; *_lo == NULL: that operand is exact in bf16), and the kernel
 * accumulates A_hi.B_hi + A_lo.B_hi + A_hi.B_lo in float32: ~2^-17 relative per product instead of 2^-9.  C_lo != NULL
 * (bf16 output only): the result is written as hi + lo planes as well, ready to be the next operand. */
int smz_gemm_bf16_split(int a_mn, int b_mn, const void *A, const void *A_lo, int64_t lda, const void *B,
                        const void *B_lo, int64_t ldb, void *C, void *C_lo, int64_t ldc, int M, int N, int K, float alpha,
                        const float *bias, const void *residual, int64_t ldr, int flags, void *stream);
int smz_split_bf16_multi(const float *const *src, void *const *hi, void *const *lo, const int64_t *n, int count,
                         void *stream);

/* ---- VASNet scorer: replaces models/vasnet.py:92-148 VASNet.forward (and, with
 *      smz_vasnet_backward, the autograd graph behind vasnet.py:209-211) -------------------------
 * Parameters are DEVICE pointers.  The four square matrices are bfloat16 copies of the module's
 * float32 nn.Linear weights ([out, in] row-major, as stored by torch):
 *   wqk [2048,1024]  rows 0..1023 = Q.weight, rows 1024..2047 = K.weight   (vasnet.py:57-58)
 *   wv, wo, w1 [1024,1024]  V.weight, attention_head_projection.weight, k1.weight (vasnet.py:59-60,64)
 *   b1 [1024], w2 [1024], b2 [1], ln_g / ln_b [1024] float32  (k1.bias, k2.weight, k2.bias and the ONE
 *   LayerNorm the reference applies twice, vasnet.py:54,137,143)
 * scale multiplies the logits (vasnet.py:34,119); aperture < 0 = global attention, else the band
 * |i-j| <= aperture of vasnet.py:124-127; ignore_self masks the diagonal (vasnet.py:121-122). */
#define SMZ_VASNET_STATUS_LOGIT_RANGE 1   /* an attention logit left [-80, 80] */
#define SMZ_VASNET_STATUS_F16_RANGE 2     /* a float16 value (features, x.(Wq^T Wk), y) exceeded the float16 range */
typedef struct smz_vasnet_params {
    const void *wqk, *wv, *wo, *w1;
    const float *b1, *w2, *b2, *ln_g, *ln_b;
    float scale, eps;
    int32_t aperture, ignore_self;
    /* optional (inference): head_gw [1024] = ln_g * w2 and head_c [2] = {sum(ln_g * w2), sum(ln_b * w2) + b2}
     * (float32, device).  When both are given the regressor head (vasnet.py:143-145) is folded into the k1
     * GEMM epilogue and the hidden activations never reach memory; NULL keeps the separate head kernel. */
    const float *head_gw, *head_c;
    /* optional (inference), all required together with head_gw / head_c for the FAST path (smz_vasnet.cu, fast_chunk):
     * the forward with its linear maps folded where no non-linearity sits between them —
     *   logits_ij = x_i^T (Wq^T Wk) x_j,   c_i = sum_j alpha_ij (Wo Wv) x_j,   W1 . LN(y) + b1 = rstd * (W1g . y - mean * ln_c) + b1f
     * — exact in real arithmetic, 22 % fewer multiply-adds, no K / output projection and no LayerNorm kernel.
     *   w1g  [1024,1024] float16(k1.weight * ln_g[None, :]);  ln_c [1024] row sums of w1g (of the float16 values, float32);
     *   b1f  [1024] = k1.weight . ln_b + k1.bias (float32);
     *   wgv  [2048,1024] bfloat16: rows 0..1023 = Wo Wv, rows 1024..2047 = Wk^T Wq (products formed in float32) — used
     *        with bfloat16 features;  wgv16: the same in float16 — used with float32 features (copied to float16);
     *   status: device word.  Softmax runs without the max subtraction (exp and row sums in the logits epilogue) and
     *        y / W1g (and, for float32 features, x / G / the folded weights) are float16: exact reformulations inside a
     *        value range the kernels check.  A violation ORs SMZ_VASNET_STATUS_* into *status (never cleared by the
     *        library), the scores of that call are void, and the caller repeats the call with status = NULL (the
     *        wide-range path: the literal chain in bf16 / fp32, max-subtracted softmax, LayerNorm kernel).  The host
     *        reads the word whenever it next synchronises — no launch waits on it. */
    const void *w1g;
    const float *ln_c, *b1f;
    const void *wgv, *wgv16;
    int32_t *status;
    /* optional, all four together: the FLOAT32-ACCURATE mode (training layout only, i.e. training != 0 in
     * smz_vasnet_forward, and smz_vasnet_backward).  The reference computes in float32 (vasnet.py:114-145); bf16 operands
     * cost 2^-9 per product.  Here every 16-bit operand becomes a hi + lo pair of bf16 arrays (hi = bf16(x),
     * lo = bf16(x - hi)) and every contraction runs the three products hi.hi + lo.hi + hi.lo into the float32 accumulator
     * (~2^-17 per product; 3 x the tensor-core work of the bf16 mode, immaterial for batch-1 training steps that are
     * launch-bound).  w*_lo = the lo planes of wqk / wv / wo / w1 (smz_split_bf16_multi makes them); the activations'
     * lo planes live in the second half of the work buffer: size it with training | SMZ_VASNET_SPLIT. */
    const void *wqk_lo, *wv_lo, *wo_lo, *w1_lo;
} smz_vasnet_params;
#define SMZ_VASNET_SPLIT 4   /* OR into `training` of smz_vasnet_workspace_bytes: room for the activations' lo planes */

/* x: packed features [sum T, 1024] (float32, or bfloat16 when x_is_bf16), video v owns rows
 * h_cu_seqlens[v] .. h_cu_seqlens[v+1]-1 (HOST array of n_videos+1 prefix offsets, [0] == 0; the
 * reference's (T, B, 1024) batch is B videos of equal length).  scores: float32 [sum T] in (0,1).
 * training != 0 keeps every intermediate in the work buffer for smz_vasnet_backward and enables the
 * three p=0.5 dropouts (vasnet.py:130,136,142) through caller-supplied KEEP masks (uint8, 1 = keep;
 * NULL = no dropout at that site): drop_att packed per video [T*T], drop_y / drop_h [sum T, 1024]. */
/* KEEP masks of the three nn.Dropout(0.5) sites (vasnet.py:130,136,142) for smz_vasnet_forward(training): n bytes,
 * 1 = keep with probability 1/2 (Philox4x32-10, one bit per byte).  state: three device uint64 words {seed, call number, 0};
 * the call number is advanced on the device, so a captured training step draws fresh masks at every graph replay. */
int smz_dropout_keep_masks(uint64_t *state, uint8_t *out, int64_t n, void *stream);
int smz_vasnet_workspace_bytes(const int32_t *h_cu_seqlens, int n_videos, int training, int x_is_bf16,
                               int64_t *bytes);
/* on != 0 forces the exact inference path for every call of this process, status word or not (testing / A-B aid). */
void smz_vasnet_set_exact_softmax(int on);
/* kernels one forward call launches (reporting); training: 1 = training, 0 = fast inference, 2 = exact inference */
int smz_vasnet_launch_count(const int32_t *h_cu_seqlens, int n_videos, int training, int x_is_bf16,
                            int64_t *launches);
int smz_vasnet_forward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos,
                       const smz_vasnet_params *p, int training, const uint8_t *drop_att, const uint8_t *drop_y,
                       const uint8_t *drop_h, float *scores, void *ws, int64_t ws_bytes, void *stream);

/* Backward of the scorer (what loss.backward() computes for vasnet.py:209-211): consumes the work buffer
 * a smz_vasnet_forward(training=1) call on the SAME batch left behind, the scores it produced and
 * d(loss)/d(scores); ACCUMULATES (+=) float32 gradients with the parameters' shapes.  wqk is
 * [2048,1024] (rows 0..1023 = d Q.weight, 1024..2047 = d K.weight).  dx (optional, [sum T, 1024])
 * receives d(loss)/d(x) — only needed when a learned positional embedding feeds x (vasnet.py:110). */
typedef struct smz_vasnet_grads {
    float *wqk, *wv, *wo, *w1, *b1, *w2, *b2, *ln_g, *ln_b;
    float *dx;
} smz_vasnet_grads;
int smz_vasnet_backward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos,
                        const smz_vasnet_params *p, const uint8_t *drop_att, const uint8_t *drop_y,
                        const uint8_t *drop_h, const float *scores, const float *dscores,
                        const smz_vasnet_grads *grads, void *ws, int64_t ws_bytes, void *stream);

/* ---- Transformer scorer: replaces models/transformer.py Transformer.forward in eval mode (no autograd graph) ----------
 * Fused variable-length multi-head attention, the encoder's hot path on its own:  out[:, h*D : (h+1)*D] =
 * softmax(Q_h K_h^T / sqrt(D)) V_h for every video and head (D = head_dim), each video attending to all of its own frames
 * and to no other video's.  qkv: bfloat16 [sum T, ld] device rows packed as nn.MultiheadAttention's in_proj output (Q
 * columns [0, n_heads*D), K [n_heads*D, 2*n_heads*D), V after them; ld >= 3*n_heads*D, multiple of 8); out: bfloat16
 * [sum T, ldo] (ldo >= n_heads*D, multiple of 8).  h_cu_seqlens as for smz_vasnet_forward.  head_dim must be 128 or 256
 * (SMZ_ERR_UNSUPPORTED otherwise).  ws: smz_mha_workspace_bytes(n_videos) bytes of device memory (the work-unit table). */
int smz_mha_workspace_bytes(int n_videos, int64_t *bytes);
int smz_mha_forward(const void *qkv, int64_t ld, const int32_t *h_cu_seqlens, int n_videos, int n_heads, int head_dim,
                    void *out, int64_t ldo, void *ws, int64_t ws_bytes, void *stream);

/* One post-norm nn.TransformerEncoderLayer(d_model=1024, nhead, dim_feedforward=1024, relu): the parameters of
 * transformer_encoder.layers.{i}.  nhead is 8 for smz_transformer_forward and smz_sumgan_att_selector_params.n_heads for
 * smz_sumgan_att_selector_forward.  Matrices are bfloat16 copies of the float32 weights ([out, in] row-major as torch
 * stores them); vectors float32.  w_qkv [3072,1024] / b_qkv [3072] = self_attn.in_proj_weight / in_proj_bias (rows q, k,
 * v); w_out = self_attn.out_proj; w1 / w2 = linear1 / linear2 [1024,1024]; norm1 / norm2 weights and biases (eps 1e-5). */
typedef struct smz_transformer_layer {
    const void *w_qkv;
    const float *b_qkv;
    const void *w_out;
    const float *b_out;
    const void *w1;
    const float *b1;
    const void *w2;
    const float *b2;
    const float *norm1_g, *norm1_b, *norm2_g, *norm2_b;
} smz_transformer_layer;
/* layers: HOST array of n_layers entries (read during the call only).  ln_g / ln_b / eps: the model's ONE layer_norm,
 * applied as the encoder's final norm and again after relu(k1(.)).  k1_w bfloat16 [1024,1024], k1_b [1024];
 * head_gw [1024] = ln_g * k2.weight, head_c [2] = {sum(ln_g * k2.weight), sum(ln_b * k2.weight) + k2.bias} (float32).
 * more_residuals != 0: the head reads encoder_out + x. */
typedef struct smz_transformer_params {
    const smz_transformer_layer *layers;
    const float *ln_g, *ln_b;
    float eps;
    int32_t more_residuals;
    const void *k1_w;
    const float *k1_b, *head_gw, *head_c;
} smz_transformer_params;
/* x: packed features [sum T, 1024] float32 (or bfloat16 when x_is_bf16), positional embeddings already added;
 * scores: float32 [sum T].  ws: smz_transformer_workspace_bytes bytes. */
int smz_transformer_workspace_bytes(const int32_t *h_cu_seqlens, int n_videos, int x_is_bf16, int64_t *bytes);
int smz_transformer_forward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos,
                            const smz_transformer_params *p, int n_layers, float *scores, void *ws, int64_t ws_bytes,
                            void *stream);

/* ---- SumGAN-att selector: replaces models/sumgan_att.py Transformer.forward in eval mode (no autograd graph) ----------
 * scores = sigmoid(out(layer_norm(TransformerEncoder(x)))).  layers: HOST array of n_layers encoder layers with n_heads
 * heads of 1024 / n_heads (n_heads 4 or 8; SMZ_ERR_UNSUPPORTED otherwise, before any device work).  ln_g / ln_b / eps:
 * the selector's layer_norm (the encoder's final norm); out_w [1024] / out_b [1]: out[0] = nn.Linear(1024, 1) (float32).
 * x, h_cu_seqlens and scores as for smz_transformer_forward.  The work buffer is the same plan as the Transformer
 * scorer's: ws: smz_transformer_workspace_bytes bytes. */
typedef struct smz_sumgan_att_selector_params {
    const smz_transformer_layer *layers;
    int32_t n_heads;
    const float *ln_g, *ln_b;
    float eps;
    const float *out_w, *out_b;
} smz_sumgan_att_selector_params;
int smz_sumgan_att_selector_forward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos,
                                    const smz_sumgan_att_selector_params *p, int n_layers, float *scores,
                                    void *ws, int64_t ws_bytes, void *stream);

/* ---- DSN scorer: replaces models/dsn.py:38-47 DSN.forward (nn.LSTM(1024, 256, bidirectional) through
 *      cuDNN + Linear(512,1) + sigmoid) and, with smz_dsn_backward, its autograd graph ---------------------
 * Device pointers:
 *   w_ih   bfloat16 [2048,1024]: rows 0..1023 = rnn.weight_ih_l0, 1024..2047 = rnn.weight_ih_l0_reverse
 *   bias   float32 [2048]: bias_ih + bias_hh of the two directions (torch gate order i,f,g,o)
 *   whh_packed / whh_t_packed: uint32 [2*8*64*256] each, W_hh / W_hh^T of both directions in the register
 *          order of the recurrence kernels — produced (on the device) by smz_dsn_pack_whh from the float32
 *          rnn.weight_hh_l0 / _reverse ([1024,256])
 *   w_out  float32 [512] (out.0.weight), b_out float32 [1] (out.0.bias)
 * x / h_cu_seqlens as for smz_vasnet_forward; probs: float32 [sum T]. */
typedef struct smz_dsn_params {
    const void *w_ih;
    const float *bias;
    const void *whh_packed, *whh_t_packed;
    const float *w_out, *b_out;
} smz_dsn_params;
int smz_dsn_pack_whh(const float *whh_fwd, const float *whh_bwd, uint32_t *out_fwd, uint32_t *out_bwd, void *stream);
int smz_dsn_workspace_bytes(int total_rows, int n_videos, int training, int x_is_bf16, int64_t *bytes);
int smz_dsn_forward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos, const smz_dsn_params *p,
                    int training, float *probs, void *ws, int64_t ws_bytes, void *stream);
/* Backward (BPTT) of a smz_dsn_forward(training=1) call on the same batch and work buffer: what
 * loss.backward() computes for dsn.py:143-144.  ACCUMULATES (+=) float32 gradients: w_ih [2048,1024] and
 * w_hh [2048,256] (rows 0..1023 = forward direction, 1024..2047 = reverse), bias [2048] (the gradient of both
 * bias_ih and bias_hh), w_out [512], b_out [1]. */
typedef struct smz_dsn_grads {
    float *w_ih, *w_hh, *bias, *w_out, *b_out;
} smz_dsn_grads;
int smz_dsn_backward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos, const smz_dsn_params *p,
                     const float *probs, const float *dprobs, const smz_dsn_grads *grads, void *ws, int64_t ws_bytes,
                     void *stream);

/* ---- DSN reward: replaces models/dsn.py:185-236 DSNTrainer.compute_reward for ALL episodes of one video ----
 * x: float32 features [T,1024]; actions: uint8 [n_episodes, T] (1 = frame picked, the Bernoulli samples of
 * dsn.py:125); rewards: float32 [n_episodes] = 0.5 * (R_div + R_rep); 0 when no frame is picked; with a single
 * picked frame R_div = 0 and R_rep is evaluated normally (the reference raises there, dsn.py:229-230).
 * n_episodes <= 8. */
int smz_dsn_reward_workspace_bytes(int T, int n_episodes, int64_t *bytes);
int smz_dsn_reward(const float *x, int T, const uint8_t *actions, int n_episodes, int temp_dist_thre, int far_sim,
                   float *rewards, void *ws, int64_t ws_bytes, void *stream);

/* ---- DSN episode sampling: replaces models/dsn.py:112,125-126 (Bernoulli(probs); dist.sample(); dist.log_prob)
 * for ALL episodes of a step in one launch.  probs: float32 [T] in (0,1); state: three device uint64 words
 * {Philox seed, call number, 0 (ticket, kept at 0 by the kernel)} — the call number is advanced on the device, so a
 * captured step draws fresh episodes at every graph replay; given: NULL, or uint8 [n_episodes,T] actions to evaluate
 * instead of drawing (tests replay the reference's draws; the call number is then left alone).  Out: actions uint8
 * [n_episodes,T] (1 = frame picked, action = u < p as torch's bernoulli), logp_mean float32 [n_episodes] = mean over
 * the frames of log_prob(action) as torch.distributions.Bernoulli computes it (probabilities clamped to
 * [2^-23, 1 - 2^-23]).
 * smz_bernoulli_logprob_backward: dprobs[t] = sum_e dlogp[e] * (a - p) / (p (1 - p)) / T, 0 where p was clamped. */
int smz_bernoulli_logprob(const float *probs, int T, int n_episodes, uint64_t *state, const uint8_t *given,
                          uint8_t *actions, float *logp_mean, void *stream);
int smz_bernoulli_logprob_backward(const float *probs, const uint8_t *actions, const float *dlogp, int T,
                                   int n_episodes, float *dprobs, void *stream);

/* ---- annotator summaries as 1 bit per frame (staging form for host -> device copies) --------------
 * evaluate_summary binarises user_summary first (utils/eval.py:148-149), so (x > 0) is all it reads.
 * smz_host_pack_user_summary runs on HOST threads over HOST pointers (it is the copy's staging step): row u of
 * video v, h_user + user_off + u*user_ld (n_frames floats), becomes ceil(n_frames/32) words at
 * h_bits + h_bits_off[v] + u*ceil(n_frames/32); bit j of word w = frame 32w+j is > 0.
 * smz_fscore_packed = smz_fscore reading those rows (device pointers); F values are bit-identical. */
int smz_host_pack_user_summary(const smz_video_desc *h_desc, int n_videos, const float *h_user,
                               const int64_t *h_bits_off, uint32_t *h_bits, int n_threads);
int smz_fscore_packed(const smz_video_desc *desc, int n_videos, const uint32_t *user_bits, const int64_t *bits_off,
                      const uint32_t *mask, const int32_t *msum, int32_t *overlap, int32_t *gsum, float *f,
                      double *avg_f, double *max_f, void *stream);

/* ---- Kernel temporal segmentation (KTS, Potapov et al. ECCV 2014): produces what the datasets hold as /change_points
 *      (datasets/README.md:24-27).  The reference ships no KTS code — it only consumes change points — so these follow
 *      the published cpd_nonlin / cpd_auto (oracle/kts_np.py); SURVEY.md §8f NEXT-4.
 *   smz_kts_gram: K = X X^T in float32, features [n, d] with row stride ld (device).
 *   smz_kts: K [n, n] device float32, or NULL to compute it from `features`; max_ncp = m of cpd_nonlin, lmin / lmax the
 *   segment length bounds; auto_select != 0 = cpd_auto's penalised choice of the number of change points (vmax,
 *   desc_rate).  Device outputs: cps [max_ncp] (ascending, first n_cps entries valid), n_cps [1], scores [max_ncp + 1]. */
int smz_kts_workspace_bytes(int n, int max_ncp, int from_features, int64_t *bytes);
int smz_kts_gram(const float *features, int n, int d, int ld, float *K, void *stream);
int smz_kts(const float *K, const float *features, int n, int d, int ld, int max_ncp, int lmin, int lmax,
            int auto_select, double vmax, int desc_rate, int32_t *cps, int32_t *n_cps, double *scores,
            void *ws, int64_t ws_bytes, void *stream);

/* ---- SumGAN LSTM recurrences: replace the cuDNN calls behind nn.LSTM in models/sumgan.py:43 (sLSTM, 2 x 1024
 *      bidirectional), :69 (eLSTM, 2 x 2048), :207 (cLSTM, 2 x 1024) and the step-wise decode loop :98-115 (dLSTM,
 *      2 x 2048), forward and BPTT, batch 1.  One call = one layer over the whole sequence (both directions of a
 *      bidirectional layer side by side).  The input projections x.W_ih^T + b, dX and the weight gradients are
 *      whole-sequence GEMMs (smz_gemm_bf16) issued by the caller.  All pointers are device memory; gate order is
 *      torch's (i, f, g, o); sync_ws = 256 bytes of device scratch for the grid barrier.
 *   forward : pre [T, ldpre] float32 pre-activations (gate g of unit u at pre[t*ldpre + g*H + u]); whh bfloat16
 *             [4H, H]; h0/c0 [H] or NULL (zeros); y[t*ldy + u] = h_t; training also fills gates (activated,
 *             [T, ldg]) and cs [T, H]; h_last/c_last [H] or NULL.  reverse != 0 walks t = T-1 .. 0.
 *   backward: whh_t bfloat16 [H, 4H] (= W_hh^T); dy [T, lddy] or NULL; dh_last/dc_last [H] or NULL; writes
 *             dgates [T, ldg] (pre-activation gradients), dh0/dc0 [H] (or NULL).
 *   B (1..4) sequences of the same length share the weights in one launch — the per-step cost is the grid barrier and
 *   the weight stream, so extra sequences are nearly free: sequence arrays are then [B][T][ld], state vectors [B][H]. */
typedef struct smz_lstm_seq {
    int32_t T, H, reverse, ldpre, ldy, lddy, ldg, B;
    const float *pre;
    const void *whh, *whh_t;
    const float *h0, *c0;
    float *y, *gates, *cs, *h_last, *c_last;
    const float *dy, *dh_last, *dc_last;
    float *dgates, *dh0, *dc0;
} smz_lstm_seq;
int smz_lstm_seq_forward(const smz_lstm_seq *dirs, int n_dir, void *sync_ws, void *stream);
int smz_lstm_seq_backward(const smz_lstm_seq *dirs, int n_dir, void *sync_ws, void *stream);

/* dLSTM decode: layer 0's input at step t is layer 1's output at step t-1 (zeros at t = 0), sumgan.py:106-112.
 *   w_* bfloat16 [4H, H], w_*_t their transposes [H, 4H] (backward only); bias0/1 float32 [4H] (b_ih + b_hh);
 *   h_init/c_init [2, H]; hs0/hs1 [T, H] layer outputs; gates0/1 [T, 4H], cs0/1 [T, H] (training);
 *   backward: dy [T, H] gradient of hs1 -> dgates0/1 [T, 4H], dh_init/dc_init [2, H].
 *   With B > 1: sequence arrays [B][T][.], h_init / c_init / dh_init / dc_init [2][B][H]. */
typedef struct smz_lstm_decode {
    int32_t T, H, B, reserved;
    const void *w_ih0, *w_hh0, *w_ih1, *w_hh1;
    const void *w_ih0_t, *w_hh0_t, *w_ih1_t, *w_hh1_t;
    const float *bias0, *bias1, *h_init, *c_init;
    float *hs0, *hs1, *gates0, *gates1, *cs0, *cs1;
    const float *dy;
    float *dgates0, *dgates1, *dh_init, *dc_init;
} smz_lstm_decode;
int smz_lstm_decode_forward(const smz_lstm_decode *d, void *sync_ws, void *stream);
int smz_lstm_decode_backward(const smz_lstm_decode *d, void *sync_ws, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SUMMARIZER_B200_H */
