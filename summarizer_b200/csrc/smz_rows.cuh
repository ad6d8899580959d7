// Row-wise kernels of the scorers (softmax with VASNet's masks, LayerNorm, regressor head, dtype
// conversion).  One warp per row, 128-bit loads; launched by smz_vasnet.cu / smz_dsn.cu.
#pragma once
#include <cuda_bf16.h>

#include "smz_gemm.cuh"

namespace smz {

constexpr int kFeat = 1024;   // feature / hidden width of VASNet (vasnet.py:18)

// lo != 0 (everywhere below): the bf16 output is written as hi + lo planes, the lo plane `lo` elements behind the hi
// plane (x - float(bf16(x)) as bf16) — the operand form of the float32-accurate GEMM mode (GemmEpilogue::a_lo)
int launch_cvt_bf16(const float *x, __nv_bfloat16 *y, int64_t n, cudaStream_t st, int64_t lo = 0);
// float32 -> float16 with a range check: |x| > 60000 or NaN ORs `bit` into *guard (the VASNet fast path's feature copy)
int launch_cvt_f16(const float *x, void *y, int64_t n, int *guard, int bit, cudaStream_t st);

// alpha = softmax(mask(S)) over the keys of each row (vasnet.py:121-130).  `probs` are the problems of
// the logits GEMM (M = N = T, c_off / ldc locate the video's block in S); alpha/P use the same offsets.
// drop (optional): keep-mask bytes of the attention dropout, video v at drop + drop_off[v]; then
// P = 2 * keep * alpha, else P == alpha (one buffer).  A row of P holds probs[v].pad zero columns, the
// T probabilities, then zeros up to the next multiple of 64 (the K extent alpha.V reads).
// gate (optional): the launch is a no-op unless *gate != 0; sum_slots (optional, [rows][n_slots][3]): the row-sum
// slots of the fused-exp logits path are overwritten with {1, 0, ...} for every row processed, so that the alpha.V
// GEMM's GEMM_SCALE_STATS row scale becomes 1 (see smz_vasnet.cu).
int launch_softmax(const GemmProblem *d_probs, int n_probs, int total_rows, const float *S, __nv_bfloat16 *alpha,
                   __nv_bfloat16 *P, const uint8_t *drop, const int64_t *d_drop_off, int aperture, int ignore_self,
                   cudaStream_t st, const int *gate = nullptr, float *sum_slots = nullptr, int n_slots = 0, int64_t lo = 0);

// yn = LayerNorm(2*keep*y or y) * g + b  (vasnet.py:136-137), rows of 1024; optional mean / rstd.
// Optional: res (float32, or bf16 with res_bf16; rows of 1024) is added to the normalised row; y32 receives the result
// in float32 as well (the transformer's residual stream); yn may then be NULL.
int launch_layernorm(const float *y, const uint8_t *keep, const float *g, const float *b, float eps, int rows,
                     __nv_bfloat16 *yn, float *mean, float *rstd, cudaStream_t st, int64_t lo = 0, float *y32 = nullptr,
                     const void *res = nullptr, bool res_bf16 = false);

// score = sigmoid(LayerNorm(2*keep*h or h) . w2 + b2)  (vasnet.py:142-145); h is post-ReLU float32.
int launch_head(const float *h, const uint8_t *keep, const float *g, const float *b, float eps,
                const float *w2, const float *b2, int rows, float *scores, float *mean, float *rstd,
                cudaStream_t st);

// score = sigmoid(LayerNorm(h) . w2 + b2) from the three row sums the k1 GEMM epilogue left behind
// (GEMM_ROWSTATS: sum h, sum h^2, sum h * (g * w2) per slot):  z = rstd * (S3 - mean * c[0]) + c[1] with
// c[0] = sum g*w2, c[1] = sum b*w2 + b2.  stats: [rows][slots][3].
int launch_head_from_stats(const float *stats, int slots, const float *c, float eps, int rows, float *scores,
                           cudaStream_t st);

// ---- backward (autograd of vasnet.py:136-145 and :129-130) -----------------------------------------
// Regressor head + second LayerNorm + ReLU: dh = d(loss)/d(k1 pre-activation) as bf16; accumulates
// (+=, float32 atomics) d_w2, d_b2, d_g, d_b (LayerNorm affine) and d_b1 (column sums of dh).
int launch_head_bwd(const float *h, const uint8_t *keep, const float *g, const float *b, const float *w2,
                    const float *mean, const float *rstd, const float *scores, const float *dscores, int rows,
                    __nv_bfloat16 *dh, float *d_w2, float *d_b2, float *d_g, float *d_b, float *d_b1, cudaStream_t st,
                    int64_t lo = 0);
// First LayerNorm (+ dropout): dy = d(loss)/d(y before dropout) as bf16 (and float32 when dy_f32 != NULL).
int launch_layernorm_bwd(const float *dyn, const float *y, const uint8_t *keep, const float *g, const float *mean,
                         const float *rstd, int rows, __nv_bfloat16 *dy, float *dy_f32, float *d_g, float *d_b,
                         cudaStream_t st, int64_t lo = 0);
// Softmax (+ attention dropout) of ONE video: dS = alpha * (dalpha - rowsum(dalpha * alpha)), dalpha = 2*keep*dP.
int launch_softmax_bwd(const float *dP, const __nv_bfloat16 *alpha, const uint8_t *keep, int T, int ld,
                       __nv_bfloat16 *dS, cudaStream_t st, int64_t lo = 0);

}  // namespace smz
