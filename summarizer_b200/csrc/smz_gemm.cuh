// Host-side interface of the tcgen05 GEMM building block (smz_gemm.cu), shared by the scorer kernels.
#pragma once
#include <cuda.h>

#include "smz_common.cuh"

namespace smz {

// One GEMM of a (possibly ragged) batch:  C[M,N] = epilogue(alpha * A[M,K] * B[N,K]^T).
// A and B are K-major (row = m resp. n, K contiguous) bf16 sub-matrices of two big 2-D arrays that
// one TMA tensor map each describes; *_row0 / *_col0 locate the sub-matrix inside them.
struct GemmProblem {
    int32_t a_row0, a_col0, b_row0, b_col0;
    int32_t M, N, K;
    int32_t tile0;       // first flat tile index of this problem (prefix sum over the batch)
    int64_t c_off;       // element offset of C[0,0] in the output array
    int64_t r_off;       // element offset of residual[0,0]
    int32_t ldc, ldr;    // leading dimensions (elements) of C and the residual
    int32_t tiles_n;     // ceil(N / BN)
    int32_t pad;         // free for the caller (VASNet: leading zero columns of the video's P block)
};
static_assert(sizeof(GemmProblem) == 64, "GemmProblem layout");

enum : int {
    GEMM_OUT_F32 = 1,    // C is float32 (default bf16)
    GEMM_RELU = 2,       // max(x, 0) last (NaN stays NaN)
    GEMM_RES_F32 = 4,    // residual is float32 (default bf16)
    GEMM_BIAS_M = 8,     // bias indexed by row m (default: by column n)
    GEMM_ROWSTATS = 16,  // per row and (n-tile, column half) slot: sum x, sum x^2, sum x * stat_w[n] of the epilogue
                         // OUTPUT x -> stat_out[(m * 2 * tiles_n + slot) * 3 + {0,1,2}] (LayerNorm + dot folded into
                         // the producer: the consumer needs three numbers per row, not the row)
    GEMM_NO_STORE = 32,  // do not write C (only meaningful with GEMM_ROWSTATS)
    GEMM_EXP = 64,       // attention logits: x = exp(mask(alpha * acc)) written as bf16 with zero columns up to the next
                         // multiple of 64 (un-normalised softmax numerators; the row sums come from GEMM_ROWSTATS).
                         // |logit| > 80 anywhere raises *guard (the caller then re-runs the exact max-subtracted path)
    GEMM_SCALE_M = 128,  // x *= bias[r_off + m]  (row scale, e.g. 1 / softmax denominator) instead of adding a bias
    GEMM_SCALE_STATS = 256,  // x *= 1 / sum_k bias[((r_off + m) * stat_slots + k) * 3]: the row scale straight from the
                         // GEMM_ROWSTATS slots of the producer (softmax denominators: no kernel in between)
    GEMM_LN_STATS = 512, // plain epilogue + per row and (n-tile, column half) slot: sum x, sum x^2 of the OUTPUT x
                         // -> stat_out[((r_off + m) * stat_slots + slot) * 3 + {0,1}] (LayerNorm statistics for the consumer)
    GEMM_OUT_F16 = 2048, // columns >= f16_col0 of C are float16 (IEEE half) instead of bf16: 3 more mantissa bits for an
                         // activation whose range is checked — |x| > 60000 raises guard_bit in *guard
    GEMM_A_F16 = 4096,   // the A operand holds float16 instead of bf16 (tcgen05 kind::f16 takes either format per operand)
    GEMM_B_F16 = 8192,   // the B operand holds float16
    GEMM_RES_AT_C = 16384,   // the residual array has C's layout: its element offset / leading dimension are c_off / ldc (r_off is
                         // then free to carry the row offset of the per-row statistics)
    GEMM_LN_FOLD = 1024, // head epilogue whose A operand is the un-normalised LayerNorm input y (bf16 / f16) and whose B is
                         // W * diag(gamma): x = rstd_m * (acc - mean_m * ln_c[n]) + bias[n], mean / rstd of row m from the
                         // GEMM_LN_STATS slots in ln_stats (ln_slots per row, rows of ln_width elements, eps ln_eps)
};

struct GemmEpilogue {
    void *C;                 // bf16 or float32
    const float *bias;       // optional
    const void *residual;    // optional, added after bias
    float alpha;
    int flags;
    const float *stat_w = nullptr;   // GEMM_ROWSTATS: weight vector [N] (optional)
    float *stat_out = nullptr;       // GEMM_ROWSTATS: [(r_off + m)][stat_slots][3] (r_off doubles as the row offset here)
    int stat_slots = 0;              // slots per row (>= 2 * tiles_n); 0 = 2 * tiles_n of the problem
    int scale_slots = 0;             // GEMM_SCALE_STATS: slots per row of the array read through `bias` (0 = stat_slots)
    int aperture = -1, ignore_self = 0;   // GEMM_EXP: VASNet's masks (vasnet.py:121-127), row / column = video-local i / j
    int *guard = nullptr;            // GEMM_EXP: |= guard_bit when a logit leaves [-80, 80]; GEMM_OUT_F16: when |x| > 60000
    int guard_bit = 1;
    int f16_col0 = 0;                // GEMM_OUT_F16: first float16 column (a multiple of 32)
    const int *gate = nullptr;       // when given: the whole launch is a no-op unless *gate != 0
    const float *ln_stats = nullptr; // GEMM_LN_FOLD: [(m)][ln_slots][3] sums written by a GEMM_LN_STATS producer
    const float *ln_c = nullptr;     // GEMM_LN_FOLD: [N] row sums of the B operand (W * diag(gamma)) as the tensor core sees it
    int ln_slots = 0, ln_width = 0;
    float ln_eps = 0.f;
    // Split-bf16 ("hi + lo planes") operands, the float32-accurate mode: element offsets (from A / B / C) of a second
    // bf16 array of the same layout holding x - float(bf16(x)); 0 = the operand has no lo plane.  The k loop then runs
    // once per product kept — A_hi.B_hi, A_lo.B_hi, A_hi.B_lo (A_lo.B_lo ~ 2^-18 is dropped) — into the same float32
    // accumulator: ~2^-17 relative per product instead of 2^-9.  c_lo (16-bit outputs of the plain epilogue only): the
    // epilogue also writes the lo plane of C.
    int64_t a_lo = 0, b_lo = 0, c_lo = 0;
};

constexpr int GEMM_BN = 256;
constexpr int GEMM_BK = 64;

// Tile rows: 256 with the default CTA-pair kernel (tcgen05 cta_group::2), 128 with SMZ_GEMM_PAIR=0.  Every
// caller sizes its tile prefix sums through gemm_tiles().
int gemm_tile_m();
int gemm_tiles(int M, int N);

// A: [a_rows, a_cols] bf16 with leading dimension lda (elements, multiple of 8), likewise B.
// probs: device array of n_probs problems (or nullptr with n_probs == 1 -> `single` is used).
int gemm_bf16_tn(const void *A, int64_t a_rows, int64_t a_cols, int64_t lda, const void *B, int64_t b_rows,
                 int64_t b_cols, int64_t ldb, const GemmProblem *d_probs, int n_probs, int total_tiles,
                 const GemmProblem &single, const GemmEpilogue &epi, cudaStream_t st);

// General form: a_mn / b_mn select MN-major storage of the operand ([K, M] resp. [K, N] arrays, m / n
// contiguous); then (*_row0, *_col0) of a problem are (first k row, first m/n column), which must be a
// multiple of 8 columns (TMA alignment).
int gemm_bf16(bool a_mn, bool b_mn, const void *A, int64_t a_rows, int64_t a_cols, int64_t lda, const void *B,
              int64_t b_rows, int64_t b_cols, int64_t ldb, const GemmProblem *d_probs, int n_probs, int total_tiles,
              const GemmProblem &single, const GemmEpilogue &epi, cudaStream_t st);

// TMA map of a bf16 [rows, cols] array (leading dimension ld elements): boxes of 64 columns x box_rows rows with the
// 128-byte swizzle, the K-major operand layout the GEMM loads (smz_attn.cu loads its Q / K / V tiles with it too).
int make_bf16_map(CUtensorMap *m, const void *base, int64_t rows, int64_t cols, int64_t ld, int box_rows);

}  // namespace smz
