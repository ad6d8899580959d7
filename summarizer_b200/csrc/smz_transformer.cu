// Transformer-encoder scorers, inference: nn.TransformerEncoder of post-norm nn.TransformerEncoderLayer(d_model=1024,
// nhead, dim_feedforward=1024, relu) layers on the tcgen05 GEMM building block and the fused attention kernel
// (smz_attn.cu), then a head:
//   smz_transformer_forward           models/transformer.py, nhead=8: the shared final LayerNorm and the regressor head
//   smz_sumgan_att_selector_forward   the selector of models/sumgan_att.py, nhead=4 or 8: final LayerNorm, Linear(1024, 1)
//                                     and sigmoid
//
// Per chunk of whole videos (<= 32 768 rows, a longer video is a chunk of its own), per layer:
//   qkv = xb . Wqkv^T + bqkv                       [R, 3072] bf16      GEMM (bias epilogue)
//   a   = attention(qkv) per (video, head)         [R, 1024] bf16      smz_attn.cu (heads 1024 / nhead wide)
//   y   = a . Wo^T + bo + x                        [R, 1024] fp32      GEMM (bias + residual epilogue)
//   x   = norm1(y) (eps 1e-5)                      fp32 + bf16 copy    LayerNorm row kernel
//   h   = relu(xb . W1^T + b1)                     [R, 1024] bf16      GEMM
//   y   = h . W2^T + b2 + x                        fp32                GEMM
//   x   = norm2(y)                                 fp32 + bf16 copy    LayerNorm row kernel
// then, for smz_transformer_forward, e = layer_norm(x) (+ the encoder input when more_residuals) as bf16, and the head:
// the k1 GEMM epilogue reduces relu(e . K1^T + k1b) to the three row sums of the shared LayerNorm + k2 dot
// (GEMM_ROWSTATS), a per-row kernel finishes sigmoid(...); for the selector, one row kernel computes
// sigmoid(layer_norm(x) . w + b) from the float32 x.  The residual stream and every LayerNorm input stay float32; bf16
// appears only as GEMM operands.
#include <vector>

#include "smz_gemm.cuh"
#include "smz_rows.cuh"

namespace smz {
int64_t mha_table_bytes(int n_videos);
int mha_forward(const void *qkv, int64_t rows, int64_t ld, const int32_t *h_cu, int v0, int v1, int n_heads, int head_dim,
                void *out, int64_t ldo, void *d_table, cudaStream_t st);
}

namespace {

using smz::GemmEpilogue;
using smz::GemmProblem;
using smz::kFeat;
typedef __nv_bfloat16 bf16;

constexpr int kRowChunk = 32768;
constexpr float kLayerEps = 1e-5f;      // nn.TransformerEncoderLayer's norm1 / norm2 (torch default)

inline int64_t up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

struct Chunk { int v0, v1, row0, rows; };

struct Plan {
    std::vector<Chunk> chunks;
    int64_t off_xb, off_xf, off_qkv, off_a, off_y, off_hstat, off_table, total;
};

int make_plan(const int32_t *cu, int n_videos, Plan *pl) {
    SMZ_REQUIRE(cu != nullptr && n_videos > 0, "transformer: empty batch");
    SMZ_REQUIRE(cu[0] == 0, "transformer: cu_seqlens[0] must be 0");
    for (int v = 0; v < n_videos; v++) SMZ_REQUIRE(cu[v + 1] > cu[v], "transformer: video %d has no frames", v);
    int v = 0, max_rows = 0;
    while (v < n_videos) {
        Chunk c;
        c.v0 = v; c.row0 = cu[v];
        int rows = 0;
        while (v < n_videos && (rows == 0 || rows + (cu[v + 1] - cu[v]) <= kRowChunk)) { rows += cu[v + 1] - cu[v]; ++v; }
        c.v1 = v; c.rows = rows;
        if (rows > max_rows) max_rows = rows;
        pl->chunks.push_back(c);
    }
    const int64_t R = up(max_rows, 8);
    int64_t o = 0;
    auto take = [&](int64_t bytes) { const int64_t at = o; o += up(bytes, 1024); return at; };
    pl->off_xb = take(R * kFeat * 2);
    pl->off_xf = take(R * kFeat * 4);
    pl->off_qkv = take(R * 3 * kFeat * 2);
    pl->off_a = take(R * kFeat * 2);
    pl->off_y = take(R * kFeat * 4);
    pl->off_hstat = take(R * (2 * kFeat / smz::GEMM_BN) * 3 * 4);
    pl->off_table = take(smz::mha_table_bytes(n_videos));     // per chunk, at the chunk's first video
    pl->total = o;
    return SMZ_OK;
}

GemmProblem dense_problem(int M, int N, int K, int ldc, int ldr) {
    GemmProblem g = {};
    g.M = M; g.N = N; g.K = K; g.ldc = ldc; g.ldr = ldr;
    g.tiles_n = (N + smz::GEMM_BN - 1) / smz::GEMM_BN;
    return g;
}

// C = epilogue(A . W^T) for a dense [R, K] x [N, K] problem
int linear(const void *A, int R, int K, const void *W, int N, const GemmEpilogue &e, int ldr, cudaStream_t st) {
    return smz::gemm_bf16_tn(A, R, K, K, W, N, K, K, nullptr, 1, smz::gemm_tiles(R, N), dense_problem(R, N, K, N, ldr), e, st);
}

// The work buffer's regions for the largest chunk of a plan
struct Work {
    bf16 *xb;           // bf16 GEMM operand
    float *xf;          // float32 residual stream
    bf16 *qkv;
    bf16 *a;            // attention output, then the feed-forward hidden layer
    float *y;           // float32 LayerNorm input
    float *hstat;       // head row statistics
    uint8_t *table;     // attention tables, chunk k's at byte v0 * 16
};

// Argument checks shared by the entry points, the plan, and the work buffer carved into its regions.
int prepare(const void *x, const int32_t *h_cu_seqlens, int n_videos, const smz_transformer_layer *layers, int n_layers,
            const void *scores, void *ws, int64_t ws_bytes, Plan *pl, Work *w) {
    SMZ_REQUIRE(x && scores && ws, "transformer_forward: NULL pointer");
    SMZ_REQUIRE(n_layers >= 1 && layers != nullptr, "transformer_forward: need at least one encoder layer");
    for (int l = 0; l < n_layers; l++) {
        const smz_transformer_layer &L = layers[l];
        SMZ_REQUIRE(L.w_qkv && L.b_qkv && L.w_out && L.b_out && L.w1 && L.b1 && L.w2 && L.b2 && L.norm1_g && L.norm1_b &&
                    L.norm2_g && L.norm2_b, "transformer_forward: NULL parameter pointer in layer %d", l);
    }
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    rc = make_plan(h_cu_seqlens, n_videos, pl);
    if (rc != SMZ_OK) return rc;
    SMZ_REQUIRE(ws_bytes >= pl->total, "transformer_forward: work buffer too small (%lld < %lld bytes)", (long long)ws_bytes,
                (long long)pl->total);
    uint8_t *b = reinterpret_cast<uint8_t *>(ws);
    w->xb = reinterpret_cast<bf16 *>(b + pl->off_xb);
    w->xf = reinterpret_cast<float *>(b + pl->off_xf);
    w->qkv = reinterpret_cast<bf16 *>(b + pl->off_qkv);
    w->a = reinterpret_cast<bf16 *>(b + pl->off_a);
    w->y = reinterpret_cast<float *>(b + pl->off_y);
    w->hstat = reinterpret_cast<float *>(b + pl->off_hstat);
    w->table = b + pl->off_table;
    return SMZ_OK;
}

// The encoder layers over chunk c: x -> the float32 output of the last norm2 in w.xf.  *xin receives the chunk's input
// rows (float32 or bf16, as x).  Heads are 1024 / n_heads wide.
int encoder_chunk(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, const Chunk &c,
                  const smz_transformer_layer *layers, int n_layers, int n_heads, const Work &w, const void **xin_out,
                  cudaStream_t st) {
    const int R = c.rows;
    const void *xin = x_is_bf16 ? (const void *)(reinterpret_cast<const bf16 *>(x) + (int64_t)c.row0 * kFeat)
                                : (const void *)(reinterpret_cast<const float *>(x) + (int64_t)c.row0 * kFeat);
    *xin_out = xin;
    const bf16 *a0 = reinterpret_cast<const bf16 *>(xin);
    int rc;
    if (!x_is_bf16) {
        rc = smz::launch_cvt_bf16(reinterpret_cast<const float *>(xin), w.xb, (int64_t)R * kFeat, st);
        if (rc != SMZ_OK) return rc;
        a0 = w.xb;
    }
    void *table = w.table + (int64_t)c.v0 * 16;
    for (int l = 0; l < n_layers; l++) {
        const smz_transformer_layer &L = layers[l];
        const bool first = l == 0, last = l == n_layers - 1;
        rc = linear(first ? (const void *)a0 : (const void *)w.xb, R, kFeat, L.w_qkv, 3 * kFeat,
                    GemmEpilogue{w.qkv, L.b_qkv, nullptr, 1.f, 0}, 0, st);
        if (rc != SMZ_OK) return rc;
        SMZ_DEBUG_STEP(st, "transformer_qkv");
        rc = smz::mha_forward(w.qkv, R, 3 * kFeat, h_cu_seqlens, c.v0, c.v1, n_heads, kFeat / n_heads, w.a, kFeat, table, st);
        if (rc != SMZ_OK) return rc;
        SMZ_DEBUG_STEP(st, "transformer_attention");
        const void *res = first ? xin : (const void *)w.xf;
        const int res_f32 = (first && x_is_bf16) ? 0 : smz::GEMM_RES_F32;
        rc = linear(w.a, R, kFeat, L.w_out, kFeat, GemmEpilogue{w.y, L.b_out, res, 1.f, smz::GEMM_OUT_F32 | res_f32}, kFeat, st);
        if (rc != SMZ_OK) return rc;
        SMZ_DEBUG_STEP(st, "transformer_out_proj");
        rc = smz::launch_layernorm(w.y, nullptr, L.norm1_g, L.norm1_b, kLayerEps, R, w.xb, nullptr, nullptr, st, 0, w.xf);
        if (rc != SMZ_OK) return rc;
        rc = linear(w.xb, R, kFeat, L.w1, kFeat, GemmEpilogue{w.a, L.b1, nullptr, 1.f, smz::GEMM_RELU}, 0, st);
        if (rc != SMZ_OK) return rc;
        rc = linear(w.a, R, kFeat, L.w2, kFeat, GemmEpilogue{w.y, L.b2, w.xf, 1.f, smz::GEMM_OUT_F32 | smz::GEMM_RES_F32},
                    kFeat, st);
        if (rc != SMZ_OK) return rc;
        SMZ_DEBUG_STEP(st, "transformer_ffn");
        rc = smz::launch_layernorm(w.y, nullptr, L.norm2_g, L.norm2_b, kLayerEps, R, last ? nullptr : w.xb, nullptr, nullptr,
                                   st, 0, w.xf);
        if (rc != SMZ_OK) return rc;
    }
    return SMZ_OK;
}

}  // namespace

extern "C" int smz_transformer_workspace_bytes(const int32_t *h_cu_seqlens, int n_videos, int x_is_bf16, int64_t *bytes) {
    SMZ_REQUIRE(bytes != nullptr, "bytes is NULL");
    (void)x_is_bf16;     // the work buffer does not depend on the feature format
    Plan pl;
    int rc = make_plan(h_cu_seqlens, n_videos, &pl);
    if (rc != SMZ_OK) return rc;
    *bytes = pl.total;
    return SMZ_OK;
}

extern "C" int smz_transformer_forward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos,
                                       const smz_transformer_params *p, int n_layers, float *scores, void *ws,
                                       int64_t ws_bytes, void *stream) {
    SMZ_REQUIRE(p != nullptr, "transformer_forward: NULL pointer");
    SMZ_REQUIRE(p->ln_g && p->ln_b && p->k1_w && p->k1_b && p->head_gw && p->head_c, "transformer_forward: NULL parameter pointer");
    Plan pl;
    Work w;
    int rc = prepare(x, h_cu_seqlens, n_videos, p->layers, n_layers, scores, ws, ws_bytes, &pl, &w);
    if (rc != SMZ_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    for (const Chunk &c : pl.chunks) {
        const int R = c.rows;
        const void *xin = nullptr;
        rc = encoder_chunk(x, x_is_bf16, h_cu_seqlens, c, p->layers, n_layers, 8, w, &xin, st);
        if (rc != SMZ_OK) return rc;
        // encoder's final norm (the model's shared layer_norm) -> bf16 operand of k1; more_residuals adds the encoder input
        rc = smz::launch_layernorm(w.xf, nullptr, p->ln_g, p->ln_b, p->eps, R, w.xb, nullptr, nullptr, st, 0, nullptr,
                                   p->more_residuals ? xin : nullptr, x_is_bf16 != 0);
        if (rc != SMZ_OK) return rc;
        {
            GemmEpilogue e{w.hstat, p->k1_b, nullptr, 1.f, smz::GEMM_RELU | smz::GEMM_OUT_F32 | smz::GEMM_ROWSTATS | smz::GEMM_NO_STORE};
            e.stat_w = p->head_gw; e.stat_out = w.hstat;
            rc = linear(w.xb, R, kFeat, p->k1_w, kFeat, e, 0, st);
            if (rc != SMZ_OK) return rc;
        }
        rc = smz::launch_head_from_stats(w.hstat, 2 * kFeat / smz::GEMM_BN, p->head_c, p->eps, R, scores + c.row0, st);
        if (rc != SMZ_OK) return rc;
        SMZ_DEBUG_STEP(st, "transformer_head");
    }
    return SMZ_OK;
}

extern "C" int smz_sumgan_att_selector_forward(const void *x, int x_is_bf16, const int32_t *h_cu_seqlens, int n_videos,
                                               const smz_sumgan_att_selector_params *p, int n_layers, float *scores,
                                               void *ws, int64_t ws_bytes, void *stream) {
    SMZ_REQUIRE(p != nullptr, "sumgan_att_selector_forward: NULL pointer");
    if (p->n_heads != 4 && p->n_heads != 8)
        return smz::fail(SMZ_ERR_UNSUPPORTED, "sumgan_att_selector_forward: n_heads %d is not supported (4 or 8)", p->n_heads);
    SMZ_REQUIRE(p->ln_g && p->ln_b && p->out_w && p->out_b, "sumgan_att_selector_forward: NULL parameter pointer");
    Plan pl;
    Work w;
    int rc = prepare(x, h_cu_seqlens, n_videos, p->layers, n_layers, scores, ws, ws_bytes, &pl, &w);
    if (rc != SMZ_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    for (const Chunk &c : pl.chunks) {
        const void *xin = nullptr;
        rc = encoder_chunk(x, x_is_bf16, h_cu_seqlens, c, p->layers, n_layers, p->n_heads, w, &xin, st);
        if (rc != SMZ_OK) return rc;
        // the encoder's final norm (the selector's layer_norm), out[0] and sigmoid, on the float32 residual stream
        rc = smz::launch_head(w.xf, nullptr, p->ln_g, p->ln_b, p->eps, p->out_w, p->out_b, c.rows, scores + c.row0, nullptr,
                              nullptr, st);
        if (rc != SMZ_OK) return rc;
        SMZ_DEBUG_STEP(st, "sumgan_att_selector_head");
    }
    return SMZ_OK;
}
