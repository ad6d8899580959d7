// Fused variable-length multi-head attention (sm_100a): softmax(scale * Q_h K_h^T) V_h for every (video, head) of a
// packed batch, without an attention mask inside a video and with no frame ever attending to another video's frames.
// This is the attention of nn.TransformerEncoderLayer(d_model=1024, nhead=8) (models/transformer.py, heads 128 wide) and
// of nhead=4 (the SumGAN-att selector, models/sumgan_att.py, heads 256 wide) in eval mode.
//
// Input: the packed Q|K|V projection rows, bf16 [R, ld] (head h: Q columns [h*HD, h*HD+HD), K at n_heads*HD + h*HD, V
// at 2*n_heads*HD + h*HD), video v owning rows cu[v] .. cu[v+1]-1.  Output: bf16 [R, ldo], head h at column h*HD.
// The kernel is a template on the head width HD (128 or 256); the key tile BKV is 128 keys for HD = 128 and 64 keys for
// HD = 256, so that Q, P and a 2-stage K/V ring fit in shared memory (208 KB at HD = 256: Q 64 KB, P 16 KB, K and V
// 32 KB per stage) and the two S buffers plus O fit the 512 TMEM columns.
//
// One work unit = one 128-row query tile of one (video, head).  Persistent grid; units are numbered longest video first
// (the host sorts the videos), a CTA takes units blockIdx.x, blockIdx.x + gridDim.x, ...
// Per CTA (192 threads, warp-specialised):
//   warps 0-3  softmax: one query row per thread.  Per key tile: tcgen05.ld of the S row, scale, keys past the video's
//              end -> -inf, online row max / row sum in fp32, P = exp2(s - max) as bf16 into shared memory (the
//              tensor core's K-major 128-byte-swizzled layout); when the row max grows, the O accumulator row is
//              rescaled in TMEM (tcgen05.ld / st).  After the last tile: O / l through a shared-memory pad to global.
//   warp 4     TMA producer: Q once per unit, then K and V tiles of BKV keys into a 2-stage ring.  Video starts are not
//              aligned: TMA takes any start row; rows of the next video are masked by the softmax, rows past the end of
//              the array arrive zero-filled.
//   warp 5     MMA issuer: S_j = Q K_j^T into one of two TMEM score buffers (the QK^T of tile j+1 is issued before the
//              P.V of tile j, so it overlaps the softmax of tile j), O += P_j V_j into a third TMEM region.
// TMEM: S0 = columns [0,BKV), S1 = [BKV,2*BKV), O = [2*BKV, 2*BKV+HD) of a 512-column allocation.
// This is a true online softmax (running max subtraction): no range assumption on the logits.
#include "smz_gemm.cuh"
#include "smz_tc.cuh"

#include <algorithm>
#include <vector>

namespace {

using namespace smztc;
typedef __nv_bfloat16 bf16;

constexpr int BQ = 128;                   // query rows per unit
constexpr int STAGES = 2;
constexpr int NUM_THREADS = 192;
constexpr int TMEM_COLS = 512;

// Tile shapes per head width.  Operands are stored as 64-column (128-byte) swizzled blocks: a K-major block of r rows
// is r * 128 bytes, an MN-major V box (64 keys x 64 d-columns) is 8 KB.
template <int HD>
struct MhaShape {
    static_assert(HD == 128 || HD == 256, "head width");
    static constexpr int BKV = HD == 128 ? 128 : 64;        // keys per tile
    static constexpr int DB = HD / 64;                       // 64-column blocks of a head
    static constexpr int KB = BKV / 64;                      // 64-key blocks of a tile
    static constexpr int Q_BYTES = BQ * HD * 2;
    static constexpr int P_BYTES = BQ * BKV * 2;
    static constexpr int KV_BYTES = BKV * HD * 2;            // one K or one V tile
    static constexpr int SMEM_BYTES = Q_BYTES + P_BYTES + 2 * STAGES * KV_BYTES + 256 + 1024;   // + barriers, alignment slack
    static_assert(2 * BKV + HD <= TMEM_COLS, "S double buffer and O exceed TMEM");
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
};

struct MhaVideo { int32_t row0, T, unit0, qtiles; };
static_assert(sizeof(MhaVideo) == 16, "MhaVideo layout");

struct MhaParams {
    const MhaVideo *videos;
    int n_videos, total_units, n_heads;
    bf16 *out;
    int64_t ldo;
    float scale_log2;     // softmax scale * log2(e): exponentials are exp2
};

struct UnitCursor {
    int v = 0;
    MhaVideo cur;
    int h = 0, qt = 0;
    __device__ __forceinline__ void seek(const MhaParams &P, int u) {
        while (v + 1 < P.n_videos && u >= __ldg(&P.videos[v + 1].unit0)) ++v;
        cur = P.videos[v];
        const int local = u - cur.unit0;
        h = local / cur.qtiles;
        qt = local - h * cur.qtiles;
    }
};

// tmQK: boxes of BKV rows x 64 columns (Q tiles are loaded as BQ / BKV boxes per column block); tmV: 64 x 64 boxes
template <int HD>
__global__ void __launch_bounds__(NUM_THREADS, 1)
mha_fwd_kernel(const __grid_constant__ CUtensorMap tmQK, const __grid_constant__ CUtensorMap tmV, const MhaParams P) {
    typedef MhaShape<HD> S;
    constexpr int BKV = S::BKV, DB = S::DB, KB = S::KB, KV_BYTES = S::KV_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SWIZZLE_128B atoms
    uint8_t *sQ = smem;                                   // [64-column block d] of BQ rows
    uint8_t *sP = smem + S::Q_BYTES;                      // [64-key block kb] of BQ rows
    uint8_t *sK = sP + S::P_BYTES;                        // STAGES tiles: [64-column block d] of BKV rows
    uint8_t *sV = sK + STAGES * KV_BYTES;                 // STAGES tiles: [key block kb][64 d-columns j] boxes of 8 KB
    uint64_t *bars = reinterpret_cast<uint64_t *>(sV + STAGES * KV_BYTES);
    uint64_t *q_full = bars, *q_empty = bars + 1;
    uint64_t *kv_full = bars + 2, *kv_empty = bars + 2 + STAGES;
    uint64_t *s_full = bars + 2 + 2 * STAGES, *s_empty = s_full + 2;
    uint64_t *p_full = s_empty + 2, *o_done = p_full + 1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(o_done + 1);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
    if (warp == 4 && lane == 0) {
        tma_prefetch_desc(&tmQK);
        tma_prefetch_desc(&tmV);
        mbar_init(q_full, 1); mbar_init(q_empty, 1);
        for (int i = 0; i < STAGES; i++) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], 128); }
        mbar_init(p_full, 128); mbar_init(o_done, 1);
        fence_mbar_init();
    }
    if (warp == 5) tmem_alloc<TMEM_COLS>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tS = tmem_base, tO = tmem_base + 2 * BKV;

    if (warp == 4) {
        // ------------------------------------------------------------------ TMA producer
        UnitCursor c;
        int stage = 0; uint32_t phase = 0, qn = 0;
        for (int u = blockIdx.x; u < P.total_units; u += gridDim.x, ++qn) {
            c.seek(P, u);
            const int nk = (c.cur.T + BKV - 1) / BKV;
            const int qcol = c.h * HD, kcol = P.n_heads * HD + c.h * HD, vcol = 2 * P.n_heads * HD + c.h * HD;
            mbar_wait(q_empty, (qn & 1u) ^ 1u);          // every QK^T of the previous unit has completed
            if (elect_one()) {
                mbar_arrive_expect_tx(q_full, S::Q_BYTES);
#pragma unroll
                for (int d = 0; d < DB; d++)
#pragma unroll
                    for (int rh = 0; rh < BQ / BKV; rh++)
                        tma_load_2d(sQ + d * BQ * 128 + rh * BKV * 128, &tmQK, q_full, qcol + 64 * d,
                                    c.cur.row0 + c.qt * BQ + rh * BKV);
            }
            __syncwarp();
            for (int j = 0; j < nk; j++) {
                mbar_wait(&kv_empty[stage], phase ^ 1u);
                if (elect_one()) {
                    const int r = c.cur.row0 + j * BKV;
                    uint8_t *k = sK + stage * KV_BYTES, *v = sV + stage * KV_BYTES;
                    mbar_arrive_expect_tx(&kv_full[stage], 2 * KV_BYTES);
#pragma unroll
                    for (int d = 0; d < DB; d++) tma_load_2d(k + d * BKV * 128, &tmQK, &kv_full[stage], kcol + 64 * d, r);
#pragma unroll
                    for (int kb = 0; kb < KB; kb++)
#pragma unroll
                        for (int jn = 0; jn < DB; jn++)
                            tma_load_2d(v + (kb * DB + jn) * 8192, &tmV, &kv_full[stage], vcol + 64 * jn, r + 64 * kb);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 5) {
        // ------------------------------------------------------------------ MMA issuer
        // whole warp walks the loop (warp-uniform descriptors), one elected lane issues
        UnitCursor c;
        const uint32_t idesc_s = make_idesc_bf16(BQ, BKV);                 // Q, K both K-major
        const uint32_t idesc_o = make_idesc_bf16(BQ, HD) | (1u << 16);     // B = V stored [key][d]: MN-major
        const uint32_t q_addr = smem_u32(sQ), p_addr = smem_u32(sP);
        int stage = 0; uint32_t phase = 0, qn = 0, sn = 0, pn = 0;
        auto issue_s = [&](int st, uint32_t ph) {     // S[sn & 1] = Q K^T of the tile in ring slot (st, phase ph)
            const uint32_t b = sn & 1u;
            mbar_wait(&s_empty[b], ((sn >> 1) & 1u) ^ 1u);
            mbar_wait(&kv_full[st], ph);
            tc_fence_after();
            const uint32_t k_addr = smem_u32(sK + st * KV_BYTES);
            if (elect_one()) {
#pragma unroll
                for (int d = 0; d < DB; d++) {
                    const uint64_t qd = make_kmajor_sw128_desc(q_addr + d * BQ * 128), kd = make_kmajor_sw128_desc(k_addr + d * BKV * 128);
#pragma unroll
                    for (int k = 0; k < 4; k++) umma_bf16<false>(tS + b * BKV, qd + 2 * k, kd + 2 * k, idesc_s, (uint32_t)((d | k) != 0));
                }
                umma_commit<false>(&s_full[b]);
            }
            __syncwarp();
            ++sn;
        };
        for (int u = blockIdx.x; u < P.total_units; u += gridDim.x, ++qn) {
            c.seek(P, u);
            const int nk = (c.cur.T + BKV - 1) / BKV;
            mbar_wait(q_full, qn & 1u);
            issue_s(stage, phase);
            for (int j = 0; j < nk; j++) {
                const bool wrap = stage + 1 == STAGES;
                if (j + 1 < nk) issue_s(wrap ? 0 : stage + 1, wrap ? phase ^ 1u : phase);                        // overlaps the softmax of tile j
                else {
                    if (elect_one()) umma_commit<false>(q_empty);    // Q is free once these QK^T MMAs complete
                    __syncwarp();
                }
                mbar_wait(p_full, pn & 1u);                           // P_j written, O rescaled
                ++pn;
                tc_fence_after();
                const uint32_t v_addr = smem_u32(sV + stage * KV_BYTES);
                if (elect_one()) {
#pragma unroll
                    for (int kb = 0; kb < KB; kb++) {
                        const uint64_t pd = make_kmajor_sw128_desc(p_addr + kb * BQ * 128), vd = make_mnmajor_sw128_desc(v_addr + kb * DB * 8192);
#pragma unroll
                        for (int k = 0; k < 4; k++) umma_bf16<false>(tO, pd + 2 * k, vd + 128 * k, idesc_o, (uint32_t)((j | kb | k) != 0));
                    }
                    umma_commit<false>(&kv_empty[stage]);
                    umma_commit<false>(o_done);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else {
        // ------------------------------------------------------------------ softmax + epilogue (warps 0-3)
        UnitCursor c;
        const int row = warp * 32 + lane;
        const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
        uint32_t sn = 0, on = 0;
        uint8_t *prow = sP + row * 128;                   // this row of P's first 64-key block (the second is 16 KB on)
        for (int u = blockIdx.x; u < P.total_units; u += gridDim.x) {
            c.seek(P, u);
            const int T = c.cur.T;
            const int nk = (T + BKV - 1) / BKV;
            float m_run = -INFINITY, l_run = 0.f;
            for (int j = 0; j < nk; j++) {
                const uint32_t b = sn & 1u;
                mbar_wait(&s_full[b], (sn >> 1) & 1u);
                ++sn;
                tc_fence_after();
                uint32_t v[BKV / 32][32];
#pragma unroll
                for (int q = 0; q < BKV / 32; q++) tmem_ld32(tS + lane_off + b * BKV + 32 * q, v[q]);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(&s_empty[b]);                  // the MMA warp may overwrite this S buffer
                const int valid = T - j * BKV;             // keys of this tile inside the video (>= 1)
                float mx = m_run;
#pragma unroll
                for (int q = 0; q < BKV / 32; q++)
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        const float s = (32 * q + i < valid) ? __uint_as_float(v[q][i]) * P.scale_log2 : -INFINITY;
                        v[q][i] = __float_as_uint(s);
                        mx = fmaxf(mx, s);
                    }
                // key 0 of every video is valid: mx is finite from the first tile on
                if (j > 0) {
                    mbar_wait(o_done, on & 1u);            // P.V of tile j-1 done: O is stable and P may be overwritten
                    ++on;
                    tc_fence_after();
                    const float alpha = exp2f(m_run - mx);
                    l_run *= alpha;
                    if (__any_sync(0xffffffffu, mx > m_run)) {      // warp-uniform: rescale the O rows of this warp
#pragma unroll 1
                        for (int q = 0; q < HD / 32; q++) {
                            uint32_t o[32];
                            tmem_ld32(tO + lane_off + 32 * q, o);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; i++) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                            tmem_st32(tO + lane_off + 32 * q, o);
                        }
                        tmem_st_wait();
                    }
                }
                m_run = mx;
                float sum = 0.f;
                // P row -> shared memory, K-major with the 128-byte swizzle: key block kb (64 keys) at kb * 16 KB, row r at
                // r * 128 B, 16-byte chunk c (keys 8c..8c+7 of the block) at chunk position c ^ (r & 7)
#pragma unroll
                for (int q = 0; q < BKV / 32; q++) {
                    uint32_t pk[16];
#pragma unroll
                    for (int i = 0; i < 32; i += 2) {
                        const float p0 = exp2f(__uint_as_float(v[q][i]) - mx), p1 = exp2f(__uint_as_float(v[q][i + 1]) - mx);
                        sum += p0 + p1;
                        pk[i >> 1] = pack_bf16x2(p0, p1);
                    }
                    const int kb = q >> 1;
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) {
                        const int chunk = (q & 1) * 4 + cc;
                        *reinterpret_cast<uint4 *>(prow + kb * 16384 + ((chunk ^ (row & 7)) << 4)) =
                            make_uint4(pk[4 * cc], pk[4 * cc + 1], pk[4 * cc + 2], pk[4 * cc + 3]);
                    }
                }
                l_run += sum;
                fence_proxy_async_smem();                  // P is read by the tensor core (async proxy)
                tc_fence_before();
                mbar_arrive(p_full);
            }
            // epilogue: O / l -> bf16 through a per-warp pad -> rows of the video.  The pad lies in this warp's own rows of P
            // (the last P.V has completed), so no other warp's next P tile can overlap it.
            mbar_wait(o_done, on & 1u);
            ++on;
            tc_fence_after();
            const float inv_l = 1.f / l_run;
            uint32_t *pad = reinterpret_cast<uint32_t *>(sP + warp * 32 * 128);   // 32 rows x 80 B inside 4 KB
            const int m_base = c.qt * BQ + warp * 32;    // video-local row of this warp's lane 0
            const int sub = lane >> 2, part = lane & 3;
            bf16 *obase = P.out + (int64_t)c.cur.row0 * P.ldo + c.h * HD + part * 8;
#pragma unroll 1
            for (int q = 0; q < HD / 32; q++) {
                uint32_t o[32];
                tmem_ld32(tO + lane_off + 32 * q, o);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; i += 8)
                    *reinterpret_cast<uint4 *>(pad + lane * 20 + (i >> 1)) =
                        make_uint4(pack_bf16x2(__uint_as_float(o[i]) * inv_l, __uint_as_float(o[i + 1]) * inv_l),
                                   pack_bf16x2(__uint_as_float(o[i + 2]) * inv_l, __uint_as_float(o[i + 3]) * inv_l),
                                   pack_bf16x2(__uint_as_float(o[i + 4]) * inv_l, __uint_as_float(o[i + 5]) * inv_l),
                                   pack_bf16x2(__uint_as_float(o[i + 6]) * inv_l, __uint_as_float(o[i + 7]) * inv_l));
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 4; i++) {              // 8 rows x 64 contiguous bytes per store instruction
                    const int r = 8 * i + sub;
                    const uint4 w4 = *reinterpret_cast<const uint4 *>(pad + r * 20 + part * 4);
                    if (m_base + r < T) *reinterpret_cast<uint4 *>(obase + (int64_t)(m_base + r) * P.ldo + 32 * q) = w4;
                }
                __syncwarp();
            }
            tc_fence_before();     // the O reads above precede the next unit's first P.V (ordered through p_full)
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

// Tensor maps, parameters and the launch of the HD-wide kernel (the table is already uploaded).
template <int HD>
int launch_mha(const void *qkv, int64_t rows, int64_t ld, int n_heads, MhaParams P, int64_t units, cudaStream_t st) {
    typedef MhaShape<HD> S;
    alignas(64) CUtensorMap mqk, mv;
    const int64_t cols = 3LL * n_heads * HD;
    int rc = smz::make_bf16_map(&mqk, qkv, rows, cols, ld, S::BKV);
    if (rc != SMZ_OK) return rc;
    rc = smz::make_bf16_map(&mv, qkv, rows, cols, ld, 64);
    if (rc != SMZ_OK) return rc;
    P.scale_log2 = 1.4426950408889634f / sqrtf((float)HD);
    static bool attr_set[64] = {false};
    int dev = 0;
    SMZ_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
        SMZ_CUDA_CHECK(cudaFuncSetAttribute((const void *)mha_fwd_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            S::SMEM_BYTES));
        attr_set[dev] = true;
    }
    const int grid = (int)std::min<int64_t>(units, (int64_t)smz::sm_count());
    mha_fwd_kernel<HD><<<grid, NUM_THREADS, S::SMEM_BYTES, st>>>(mqk, mv, P);
    SMZ_CUDA_CHECK(cudaGetLastError());
    return SMZ_OK;
}

}  // namespace

namespace smz {

int64_t mha_table_bytes(int n_videos) { return ((int64_t)n_videos * (int64_t)sizeof(MhaVideo) + 1023) / 1024 * 1024; }

// Builds the unit table of videos [v0, v1) of h_cu (rows relative to h_cu[v0]), longest video first, uploads it to
// d_table (mha_table_bytes(v1 - v0) bytes) and launches the kernel on qkv rows [0, rows).
// head_dim: 128 or 256.
int mha_forward(const void *qkv, int64_t rows, int64_t ld, const int32_t *h_cu, int v0, int v1, int n_heads, int head_dim,
                void *out, int64_t ldo, void *d_table, cudaStream_t st) {
    const int n = v1 - v0;
    if (n <= 0) return SMZ_OK;
    if (head_dim != 128 && head_dim != 256)
        return fail(SMZ_ERR_UNSUPPORTED, "mha: head_dim %d is not supported (128 or 256)", head_dim);
    SMZ_REQUIRE(qkv && out && d_table && h_cu, "mha_forward: NULL pointer");
    const int64_t w = (int64_t)n_heads * head_dim;
    SMZ_REQUIRE(n_heads > 0 && ld >= 3 * w && ldo >= w && (ldo & 7) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "mha_forward: need ld >= 3 * n_heads * head_dim, ldo >= n_heads * head_dim, ldo %% 8 == 0 and a 16-byte "
                "aligned output");
    std::vector<int> order((size_t)n);
    for (int i = 0; i < n; i++) {
        order[i] = i;
        SMZ_REQUIRE(h_cu[v0 + i + 1] > h_cu[v0 + i], "mha_forward: video %d has no frames", v0 + i);
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        return h_cu[v0 + a + 1] - h_cu[v0 + a] > h_cu[v0 + b + 1] - h_cu[v0 + b];
    });
    std::vector<MhaVideo> tab((size_t)n);
    int64_t units = 0;
    for (int i = 0; i < n; i++) {
        const int v = v0 + order[i];
        MhaVideo &e = tab[i];
        e.row0 = h_cu[v] - h_cu[v0];
        e.T = h_cu[v + 1] - h_cu[v];
        e.qtiles = (e.T + BQ - 1) / BQ;
        e.unit0 = (int32_t)units;
        units += (int64_t)e.qtiles * n_heads;
    }
    SMZ_REQUIRE(units < (1LL << 31), "mha_forward: too many work units");
    SMZ_REQUIRE(rows >= h_cu[v1] - h_cu[v0], "mha_forward: fewer rows than the videos cover");
    int rc = upload_small(d_table, tab.data(), tab.size() * sizeof(MhaVideo), st);
    if (rc != SMZ_OK) return rc;
    MhaParams P;
    P.videos = reinterpret_cast<const MhaVideo *>(d_table);
    P.n_videos = n;
    P.total_units = (int)units;
    P.n_heads = n_heads;
    P.out = reinterpret_cast<bf16 *>(out);
    P.ldo = ldo;
    return head_dim == 128 ? launch_mha<128>(qkv, rows, ld, n_heads, P, units, st)
                           : launch_mha<256>(qkv, rows, ld, n_heads, P, units, st);
}

}  // namespace smz

extern "C" int smz_mha_workspace_bytes(int n_videos, int64_t *bytes) {
    SMZ_REQUIRE(bytes != nullptr, "bytes is NULL");
    SMZ_REQUIRE(n_videos > 0, "mha: empty batch");
    *bytes = smz::mha_table_bytes(n_videos);
    return SMZ_OK;
}

extern "C" int smz_mha_forward(const void *qkv, int64_t ld, const int32_t *h_cu_seqlens, int n_videos, int n_heads,
                               int head_dim, void *out, int64_t ldo, void *ws, int64_t ws_bytes, void *stream) {
    if (head_dim != 128 && head_dim != 256)
        return smz::fail(SMZ_ERR_UNSUPPORTED, "mha: head_dim %d is not supported (128 or 256)", head_dim);
    SMZ_REQUIRE(h_cu_seqlens != nullptr && n_videos > 0, "mha: empty batch");
    SMZ_REQUIRE(h_cu_seqlens[0] == 0, "mha: cu_seqlens[0] must be 0");
    SMZ_REQUIRE(ws != nullptr && ws_bytes >= smz::mha_table_bytes(n_videos), "mha: work buffer too small (%lld < %lld bytes)",
                (long long)ws_bytes, (long long)smz::mha_table_bytes(n_videos));
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    return smz::mha_forward(qkv, h_cu_seqlens[n_videos], ld, h_cu_seqlens, 0, n_videos, n_heads, head_dim, out, ldo,
                            ws, (cudaStream_t)stream);
}
