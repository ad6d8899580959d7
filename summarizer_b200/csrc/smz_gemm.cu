// tcgen05 GEMM building block (sm_100a):  C = epilogue(alpha * A * B^T), bf16 operands, fp32
// accumulation in tensor memory.  Every dense contraction of the scorers goes through this kernel:
// VASNet's packed Q|K projection, V^T projection, Q.K^T logits, alpha.V, output projection and k1
// (vasnet.py:114-140), DSN's LSTM input projection (dsn.py:45) and the reward Gram matrix
// (dsn.py:215-216,226-228).
//
// Structure (persistent, 320 threads per CTA, warp-specialised; default = CTA PAIRS, see Cfg<PAIR> below):
//   warp 0      TMA producer (every CTA): its 128 A rows and its share of the B rows per 64-wide k block, bf16
//               boxes with the 128-byte swizzle, mbarrier ring (5 x 32 KB per CTA in pair mode).
//   warp 1      MMA issuer (leader CTA of the pair): one thread issues tcgen05.mma cta_group::2 (M=256, N=256,
//               K=16) reading both CTAs' shared memory and accumulating in both CTAs' tensor memory (two 256-column
//               accumulators per CTA, double buffered); tcgen05.commit multicasts "stage free" / "tile ready".
//   warps 2-9   epilogue (two per TMEM lane quadrant, 128 columns each): tcgen05.ld 32 lanes x 32 columns, then one
//               of three COMPILE-TIME epilogues (plain: alpha / bias or row scale / residual / ReLU / store with
//               prefetched residual and smem-transposed fp32 stores; head: bias + ReLU + three row sums, no store;
//               exp: masked exp + row sum + bf16 store + logit-range guard); overlaps the next tile's main loop.
// Operands may be K-major or MN-major (k rows, m/n contiguous): the backward GEMMs read row-major activations.
// Tiles are enumerated problem-major over a ragged batch (one problem per video for the attention
// contractions), N fastest so that CTAs running concurrently share the A tile and the weights in L2.
#include "smz_gemm.cuh"
#include "smz_tc.cuh"

#include <cudaTypedefs.h>
#include <stdlib.h>

namespace {

using namespace smztc;
using smz::GemmEpilogue;
using smz::GemmProblem;

constexpr int BM = 128;                // accumulator rows per CTA (TMEM lanes)
constexpr int BN = smz::GEMM_BN, BK = smz::GEMM_BK;
constexpr int A_STAGE = BM * BK * 2;   // 16 KB
constexpr int EPI_WARPS = 8;           // two warps per TMEM lane quadrant, each drains half of the 256 columns
constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
constexpr int TMEM_COLS = 2 * BN;      // two accumulators
constexpr int BAR_BYTES = 256;
constexpr int STG_BYTES = EPI_WARPS * 32 * 33 * 4;   // per epilogue warp: a 32 x 32 fp32 transposition pad (row stride 33 words)
static_assert(TMEM_COLS == 512, "TMEM allocation must be a power of two <= 512 columns");
// PAIR = false: one CTA per 128 x 256 tile, 4 stages of 16 KB (A) + 32 KB (B).
// PAIR = true : a cluster of two CTAs (one TPC) per 256 x 256 tile with tcgen05 cta_group::2: each CTA loads ITS
//               128 rows of A and ITS 128 of the 256 B rows (16 + 16 KB per stage, 6 stages), the leader CTA issues
//               M=256 MMAs that read both CTAs' shared memory and write both CTAs' tensor memory.  Per MMA the
//               pair moves 2/3 of the L2->SM bytes of two independent CTAs — the operand traffic, not the tensor
//               pipe, is what caps the one-CTA kernel at ~1.1 PFLOP/s.
template <bool PAIR> struct Cfg {
    static constexpr int STAGES = PAIR ? 5 : 3;               // 32 KB / 48 KB per stage
    static constexpr int B_ROWS = PAIR ? BN / 2 : BN;          // B rows (n) loaded by one CTA
    static constexpr int B_STAGE = B_ROWS * BK * 2;
    static constexpr int TILE_M = PAIR ? 2 * BM : BM;
    static constexpr int SMEM_BYTES = STAGES * (A_STAGE + B_STAGE) + BAR_BYTES + STG_BYTES + 1024;   // + alignment slack
};

struct Params {
    const GemmProblem *probs;
    GemmProblem single;
    int n_probs, total_tiles;
    GemmEpilogue epi;
};

struct Cursor {
    int p = -1;
    GemmProblem cur;
    __device__ __forceinline__ void seek(const Params &P, int tile) {
        if (P.probs == nullptr) { cur = P.single; return; }
        int q = p < 0 ? 0 : p;
        while (q + 1 < P.n_probs && tile >= __ldg(&P.probs[q + 1].tile0)) ++q;
        if (q != p) { p = q; cur = P.probs[q]; }
    }
};

__device__ __forceinline__ float4 ld_f4(const float *p) { return *reinterpret_cast<const float4 *>(p); }

// A_MN / B_MN: the operand is stored "MN-major" (k rows, m resp. n contiguous) instead of K-major; it is
// then loaded as 64x64 boxes (64 k-rows of 128 bytes, one box per 64 m/n) and described to the tensor
// core with the MN-major canonical layout (LBO = one box = 8 KB between 64-element m/n groups, SBO =
// 1 KB between 8-row k groups, +2 KB per K=16 slice).  This is what lets the backward pass run
// dX = dY.W and dW = dY^T.X on the row-major activations without materialising any transpose.
// EPI selects the epilogue at COMPILE time (the epilogue must stay shorter than the MMA time of a tile, so the
// special modes cannot be paid for by the plain one): EPI_PLAIN = alpha / bias or row scale / residual / ReLU /
// store; EPI_HEAD = bias + ReLU + three row sums, no store (GEMM_ROWSTATS | GEMM_NO_STORE); EPI_EXP = masked exp +
// row sum + bf16 store (GEMM_EXP | GEMM_ROWSTATS).
// EPI_SPLIT = the plain epilogue whose 16-bit output is written as hi + lo planes (GemmEpilogue::c_lo): its own
// instantiation so that the tuned plain epilogue carries none of its registers.
enum { EPI_PLAIN = 0, EPI_HEAD = 1, EPI_EXP = 2, EPI_SPLIT = 3 };

template <bool A_MN, bool B_MN, bool PAIR, int EPI_T>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmA_lo, const __grid_constant__ CUtensorMap tmB_lo, const Params P) {
    constexpr bool SPLIT_OUT = EPI_T == EPI_SPLIT;
    constexpr int EPI = SPLIT_OUT ? (int)EPI_PLAIN : EPI_T;
    // passes of the k loop: hi.hi, then A_lo.B_hi (when A has a lo plane), then A_hi.B_lo (when B has one)
    const int pass_a = P.epi.a_lo != 0 ? 1 : -1;
    const int pass_b = P.epi.b_lo != 0 ? (P.epi.a_lo != 0 ? 2 : 1) : -1;
    const int npass = 1 + (P.epi.a_lo != 0 ? 1 : 0) + (P.epi.b_lo != 0 ? 1 : 0);
    constexpr int STAGES = Cfg<PAIR>::STAGES, B_STAGE = Cfg<PAIR>::B_STAGE, B_ROWS = Cfg<PAIR>::B_ROWS;
    constexpr int TILE_M = Cfg<PAIR>::TILE_M;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SWIZZLE_128B atoms
    uint8_t *sA = smem;
    uint8_t *sB = smem + STAGES * A_STAGE;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + STAGES * (A_STAGE + B_STAGE));
    uint64_t *empty = full + STAGES;
    uint64_t *tfull = empty + STAGES;
    uint64_t *tempty = tfull + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
    float *stg_all = reinterpret_cast<float *>(smem + STAGES * (A_STAGE + B_STAGE) + BAR_BYTES);

    smz::pdl_trigger();                                           // the next kernel of the stream may set itself up under this one
    if (P.epi.gate != nullptr) {                                  // gated launch (fallback path not needed): every CTA leaves
        smz::pdl_wait();
        if (__ldg(P.epi.gate) == 0) return;
    }
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;     // warp index, provably uniform
    const int rank = PAIR ? (int)cluster_ctarank() : 0;           // 0 = leader CTA of the pair
    const int first_tile = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tile_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    if (PAIR) cluster_sync_all();                                 // both CTAs alive before the pair allocates TMEM
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if (npass > 1) { tma_prefetch_desc(&tmA_lo); tma_prefetch_desc(&tmB_lo); }
        for (int i = 0; i < STAGES; i++) { mbar_init(&full[i], PAIR ? 2 : 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], (PAIR ? 2 : 1) * 32 * EPI_WARPS); }
        fence_mbar_init();
    }
    if (warp == 1) { if (PAIR) tmem_alloc_pair<TMEM_COLS>(tmem_slot); else tmem_alloc<TMEM_COLS>(tmem_slot); }
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // everything above (barriers, TMEM, descriptor prefetch) may run under the previous kernel of the stream; from here on
    // global memory is read (problem table, operands, residual) and written
    smz::pdl_wait();

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (every CTA)
        // whole warp in the loop, one elected lane issues (see the MMA issuer below)
        {
            Cursor c;
            int stage = 0; uint32_t phase = 0;
            for (int tile = first_tile; tile < P.total_tiles; tile += tile_step) {
                c.seek(P, tile);
                const int lt = tile - c.cur.tile0;
                const int mt = lt / c.cur.tiles_n, nt = lt - mt * c.cur.tiles_n;
                const int nkb = (c.cur.K + BK - 1) / BK;
                // K-major: (row0, col0) = (first m/n row, first k column); MN-major: (first k row, first m/n column)
                const int a_mn = (A_MN ? c.cur.a_col0 : c.cur.a_row0) + mt * TILE_M + rank * BM;
                const int b_mn = (B_MN ? c.cur.b_col0 : c.cur.b_row0) + nt * BN + rank * B_ROWS;
                const int a_k = A_MN ? c.cur.a_row0 : c.cur.a_col0, b_k = B_MN ? c.cur.b_row0 : c.cur.b_col0;
                for (int kbp = 0; kbp < nkb * npass; kbp++) {
                    const int pass = kbp / nkb, kb = kbp - pass * nkb;
                    const CUtensorMap *mapA = pass == pass_a ? &tmA_lo : &tmA, *mapB = pass == pass_b ? &tmB_lo : &tmB;
                    mbar_wait(&empty[stage], phase ^ 1u);
                    if (elect_one()) {
                        // the bytes of BOTH CTAs are accounted on the leader's barrier, which the MMA thread waits on
                        if (!PAIR) mbar_arrive_expect_tx(&full[stage], A_STAGE + B_STAGE);
                        else if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * (A_STAGE + B_STAGE));
                        else mbar_arrive_remote(&full[stage], 0);
                        if (A_MN) {
#pragma unroll
                            for (int j = 0; j < BM / 64; j++)
                                tma_load<PAIR>(sA + stage * A_STAGE + j * 8192, mapA, &full[stage], a_mn + 64 * j, a_k + kb * BK);
                        } else {
                            tma_load<PAIR>(sA + stage * A_STAGE, mapA, &full[stage], a_k + kb * BK, a_mn);
                        }
                        if (B_MN) {
#pragma unroll
                            for (int j = 0; j < B_ROWS / 64; j++)
                                tma_load<PAIR>(sB + stage * B_STAGE + j * 8192, mapB, &full[stage], b_mn + 64 * j, b_k + kb * BK);
                        } else {
                            tma_load<PAIR>(sB + stage * B_STAGE, mapB, &full[stage], b_k + kb * BK, b_mn);
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        // The whole warp walks the loop and waits on the barriers; one elected lane issues.  With a single-lane branch
        // around the loop the compiler must treat every descriptor as divergent and wraps each tcgen05.mma in an
        // ELECT / R2UR waterfall loop: ~110 dependent instructions per k block against 512 cycles of tensor work,
        // which held the tensor pipe at 65-75 % (profiles/r02c).
        if (rank == 0) {
            Cursor c;
            // operand format fields ([7,10) A, [10,13) B): 1 = bf16 (make_idesc_bf16's default), 0 = f16
            const uint32_t idesc = (make_idesc_bf16(TILE_M, BN) | (A_MN ? (1u << 15) : 0u) | (B_MN ? (1u << 16) : 0u))
                                   & ~(((P.epi.flags & smz::GEMM_A_F16) ? (1u << 7) : 0u) | ((P.epi.flags & smz::GEMM_B_F16) ? (1u << 10) : 0u));
            const uint32_t a_base = smem_u32(sA), b_base = smem_u32(sB);
            int stage = 0; uint32_t phase = 0;
            int it = 0;
            for (int tile = first_tile; tile < P.total_tiles; tile += tile_step, ++it) {
                c.seek(P, tile);
                const int nkb = ((c.cur.K + BK - 1) / BK) * npass;     // split operands: the k extent once per kept product
                const int as = it & 1;
                mbar_wait(&tempty[as], (((uint32_t)it >> 1) & 1u) ^ 1u);   // epilogue(s) drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
                for (int kb = 0; kb < nkb; kb++) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = a_base + stage * A_STAGE, b_addr = b_base + stage * B_STAGE;
                    const uint64_t adesc = A_MN ? make_mnmajor_sw128_desc(a_addr) : make_kmajor_sw128_desc(a_addr);
                    const uint64_t bdesc = B_MN ? make_mnmajor_sw128_desc(b_addr) : make_kmajor_sw128_desc(b_addr);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BK / 16; k++)   // per K=16 slice: +32 B inside the swizzle atom (K-major), +2 KB (MN-major)
                            umma_bf16<PAIR>(d_tmem, adesc + (A_MN ? 128 : 2) * k, bdesc + (B_MN ? 128 : 2) * k, idesc,
                                            (uint32_t)((kb | k) != 0));
                        umma_commit<PAIR>(&empty[stage]);       // PAIR: multicast to the same barrier of both CTAs
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                if (elect_one()) umma_commit<PAIR>(&tfull[as]);
                __syncwarp();
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 2..9)
        Cursor c;
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read
        const int half = (warp - 2) >> 2;       // which 128 of the 256 accumulator columns this warp drains
        float *stg = stg_all + (warp - 2) * (32 * 33);
        const int row = q * 32 + lane;
        const float alpha = P.epi.alpha;
        const int flags = P.epi.flags;
        int it = 0;
        for (int tile = first_tile; tile < P.total_tiles; tile += tile_step, ++it) {
            c.seek(P, tile);
            const GemmProblem &g = c.cur;
            const int lt = tile - g.tile0;
            const int mt = lt / g.tiles_n, nt = lt - mt * g.tiles_n;
            const int as = it & 1;
            const int m = mt * TILE_M + rank * BM + row;
            const bool row_ok = m < g.M;
            const float bias_m = (P.epi.bias != nullptr && (flags & smz::GEMM_BIAS_M) && !(flags & (smz::GEMM_SCALE_M | smz::GEMM_SCALE_STATS)) && row_ok) ? __ldg(P.epi.bias + m) : 0.f;
            const bool out_f32 = flags & smz::GEMM_OUT_F32;
            const bool res_f32 = flags & smz::GEMM_RES_F32;
            const bool c_vec = ((g.c_off | (int64_t)g.ldc) & 7) == 0 && (reinterpret_cast<uintptr_t>(P.epi.C) & 15) == 0;
            const int64_t res_off = (flags & smz::GEMM_RES_AT_C) ? g.c_off : g.r_off;
            const int res_ld = (flags & smz::GEMM_RES_AT_C) ? g.ldc : g.ldr;
            const bool r_vec = ((res_off | (int64_t)res_ld) & 7) == 0 && (reinterpret_cast<uintptr_t>(P.epi.residual) & 15) == 0;
            // The residual of the NEXT 32-column chunk is fetched while the current one is processed (and the
            // first one while the MMAs of this tile are still running): its ~1 us L2/HBM latency would otherwise
            // serialise 8 times per tile and make the epilogue, not the tensor pipe, the pace of the kernel.
            const char *res_row = P.epi.residual == nullptr ? nullptr
                : reinterpret_cast<const char *>(P.epi.residual) + (res_off + (int64_t)m * res_ld) * (res_f32 ? 4 : 2);
            auto res_vec_ok = [&](int n0) { return res_row != nullptr && row_ok && r_vec && n0 + 32 <= g.N; };
            auto res_fetch = [&](int n0, uint4 (&buf)[8]) {
                if (!res_vec_ok(n0)) return;
                const uint4 *src = reinterpret_cast<const uint4 *>(res_row + (int64_t)n0 * (res_f32 ? 4 : 2));
#pragma unroll
                for (int j = 0; j < 8; j++)
                    if (res_f32 || j < 4) buf[j] = src[j];
            };
            uint4 rcur[8], rnext[8];
            float st1 = 0.f, st2 = 0.f, st3 = 0.f;      // GEMM_ROWSTATS accumulators of this thread's row
            constexpr bool do_exp = EPI == EPI_EXP;
            const int n_store = do_exp ? ((g.N + 63) & ~63) : g.N;   // GEMM_EXP also writes the zero padding columns
            float amax = 0.f;
            if (EPI == EPI_PLAIN && res_row != nullptr && row_ok) {     // pull this thread's residual segment towards L2 while the MMAs run
                const char *pf = res_row + (int64_t)(nt * BN + half * (BN / 2)) * (res_f32 ? 4 : 2);
                const int bytes = (BN / 2) * (res_f32 ? 4 : 2);
                for (int b = 0; b < bytes; b += 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(pf + b));
            }
            res_fetch(nt * BN + half * (BN / 2), rcur);
            // per-row constants, fetched while the MMAs of this tile are still running
            float row_scale = 1.f, ln_mean = 0.f, ln_rstd = 1.f;
            if (EPI == EPI_PLAIN && row_ok && (flags & smz::GEMM_SCALE_M)) row_scale = __ldg(P.epi.bias + g.r_off + m);
            if (EPI == EPI_PLAIN && row_ok && (flags & smz::GEMM_SCALE_STATS)) {
                const int ns = P.epi.scale_slots > 0 ? P.epi.scale_slots : P.epi.stat_slots;
                const float *sp = P.epi.bias + (g.r_off + m) * ns * 3;
                float ssum = 0.f;
                for (int k = 0; k < ns; k++) ssum += __ldg(sp + 3 * k);
                row_scale = 1.f / ssum;       // a fully masked row: 1/0 = inf -> NaN scores, as torch's softmax of all -inf
            }
            if (EPI == EPI_HEAD && row_ok && (flags & smz::GEMM_LN_FOLD)) {
                const float *sp = P.epi.ln_stats + (g.r_off + m) * P.epi.ln_slots * 3;
                float s1 = 0.f, s2 = 0.f;
                for (int k = 0; k < P.epi.ln_slots; k++) { s1 += __ldg(sp + 3 * k); s2 += __ldg(sp + 3 * k + 1); }
                const float inv_w = 1.f / (float)P.epi.ln_width;
                ln_mean = s1 * inv_w;
                ln_rstd = rsqrtf(fmaxf(s2 * inv_w - ln_mean * ln_mean, 0.f) + P.epi.ln_eps);
            }
            mbar_wait(&tfull[as], ((uint32_t)it >> 1) & 1u);
            tc_fence_after();
            for (int c0 = half * (BN / 2); c0 < (half + 1) * (BN / 2); c0 += 32) {
                const int n0 = nt * BN + c0;
                if (n0 >= n_store) break;   // warp-uniform
                uint32_t v[32];
                uint32_t lo_pk[SPLIT_OUT ? 16 : 1];     // EPI_SPLIT: the lo plane of this thread's 32 outputs, packed
                __syncwarp();           // tcgen05.ld is .sync.aligned: reconverge after the row mask
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + c0), v);
                if (c0 + 32 < (half + 1) * (BN / 2)) res_fetch(n0 + 32, rnext);
                tmem_ld_wait();
                if (row_ok) {
                float x[32];
#pragma unroll
                for (int j = 0; j < 32; j++) x[j] = alpha * __uint_as_float(v[j]);
                const bool full32 = n0 + 32 <= n_store;
                if constexpr (do_exp) {
                    const int ap = P.epi.aperture, ig = P.epi.ignore_self;
                    if (ap < 0 && !ig && n0 + 32 <= g.N) {      // warp-uniform common case: no masks, no column tail
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            amax = fmaxf(amax, fabsf(x[j]));
                            x[j] = __expf(x[j]);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const int col = n0 + j;
                            float e = x[j];
                            bool live = col < g.N;
                            if (ig && col == m) live = false;                                   // vasnet.py:121-122
                            if (ap >= 0) {                                                      // vasnet.py:124-127
                                int d = m - col; d = d < 0 ? -d : d;
                                if (d > ap || e * e == 0.f) live = false;
                            }
                            if (live) amax = fmaxf(amax, fabsf(e));
                            x[j] = live ? __expf(e) : 0.f;
                        }
                    }
                }
                if (EPI == EPI_PLAIN && (flags & (smz::GEMM_SCALE_M | smz::GEMM_SCALE_STATS))) {
#pragma unroll
                    for (int j = 0; j < 32; j++) x[j] *= row_scale;
                }
                if (EPI == EPI_HEAD && (flags & smz::GEMM_LN_FOLD)) {       // N is a multiple of 32 in this mode
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 cc = ld_f4(P.epi.ln_c + n0 + j);
                        x[j] = ln_rstd * fmaf(-ln_mean, cc.x, x[j]); x[j + 1] = ln_rstd * fmaf(-ln_mean, cc.y, x[j + 1]);
                        x[j + 2] = ln_rstd * fmaf(-ln_mean, cc.z, x[j + 2]); x[j + 3] = ln_rstd * fmaf(-ln_mean, cc.w, x[j + 3]);
                    }
                }
                if (EPI != EPI_EXP && P.epi.bias != nullptr && !(flags & (smz::GEMM_SCALE_M | smz::GEMM_SCALE_STATS))) {
                    if (flags & smz::GEMM_BIAS_M) {
#pragma unroll
                        for (int j = 0; j < 32; j++) x[j] += bias_m;
                    } else if (full32) {
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 b = ld_f4(P.epi.bias + n0 + j);
                            x[j] += b.x; x[j + 1] += b.y; x[j + 2] += b.z; x[j + 3] += b.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++) if (n0 + j < g.N) x[j] += __ldg(P.epi.bias + n0 + j);
                    }
                }
                if (EPI == EPI_PLAIN && res_row != nullptr) {
                    if (res_vec_ok(n0)) {
                        if (res_f32) {
#pragma unroll
                            for (int j = 0; j < 8; j++) {
                                x[4 * j] += __uint_as_float(rcur[j].x); x[4 * j + 1] += __uint_as_float(rcur[j].y);
                                x[4 * j + 2] += __uint_as_float(rcur[j].z); x[4 * j + 3] += __uint_as_float(rcur[j].w);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                const uint32_t w4[4] = {rcur[j].x, rcur[j].y, rcur[j].z, rcur[j].w};
#pragma unroll
                                for (int t = 0; t < 4; t++) {
                                    x[8 * j + 2 * t] += __uint_as_float(w4[t] << 16);
                                    x[8 * j + 2 * t + 1] += __uint_as_float(w4[t] & 0xffff0000u);
                                }
                            }
                        }
                    } else if (res_f32) {
                        const float *r = reinterpret_cast<const float *>(res_row) + n0;
#pragma unroll
                        for (int j = 0; j < 32; j++) if (n0 + j < g.N) x[j] += r[j];
                    } else {
                        const __nv_bfloat16 *r = reinterpret_cast<const __nv_bfloat16 *>(res_row) + n0;
#pragma unroll
                        for (int j = 0; j < 32; j++) if (n0 + j < g.N) x[j] += __bfloat162float(r[j]);
                    }
                }
                if (EPI != EPI_EXP && (flags & smz::GEMM_RELU)) {    // NaN passes, as torch.relu (fmaxf would turn it into 0)
#pragma unroll
                    for (int j = 0; j < 32; j++) x[j] = x[j] < 0.f ? 0.f : x[j];
                }
                const bool f16 = EPI == EPI_PLAIN && (flags & smz::GEMM_OUT_F16) && n0 >= P.epi.f16_col0;     // warp-uniform
                if (f16 && !(flags & smz::GEMM_LN_STATS)) {     // range check (with GEMM_LN_STATS the sum of squares does it)
#pragma unroll
                    for (int j = 0; j < 32; j += 2) amax = fmaxf(amax, fmaxf(fabsf(x[j]), fabsf(x[j + 1])));
                }
                if (EPI == EPI_PLAIN && (flags & smz::GEMM_LN_STATS)) {      // N is a multiple of 32 in this mode
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        st1 += (x[j] + x[j + 1]) + (x[j + 2] + x[j + 3]);
                        st2 = fmaf(x[j], x[j], st2); st2 = fmaf(x[j + 1], x[j + 1], st2);
                        st2 = fmaf(x[j + 2], x[j + 2], st2); st2 = fmaf(x[j + 3], x[j + 3], st2);
                    }
                }
                if constexpr (EPI == EPI_HEAD) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 sw = ld_f4(P.epi.stat_w + n0 + j);      // N is a multiple of 32 in this mode
                        st1 += (x[j] + x[j + 1]) + (x[j + 2] + x[j + 3]);
                        st2 = fmaf(x[j], x[j], st2); st2 = fmaf(x[j + 1], x[j + 1], st2);
                        st2 = fmaf(x[j + 2], x[j + 2], st2); st2 = fmaf(x[j + 3], x[j + 3], st2);
                        st3 = fmaf(x[j], sw.x, st3); st3 = fmaf(x[j + 1], sw.y, st3);
                        st3 = fmaf(x[j + 2], sw.z, st3); st3 = fmaf(x[j + 3], sw.w, st3);
                    }
                }
                if constexpr (EPI == EPI_EXP) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) st1 += (x[j] + x[j + 1]) + (x[j + 2] + x[j + 3]);   // dead columns hold 0
                }
                if constexpr (EPI != EPI_HEAD) {
                const int64_t co = g.c_off + (int64_t)m * g.ldc + n0;
                if (out_f32) {
                    float *dst = reinterpret_cast<float *>(P.epi.C) + co;
                    if (full32) {
                        // float32 tiles leave through the transposition pad (below): a thread owns a ROW of the
                        // accumulator, so direct 16-byte stores would touch 32 different 128-byte lines per
                        // instruction and make the store unit, not the tensor pipe, the pace of the kernel
#pragma unroll
                        for (int j = 0; j < 32; j++) stg[lane * 33 + j] = x[j];
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++) if (n0 + j < g.N) dst[j] = x[j];
                    }
                } else {
                    __nv_bfloat16 *dst = reinterpret_cast<__nv_bfloat16 *>(P.epi.C) + co;
                    if (full32 && c_vec) {
                        // 16-bit tiles leave through the pad as well (below): 8 rows x 64 contiguous bytes per store
                        // instruction instead of 32 rows x 16 bytes (half-used sectors on 32 different lines)
                        uint4 *pad = reinterpret_cast<uint4 *>(reinterpret_cast<uint32_t *>(stg) + lane * 20);
#pragma unroll
                        for (int j = 0; j < 32; j += 8)
                            pad[j >> 3] = f16 ?
                                make_uint4(pack_f16x2(x[j], x[j + 1]), pack_f16x2(x[j + 2], x[j + 3]),
                                           pack_f16x2(x[j + 4], x[j + 5]), pack_f16x2(x[j + 6], x[j + 7])) :
                                make_uint4(pack_bf16x2(x[j], x[j + 1]), pack_bf16x2(x[j + 2], x[j + 3]),
                                           pack_bf16x2(x[j + 4], x[j + 5]), pack_bf16x2(x[j + 6], x[j + 7]));
                        if constexpr (SPLIT_OUT) {
#pragma unroll
                            for (int j = 0; j < 32; j += 2) {
                                const uint32_t hi = pack_bf16x2(x[j], x[j + 1]);
                                lo_pk[j >> 1] = pack_bf16x2(x[j] - __uint_as_float(hi << 16), x[j + 1] - __uint_as_float(hi & 0xffff0000u));
                            }
                        }
                    } else if (f16) {
#pragma unroll
                        for (int j = 0; j < 32; j++) if (n0 + j < g.N) reinterpret_cast<__half *>(dst)[j] = __float2half_rn(x[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++) if (n0 + j < g.N) {
                            const __nv_bfloat16 hi = __float2bfloat16_rn(x[j]);
                            dst[j] = hi;
                            if (SPLIT_OUT) dst[P.epi.c_lo + j] = __float2bfloat16_rn(x[j] - __bfloat162float(hi));
                        }
                    }
                }
                }   // !GEMM_NO_STORE
                }   // row_ok
                if (EPI == EPI_PLAIN && out_f32 && n0 + 32 <= g.N) {   // warp-uniform: coalesced 128-byte row stores
                    __syncwarp();
                    const int m_base = m - lane;       // first row of this warp's 32 accumulator rows
                    float *base = reinterpret_cast<float *>(P.epi.C) + g.c_off + n0 + lane;
#pragma unroll 8
                    for (int r = 0; r < 32; r++)
                        if (m_base + r < g.M) base[(int64_t)(m_base + r) * g.ldc] = stg[r * 33 + lane];
                    __syncwarp();
                }
                if (EPI != EPI_HEAD && !out_f32 && n0 + 32 <= n_store && c_vec) {   // warp-uniform: 16-bit rows, 64 contiguous bytes each
                    __syncwarp();
                    const int m_base = m - lane;
                    const int sub = lane >> 2, part = lane & 3;
                    __nv_bfloat16 *base = reinterpret_cast<__nv_bfloat16 *>(P.epi.C) + g.c_off + n0 + part * 8;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int r = 8 * i + sub;
                        const uint4 w4 = *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint32_t *>(stg) + r * 20 + part * 4);
                        if (m_base + r < g.M) *reinterpret_cast<uint4 *>(base + (int64_t)(m_base + r) * g.ldc) = w4;
                    }
                    __syncwarp();
                    if constexpr (SPLIT_OUT) {      // the lo plane leaves the same way
                        if (row_ok) {
                            uint4 *pad = reinterpret_cast<uint4 *>(reinterpret_cast<uint32_t *>(stg) + lane * 20);
#pragma unroll
                            for (int j = 0; j < 4; j++) pad[j] = make_uint4(lo_pk[4 * j], lo_pk[4 * j + 1], lo_pk[4 * j + 2], lo_pk[4 * j + 3]);
                        }
                        __syncwarp();
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const int r = 8 * i + sub;
                            const uint4 w4 = *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint32_t *>(stg) + r * 20 + part * 4);
                            if (m_base + r < g.M) *reinterpret_cast<uint4 *>(base + P.epi.c_lo + (int64_t)(m_base + r) * g.ldc) = w4;
                        }
                        __syncwarp();
                    }
                }
#pragma unroll
                for (int j = 0; j < 8; j++) rcur[j] = rnext[j];
            }
            if ((EPI != EPI_PLAIN || (flags & smz::GEMM_LN_STATS)) && row_ok) {
                const int slots = P.epi.stat_slots > 0 ? P.epi.stat_slots : 2 * g.tiles_n;
                float *so = P.epi.stat_out + ((g.r_off + m) * slots + (nt * 2 + half)) * 3;
                so[0] = st1; so[1] = st2; so[2] = st3;
            }
            if (do_exp && P.epi.guard != nullptr && !(amax <= 80.f)) atomicOr(P.epi.guard, P.epi.guard_bit);   // also catches NaN
            // float16 range: sum x^2 < 60000^2 bounds every |x| of the slot (conservative: tripping it costs a repeat on the
            // exact path, never a wrong result)
            if (EPI == EPI_PLAIN && (flags & smz::GEMM_OUT_F16) && P.epi.guard != nullptr && row_ok &&
                !(((flags & smz::GEMM_LN_STATS) ? st2 : amax * amax) <= 3.6e9f))
                atomicOr(P.epi.guard, P.epi.guard_bit);
            tc_fence_before();
            if (PAIR) mbar_arrive_remote(&tempty[as], 0); else mbar_arrive(&tempty[as]);
        }
    }
    __syncwarp();          // the single-lane roles rejoin their warps before the block / cluster barrier
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if (PAIR) tmem_dealloc_pair<TMEM_COLS>(tmem_base); else tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

// ---- host ---------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (fn == nullptr) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

// K-major operand: box = 64 k-columns x box_rows rows.  MN-major operand: box = 64 m/n-columns x 64 k-rows.
int make_map(CUtensorMap *m, const void *base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
    PFN_cuTensorMapEncodeTiled_v12000 enc = encode_fn();
    if (enc == nullptr) return smz::fail(SMZ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld & 7) != 0 || rows <= 0 || cols <= 0)
        return smz::fail(SMZ_ERR_ARG, "gemm operand must be 16-byte aligned with a leading dimension multiple of 8 "
                         "(base %p, ld %lld, %lld x %lld)", base, (long long)ld, (long long)rows, (long long)cols);
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return smz::fail(SMZ_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return SMZ_OK;
}

}  // namespace

namespace smz {

int make_bf16_map(CUtensorMap *m, const void *base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
    return make_map(m, base, rows, cols, ld, box_rows);
}

int gemm_bf16_tn(const void *A, int64_t a_rows, int64_t a_cols, int64_t lda, const void *B, int64_t b_rows,
                 int64_t b_cols, int64_t ldb, const GemmProblem *d_probs, int n_probs, int total_tiles,
                 const GemmProblem &single, const GemmEpilogue &epi, cudaStream_t st) {
    return gemm_bf16(false, false, A, a_rows, a_cols, lda, B, b_rows, b_cols, ldb, d_probs, n_probs, total_tiles, single,
                     epi, st);
}

bool gemm_pair_mode() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("SMZ_GEMM_PAIR"); v = (e != nullptr && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

int gemm_tile_m() { return gemm_pair_mode() ? 2 * BM : BM; }

int gemm_tiles(int M, int N) { return ((M + gemm_tile_m() - 1) / gemm_tile_m()) * ((N + GEMM_BN - 1) / GEMM_BN); }

template <bool PAIR>
static int launch_variant(bool a_mn, bool b_mn, const CUtensorMap &ma, const CUtensorMap &mb, const CUtensorMap &ma_lo,
                          const CUtensorMap &mb_lo, const Params &P, int total_tiles, cudaStream_t st) {
    typedef void (*kern_t)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const Params);
    const int f = P.epi.flags;
    const int epi = (f & GEMM_EXP) ? EPI_EXP : (f & GEMM_ROWSTATS) ? EPI_HEAD
                    : (P.epi.c_lo != 0 && !(f & GEMM_OUT_F32)) ? EPI_SPLIT : EPI_PLAIN;
    kern_t kern;
    if (epi == EPI_SPLIT) {
        if (f & (GEMM_OUT_F16 | GEMM_LN_STATS)) return fail(SMZ_ERR_UNSUPPORTED, "gemm: hi + lo output planes are bf16, without row statistics");
        if ((P.epi.c_lo & 7) != 0) return fail(SMZ_ERR_ARG, "gemm: c_lo must be a multiple of 8 elements");
        kern = a_mn ? (b_mn ? (kern_t)gemm_kernel<true, true, PAIR, EPI_SPLIT> : (kern_t)gemm_kernel<true, false, PAIR, EPI_SPLIT>)
                    : (b_mn ? (kern_t)gemm_kernel<false, true, PAIR, EPI_SPLIT> : (kern_t)gemm_kernel<false, false, PAIR, EPI_SPLIT>);
    } else if (epi != EPI_PLAIN) {
        if (a_mn || b_mn) return fail(SMZ_ERR_UNSUPPORTED, "gemm: the fused head / exp epilogues exist for K-major operands only");
        if (epi == EPI_HEAD && (!(f & GEMM_NO_STORE) || P.epi.stat_w == nullptr || P.epi.stat_out == nullptr))
            return fail(SMZ_ERR_ARG, "gemm: GEMM_ROWSTATS needs GEMM_NO_STORE, stat_w and stat_out");
        if (epi == EPI_EXP && (!(f & GEMM_ROWSTATS) || (f & GEMM_OUT_F32) || P.epi.stat_out == nullptr))
            return fail(SMZ_ERR_ARG, "gemm: GEMM_EXP writes bf16 and needs GEMM_ROWSTATS + stat_out");
        kern = epi == EPI_HEAD ? (kern_t)gemm_kernel<false, false, PAIR, EPI_HEAD> : (kern_t)gemm_kernel<false, false, PAIR, EPI_EXP>;
    } else {
        kern = a_mn ? (b_mn ? (kern_t)gemm_kernel<true, true, PAIR, EPI_PLAIN> : (kern_t)gemm_kernel<true, false, PAIR, EPI_PLAIN>)
                    : (b_mn ? (kern_t)gemm_kernel<false, true, PAIR, EPI_PLAIN> : (kern_t)gemm_kernel<false, false, PAIR, EPI_PLAIN>);
    }
    const int variant = epi == EPI_SPLIT ? 6 + (a_mn ? 2 : 0) + (b_mn ? 1 : 0) : epi != EPI_PLAIN ? 3 + epi : (a_mn ? 2 : 0) + (b_mn ? 1 : 0);
    static bool attr_set[64][10] = {{false}};
    int dev = 0;
    SMZ_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_set[dev][variant]) {
        SMZ_CUDA_CHECK(cudaFuncSetAttribute((const void *)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<PAIR>::SMEM_BYTES));
        attr_set[dev][variant] = true;
    }
    const int sms = sm_count();
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg<PAIR>::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int n_attr = 0;
    if (PAIR) {
        const int pairs = total_tiles < sms / 2 ? total_tiles : sms / 2;
        cfg.gridDim = dim3(2 * pairs);
        attr[n_attr].id = cudaLaunchAttributeClusterDimension;
        attr[n_attr].val.clusterDim.x = 2; attr[n_attr].val.clusterDim.y = 1; attr[n_attr].val.clusterDim.z = 1;
        ++n_attr;
    } else {
        cfg.gridDim = dim3(total_tiles < sms ? total_tiles : sms);
    }
    // Programmatic dependent launch (smz_common.cuh): the prologue overlaps the previous kernel's tail.  Only for grids
    // that leave SMs free (the few-tile GEMMs of a batch-1 training step: +5 % on the replayed step) — a full persistent
    // grid gains nothing, and in the two-lane inference sweep its early-resident CTAs sit on SMs the OTHER lane's kernel
    // could use (measured: -1.7 % on the sweep).
    if (pdl_enabled() && total_tiles < (PAIR ? sms / 2 : sms)) {
        attr[n_attr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n_attr].val.programmaticStreamSerializationAllowed = 1;
        ++n_attr;
    }
    cfg.attrs = attr; cfg.numAttrs = n_attr;
    SMZ_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, ma, mb, ma_lo, mb_lo, P));
    return SMZ_OK;
}

int gemm_bf16(bool a_mn, bool b_mn, const void *A, int64_t a_rows, int64_t a_cols, int64_t lda, const void *B,
              int64_t b_rows, int64_t b_cols, int64_t ldb, const GemmProblem *d_probs, int n_probs, int total_tiles,
              const GemmProblem &single, const GemmEpilogue &epi, cudaStream_t st) {
    if (total_tiles <= 0) return SMZ_OK;
    SMZ_REQUIRE(A && B && epi.C, "gemm: NULL operand");
    SMZ_REQUIRE(d_probs != nullptr || n_probs == 1, "gemm: a batch needs a device problem array");
    alignas(64) CUtensorMap ma, mb;
    const bool pair = gemm_pair_mode();
    int rc = make_map(&ma, A, a_rows, a_cols, lda, a_mn ? 64 : BM);
    if (rc != SMZ_OK) return rc;
    rc = make_map(&mb, B, b_rows, b_cols, ldb, b_mn ? 64 : (pair ? BN / 2 : BN));
    if (rc != SMZ_OK) return rc;
    alignas(64) CUtensorMap ma_lo = ma, mb_lo = mb;       // the lo planes of split-bf16 operands: same shape, other base
    if (epi.a_lo != 0) {
        rc = make_map(&ma_lo, reinterpret_cast<const uint16_t *>(A) + epi.a_lo, a_rows, a_cols, lda, a_mn ? 64 : BM);
        if (rc != SMZ_OK) return rc;
    }
    if (epi.b_lo != 0) {
        rc = make_map(&mb_lo, reinterpret_cast<const uint16_t *>(B) + epi.b_lo, b_rows, b_cols, ldb, b_mn ? 64 : (pair ? BN / 2 : BN));
        if (rc != SMZ_OK) return rc;
    }
    Params P;
    P.probs = d_probs;
    P.single = single;
    P.n_probs = n_probs;
    P.total_tiles = total_tiles;
    P.epi = epi;
    return pair ? launch_variant<true>(a_mn, b_mn, ma, mb, ma_lo, mb_lo, P, total_tiles, st)
                : launch_variant<false>(a_mn, b_mn, ma, mb, ma_lo, mb_lo, P, total_tiles, st);
}

}  // namespace smz

// C[M,N] = epilogue(alpha * A[M,K] * B[N,K]^T): the stand-alone entry point (tests, host-side reuse).
extern "C" int smz_gemm_bf16_tn(const void *A, int64_t lda, const void *B, int64_t ldb, void *C, int64_t ldc, int M,
                                int N, int K, float alpha, const float *bias, const void *residual, int64_t ldr,
                                int flags, void *stream) {
    if (M == 0 || N == 0) return SMZ_OK;
    SMZ_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: bad shape %d x %d x %d", M, N, K);
    SMZ_REQUIRE(ldc >= N && lda >= K && ldb >= K, "gemm: leading dimension smaller than the row length");
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    smz::GemmProblem g = {};
    g.M = M; g.N = N; g.K = K;
    g.ldc = (int32_t)ldc; g.ldr = (int32_t)ldr;
    g.tiles_n = (N + smz::GEMM_BN - 1) / smz::GEMM_BN;
    smz::GemmEpilogue e = {C, bias, residual, alpha, flags};
    return smz::gemm_bf16_tn(A, M, K, lda, B, N, K, ldb, nullptr, 1, smz::gemm_tiles(M, N), g, e, (cudaStream_t)stream);
}

// General form: op(A) / op(B) may be stored MN-major (k rows, m resp. n contiguous):
//   a_mn == 0: A is [M, K] (lda >= K);  a_mn != 0: A is [K, M] (lda >= M).  Likewise B with N.
extern "C" int smz_gemm_bf16(int a_mn, int b_mn, const void *A, int64_t lda, const void *B, int64_t ldb, void *C,
                             int64_t ldc, int M, int N, int K, float alpha, const float *bias, const void *residual,
                             int64_t ldr, int flags, void *stream) {
    if (M == 0 || N == 0) return SMZ_OK;
    SMZ_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: bad shape %d x %d x %d", M, N, K);
    SMZ_REQUIRE(ldc >= N && lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "gemm: leading dimension smaller than the row length");
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    smz::GemmProblem g = {};
    g.M = M; g.N = N; g.K = K;
    g.ldc = (int32_t)ldc; g.ldr = (int32_t)ldr;
    g.tiles_n = (N + smz::GEMM_BN - 1) / smz::GEMM_BN;
    smz::GemmEpilogue e = {C, bias, residual, alpha, flags};
    return smz::gemm_bf16(a_mn != 0, b_mn != 0, A, a_mn ? K : M, a_mn ? M : K, lda, B, b_mn ? K : N, b_mn ? N : K, ldb,
                          nullptr, 1, smz::gemm_tiles(M, N), g, e, (cudaStream_t)stream);
}

// Split-bf16 form of smz_gemm_bf16 (float32-accurate products): every operand is a pair of bf16 arrays of the same
// layout, hi = bf16(x) and lo = bf16(x - hi) (smz_split_bf16_multi makes them); A_lo / B_lo may be NULL (that operand
// is exact in bf16).  C_lo != NULL with a bf16 output: the result is written as hi + lo planes too.
extern "C" int smz_gemm_bf16_split(int a_mn, int b_mn, const void *A, const void *A_lo, int64_t lda, const void *B,
                                   const void *B_lo, int64_t ldb, void *C, void *C_lo, int64_t ldc, int M, int N, int K,
                                   float alpha, const float *bias, const void *residual, int64_t ldr, int flags,
                                   void *stream) {
    if (M == 0 || N == 0) return SMZ_OK;
    SMZ_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: bad shape %d x %d x %d", M, N, K);
    SMZ_REQUIRE(ldc >= N && lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "gemm: leading dimension smaller than the row length");
    SMZ_REQUIRE(C_lo == nullptr || !(flags & smz::GEMM_OUT_F32), "gemm: a float32 output has no lo plane");
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    smz::GemmProblem g = {};
    g.M = M; g.N = N; g.K = K;
    g.ldc = (int32_t)ldc; g.ldr = (int32_t)ldr;
    g.tiles_n = (N + smz::GEMM_BN - 1) / smz::GEMM_BN;
    smz::GemmEpilogue e = {C, bias, residual, alpha, flags};
    auto delta = [](const void *lo, const void *hi) -> int64_t {
        return lo == nullptr ? 0 : (reinterpret_cast<const char *>(lo) - reinterpret_cast<const char *>(hi)) / 2;
    };
    e.a_lo = delta(A_lo, A); e.b_lo = delta(B_lo, B); e.c_lo = delta(C_lo, C);
    SMZ_REQUIRE((A_lo == nullptr || e.a_lo != 0) && (B_lo == nullptr || e.b_lo != 0) && (C_lo == nullptr || e.c_lo != 0),
                "gemm: a lo plane must be a different array than its hi plane");
    return smz::gemm_bf16(a_mn != 0, b_mn != 0, A, a_mn ? K : M, a_mn ? M : K, lda, B, b_mn ? K : N, b_mn ? N : K, ldb,
                          nullptr, 1, smz::gemm_tiles(M, N), g, e, (cudaStream_t)stream);
}
