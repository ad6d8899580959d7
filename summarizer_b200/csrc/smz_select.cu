// Shot selection kernels (sm_100a) + their C ABI:  utils/eval.py:74-123 generate_summary and
// utils/knapsack.py:5-23 knapsack_ortools (OR-tools 7.5 KnapsackDynamicProgrammingSolver).
//
// Fast path (capacity+1 <= 27*256 cells), three kernels per batch:
//   pool_kernel     grid (segment tile, video), 8 lanes per segment: float32 segment means in
//                   numpy's pairwise summation order, values = trunc(double(mean) * 1000).
//   dp_kernel<K>    persistent CTAs (256 threads, K cells per thread held in registers), one
//                   video at a time: forward DP with ONE __syncthreads per item; the shared row
//                   only serves the shifted read dp[c-w] (front pad of -2^30 removes the c>=w
//                   test); improvement bits are accumulated per cell in registers (32 items per
//                   word) and flushed coalesced to an L2-resident work buffer; warp 0 then walks
//                   the OR-tools extraction loop (one L2 round trip per picked item).
//   summary_kernel  one CTA per video: prefix of nfps -> float summary vector, bit mask, popcount.
//   dp16_kernel<KW,MK>  the same DP on 16-bit cells, two per 32-bit shared-memory word (cells c and c + H share
//                   word c, so a shift by any weight is ONE aligned LDS per two cells), DPX VIADDMNMX.U16x2 for
//                   max(cand + p, val) on both halves: half the shared-memory bytes and 3 instead of 5
//                   instructions per cell.  Exact: it only runs while every row value provably fits 16 bits and
//                   hands the video to dp_kernel<K> (through a fallback list) otherwise.
// Generic path: select_generic_kernel (monolithic, rows of any size up to shared memory).
#include "smz_common.cuh"
#include "smz_fscore_dev.cuh"

#include <limits.h>
#include <stdlib.h>

#include <mutex>

namespace {

using namespace smzdev;

constexpr int SELECT_THREADS = 512;   // generic kernel
constexpr int DP_THREADS = 256;       // register-DP kernel
constexpr int POOL_THREADS = 256;     // 32 segments per CTA, 8 lanes each
constexpr int SUMMARY_THREADS = 256;
constexpr int kDpNeg = -(1 << 29) - 1;   // front-pad value of the DP rows: pad + value <= -1 never improves a cell (rows are >= 0)

// |value| limit of the int32 DP: n * limit <= 2^29, so that the take test val - cand - value (dp_kernel) stays
// inside int32 even against the pad:  2^29 + (2^29 + 1) + 2^29 < 2^31.  Values beyond it are clipped and flagged.
__host__ __device__ inline int value_limit(int n) { return (1 << 29) / (n > 0 ? n : 1); }

// ------------------------------------------------------------------------------------------
// pool_kernel: utils/eval.py:87-94 (segment means) + utils/knapsack.py:11-15 (quantisation)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(POOL_THREADS)
pool_kernel(const smz_video_desc *__restrict__ desc, int v0, const float *__restrict__ scores,
            const int32_t *__restrict__ picks, const int32_t *__restrict__ cps,
            float *__restrict__ out_mean, int32_t *__restrict__ out_values, int32_t *__restrict__ status) {
    const int v = v0 + blockIdx.y;
    const smz_video_desc d = desc[v];
    const int n = d.n_segs;
    const int s = blockIdx.x * (POOL_THREADS / 8) + (threadIdx.x >> 3);
    if (blockIdx.x * (POOL_THREADS / 8) >= n) return;
    const int lane = threadIdx.x & 31;
    const int gl = lane & 7, lane0 = lane & ~7;
    const unsigned gmask = 0xffu << lane0;
    FrameCursor cur;
    cur.init(scores + d.score_off, picks + d.picks_off, d.n_scores, d.n_picks, d.n_frames);
    if (blockIdx.x == 0 && threadIdx.x == 0 && cur.n_bound - 1 > d.n_scores + 1)
        atomicOr(status + v, SMZ_STATUS_INTERVALS);
    if (s >= n) return;                                   // uniform within an 8-lane group
    const int start = __ldg(cps + 2 * (d.seg_off + s));
    int end = __ldg(cps + 2 * (d.seg_off + s) + 1) + 1;
    end = min(end, d.n_frames);
    const int len = end - start;
    cur.seek(start + (len >= 8 ? gl : 0));
    const float sum = pw_sum_group(cur, start, len, gl, gmask, lane0);
    if (gl == 0) {
        const float mean = __fdiv_rn(sum, (float)len);
        long long val = __double2ll_rz(__dmul_rn((double)mean, 1000.0));
        const int vlim = value_limit(n);
        if (val > vlim || val < -vlim) { atomicOr(status + v, SMZ_STATUS_VALUE_RANGE); val = val > 0 ? vlim : -vlim; }
        if (out_mean) out_mean[d.seg_off + s] = mean;
        out_values[d.seg_off + s] = (int)val;
    }
}

// Same result, one CTA per video: the upsample (utils/eval.py:15-35) is first expanded into shared memory as one
// 16-bit score index per frame, so that the pairwise sums read shared memory + an L1-resident score instead of
// walking the picks cursor through global memory — ~20x fewer instructions.  2 bytes per frame keeps three CTAs
// per SM at 30 000 frames.  Used whenever the frames fit and there are fewer than 65 535 intervals.
constexpr int POOL_SMEM_THREADS = 512;

__global__ void __launch_bounds__(POOL_SMEM_THREADS)
pool_smem_kernel(const smz_video_desc *__restrict__ desc, int v0, const float *__restrict__ scores,
                 const int32_t *__restrict__ picks, const int32_t *__restrict__ cps,
                 float *__restrict__ out_mean, int32_t *__restrict__ out_values, int32_t *__restrict__ status) {
    extern __shared__ unsigned short frames[];
    constexpr int NT = POOL_SMEM_THREADS;
    const int v = v0 + blockIdx.x, tid = threadIdx.x;
    const smz_video_desc d = desc[v];
    const int n = d.n_segs, n_frames = d.n_frames, n_picks = d.n_picks;
    const int32_t *pk = picks + d.picks_off;
    const float *sc = scores + d.score_off;
    const int n_bound = n_picks + ((n_picks > 0 && __ldg(pk + n_picks - 1) != n_frames) ? 1 : 0);
    if (tid == 0 && n_bound - 1 > d.n_scores + 1) atomicOr(status + v, SMZ_STATUS_INTERVALS);
    {   // before picks[0], after the last boundary, zero-filled intervals: index 0xffff
        uint32_t *w = reinterpret_cast<uint32_t *>(frames);
        for (int f = tid; f < (n_frames + 1) / 2; f += NT) w[f] = 0xffffffffu;
    }
    __syncthreads();
    for (int i = tid; i + 1 < n_bound && i < d.n_scores && i < 0xffff; i += NT) {  // interval i = [bound(i), bound(i+1))
        const int lo = max(__ldg(pk + i), 0);
        const int hi = min(i + 1 < n_picks ? __ldg(pk + i + 1) : n_frames, n_frames);
        for (int f = lo; f < hi; f++) frames[f] = (unsigned short)i;
    }
    __syncthreads();
    SmemFrames cur{frames, sc};
    const int lane = tid & 31, gl = lane & 7, lane0 = lane & ~7;
    const unsigned gmask = 0xffu << lane0;
    const int vlim = value_limit(n);
    for (int s = tid >> 3; s < n; s += NT / 8) {                    // uniform within an 8-lane group
        const int start = __ldg(cps + 2 * (d.seg_off + s));
        int end = __ldg(cps + 2 * (d.seg_off + s) + 1) + 1;
        end = min(end, n_frames);
        const int len = end - start;
        const float sum = pw_sum_group(cur, start, len, gl, gmask, lane0);
        if (gl == 0) {
            const float mean = __fdiv_rn(sum, (float)len);
            long long val = __double2ll_rz(__dmul_rn((double)mean, 1000.0));
            if (val > vlim || val < -vlim) { atomicOr(status + v, SMZ_STATUS_VALUE_RANGE); val = val > 0 ? vlim : -vlim; }
            if (out_mean) out_mean[d.seg_off + s] = mean;
            out_values[d.seg_off + s] = (int)val;
        }
    }
}

// Same result again for the common dataset layout — picks on a regular grid, picks[i] = i * stride
// (datasets/README.md:36-41: every 15th frame): the upsample needs no per-frame table at all, frame f belongs to
// interval min(f / stride, last), the division is one multiply-high by a per-video constant, and the scores sit in
// shared memory (4 bytes per STEP, 8 KB for 2 000 steps: many CTAs per SM).  ~6 instructions per frame instead of ~55.
// Videos whose picks are not such a grid take the cursor walk over global memory (pool_kernel's path) in the same CTA.
constexpr int POOL_REG_THREADS = 256;

struct RegularFrames {   // upsample of a regular pick grid: scores staged in shared memory (zero-filled past n_scores)
    const float *sc;
    uint32_t magic;      // floor(2^32 / stride) + 1: f / stride == umulhi(f, magic) for f < 65536, 2 <= stride < 65536
    int last;            // index of the last interval
    __device__ __forceinline__ float at(int f) const { return sc[min((int)__umulhi((uint32_t)f, magic), last)]; }
};

// One video, all POOL_REG_THREADS threads of the CTA; s_sc: max_intervals + 4 * d.n_segs words of shared memory (scores,
// then the segment lists).  Also called by the 16-bit knapsack kernel for the video it is about to solve (fused pooling).
__device__ void pool_regular_video(const smz_video_desc &d, int v, const float *__restrict__ scores,
                                   const int32_t *__restrict__ picks, const int32_t *__restrict__ cps, int max_intervals,
                                   float *s_sc, float *__restrict__ out_mean, int32_t *__restrict__ out_values,
                                   int32_t *__restrict__ status) {
    __shared__ int s_class[4];
    constexpr int NT = POOL_REG_THREADS;
    const int tid = threadIdx.x;
    const int n = d.n_segs, n_frames = d.n_frames, n_picks = d.n_picks;
    const int32_t *pk = picks + d.picks_off;
    const float *sc = scores + d.score_off;
    const int n_bound = n_picks + ((n_picks > 0 && __ldg(pk + n_picks - 1) != n_frames) ? 1 : 0);
    const int n_int = n_bound - 1;                                   // intervals [bound(i), bound(i+1))
    if (tid == 0 && n_int > d.n_scores + 1) atomicOr(status + v, SMZ_STATUS_INTERVALS);
    const int stride = n_picks >= 2 ? __ldg(pk + 1) - __ldg(pk) : n_frames;
    // stride 1 (a pick on every frame) takes the cursor walk: 2^32 / 1 does not fit the 32-bit multiplier
    int ok = n_picks >= 1 && n_int >= 1 && n_int <= max_intervals && stride >= 2 && stride < 65536 && n_frames < 65536;
    for (int i = tid; i < n_picks && ok; i += NT) ok = __ldg(pk + i) == i * stride;
    for (int i = tid; i < n_int && i < max_intervals; i += NT) s_sc[i] = i < d.n_scores ? __ldg(sc + i) : 0.f;
    ok = __syncthreads_and(ok);
    const int lane = tid & 31, gl = lane & 7, lane0 = lane & ~7;
    const unsigned gmask = 0xffu << lane0;
    const int vlim = value_limit(n);
    RegularFrames reg{s_sc, (uint32_t)(0x100000000ull / (uint32_t)max(stride, 2)) + 1u, n_int - 1};
    FrameCursor cur;
    if (!ok) cur.init(sc, pk, d.n_scores, n_picks, n_frames);
    // Segments are handed to the 8-lane groups sorted by the SHAPE of their pairwise-summation tree (one block up to
    // 128 frames, two up to 256, four up to 512, deeper beyond): the four groups of a warp then run the same code path
    // instead of four different ones one after the other.
    int *s_list = reinterpret_cast<int *>(s_sc + max_intervals);    // 4 lists of up to n segment indices
    if (tid < 4) s_class[tid] = 0;
    __syncthreads();
    for (int s = tid; s < n; s += NT) {
        const int start = __ldg(cps + 2 * (d.seg_off + s));
        const int len = min(__ldg(cps + 2 * (d.seg_off + s) + 1) + 1, n_frames) - start;
        const int c = len <= 128 ? 0 : (len <= 256 ? 1 : (len <= 512 ? 2 : 3));
        s_list[c * n + atomicAdd(&s_class[c], 1)] = s;
    }
    __syncthreads();
    const int c0 = s_class[0], c1 = c0 + s_class[1], c2 = c1 + s_class[2];
    for (int t = tid >> 3; t < n; t += NT / 8) {                    // uniform within an 8-lane group
        const int s = t < c0 ? s_list[t] : (t < c1 ? s_list[n + t - c0] : (t < c2 ? s_list[2 * n + t - c1] : s_list[3 * n + t - c2]));
        const int start = __ldg(cps + 2 * (d.seg_off + s));
        int end = __ldg(cps + 2 * (d.seg_off + s) + 1) + 1;
        end = min(end, n_frames);
        const int len = end - start;
        float sum;
        if (ok) {
            sum = pw_sum_group(reg, start, len, gl, gmask, lane0);
        } else {
            cur.seek(start + (len >= 8 ? gl : 0));
            sum = pw_sum_group(cur, start, len, gl, gmask, lane0);
        }
        if (gl == 0) {
            const float mean = __fdiv_rn(sum, (float)len);
            long long val = __double2ll_rz(__dmul_rn((double)mean, 1000.0));
            if (val > vlim || val < -vlim) { atomicOr(status + v, SMZ_STATUS_VALUE_RANGE); val = val > 0 ? vlim : -vlim; }
            if (out_mean) out_mean[d.seg_off + s] = mean;
            out_values[d.seg_off + s] = (int)val;
        }
    }
}

__global__ void __launch_bounds__(POOL_REG_THREADS)
pool_regular_kernel(const smz_video_desc *__restrict__ desc, int v0, const float *__restrict__ scores,
                    const int32_t *__restrict__ picks, const int32_t *__restrict__ cps, int max_intervals,
                    float *__restrict__ out_mean, int32_t *__restrict__ out_values, int32_t *__restrict__ status) {
    extern __shared__ float s_pool[];        // max_intervals scores, then 4 * max_n_segs ints (segment lists)
    const int v = v0 + blockIdx.x;
    const smz_video_desc d = desc[v];
    pool_regular_video(d, v, scores, picks, cps, max_intervals, s_pool, out_mean, out_values, status);
}

// ------------------------------------------------------------------------------------------
// evaluation tail fused into the knapsack kernels: summary vector + mask (utils/eval.py:111-122) and
// the per-annotator F-score (utils/eval.py:125-165) of the video the CTA has just solved
// ------------------------------------------------------------------------------------------
// The knapsack DP is shared-memory bound and takes ~200 us per video and CTA; the F-score streams 4*n_users*n_frames
// bytes of annotator rows and is HBM bound.  Run as separate kernels the two add up; run by the SAME persistent CTA,
// video after video, the CTAs of an SM are in different phases at any time, so the DP of some videos overlaps the
// streaming of others and the stage costs about max(DP, stream) instead of the sum.  No mask round trip through
// global memory either: the summary mask is built and consumed in shared memory.
struct EvalTail {
    int enabled;                    // 0: the kernels stop after out_picked
    int n_videos_total;             // unused by the device code (kept for debugging)
    const float *user;              // annotator rows (float32), or
    const uint32_t *user_bits;      // ... 1 bit per frame with
    const int64_t *bits_off;        //     per-video word offsets; both NULL: summary / mask only
    float *summary;                 // may be NULL
    uint32_t *mask;
    int32_t *msum;
    int32_t *overlap, *gsum;
    float *f;
    double *avg_f, *max_f;
    // fused segment pooling (16-bit knapsack kernel only): when pool_scores is given the CTA pools the video it is about
    // to solve itself (pool_regular_video) — no pooling kernel runs in front, its latency-bound work hides behind the
    // other CTAs' DP / streaming
    const float *pool_scores;
    const int32_t *pool_picks, *pool_cps;
    int pool_max_intervals;
    float *pool_seg_mean;
    int32_t *pool_values, *pool_status;
};

__host__ __device__ inline int tail_words(int max_n_segs, int max_n_frames) {
    return (max_n_segs + 1) + (max_n_frames + 31) / 32 + 2 * FSCORE_MAX_USERS;
}

// Called by all DP_THREADS (= FSCORE_THREADS) threads.  spk: picked flags, swp: (weight, value) per segment, both in
// shared memory; mem: tail_words() words of shared memory that the DP no longer needs.  v: index of the video in the
// arrays that are indexed per video (msum, avg_f, max_f).
static_assert(DP_THREADS == POOL_REG_THREADS, "the 16-bit knapsack kernel runs pool_regular_video on its own CTA");
static_assert(DP_THREADS == FSCORE_THREADS, "the fused tail runs the F-score chunk code on the DP kernel's CTA");
__device__ void eval_tail_video(const EvalTail &t, const smz_video_desc &d, int v, const int *spk, const int2 *swp,
                                uint32_t *mem) {
    __shared__ int swarp[DP_THREADS / 32];
    __shared__ int s_msum;
    constexpr int NT = DP_THREADS, NW = DP_THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = d.n_segs, n_frames = d.n_frames;
    const int mwords = (n_frames + 31) >> 5;
    int *spre = reinterpret_cast<int *>(mem);                 // n + 1
    uint32_t *smask = mem + n + 1;                            // mwords
    uint32_t *s_ov = smask + mwords, *s_gs = s_ov + FSCORE_MAX_USERS;
    const int n_users = min(d.n_users, FSCORE_MAX_USERS);
    for (int j = tid; j < mwords; j += NT) smask[j] = 0u;
    for (int u = tid; u < n_users; u += NT) { s_ov[u] = 0u; s_gs[u] = 0u; }
    // exclusive prefix of nfps = positions in the summary vector
    int carry = 0;
    for (int base = 0; base < n; base += NT) {
        const int i = base + tid;
        const int x = i < n ? swp[i].x : 0;
        int incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) swarp[warp] = incl;
        __syncthreads();
        int woff = 0, tile_total = 0;
#pragma unroll
        for (int k = 0; k < NW; k++) { const int w = swarp[k]; if (k < warp) woff += w; tile_total += w; }
        if (i < n) spre[i] = carry + woff + incl - x;
        carry += tile_total;
        __syncthreads();
    }
    if (tid == 0) spre[n] = carry;
    __syncthreads();
    for (int s = tid; s < n; s += NT) {
        if (spk[s]) {
            const int a = spre[s];
            const int b = min(spre[s + 1], n_frames);
            if (a < b) {
                const int wa = a >> 5, wb = (b - 1) >> 5;
                for (int wd = wa; wd <= wb; wd++) {
                    const int lo = max(a, wd << 5) & 31;
                    const int hi = min(b, (wd + 1) << 5) - (wd << 5);  // 1..32
                    const uint32_t m = (hi >= 32 ? 0xffffffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
                    atomicOr(&smask[wd], m);
                }
            }
        }
    }
    if (t.summary != nullptr) {
        float *dst = t.summary + d.summ_off;
        for (int s = warp; s < n; s += NW) {
            const int a = spre[s], nf = spre[s + 1] - a;
            const float val = spk[s] ? 1.f : 0.f;
            for (int j = lane; j < nf; j += 32) dst[a + j] = val;
        }
    }
    __syncthreads();
    int cnt = 0;
    for (int j = tid; j < mwords; j += NT) {
        const uint32_t m = smask[j];
        t.mask[d.mask_off + j] = m;
        cnt += __popc(m);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) swarp[warp] = cnt;
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
#pragma unroll
        for (int k = 0; k < NW; k++) tot += swarp[k];
        t.msum[v] = tot;
        s_msum = tot;
    }
    if (t.user == nullptr && t.user_bits == nullptr) { __syncthreads(); return; }
    // ---- F-score: stream the annotator rows once against the mask in shared memory
    if (t.user != nullptr) {
        fscore_rows_acc<FSCORE_UNROLL>(d, 0, n_frames, t.user, smask, s_ov, s_gs);
    } else {
        const uint32_t *ub = t.user_bits + t.bits_off[v];
        for (int u = warp; u < n_users; u += NW) {
            const uint32_t *row = ub + (int64_t)u * mwords;
            int ov = 0, gs = 0;
            for (int w = lane; w < mwords; w += 32) {
                const uint32_t x = __ldg(row + w);
                ov += __popc(x & smask[w]);
                gs += __popc(x);
            }
            ov = __reduce_add_sync(0xffffffffu, ov);
            gs = __reduce_add_sync(0xffffffffu, gs);
            if (lane == 0) { s_ov[u] = (uint32_t)ov; s_gs[u] = (uint32_t)gs; }
        }
    }
    __syncthreads();
    for (int u = tid; u < n_users; u += NT) {
        t.overlap[d.ucount_off + u] = (int)s_ov[u];
        t.gsum[d.ucount_off + u] = (int)s_gs[u];
    }
    if (tid == 0)
        fscore_final_video(n_users, s_msum, reinterpret_cast<const int32_t *>(s_ov), reinterpret_cast<const int32_t *>(s_gs),
                           t.f + d.ucount_off, t.avg_f ? t.avg_f + v : nullptr, t.max_f ? t.max_f + v : nullptr,
                           d.summ_len < d.n_frames);
    __syncthreads();
}

// ------------------------------------------------------------------------------------------
// dp_kernel<K>: knapsack DP + OR-tools extraction (or the 'rank' greedy) -> picked[]
// ------------------------------------------------------------------------------------------
// Longest-first order of the videos for the dp_kernel queue (cost ~ n_segs x capacity): a counting sort over 64
// cost buckets, so that the tail of the persistent kernel is a cheap video, not an expensive one.
constexpr int ORDER_BUCKETS = 64;

__device__ __forceinline__ int cost_bucket(const smz_video_desc &d, int max_n_segs) {
    const int b = (int)(((int64_t)d.n_segs * ORDER_BUCKETS) / (max_n_segs + 1));
    return ORDER_BUCKETS - 1 - min(max(b, 0), ORDER_BUCKETS - 1);             // bucket 0 = most segments
}

__global__ void order_count_kernel(const smz_video_desc *__restrict__ desc, int n_videos, int max_n_segs, int *__restrict__ counters) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n_videos) atomicAdd(counters + 1 + cost_bucket(desc[v], max_n_segs), 1);
}

__global__ void order_fill_kernel(const smz_video_desc *__restrict__ desc, int n_videos, int max_n_segs, int *__restrict__ counters,
                                  int *__restrict__ order) {
    __shared__ int base[ORDER_BUCKETS];
    if (threadIdx.x == 0) {
        int run = 0;
        for (int b = 0; b < ORDER_BUCKETS; b++) { base[b] = run; run += counters[1 + b]; }
    }
    __syncthreads();
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n_videos) {
        const int b = cost_bucket(desc[v], max_n_segs);
        order[base[b] + atomicAdd(counters + 1 + ORDER_BUCKETS + b, 1)] = v;
    }
}

struct DpSmem { int dp0, dp1, wp, pk, red, total, row, pad; };

// front_words: minimum size of the region in front of wp (the DP rows; the fused evaluation tail reuses it)
__host__ __device__ inline DpSmem dp_layout(int K, int max_n_segs, int max_weight, int front_words) {
    DpSmem L;
    L.row = K * DP_THREADS;
    L.pad = (max_weight + 31) / 32 * 32;
    if (L.pad < 32) L.pad = 32;
    int o = 0;
    o += L.pad; L.dp0 = o; o += L.row;      // [pad][row0][pad][row1]
    o += L.pad; L.dp1 = o; o += L.row;
    if (o < front_words) o = front_words;
    o = (o + 1) & ~1;                       // int2 alignment
    L.wp = o; o += 2 * max_n_segs;          // int2 (weight, value)
    L.pk = o; o += max_n_segs;              // picked flags; 'rank': order
    L.red = o; o += 32;
    L.total = o;
    return L;
}

template <int K>
__global__ void __launch_bounds__(DP_THREADS, K <= 18 ? 4 : 1)
dp_kernel(const smz_video_desc *__restrict__ desc, int n_videos, const int32_t *__restrict__ nfps,
          const int32_t *__restrict__ values, const float *__restrict__ seg_mean, int method, int max_n_segs,
          int max_weight, uint8_t *__restrict__ out_picked, int32_t *__restrict__ status,
          uint32_t *__restrict__ ws, int64_t ws_words_per_cta, int *__restrict__ queue, const int *__restrict__ order,
          const int *__restrict__ list_count, int front_words, const EvalTail tail) {
    extern __shared__ uint32_t smem[];
    __shared__ int s_next;
    // list_count != NULL: `order` is the fallback list dp16_kernel left behind and *list_count its length
    if (list_count != nullptr) n_videos = __ldcg(list_count);
    const DpSmem L = dp_layout(K, max_n_segs, max_weight, front_words);
    int *dp0 = reinterpret_cast<int *>(smem + L.dp0);
    int *dp1 = reinterpret_cast<int *>(smem + L.dp1);
    int2 *swp = reinterpret_cast<int2 *>(smem + L.wp);
    int *spk = reinterpret_cast<int *>(smem + L.pk);
    int *sred = reinterpret_cast<int *>(smem + L.red);
    uint32_t *bits = ws + (int64_t)blockIdx.x * ws_words_per_cta;   // [item/32][L.row]
    constexpr int NT = DP_THREADS, NW = DP_THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // videos are handed out through an atomic queue: their cost (n_segs x capacity) varies several-fold
    while (true) {
        if (tid == 0) s_next = atomicAdd(queue, 1);
        __syncthreads();
        if (s_next >= n_videos) break;
        const int v = order[s_next];
        const smz_video_desc d = desc[v];
        const int n = d.n_segs, cap = d.capacity;
        for (int j = tid; j < L.pad; j += NT) { dp0[j - L.pad] = kDpNeg; dp1[j - L.pad] = kDpNeg; }   // (the tail reuses the rows)
        // ---- weights / values, sum of weights, weight-range check
        int wsum = 0, bad = 0;
        const int vlim = value_limit(n);
        for (int i = tid; i < n; i += NT) {
            const int w = __ldg(nfps + d.seg_off + i);
            int p = __ldg(values + d.seg_off + i);
            if (p > vlim || p < -vlim) { bad |= SMZ_STATUS_VALUE_RANGE; p = p > 0 ? vlim : -vlim; }
            if (w <= cap && w > L.pad) bad |= SMZ_STATUS_WEIGHT_RANGE;   // host passed a wrong max_weight
            swp[i] = make_int2(w, p);
            spk[i] = 0;
            wsum += w;
        }
        wsum = __reduce_add_sync(0xffffffffu, wsum);
        bad = __reduce_or_sync(0xffffffffu, bad);
        if (lane == 0) { sred[warp] = wsum; sred[NW + warp] = bad; }
        __syncthreads();
        wsum = 0; bad = 0;
#pragma unroll
        for (int k = 0; k < NW; k++) { wsum += sred[k]; bad |= sred[NW + k]; }
        if (bad && tid == 0) atomicOr(status + v, bad);
        __syncthreads();   // sred is reused below

        if (method == SMZ_METHOD_KNAPSACK) {
            if (wsum <= cap) {
                // KnapsackSolver::ReduceCapacities: the capacity constraint is inactive, all items in
                for (int i = tid; i < n; i += NT) spk[i] = 1;
            } else if (cap > 0 && n > 0 && !(bad & SMZ_STATUS_WEIGHT_RANGE)) {
                // forward DP == KnapsackDynamicProgrammingSolver::SolveSubProblem over ALL items.
                // Thread t owns cells t, t+NT, ...: values in registers; cells above the capacity
                // (row padding) are ordinary cells of a larger knapsack: harmless.
                int val[K];
                uint32_t acc[K];
                int *cur = dp0, *nxt = dp1;
#pragma unroll
                for (int k = 0; k < K; k++) { val[k] = 0; acc[k] = 0u; cur[tid + k * NT] = 0; }
                __syncthreads();
                for (int i = 0; i < n; i++) {
                    const int2 wp = swp[i];
                    if (wp.x <= cap) {                         // uniform: upstream's loop body is empty otherwise
                        const int *src = cur + (tid - wp.x);   // c < w lands in the kDpNeg pad
#pragma unroll
                        for (int k0 = 0; k0 < K; k0 += 9) {
                            int cand[9];
#pragma unroll
                            for (int k = k0; k < K && k < k0 + 9; k++) cand[k - k0] = src[k * NT];
#pragma unroll
                            for (int k = k0; k < K && k < k0 + 9; k++) {
                                const int d = val[k] - cand[k - k0] - wp.y;                  // < 0 iff cand + p > val: the strict '>' of upstream
                                val[k] = __viaddmax_s32(cand[k - k0], wp.y, val[k]);          // DPX: max(cand + p, val)
                                acc[k] = __funnelshift_l((unsigned)d, acc[k], 1);             // take bit shifted in from the sign
                                nxt[tid + k * NT] = val[k];
                            }
                        }
                        __syncthreads();
                        int *t = cur; cur = nxt; nxt = t;
                    } else {
#pragma unroll
                        for (int k = 0; k < K; k++) acc[k] <<= 1;          // item not taken anywhere: a zero bit
                    }
                    if ((i & 31) == 31 || i == n - 1) {        // flush 32 items' take bits (item j of the word -> bit j), coalesced
                        uint32_t *dst = bits + (int64_t)(i >> 5) * L.row + tid;
                        const int sh = 31 - (i & 31);
#pragma unroll
                        for (int k = 0; k < K; k++) { dst[k * NT] = __brev(acc[k]) >> sh; acc[k] = 0u; }
                    }
                }
                __syncthreads();   // take bits visible to warp 0
                // KnapsackDynamicProgrammingSolver::Solve extraction loop.  SolveSubProblem(c, k)
                // == highest item < k whose take bit at cell c is set, else 0 (ids[] default).
                if (warp == 0) {
                    int remaining = cap, num = n;
                    while (remaining > 0 && num > 0) {
                        const int last = (num - 1) >> 5;
                        int sel = -1;
                        for (int j0 = 0; j0 <= last; j0 += 32) {
                            const int j = j0 + lane;
                            uint32_t wv = 0u;
                            if (j <= last) {
                                wv = __ldcg(bits + (int64_t)j * L.row + remaining);
                                const int nb = num - (j << 5);
                                if (nb < 32) wv &= (1u << nb) - 1u;
                            }
                            const int c = wv ? (j << 5) + 31 - __clz(wv) : -1;
                            sel = max(sel, warp_max(c));
                        }
                        sel = max(sel, 0);
                        remaining -= swp[sel].x;
                        num = sel;
                        if (remaining >= 0 && lane == 0) spk[sel] = 1;
                    }
                }
            }
        } else {
            // utils/eval.py:100-107: descending score, ties -> higher index first (see oracle);
            // strict '<' against the budget, no early break.
            int *order = dp0, *rank = dp1;        // n <= max_n_segs <= row is enforced by the host plan
            for (int i = tid; i < n; i += NT) {
                const float mi = __ldg(seg_mean + d.seg_off + i);
                int r = 0;
                for (int j = 0; j < n; j++) {
                    const float mj = __ldg(seg_mean + d.seg_off + j);
                    r += (mj > mi) || (mj == mi && j > i);
                }
                rank[i] = r;
            }
            __syncthreads();
            for (int i = tid; i < n; i += NT) order[rank[i]] = i;
            __syncthreads();
            if (tid == 0) {
                long long total = 0;
                for (int r = 0; r < n; r++) {
                    const int i = order[r];
                    if (total + swp[i].x < (long long)cap) { spk[i] = 1; total += swp[i].x; }
                }
            }
        }
        __syncthreads();
        for (int i = tid; i < n; i += NT) out_picked[d.seg_off + i] = (uint8_t)spk[i];
        if (tail.enabled) eval_tail_video(tail, d, v, spk, swp, smem);
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// dp16_kernel<KW, MK>: the knapsack DP of dp_kernel on 16-bit cells
// ------------------------------------------------------------------------------------------
// Row of 2H cells (H = KW * 256) stored as H words: word j = (cell j | cell j + H << 16).  The shifted read of item
// weight w is word j - w for BOTH halves: for j >= w that is (cell j - w, cell j + H - w); for j < w the low cell does
// not exist (the item cannot be packed below its weight: masked) and the high cell j + H - w < H is the LOW half of
// word j + H - w — so the P words in front of the row mirror the low halves of the last P row words in their HIGH
// halves (one extra 16-bit store for the threads that own those words).  Needs w <= P = MK * 256 for every usable
// item; the low-cell mask is only compiled for the first MK words of a thread (k * 256 + tid < w <= MK * 256).
// Values are unsigned 16 bit: p in [0, 32767] and no row value above 65535.  The second condition is checked
// exactly while running: rows are non-decreasing in the cell index, so the top cell bounds the row, and an item adds
// at most max(p): after every item the thread that owns the top cell tests top + max(p) <= 65535 (folded into the
// barrier, BAR.RED.OR); when it fails the video goes to the fallback list and dp_kernel<K> solves it in 32 bits.
// Take bits: per word a 2 x 16-bit shift register (item i of a group of 16 -> bit i of each half), flushed to the
// work buffer every 16 items as [group][H] words.
struct Dp16Smem { int row0, row1, wp, dpi, pk, total; };

__host__ __device__ inline Dp16Smem dp16_layout(int KW, int MK, int max_n_segs, int front_words) {
    Dp16Smem L;
    const int H = KW * DP_THREADS, P = MK * DP_THREADS;
    int o = 0;
    o += P; L.row0 = o; o += H;             // [mirror pad][row0][mirror pad][row1]
    o += P; L.row1 = o; o += H;
    if (o < front_words) o = front_words;   // the fused evaluation tail reuses the rows
    o = (o + 1) & ~1;
    L.wp = o; o += 2 * max_n_segs;          // int2 (weight, value)
    L.dpi = o; o += 2 * max_n_segs;         // int2 (weight, value) as the DP loop sees them
    L.pk = o; o += max_n_segs;              // picked flags
    L.total = o;
    return L;
}

__device__ __forceinline__ uint32_t add_u16x2(uint32_t a, uint32_t b) {
    uint32_t r;
    asm("add.u16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}
__device__ __forceinline__ uint32_t max_u16x2(uint32_t a, uint32_t b) {
    uint32_t r;
    asm("max.u16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}

constexpr int dp16_min_blocks(int KW) { return KW <= 5 ? 6 : (KW <= 9 ? 5 : (KW <= 14 ? 3 : (KW <= 18 ? 2 : 1))); }

template <int KW, int MK>
__global__ void __launch_bounds__(DP_THREADS, dp16_min_blocks(KW))
dp16_kernel(const smz_video_desc *__restrict__ desc, int n_videos, const int32_t *__restrict__ nfps,
            const int32_t *__restrict__ values, int max_n_segs, uint8_t *__restrict__ out_picked,
            uint32_t *__restrict__ ws, int64_t ws_words_per_cta, int *__restrict__ queue, const int *__restrict__ order,
            int *__restrict__ fallback, int front_words, const EvalTail tail) {
    extern __shared__ uint32_t smem[];
    __shared__ int s_next;
    constexpr int NT = DP_THREADS, NW = DP_THREADS / 32;
    constexpr int H = KW * NT, P = MK * NT;
    __shared__ int sred[6 * NW];
    const Dp16Smem L = dp16_layout(KW, MK, max_n_segs, front_words);
    uint32_t *row0 = smem + L.row0, *row1 = smem + L.row1;
    int2 *swp = reinterpret_cast<int2 *>(smem + L.wp);
    int2 *sdp = reinterpret_cast<int2 *>(smem + L.dpi);
    int *spk = reinterpret_cast<int *>(smem + L.pk);
    uint32_t *bits = ws + (int64_t)blockIdx.x * ws_words_per_cta;   // [item / 16][H]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    while (true) {
        if (tid == 0) s_next = atomicAdd(queue, 1);
        __syncthreads();
        if (s_next >= n_videos) break;
        const int v = order[s_next];
        const smz_video_desc d = desc[v];
        const int n = d.n_segs, cap = d.capacity;
        if (tail.pool_scores != nullptr) {          // fused pooling: segment means -> integer values of THIS video
            pool_regular_video(d, v, tail.pool_scores, tail.pool_picks, tail.pool_cps, tail.pool_max_intervals,
                               reinterpret_cast<float *>(smem), tail.pool_seg_mean, tail.pool_values, tail.pool_status);
            __syncthreads();                        // the values this CTA just wrote are read (through L2) below
        }
        // ---- weights / values and what decides the path: sum of weights, value / weight ranges of the usable items
        int wsum = 0, bad = 0, maxw = 0, maxp = 0, minp = 0, psum = 0;
        const int vlim = value_limit(n);
        for (int i = tid; i < n; i += NT) {
            const int w = __ldg(nfps + d.seg_off + i);
            const int p = __ldcg(values + d.seg_off + i);
            if (p > vlim || p < -vlim || w < 0) bad = 1;        // dp_kernel flags and clips these
            swp[i] = make_int2(w, p);
            sdp[i] = w <= cap ? make_int2(w, p) : make_int2(0, 0);
            spk[i] = 0;
            wsum += w;
            if (w <= cap) { maxw = max(maxw, w); maxp = max(maxp, p); minp = min(minp, p); psum += min(max(p, 0), 32767); }
        }
        wsum = __reduce_add_sync(0xffffffffu, wsum);
        psum = __reduce_add_sync(0xffffffffu, psum);
        bad = __reduce_or_sync(0xffffffffu, bad);
        maxw = __reduce_max_sync(0xffffffffu, maxw);
        maxp = __reduce_max_sync(0xffffffffu, maxp);
        minp = __reduce_min_sync(0xffffffffu, minp);
        if (lane == 0) {
            sred[warp] = wsum; sred[NW + warp] = bad; sred[2 * NW + warp] = maxw;
            sred[3 * NW + warp] = maxp; sred[4 * NW + warp] = minp; sred[5 * NW + warp] = psum;
        }
        __syncthreads();
        wsum = 0; bad = 0; maxw = 0; maxp = 0; minp = 0; psum = 0;
#pragma unroll
        for (int k = 0; k < NW; k++) {
            wsum += sred[k]; bad |= sred[NW + k]; maxw = max(maxw, sred[2 * NW + k]);
            maxp = max(maxp, sred[3 * NW + k]); minp = min(minp, sred[4 * NW + k]); psum += sred[5 * NW + k];
        }
        // 0: nothing packed, 1: everything packed (KnapsackSolver::ReduceCapacities), 2: 16-bit DP, 3: dp_kernel<K>
        int mode;
        if (bad) mode = 3;
        else if (n == 0) mode = 0;
        else if (wsum <= cap) mode = 1;
        else if (cap <= 0) mode = 0;
        else {
            // exact conditions (cells, pad, value range) + a guess that spares a doomed attempt: the optimum is at
            // least about the average value density times the capacity
            const bool fits = cap < 2 * H && maxw <= (P < H ? P : H) && minp >= 0 && maxp <= 32767;
            const bool hopeless = (long long)psum * cap > 45000ll * wsum;
            mode = (fits && !hopeless) ? 2 : 3;
        }
        if (mode == 1)
            for (int i = tid; i < n; i += NT) spk[i] = 1;
        if (mode == 2) {
            uint32_t val[KW], acc[KW];
#pragma unroll
            for (int k = 0; k < KW; k++) { val[k] = 0u; acc[k] = 0u; row0[tid + k * NT] = 0u; }
            for (int j = tid; j < P; j += NT) { row0[j - P] = 0u; row1[j - P] = 0u; }
            __syncthreads();
            const uint32_t top_limit = 65535u - (uint32_t)maxp;
            int aborted = 0;
            // One item: row CUR -> row NXT.  sdp[] is the DP's view of the items: (w, p), (0, 0) for an item heavier than
            // the capacity (upstream's loop body is empty for it; with w = p = 0 every cell compares against itself and
            // nothing is taken, so the row ping-pong keeps its parity), w < 0 = stop marker left by the top-cell check.
#define SMZ_DP16_STEP(CUR, NXT, I)                                                                                   \
            {                                                                                                        \
                const int2 wp = sdp[I];                                                                              \
                if (wp.x < 0) { aborted = 1; break; }                                                                \
                const uint32_t *src = (CUR) + (tid - wp.x);       /* word j - w; j < w lands in the mirror pad */    \
                const uint32_t pp = (uint32_t)wp.y * 0x10001u;                                                       \
                uint32_t cand[KW];                                                                                   \
                _Pragma("unroll") for (int k = 0; k < KW; k++) cand[k] = src[k * NT];                                \
                _Pragma("unroll") for (int k = 0; k < KW; k++) {                                                     \
                    uint32_t nv;                                                                                     \
                    if (k < MK) {                                                                                    \
                        uint32_t t = add_u16x2(cand[k], pp);                                                         \
                        if (tid + k * NT < wp.x) t &= 0xffff0000u;     /* cell j < w: the item does not fit */       \
                        nv = max_u16x2(t, val[k]);                                                                   \
                    } else {                                                                                         \
                        nv = __viaddmax_u16x2(cand[k], pp, val[k]);     /* DPX: max(cand + p, val), both halves */   \
                    }                                                                                                \
                    /* improved halves differ by 1..32767: + 0x7fff sets bit 15 of exactly those (no carries) */     \
                    const uint32_t y = nv - val[k] + 0x7fff7fffu;                                                    \
                    acc[k] = (acc[k] >> 1) | (y & 0x80008000u);                                                      \
                    val[k] = nv;                                                                                     \
                    (NXT)[tid + k * NT] = nv;                                                                        \
                    if (k >= KW - MK)                                   /* words [H - P, H): mirror the low half */  \
                        reinterpret_cast<unsigned short *>((NXT) + (tid + k * NT - H))[1] = (unsigned short)nv;      \
                }                                                                                                    \
                if (tid == NT - 1 && val[KW - 1] > ((top_limit << 16) | 0xffffu) && (I) + 1 < n) sdp[(I) + 1].x = -1; \
                __syncthreads();                                                                                     \
            }
            // flush `cnt` items' take bits of group G (item j of the group -> bit j of each half), coalesced
#define SMZ_DP16_FLUSH(G, CNT)                                                                                        \
            {                                                                                                        \
                uint32_t *dst = bits + (int64_t)(G) * H + tid;                                                       \
                const int sh = 16 - (CNT);                                                                           \
                const uint32_t m = (0xffffu >> sh) * 0x10001u;                                                       \
                _Pragma("unroll") for (int k = 0; k < KW; k++) { dst[k * NT] = (acc[k] >> sh) & m; acc[k] = 0u; }    \
            }
            int i = 0;
            for (; i + 1 < n; i += 2) {                     // two items per trip: the rows (and the registers) ping-pong
                SMZ_DP16_STEP(row0, row1, i)
                SMZ_DP16_STEP(row1, row0, i + 1)
                if ((i & 15) == 14) SMZ_DP16_FLUSH(i >> 4, 16)
            }
            if (!aborted && i < n) {
                do { SMZ_DP16_STEP(row0, row1, i) } while (0);
            }
            if (!aborted && (n & 15)) SMZ_DP16_FLUSH((n - 1) >> 4, n & 15)
#undef SMZ_DP16_STEP
#undef SMZ_DP16_FLUSH
            if (aborted) mode = 3;
            __syncthreads();   // take bits visible to warp 0
            // KnapsackDynamicProgrammingSolver::Solve extraction loop (see dp_kernel)
            if (mode == 2 && warp == 0) {
                int remaining = cap, num = n;
                while (remaining > 0 && num > 0) {
                    const int j = remaining >= H ? remaining - H : remaining;
                    const int hs = remaining >= H ? 16 : 0;
                    const int last = (num - 1) >> 4;
                    int sel = -1;
                    for (int g0 = 0; g0 <= last; g0 += 32) {
                        const int g = g0 + lane;
                        uint32_t wv = 0u;
                        if (g <= last) {
                            wv = (__ldcg(bits + (int64_t)g * H + j) >> hs) & 0xffffu;
                            const int nb = num - (g << 4);
                            if (nb < 16) wv &= (1u << nb) - 1u;
                        }
                        const int c = wv ? (g << 4) + 31 - __clz(wv) : -1;
                        sel = max(sel, warp_max(c));
                    }
                    sel = max(sel, 0);
                    remaining -= swp[sel].x;
                    num = sel;
                    if (remaining >= 0 && lane == 0) spk[sel] = 1;
                }
            }
        }
        if (mode == 3) {
            if (tid == 0) { const int k = atomicAdd(fallback, 1); fallback[1 + k] = v; }
        } else {
            __syncthreads();
            for (int i = tid; i < n; i += NT) out_picked[d.seg_off + i] = (uint8_t)spk[i];
            if (tail.enabled) eval_tail_video(tail, d, v, spk, swp, smem);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// summary_kernel: utils/eval.py:111-122 summary vector (+ bit mask truncated to n_frames, msum)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SUMMARY_THREADS)
summary_kernel(const smz_video_desc *__restrict__ desc, int v0, const int32_t *__restrict__ nfps,
               const uint8_t *__restrict__ picked, int max_n_segs, int max_n_frames,
               float *__restrict__ out_summary, uint32_t *__restrict__ out_mask, int32_t *__restrict__ out_msum) {
    extern __shared__ uint32_t smem[];
    int *spre = reinterpret_cast<int *>(smem);                  // max_n_segs + 1
    uint32_t *smask = smem + max_n_segs + 1;                    // ceil(max_n_frames / 32)
    __shared__ int swarp[SUMMARY_THREADS / 32];
    constexpr int NT = SUMMARY_THREADS, NW = SUMMARY_THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int v = v0 + blockIdx.x;
    const smz_video_desc d = desc[v];
    const int n = d.n_segs, n_frames = d.n_frames;
    const int mwords = (n_frames + 31) >> 5;
    for (int j = tid; j < mwords; j += NT) smask[j] = 0u;
    // exclusive prefix of nfps = positions in the summary vector
    int carry = 0;
    for (int base = 0; base < n; base += NT) {
        const int i = base + tid;
        const int x = i < n ? __ldg(nfps + d.seg_off + i) : 0;
        int incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) swarp[warp] = incl;
        __syncthreads();
        int woff = 0, tile_total = 0;
#pragma unroll
        for (int k = 0; k < NW; k++) { const int t = swarp[k]; if (k < warp) woff += t; tile_total += t; }
        if (i < n) spre[i] = carry + woff + incl - x;
        carry += tile_total;
        __syncthreads();
    }
    if (tid == 0) spre[n] = carry;
    __syncthreads();
    for (int s = tid; s < n; s += NT) {
        if (picked[d.seg_off + s]) {
            const int a = spre[s];
            const int b = min(spre[s + 1], n_frames);
            if (a < b) {
                const int wa = a >> 5, wb = (b - 1) >> 5;
                for (int wd = wa; wd <= wb; wd++) {
                    const int lo = max(a, wd << 5) & 31;
                    const int hi = min(b, (wd + 1) << 5) - (wd << 5);  // 1..32
                    const uint32_t m = (hi >= 32 ? 0xffffffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
                    atomicOr(&smask[wd], m);
                }
            }
        }
    }
    if (out_summary) {
        float *dst = out_summary + d.summ_off;
        for (int s = warp; s < n; s += NW) {
            const int a = spre[s], nf = spre[s + 1] - a;
            const float val = picked[d.seg_off + s] ? 1.f : 0.f;
            for (int j = lane; j < nf; j += 32) dst[a + j] = val;
        }
    }
    __syncthreads();
    int cnt = 0;
    for (int j = tid; j < mwords; j += NT) {
        const uint32_t m = smask[j];
        out_mask[d.mask_off + j] = m;
        cnt += __popc(m);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) swarp[warp] = cnt;
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
#pragma unroll
        for (int k = 0; k < NW; k++) tot += swarp[k];
        out_msum[v] = tot;
    }
}

// ------------------------------------------------------------------------------------------
// select_generic_kernel — one persistent CTA does everything for a video.  Fallback for
// capacities whose DP row does not fit the register-DP plan (very long videos).
// ------------------------------------------------------------------------------------------
struct SelectSmem {  // word offsets into dynamic shared memory (generic kernel)
    int dp0, dp1, w, p, wp, pk, mean, pre, mask, sel, bits, total, row;
};

__host__ __device__ inline SelectSmem select_layout(int max_n_segs, int max_capacity, int max_n_frames,
                                                    bool bits_in_smem) {
    SelectSmem L;
    const int ncell = max_capacity + 1;
    // the dp rows double as scratch (warp totals, 'rank' order): at least 32 and max_n_segs words
    int row = ncell > max_n_segs ? ncell : max_n_segs;
    row = row > 32 ? row : 32;
    L.row = row;
    int o = 0;
    L.dp0 = o; o += row;
    L.dp1 = o; o += row;
    L.w = o; o += max_n_segs;
    L.p = o; o += max_n_segs;
    L.wp = o; o += 2 * max_n_segs;
    L.pk = o; o += max_n_segs;
    L.mean = o; o += max_n_segs;
    L.pre = o; o += max_n_segs + 1;
    L.mask = o; o += (max_n_frames + 31) / 32;
    L.sel = o; o += 4;
    L.bits = o;
    if (bits_in_smem) o += max_n_segs * ((ncell + 31) / 32);
    L.total = o;
    return L;
}

template <bool BITS_IN_SMEM>
__global__ void __launch_bounds__(SELECT_THREADS)
select_generic_kernel(const smz_video_desc *__restrict__ desc, int n_videos, const float *__restrict__ scores,
              const int32_t *__restrict__ picks, const int32_t *__restrict__ cps,
              const int32_t *__restrict__ nfps, const int32_t *__restrict__ values_in, int method,
              int max_n_segs, int max_capacity, int max_n_frames, float *__restrict__ out_mean, int32_t *__restrict__ out_values,
              uint8_t *__restrict__ out_picked, float *__restrict__ out_summary,
              uint32_t *__restrict__ out_mask, int32_t *__restrict__ out_msum,
              int32_t *__restrict__ out_status, uint32_t *__restrict__ ws, int64_t ws_words_per_cta) {
    extern __shared__ uint32_t smem[];
    const SelectSmem L = select_layout(max_n_segs, max_capacity, max_n_frames, BITS_IN_SMEM);
    int *dp0 = reinterpret_cast<int *>(smem + L.dp0);
    int *dp1 = reinterpret_cast<int *>(smem + L.dp1);
    int *sw = reinterpret_cast<int *>(smem + L.w);
    int *sp = reinterpret_cast<int *>(smem + L.p);
    int *spk = reinterpret_cast<int *>(smem + L.pk);
    float *smean = reinterpret_cast<float *>(smem + L.mean);
    int *spre = reinterpret_cast<int *>(smem + L.pre);
    uint32_t *smask = smem + L.mask;
    int *ssel = reinterpret_cast<int *>(smem + L.sel);
    int2 *swp = reinterpret_cast<int2 *>(smem + L.wp);
    uint32_t *bits = BITS_IN_SMEM ? (smem + L.bits) : (ws + (int64_t)blockIdx.x * ws_words_per_cta);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NT = SELECT_THREADS, NW = SELECT_THREADS / 32;

    for (int v = blockIdx.x; v < n_videos; v += gridDim.x) {
        const smz_video_desc d = desc[v];
        const int n = d.n_segs;
        const int cap = d.capacity;
        const int n_frames = d.n_frames;
        int status = 0;

        // ---- A. segment pooling (utils/eval.py:87-94) + value quantisation (knapsack.py:11-15)
        if (values_in != nullptr) {
            // stand-alone knapsack (utils/knapsack.py:5-23): values already quantised by the caller
            const int vlim = value_limit(n);
            for (int s = tid; s < n; s += NT) {
                int val = __ldg(values_in + d.seg_off + s);
                if (val > vlim || val < -vlim) { status |= SMZ_STATUS_VALUE_RANGE; val = val > 0 ? vlim : -vlim; }
                smean[s] = (float)val;
                sp[s] = val;
                sw[s] = __ldg(nfps + d.seg_off + s);
                spk[s] = 0;
            }
            if (tid == 0) { ssel[0] = -1; ssel[1] = -1; ssel[2] = -1; }
        } else {
            FrameCursor cur;
            cur.init(scores + d.score_off, picks + d.picks_off, d.n_scores, d.n_picks, n_frames);
            if (cur.n_bound - 1 > d.n_scores + 1) status |= SMZ_STATUS_INTERVALS;
            const int vlim = value_limit(n);
            const int gl = lane & 7, lane0 = lane & ~7;
            const unsigned gmask = 0xffu << lane0;
            for (int s0 = 0; s0 < n; s0 += NT / 8) {        // 8 lanes per segment
                const int s = s0 + (tid >> 3);
                if (s < n) {                                 // uniform within a group
                    const int start = __ldg(cps + 2 * (d.seg_off + s));
                    int end = __ldg(cps + 2 * (d.seg_off + s) + 1) + 1;
                    end = min(end, n_frames);
                    const int len = end - start;
                    cur.seek(start + (len >= 8 ? gl : 0));
                    const float sum = pw_sum_group(cur, start, len, gl, gmask, lane0);
                    if (gl == 0) {
                        const float mean = __fdiv_rn(sum, (float)len);
                        long long val = __double2ll_rz(__dmul_rn((double)mean, 1000.0));
                        if (val > vlim || val < -vlim) { status |= SMZ_STATUS_VALUE_RANGE; val = val > 0 ? vlim : -vlim; }
                        smean[s] = mean;
                        sp[s] = (int)val;
                        sw[s] = __ldg(nfps + d.seg_off + s);
                        spk[s] = 0;
                        if (out_mean) out_mean[d.seg_off + s] = mean;
                        if (out_values) out_values[d.seg_off + s] = (int)val;
                    }
                }
            }
            if (tid == 0) { ssel[0] = -1; ssel[1] = -1; ssel[2] = -1; }
        }
        {
            const int s1 = __syncthreads_or(status & SMZ_STATUS_VALUE_RANGE);
            const int s2 = __syncthreads_or(status & SMZ_STATUS_INTERVALS);
            status = (s1 ? SMZ_STATUS_VALUE_RANGE : 0) | (s2 ? SMZ_STATUS_INTERVALS : 0);
        }

        // ---- B. exclusive prefix of nfps (positions in the summary vector, utils/eval.py:111-122)
        {
            int carry = 0;
            for (int base = 0; base < n; base += NT) {
                const int i = base + tid;
                const int x = i < n ? sw[i] : 0;
                int incl = x;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += y;
                }
                if (lane == 31) dp0[warp] = incl;  // dp rows are not live yet (rows hold >= 32 words)
                __syncthreads();
                int woff = 0;
                for (int k = 0; k < warp; k++) woff += dp0[k];
                int tile_total = 0;
                for (int k = 0; k < NW; k++) tile_total += dp0[k];
                if (i < n) spre[i] = carry + woff + incl - x;
                carry += tile_total;
                __syncthreads();
            }
            if (tid == 0) spre[n] = carry;
            for (int i = tid; i < n; i += NT) swp[i] = make_int2(sw[i], sp[i]);
            const int mwords = (n_frames + 31) >> 5;
            for (int j = tid; j < mwords; j += NT) smask[j] = 0u;
        }
        __syncthreads();

        // ---- C. selection
        if (method == SMZ_METHOD_KNAPSACK) {
            if (spre[n] <= cap) {
                // KnapsackSolver::ReduceCapacities: the capacity constraint is inactive, all items in
                for (int s = tid; s < n; s += NT) spk[s] = 1;
            } else if (cap > 0 && n > 0) {
                const int ncell = cap + 1;
                // take-bit row stride: the register DP writes one word per (warp, k) pass
                const int words = (ncell + 31) >> 5;
                int *cur = dp0, *nxt = dp1;
                // forward DP, KnapsackDynamicProgrammingSolver::SolveSubProblem for ALL items; the
                // strict '>' of upstream is kept per cell in the take-bit row of the item
                {
                    for (int c = tid; c < ncell; c += NT) cur[c] = 0;
                    __syncthreads();
                    for (int i = 0; i < n; i++) {
                        const int w = sw[i], p = sp[i];
                        uint32_t *row = bits + (int64_t)i * words;
                        if (w > cap) {
                            for (int j = tid; j < words; j += NT) row[j] = 0u;
                            continue;
                        }
                        for (int base = warp * 32; base < ncell; base += NT) {
                            const int c = base + lane;
                            bool imp = false;
                            if (c < ncell) {
                                const int old = cur[c];
                                int v2 = old;
                                if (c >= w) {
                                    const int cand = cur[c - w] + p;
                                    if (cand > old) { v2 = cand; imp = true; }
                                }
                                nxt[c] = v2;
                            }
                            const uint32_t b = __ballot_sync(0xffffffffu, imp);
                            if (lane == 0) row[base >> 5] = b;
                        }
                        __syncthreads();
                        int *t = cur; cur = nxt; nxt = t;
                    }
                }
                __syncthreads();
                // KnapsackDynamicProgrammingSolver::Solve extraction loop.  SolveSubProblem(c, k)
                // == highest item < k whose take bit at cell c is set, else 0 (ids[] default).
                int remaining = cap, num = n, round = 0;
                while (remaining > 0 && num > 0) {
                    const int slot = round % 3;
                    if (tid == 0) ssel[(round + 1) % 3] = -1;
                    const int widx = remaining >> 5, bit = remaining & 31;
                    int local = -1;
                    for (int i = tid; i < num; i += NT)
                        if ((bits[(int64_t)i * words + widx] >> bit) & 1u) local = i;
                    local = warp_max(local);
                    if (lane == 0 && local >= 0) atomicMax(&ssel[slot], local);
                    __syncthreads();
                    const int sel = max(ssel[slot], 0);
                    remaining -= sw[sel];
                    num = sel;
                    if (remaining >= 0 && tid == 0) spk[sel] = 1;
                    ++round;
                }
            }
        } else {
            // utils/eval.py:100-107: descending score, ties -> higher index first (see oracle);
            // strict '<' against the budget, no early break.
            int *order = sp;  // values are not needed by 'rank'
            int *rank = dp1;  // n <= max_n_segs; dp1 is sized below to hold it
            for (int i = tid; i < n; i += NT) {
                const float mi = smean[i];
                int r = 0;
                for (int j = 0; j < n; j++) {
                    const float mj = smean[j];
                    r += (mj > mi) || (mj == mi && j > i);
                }
                rank[i] = r;
            }
            __syncthreads();
            for (int i = tid; i < n; i += NT) order[rank[i]] = i;
            __syncthreads();
            if (tid == 0) {
                long long total = 0;
                for (int r = 0; r < n; r++) {
                    const int i = order[r];
                    if (total + sw[i] < (long long)cap) { spk[i] = 1; total += sw[i]; }
                }
            }
        }
        __syncthreads();

        // ---- D. outputs: picked flags, float summary vector, bit mask (truncated to n_frames)
        for (int s = tid; s < n; s += NT) {
            const int pk = spk[s];
            out_picked[d.seg_off + s] = (uint8_t)pk;
            if (pk) {
                const int a = spre[s];
                const int b = min(a + sw[s], n_frames);
                if (a < b) {
                    const int wa = a >> 5, wb = (b - 1) >> 5;
                    for (int wd = wa; wd <= wb; wd++) {
                        const int lo = max(a, wd << 5) & 31;
                        const int hi = min(b, (wd + 1) << 5) - (wd << 5);  // 1..32
                        const uint32_t m = (hi >= 32 ? 0xffffffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
                        atomicOr(&smask[wd], m);
                    }
                }
            }
        }
        if (out_summary) {
            float *dst = out_summary + d.summ_off;
            for (int s = warp; s < n; s += NW) {
                const int a = spre[s], nf = sw[s];
                const float val = spk[s] ? 1.f : 0.f;
                for (int j = lane; j < nf; j += 32) dst[a + j] = val;
            }
        }
        __syncthreads();
        {
            const int mwords = (n_frames + 31) >> 5;
            int cnt = 0;
            for (int j = tid; j < mwords; j += NT) {
                const uint32_t m = smask[j];
                out_mask[d.mask_off + j] = m;
                cnt += __popc(m);
            }
            cnt = __reduce_add_sync(0xffffffffu, cnt);
            if (lane == 0) dp1[warp] = cnt;
            __syncthreads();
            if (tid == 0) {
                int tot = 0;
                for (int k = 0; k < NW; k++) tot += dp1[k];
                out_msum[v] = tot;
                if (out_status) out_status[v] = status;
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// host side: plan + launch
// ------------------------------------------------------------------------------------------
struct SelectPlan {
    int k;               // cells per thread of dp_kernel; 0 = generic monolithic kernel
    bool bits_in_smem;   // generic kernel only
    int smem_bytes;
    int grid;
    int64_t ws_words_per_cta;
    int pad_weight;      // max weight the dp rows' front pad is sized for
    int kw16, mk16;      // words per thread / masked words of dp16_kernel; kw16 == 0: no 16-bit pass
    int smem16_bytes, grid16;
    int64_t ws16_words_per_cta;
    int front_words;     // > 0: the DP kernels' shared memory also holds the fused evaluation tail (summary + F-score)
    int64_t ws_bits_bytes() const {
        const int64_t a = (int64_t)grid * ws_words_per_cta, b = kw16 ? (int64_t)grid16 * ws16_words_per_cta : 0;
        return (a > b ? a : b) * 4;      // the two DP passes run one after the other and share the take-bit buffer
    }
};

constexpr int kDpK[] = {2, 5, 9, 18, 27, 36, 54};

typedef void (*dp_fn)(const smz_video_desc *, int, const int32_t *, const int32_t *, const float *, int, int, int,
                      uint8_t *, int32_t *, uint32_t *, int64_t, int *, const int *, const int *, int, const EvalTail);
typedef void (*dp16_fn)(const smz_video_desc *, int, const int32_t *, const int32_t *, int, uint8_t *, uint32_t *, int64_t,
                        int *, const int *, int *, int, const EvalTail);
typedef void (*generic_fn)(const smz_video_desc *, int, const float *, const int32_t *, const int32_t *,
                           const int32_t *, const int32_t *, int, int, int, int, float *, int32_t *, uint8_t *,
                           float *, uint32_t *, int32_t *, int32_t *, uint32_t *, int64_t);

dp_fn dp_fn_for(int k) {
    switch (k) {
        case 2: return dp_kernel<2>;
        case 5: return dp_kernel<5>;
        case 9: return dp_kernel<9>;
        case 18: return dp_kernel<18>;
        case 27: return dp_kernel<27>;
        case 36: return dp_kernel<36>;
        case 54: return dp_kernel<54>;
        default: return nullptr;
    }
}

dp16_fn dp16_fn_for(int kw, int mk) {
#define SMZ_DP16_CASE(KW, MK) if (kw == KW && mk == MK) return dp16_kernel<KW, MK>;
    SMZ_DP16_CASE(1, 1) SMZ_DP16_CASE(3, 2) SMZ_DP16_CASE(3, 3) SMZ_DP16_CASE(5, 2) SMZ_DP16_CASE(5, 5)
    SMZ_DP16_CASE(9, 2) SMZ_DP16_CASE(9, 9) SMZ_DP16_CASE(14, 2) SMZ_DP16_CASE(14, 14) SMZ_DP16_CASE(18, 2)
    SMZ_DP16_CASE(18, 18) SMZ_DP16_CASE(27, 2) SMZ_DP16_CASE(27, 27)
#undef SMZ_DP16_CASE
    return nullptr;
}

generic_fn generic_fn_for(bool bits_in_smem) {
    return bits_in_smem ? (generic_fn)select_generic_kernel<true> : (generic_fn)select_generic_kernel<false>;
}

}  // namespace

// int32 words behind the take-bit buffer: [0] dp16 queue head, [1..64] bucket counts, [65..128] bucket fills,
// [129] dp_kernel queue head, [130] fallback count, [131, 131 + n) fallback list, then order[n]
constexpr int kQueueHead32 = 1 + 2 * ORDER_BUCKETS, kFallback = kQueueHead32 + 1, kQueueInts = kFallback + 1;
static int64_t queue_bytes(int n_videos) { return (int64_t)(kQueueInts + 2 * (int64_t)n_videos) * 4 + 256; }

// cudaFuncSetAttribute + occupancy query once per (device, kernel, dynamic shared memory): the plan is rebuilt on every
// call and these two driver calls would otherwise dominate its host time.  Callers may plan from several host threads
// at once (ctypes releases the GIL): the table and the attribute it tracks change under one lock, so one thread cannot
// lower a kernel's shared-memory limit below what another has planned a launch with.
static int cached_occupancy(const void *fn, int threads, int smem_bytes, int *per_sm) {
    struct Entry { int dev; const void *fn; int smem, per_sm; };
    static std::mutex mu;
    static Entry table[96];
    static int used = 0;
    std::lock_guard<std::mutex> lock(mu);
    int dev = 0;
    SMZ_CUDA_CHECK(cudaGetDevice(&dev));
    int attr = -1;                       // largest dynamic size this kernel's attribute was raised to on this device
    for (int i = 0; i < used; i++) {
        if (table[i].dev != dev || table[i].fn != fn) continue;
        if (table[i].smem == smem_bytes) { *per_sm = table[i].per_sm; return SMZ_OK; }
        if (table[i].smem > attr) attr = table[i].smem;
    }
    if (used >= 96) {                    // a full table no longer knows every size the attribute was raised to: ask
        cudaFuncAttributes fa;
        SMZ_CUDA_CHECK(cudaFuncGetAttributes(&fa, fn));
        attr = fa.maxDynamicSharedSizeBytes;
    }
    if (smem_bytes > attr)               // only ever raised, so launches planned earlier (on any thread) stay valid
        SMZ_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    SMZ_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, fn, threads, smem_bytes));
    if (used < 96) table[used++] = Entry{dev, fn, smem_bytes, *per_sm};
    return SMZ_OK;
}

static int select_plan(int n_videos, int max_n_segs, int max_capacity, int max_n_frames, int max_weight,
                       SelectPlan *plan) {
    if (max_n_segs < 0 || max_capacity < 0 || max_n_frames < 0 || max_weight < 0)
        return smz::fail(SMZ_ERR_ARG, "negative batch maxima");
    const int optin = smz::max_smem_optin();
    const int ncell = max_capacity + 1;
    const int need = ncell > max_n_segs ? ncell : max_n_segs;
    plan->pad_weight = max_weight < max_capacity ? max_weight : max_capacity;   // heavier items are never read
    plan->k = 0;
    plan->kw16 = plan->mk16 = plan->smem16_bytes = plan->grid16 = 0;
    plan->ws16_words_per_cta = 0;
    plan->front_words = 0;
    for (int k : kDpK)
        if (k * DP_THREADS >= need) { plan->k = k; break; }
    int per_sm = 0;
    if (plan->k > 0) {
        // with the evaluation tail when it fits next to the rows (it reuses them), without it otherwise
        const int fw = getenv("SMZ_NO_FUSED_TAIL") ? 0 : tail_words(max_n_segs, max_n_frames);
        plan->smem_bytes = dp_layout(plan->k, max_n_segs, plan->pad_weight, fw).total * 4;
        if (plan->smem_bytes <= optin) plan->front_words = fw;
        else plan->smem_bytes = dp_layout(plan->k, max_n_segs, plan->pad_weight, 0).total * 4;
        if (plan->smem_bytes > optin) plan->k = 0;
    }
    if (plan->k > 0) {
        dp_fn fn = dp_fn_for(plan->k);
        plan->bits_in_smem = false;
        { const int rc = cached_occupancy((const void *)fn, DP_THREADS, plan->smem_bytes, &per_sm); if (rc != SMZ_OK) return rc; }
        plan->ws_words_per_cta = (int64_t)((max_n_segs + 31) / 32) * plan->k * DP_THREADS;
        // 16-bit pass in front of it (same cell count: 2 * kw16 * 256 >= k * 256)
        const int kw = (plan->k + 1) / 2;
        const int mk = (kw >= 2 && plan->pad_weight <= 2 * DP_THREADS) ? 2 : kw;
        dp16_fn fn16 = getenv("SMZ_NO_DP16") ? nullptr : dp16_fn_for(kw, mk);
        const int smem16 = dp16_layout(kw, mk, max_n_segs, plan->front_words).total * 4;
        if (fn16 != nullptr && smem16 <= optin) {
            int per_sm16 = 0;
            { const int rc = cached_occupancy((const void *)fn16, DP_THREADS, smem16, &per_sm16); if (rc != SMZ_OK) return rc; }
            if (per_sm16 >= 1) {
                plan->kw16 = kw; plan->mk16 = mk; plan->smem16_bytes = smem16;
                const int g16 = smz::sm_count() * per_sm16;
                plan->grid16 = n_videos < g16 ? n_videos : g16;
                // More videos than resident CTAs: every CTA works through ceil(n / grid) videos of near-equal cost, so a
                // grid that does not divide n leaves a last round in which part of the CTAs idle (10 000 videos on 740
                // CTAs: 13.5 rounds).  Shrink the grid to the smallest one with the same number of rounds.
                if (n_videos > g16 && !getenv("SMZ_EVAL_FULL_GRID")) {
                    const int rounds = (n_videos + g16 - 1) / g16;
                    plan->grid16 = (n_videos + rounds - 1) / rounds;
                }
                plan->ws16_words_per_cta = (int64_t)((max_n_segs + 15) / 16) * kw * DP_THREADS;
            }
        }
    } else {
        const int with_bits = select_layout(max_n_segs, max_capacity, max_n_frames, true).total * 4;
        const int without = select_layout(max_n_segs, max_capacity, max_n_frames, false).total * 4;
        if (with_bits <= optin) { plan->bits_in_smem = true; plan->smem_bytes = with_bits; }
        else if (without <= optin) { plan->bits_in_smem = false; plan->smem_bytes = without; }
        else
            return smz::fail(SMZ_ERR_UNSUPPORTED,
                             "select_shots: DP rows for capacity %d, %d segments and %d frames need %d B of shared "
                             "memory (> %d B per CTA)", max_capacity, max_n_segs, max_n_frames, without, optin);
        generic_fn fn = generic_fn_for(plan->bits_in_smem);
        { const int rc = cached_occupancy((const void *)fn, SELECT_THREADS, plan->smem_bytes, &per_sm); if (rc != SMZ_OK) return rc; }
        plan->ws_words_per_cta = plan->bits_in_smem ? 0 : (int64_t)max_n_segs * ((ncell + 31) / 32);
    }
    if (per_sm < 1) per_sm = 1;
    const int g = smz::sm_count() * per_sm;
    plan->grid = n_videos < g ? n_videos : g;
    return SMZ_OK;
}

extern "C" int smz_select_workspace_bytes(int n_videos, int max_n_segs, int max_capacity, int max_n_frames,
                                          int max_seg_frames, int64_t *bytes) {
    SMZ_REQUIRE(bytes != nullptr, "bytes is NULL");
    *bytes = 0;
    if (n_videos <= 0) return SMZ_OK;
    SelectPlan plan;
    int rc = select_plan(n_videos, max_n_segs, max_capacity, max_n_frames, max_seg_frames, &plan);
    if (rc != SMZ_OK) return rc;
    *bytes = plan.ws_bits_bytes() + queue_bytes(n_videos);   // + queue counters, sort counters, fallback list, order
    return SMZ_OK;
}

static int select_launch(const smz_video_desc *desc, int n_videos, const float *scores, const int32_t *picks,
                         const int32_t *cps, const int32_t *nfps, const int32_t *values_in, int method,
                         int max_n_segs, int max_capacity, int max_n_frames, int max_weight, float *seg_mean,
                         int32_t *values, uint8_t *picked, float *summary, uint32_t *mask, int32_t *msum,
                         int32_t *status, void *ws, int64_t ws_bytes, void *stream, const EvalTail *fscore_tail = nullptr,
                         bool *fscore_done = nullptr) {
    if (fscore_done) *fscore_done = false;
    if (n_videos == 0) return SMZ_OK;
    SMZ_REQUIRE(n_videos > 0, "n_videos < 0");
    SMZ_REQUIRE(desc && nfps && picked && status, "NULL pointer (desc, nfps, picked and status are required)");
    SMZ_REQUIRE(method == SMZ_METHOD_KNAPSACK || method == SMZ_METHOD_RANK, "unknown method %d", method);
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    SelectPlan plan;
    rc = select_plan(n_videos, max_n_segs, max_capacity, max_n_frames, max_weight, &plan);
    if (rc != SMZ_OK) return rc;
    const int64_t need = plan.ws_bits_bytes();
    SMZ_REQUIRE(ws != nullptr && ws_bytes >= need + queue_bytes(n_videos), "work buffer too small: need %lld bytes",
                (long long)(need + queue_bytes(n_videos)));
    int *queue = reinterpret_cast<int *>(reinterpret_cast<uint8_t *>(ws) + need);   // layout: see queue_bytes
    int *fallback = queue + kFallback;
    int *order = queue + kQueueInts + n_videos;
    cudaStream_t st = (cudaStream_t)stream;
    SMZ_CUDA_CHECK(cudaMemsetAsync(status, 0, sizeof(int32_t) * (size_t)n_videos, st));
    if (plan.k == 0) {
        SMZ_REQUIRE(mask && msum, "mask and msum outputs are required on the generic path");
        generic_fn fn = generic_fn_for(plan.bits_in_smem);
        fn<<<plan.grid, SELECT_THREADS, plan.smem_bytes, st>>>(
            desc, n_videos, scores, picks, cps, nfps, values_in, method, max_n_segs, max_capacity, max_n_frames,
            seg_mean, values, picked, summary, mask, msum, status, (uint32_t *)ws, plan.ws_words_per_cta);
        SMZ_CUDA_CHECK(cudaGetLastError());
        return SMZ_OK;
    }
    const int32_t *vals = values_in;
    bool fused_pool = false;
    int fused_pool_intervals = 0;
    if (values_in == nullptr) {
        SMZ_REQUIRE(values != nullptr, "values output is required (it feeds the DP kernel)");
        SMZ_REQUIRE(method == SMZ_METHOD_KNAPSACK || seg_mean != nullptr, "seg_mean output is required by method 'rank'");
        const int tiles = (max_n_segs + POOL_THREADS / 8 - 1) / (POOL_THREADS / 8);
        const int64_t frame_bytes = ((int64_t)max_n_frames + 1) / 2 * 4;      // one 16-bit score index per frame
        constexpr int kPoolWords = 12288 - 16;       // 48 KB less the kernel's static shared memory (s_class)
        int max_intervals = max_n_frames + 1 < kPoolWords ? max_n_frames + 1 : kPoolWords;  // staged scores per CTA, with the
        if (max_intervals + 4 * max_n_segs > kPoolWords) max_intervals = kPoolWords - 4 * max_n_segs > 0 ? kPoolWords - 4 * max_n_segs : 0;   // segment lists <= 48 KB
        // 16-bit knapsack plan: the DP kernel pools each video itself (pool_regular_video on the rows region of its shared
        // memory, before the rows are needed) — no pooling kernel in front
        if (tiles > 0 && max_n_segs <= 2048 && !getenv("SMZ_NO_POOL_REGULAR") && method == SMZ_METHOD_KNAPSACK && plan.kw16 > 0 &&
            !getenv("SMZ_NO_FUSED_POOL")) {
            const Dp16Smem L = dp16_layout(plan.kw16, plan.mk16, max_n_segs, plan.front_words);
            int mi = max_intervals;
            if (mi + 4 * max_n_segs > L.wp) mi = L.wp - 4 * max_n_segs;
            if (mi >= 64) { fused_pool = true; fused_pool_intervals = mi; }
        }
        if (fused_pool) {
        } else if (tiles > 0 && max_n_segs <= 2048 && !getenv("SMZ_NO_POOL_REGULAR")) {
            for (int v0 = 0; v0 < n_videos; v0 += 65535) {
                const int nv = n_videos - v0 < 65535 ? n_videos - v0 : 65535;
                pool_regular_kernel<<<nv, POOL_REG_THREADS, ((size_t)max_intervals + 4 * (size_t)max_n_segs) * sizeof(float), st>>>(
                    desc, v0, scores, picks, cps, max_intervals, seg_mean, values, status);
            }
        } else if (tiles > 0 && frame_bytes <= smz::max_smem_optin() - 1024 && max_n_frames < 65535) {
            { int unused = 0; const int rc2 = cached_occupancy((const void *)pool_smem_kernel, POOL_SMEM_THREADS, (int)frame_bytes, &unused); if (rc2 != SMZ_OK) return rc2; }
            pool_smem_kernel<<<n_videos, POOL_SMEM_THREADS, (size_t)frame_bytes, st>>>(desc, 0, scores, picks, cps, seg_mean,
                                                                                     values, status);
        } else {
            for (int v0 = 0; v0 < n_videos && tiles > 0; v0 += 65535) {
                const int nv = n_videos - v0 < 65535 ? n_videos - v0 : 65535;
                pool_kernel<<<dim3(tiles, nv), POOL_THREADS, 0, st>>>(desc, v0, scores, picks, cps, seg_mean, values, status);
            }
        }
        SMZ_CUDA_CHECK(cudaGetLastError());
        vals = values;
    }
    dp_fn fn = dp_fn_for(plan.k);
    // evaluation tail inside the DP kernels: summary vector + mask (+ the F-score when the caller asked for it)
    EvalTail tail = {};
    if (plan.front_words > 0 && mask != nullptr) {
        SMZ_REQUIRE(msum != nullptr, "msum is required with mask");
        if (fscore_tail != nullptr) { tail = *fscore_tail; if (fscore_done) *fscore_done = true; }
        tail.enabled = 1; tail.summary = summary; tail.mask = mask; tail.msum = msum;
    }
    SMZ_CUDA_CHECK(cudaMemsetAsync(queue, 0, sizeof(int) * kQueueInts, st));
    order_count_kernel<<<(n_videos + 255) / 256, 256, 0, st>>>(desc, n_videos, max_n_segs, queue);
    order_fill_kernel<<<(n_videos + 255) / 256, 256, 0, st>>>(desc, n_videos, max_n_segs, queue, order);
    if (method == SMZ_METHOD_KNAPSACK && plan.kw16 > 0) {
        // 16-bit pass over every video, then the 32-bit kernel over whatever it handed back (usually nothing)
        dp16_fn fn16 = dp16_fn_for(plan.kw16, plan.mk16);
        if (fused_pool) {
            tail.pool_scores = scores; tail.pool_picks = picks; tail.pool_cps = cps; tail.pool_max_intervals = fused_pool_intervals;
            tail.pool_seg_mean = seg_mean; tail.pool_values = values; tail.pool_status = status;
        }
        fn16<<<plan.grid16, DP_THREADS, plan.smem16_bytes, st>>>(desc, n_videos, nfps, vals, max_n_segs, picked,
                                                                 (uint32_t *)ws, plan.ws16_words_per_cta, queue, order, fallback,
                                                                 plan.front_words, tail);
        fn<<<plan.grid, DP_THREADS, plan.smem_bytes, st>>>(desc, n_videos, nfps, vals, seg_mean, method, max_n_segs,
                                                          plan.pad_weight, picked, status, (uint32_t *)ws,
                                                          plan.ws_words_per_cta, queue + kQueueHead32, fallback + 1, fallback,
                                                          plan.front_words, tail);
    } else {
        fn<<<plan.grid, DP_THREADS, plan.smem_bytes, st>>>(desc, n_videos, nfps, vals, seg_mean, method, max_n_segs,
                                                          plan.pad_weight, picked, status, (uint32_t *)ws,
                                                          plan.ws_words_per_cta, queue, order, nullptr, plan.front_words, tail);
    }
    SMZ_CUDA_CHECK(cudaGetLastError());
    if (mask != nullptr && !tail.enabled) {
        SMZ_REQUIRE(msum != nullptr, "msum is required with mask");
        const int sm_bytes = (max_n_segs + 1 + (max_n_frames + 31) / 32) * 4;
        SMZ_REQUIRE(sm_bytes <= smz::max_smem_optin(), "summary: %d B of shared memory needed", sm_bytes);
        { int unused = 0; const int rc2 = cached_occupancy((const void *)summary_kernel, SUMMARY_THREADS, sm_bytes, &unused); if (rc2 != SMZ_OK) return rc2; }
        summary_kernel<<<n_videos, SUMMARY_THREADS, sm_bytes, st>>>(desc, 0, nfps, picked, max_n_segs, max_n_frames,
                                                                   summary, mask, msum);
        SMZ_CUDA_CHECK(cudaGetLastError());
    }
    return SMZ_OK;
}

extern "C" int smz_select_shots(const smz_video_desc *desc, int n_videos, const float *scores,
                                const int32_t *picks, const int32_t *cps, const int32_t *nfps, int method,
                                int max_n_segs, int max_capacity, int max_n_frames, int max_seg_frames,
                                float *seg_mean, int32_t *values, uint8_t *picked, float *summary, uint32_t *mask,
                                int32_t *msum, int32_t *status, void *ws, int64_t ws_bytes, void *stream) {
    SMZ_REQUIRE(n_videos == 0 || (scores && picks && cps), "NULL input pointer");
    SMZ_REQUIRE(n_videos == 0 || (mask && msum), "mask and msum outputs are required");
    return select_launch(desc, n_videos, scores, picks, cps, nfps, nullptr, method, max_n_segs, max_capacity,
                         max_n_frames, max_seg_frames, seg_mean, values, picked, summary, mask, msum, status, ws,
                         ws_bytes, stream);
}

extern "C" int smz_knapsack(const smz_video_desc *desc, int n_videos, const int32_t *values, const int32_t *nfps,
                            int max_n_segs, int max_capacity, int max_n_frames, int max_seg_frames,
                            uint8_t *picked, uint32_t *mask, int32_t *msum, int32_t *status, void *ws,
                            int64_t ws_bytes, void *stream) {
    SMZ_REQUIRE(n_videos == 0 || values, "NULL values pointer");
    return select_launch(desc, n_videos, nullptr, nullptr, nullptr, nfps, values, SMZ_METHOD_KNAPSACK, max_n_segs,
                         max_capacity, max_n_frames, max_seg_frames, nullptr, nullptr, picked, nullptr, mask, msum,
                         status, ws, ws_bytes, stream);
}

// ------------------------------------------------------------------------------------------
// smz_eval_batch: shot selection + F-score of a whole batch in one pass
// ------------------------------------------------------------------------------------------
namespace smz {
int launch_fscore_counts(const smz_video_desc *desc, int n_videos, int max_n_frames, const float *user_summary,
                         const uint32_t *mask, int32_t *overlap, int32_t *gsum, cudaStream_t st);
int launch_fscore_bits(const smz_video_desc *desc, int n_videos, const uint32_t *user_bits, const int64_t *bits_off,
                       const uint32_t *mask, int32_t *overlap, int32_t *gsum, cudaStream_t st);
int launch_fscore_final(const smz_video_desc *desc, int n_videos, const int32_t *msum, const int32_t *overlap,
                        const int32_t *gsum, float *f, double *avg_f, double *max_f, cudaStream_t st);
}  // namespace smz

extern "C" int smz_eval_batch(const smz_video_desc *desc, int n_videos, int total_users, const float *scores,
                              const int32_t *picks, const int32_t *cps, const int32_t *nfps, int method,
                              int max_n_segs, int max_capacity, int max_n_frames, int max_seg_frames,
                              const float *user_summary, const uint32_t *user_bits, const int64_t *bits_off,
                              float *seg_mean, int32_t *values, uint8_t *picked, float *summary, uint32_t *mask,
                              int32_t *msum, int32_t *status, int32_t *overlap, int32_t *gsum, float *f, double *avg_f,
                              double *max_f, void *ws, int64_t ws_bytes, void *stream) {
    if (n_videos == 0) return SMZ_OK;
    SMZ_REQUIRE(n_videos > 0 && total_users >= 0, "negative size");
    SMZ_REQUIRE(desc && scores && picks && cps && nfps && mask && msum && picked && status, "NULL pointer");
    SMZ_REQUIRE((user_summary != nullptr) != (user_bits != nullptr), "exactly one of user_summary / user_bits");
    SMZ_REQUIRE(user_bits == nullptr || bits_off != nullptr, "bits_off is required with user_bits");
    SMZ_REQUIRE(overlap && gsum && f, "NULL output pointer");
    cudaStream_t st = (cudaStream_t)stream;
    EvalTail tail = {};
    tail.user = user_summary; tail.user_bits = user_bits; tail.bits_off = bits_off;
    tail.overlap = overlap; tail.gsum = gsum; tail.f = f; tail.avg_f = avg_f; tail.max_f = max_f;
    bool fused = false;
    int rc = select_launch(desc, n_videos, scores, picks, cps, nfps, nullptr, method, max_n_segs, max_capacity, max_n_frames,
                           max_seg_frames, seg_mean, values, picked, summary, mask, msum, status, ws, ws_bytes, stream,
                           &tail, &fused);
    if (rc != SMZ_OK || fused) return rc;
    // rows that do not fit the register-DP plan (very long videos): the stand-alone F-score kernels behind the selection
    if (user_summary != nullptr) {
        SMZ_CUDA_CHECK(cudaMemsetAsync(overlap, 0, sizeof(int32_t) * (size_t)total_users, st));
        SMZ_CUDA_CHECK(cudaMemsetAsync(gsum, 0, sizeof(int32_t) * (size_t)total_users, st));
        rc = smz::launch_fscore_counts(desc, n_videos, max_n_frames, user_summary, mask, overlap, gsum, st);
    } else {
        rc = smz::launch_fscore_bits(desc, n_videos, user_bits, bits_off, mask, overlap, gsum, st);
    }
    if (rc != SMZ_OK) return rc;
    return smz::launch_fscore_final(desc, n_videos, msum, overlap, gsum, f, avg_f, max_f, st);
}
