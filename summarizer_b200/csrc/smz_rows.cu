// Row-wise kernels of the scorers: softmax with VASNet's masks (vasnet.py:121-130), LayerNorm
// (vasnet.py:137,143), regressor head k2 + sigmoid (vasnet.py:144-145), fp32 -> bf16 conversion.
// One warp per row, 128-bit accesses, fp32 arithmetic.  All of them are L2/HBM-bandwidth bound.
#include <cuda_fp16.h>
#include "smz_rows.cuh"

#include <math.h>

namespace {

using smz::GemmProblem;
using smz::kFeat;

constexpr int ROW_WARPS = 8;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&t);
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
// four consecutive bf16 outputs; lo != 0: also the lo plane (x - float(bf16(x))) at p + lo (float32-accurate mode)
__device__ __forceinline__ void st_bf16x4(__nv_bfloat16 *p, int64_t lo, float a, float b, float c, float d) {
    const uint32_t w0 = pack2(a, b), w1 = pack2(c, d);
    *reinterpret_cast<uint2 *>(p) = make_uint2(w0, w1);
    if (lo != 0)
        *reinterpret_cast<uint2 *>(p + lo) = make_uint2(pack2(a - bf_lo(w0), b - bf_hi(w0)), pack2(c - bf_lo(w1), d - bf_hi(w1)));
}

__global__ void cvt_bf16_kernel(const float *__restrict__ x, __nv_bfloat16 *__restrict__ y, int64_t n, int64_t lo) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i + 8 <= n) {
        const float4 a = *reinterpret_cast<const float4 *>(x + i);
        const float4 b = *reinterpret_cast<const float4 *>(x + i + 4);
        st_bf16x4(y + i, lo, a.x, a.y, a.z, a.w);
        st_bf16x4(y + i + 4, lo, b.x, b.y, b.z, b.w);
    } else {
        for (int64_t j = i; j < n; j++) {
            const __nv_bfloat16 h = __float2bfloat16_rn(x[j]);
            y[j] = h;
            if (lo != 0) y[lo + j] = __float2bfloat16_rn(x[j] - __bfloat162float(h));
        }
    }
}

// float32 -> float16 with a range check: |x| > 60000 (or NaN) ORs `bit` into *guard
__global__ void cvt_f16_kernel(const float *__restrict__ x, __half *__restrict__ y, int64_t n, int *__restrict__ guard, int bit) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    float amax = 0.f;
    if (i + 8 <= n) {
        const float4 a = *reinterpret_cast<const float4 *>(x + i);
        const float4 b = *reinterpret_cast<const float4 *>(x + i + 4);
        amax = fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w))),
                     fmaxf(fmaxf(fabsf(b.x), fabsf(b.y)), fmaxf(fabsf(b.z), fabsf(b.w))));
        if (!(a.x == a.x && a.y == a.y && a.z == a.z && a.w == a.w && b.x == b.x && b.y == b.y && b.z == b.z && b.w == b.w)) amax = INFINITY;
        const __half2 h0 = __floats2half2_rn(a.x, a.y), h1 = __floats2half2_rn(a.z, a.w);
        const __half2 h2 = __floats2half2_rn(b.x, b.y), h3 = __floats2half2_rn(b.z, b.w);
        *reinterpret_cast<uint4 *>(y + i) = make_uint4(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1),
                                                       *reinterpret_cast<const uint32_t *>(&h2), *reinterpret_cast<const uint32_t *>(&h3));
    } else {
        for (int64_t j = i; j < n; j++) { y[j] = __float2half_rn(x[j]); amax = (x[j] == x[j]) ? fmaxf(amax, fabsf(x[j])) : INFINITY; }
    }
    if (guard != nullptr && !(amax <= 60000.f)) atomicOr(guard, bit);
}

// up to 8 float32 -> bfloat16 conversions in one launch (the parameter copies of a training step): blockIdx.y = segment
// lo[i] (optional): the segment is split into hi + lo planes (hi = bf16(x), lo = bf16(x - hi)), the operand form of
// the float32-accurate GEMM mode
struct CvtSegments { const float *src[8]; __nv_bfloat16 *dst[8]; __nv_bfloat16 *lo[8]; long long n[8]; };
__global__ void cvt_bf16_segments_kernel(const CvtSegments seg) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const float *x = seg.src[blockIdx.y];
    __nv_bfloat16 *y = seg.dst[blockIdx.y];
    __nv_bfloat16 *yl = seg.lo[blockIdx.y];
    const long long n = seg.n[blockIdx.y];
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += (long long)gridDim.x * blockDim.x * 8) {
        if (i + 8 <= n) {
            const float4 a = *reinterpret_cast<const float4 *>(x + i);
            const float4 b = *reinterpret_cast<const float4 *>(x + i + 4);
            const uint4 h = make_uint4(pack2(a.x, a.y), pack2(a.z, a.w), pack2(b.x, b.y), pack2(b.z, b.w));
            *reinterpret_cast<uint4 *>(y + i) = h;
            if (yl != nullptr)
                *reinterpret_cast<uint4 *>(yl + i) = make_uint4(pack2(a.x - bf_lo(h.x), a.y - bf_hi(h.x)), pack2(a.z - bf_lo(h.y), a.w - bf_hi(h.y)),
                                                                pack2(b.x - bf_lo(h.z), b.y - bf_hi(h.z)), pack2(b.z - bf_lo(h.w), b.w - bf_hi(h.w)));
        } else {
            for (long long j = i; j < n; j++) {
                const __nv_bfloat16 h = __float2bfloat16_rn(x[j]);
                y[j] = h;
                if (yl != nullptr) yl[j] = __float2bfloat16_rn(x[j] - __bfloat162float(h));
            }
        }
    }
}

// vasnet.py:121-127 — masks are applied AFTER scaling: diagonal (ignore_self), then the aperture
// band; inside the band an entry whose square is 0 is masked too (tril(e)*triu(e) == 0 quirk).
__device__ __forceinline__ float mask_logit(float e, int i, int j, int aperture, int ignore_self) {
    if (ignore_self && j == i) e = -INFINITY;
    if (aperture >= 0) {
        int d = i - j;
        d = d < 0 ? -d : d;
        if (d > aperture || e * e == 0.f) e = -INFINITY;
    }
    return e;
}

// One warp per query row.  Fast path (row fits 16 float4 per lane, no leading pad, no dropout): the
// logits are read ONCE into registers (16 independent 128-bit loads in flight per lane), max / exp /
// sum / normalise happen there, P is written once.  Other rows take the three-pass path.
__global__ void __launch_bounds__(ROW_WARPS * 32)
softmax_kernel(const GemmProblem *__restrict__ probs, int n_probs, int total_rows, const float *__restrict__ S,
               __nv_bfloat16 *__restrict__ alpha, __nv_bfloat16 *__restrict__ P, const uint8_t *__restrict__ drop,
               const int64_t *__restrict__ drop_off, int aperture, int ignore_self, const int *__restrict__ gate,
               float *__restrict__ sum_slots, int n_slots, int64_t lop) {
    smz::pdl_trigger();
    smz::pdl_wait();
    if (gate != nullptr && __ldg(gate) == 0) return;
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
    if (r >= total_rows) return;
    if (sum_slots != nullptr)       // P is normalised here: the row-sum slots alpha.V scales by (GEMM_SCALE_STATS) become {1, 0, ...}
        for (int k = lane; k < n_slots; k += 32) sum_slots[((int64_t)r * n_slots + k) * 3] = k == 0 ? 1.f : 0.f;
    int lo = 0, hi = n_probs - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (probs[mid].c_off / probs[mid].ldc <= r) lo = mid; else hi = mid - 1;
    }
    const GemmProblem g = probs[lo];
    const int T = g.M, ld = g.ldc;
    const int i = r - (int)(g.c_off / ld);
    const int64_t off = g.c_off + (int64_t)i * ld;
    const float *s = S + off;
    const bool plain = aperture < 0 && !ignore_self;
    const int lead = g.pad;
    const int W64 = (lead + T + 63) & ~63;

    if (T <= 2048 && lead == 0 && drop == nullptr) {
        constexpr int NV = 16;
        float v[NV][4];
        // all loads first, nothing consumes them inside this loop: 16 independent 128-bit requests in flight per
        // lane (a load-use pair per iteration serialises 16 DRAM round trips per row)
#pragma unroll
        for (int k = 0; k < NV; k++) {
            const int j = lane * 4 + 128 * k;
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j < ld) e = *reinterpret_cast<const float4 *>(s + j);     // [T, ld) is allocated padding
            v[k][0] = e.x; v[k][1] = e.y; v[k][2] = e.z; v[k][3] = e.w;
        }
        float m = -INFINITY;
#pragma unroll
        for (int k = 0; k < NV; k++) {
            const int j = lane * 4 + 128 * k;
            if (j < T) {
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    if (j + t >= T) v[k][t] = -INFINITY;
                    else if (!plain) v[k][t] = mask_logit(v[k][t], i, j + t, aperture, ignore_self);
                    m = fmaxf(m, v[k][t]);
                }
            }
        }
        m = warp_max(m);
        float l = 0.f;
#pragma unroll
        for (int k = 0; k < NV; k++) {
            const int j = lane * 4 + 128 * k;
            if (j < T) {
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    v[k][t] = (j + t < T) ? __expf(v[k][t] - m) : 0.f;   // a fully masked row gives NaN, as torch does
                    l += v[k][t];
                }
            }
        }
        l = warp_sum(l);
        const float inv = 1.f / l;
#pragma unroll
        for (int k = 0; k < NV; k++) {
            const int j = lane * 4 + 128 * k;
            if (j < W64) {
                if (j < T) st_bf16x4(P + off + j, lop, v[k][0] * inv, v[k][1] * inv, v[k][2] * inv, v[k][3] * inv);
                else st_bf16x4(P + off + j, lop, 0.f, 0.f, 0.f, 0.f);
            }
        }
        return;
    }

    float m = -INFINITY;
    for (int j = lane * 4; j < T; j += 128) {
        const float4 e = *reinterpret_cast<const float4 *>(s + j);
        const float v[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
        for (int t = 0; t < 4; t++)
            if (j + t < T) m = fmaxf(m, plain ? v[t] : mask_logit(v[t], i, j + t, aperture, ignore_self));
    }
    m = warp_max(m);
    float l = 0.f;
    for (int j = lane * 4; j < T; j += 128) {
        const float4 e = *reinterpret_cast<const float4 *>(s + j);
        const float v[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
        for (int t = 0; t < 4; t++)
            if (j + t < T) l += __expf((plain ? v[t] : mask_logit(v[t], i, j + t, aperture, ignore_self)) - m);
    }
    l = warp_sum(l);
    const float inv = 1.f / l;
    const uint8_t *keep = drop != nullptr ? drop + drop_off[lo] + (int64_t)i * T : nullptr;
    // P / alpha rows: `lead` zero columns, the T probabilities, zeros up to the next multiple of 64
    for (int jo = lane * 4; jo < W64; jo += 128) {
        float a[4], p[4];
#pragma unroll
        for (int t = 0; t < 4; t++) {
            const int j = jo + t - lead;
            a[t] = 0.f;
            if (j >= 0 && j < T) a[t] = __expf((plain ? s[j] : mask_logit(s[j], i, j, aperture, ignore_self)) - m) * inv;
            p[t] = a[t];
            if (keep != nullptr && j >= 0 && j < T) p[t] = keep[j] ? 2.f * a[t] : 0.f;   // nn.Dropout(0.5), vasnet.py:130
        }
        if (alpha != nullptr && alpha != P) st_bf16x4(alpha + off + jo, lop, a[0], a[1], a[2], a[3]);
        st_bf16x4(P + off + jo, lop, p[0], p[1], p[2], p[3]);
    }
}

// torch.nn.LayerNorm(1024, eps): biased variance, eps inside the square root.
__global__ void __launch_bounds__(ROW_WARPS * 32)
layernorm_kernel(const float *__restrict__ y, const uint8_t *__restrict__ keep, const float *__restrict__ g,
                 const float *__restrict__ b, float eps, int rows, __nv_bfloat16 *__restrict__ yn,
                 float *__restrict__ mean, float *__restrict__ rstd, int64_t lo, float *__restrict__ y32,
                 const void *__restrict__ res, int res_bf16) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
    if (r >= rows) return;
    const float *row = y + (int64_t)r * kFeat;
    float x[32];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int c = lane * 4 + 128 * k;
        const float4 v = *reinterpret_cast<const float4 *>(row + c);
        x[4 * k] = v.x; x[4 * k + 1] = v.y; x[4 * k + 2] = v.z; x[4 * k + 3] = v.w;
        if (keep != nullptr) {
            const uchar4 kp = *reinterpret_cast<const uchar4 *>(keep + (int64_t)r * kFeat + c);
            x[4 * k] = kp.x ? 2.f * x[4 * k] : 0.f; x[4 * k + 1] = kp.y ? 2.f * x[4 * k + 1] : 0.f;
            x[4 * k + 2] = kp.z ? 2.f * x[4 * k + 2] : 0.f; x[4 * k + 3] = kp.w ? 2.f * x[4 * k + 3] : 0.f;
        }
        sum += (x[4 * k] + x[4 * k + 1]) + (x[4 * k + 2] + x[4 * k + 3]);
    }
    const float mu = warp_sum(sum) * (1.f / kFeat);
    float var = 0.f;
#pragma unroll
    for (int k = 0; k < 32; k++) { const float d = x[k] - mu; var += d * d; }
    const float rs = rsqrtf(warp_sum(var) * (1.f / kFeat) + eps);
    if (lane == 0) {
        if (mean != nullptr) mean[r] = mu;
        if (rstd != nullptr) rstd[r] = rs;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int c = lane * 4 + 128 * k;
        const float4 gg = *reinterpret_cast<const float4 *>(g + c);
        const float4 bb = *reinterpret_cast<const float4 *>(b + c);
        float o0 = (x[4 * k] - mu) * rs * gg.x + bb.x, o1 = (x[4 * k + 1] - mu) * rs * gg.y + bb.y;
        float o2 = (x[4 * k + 2] - mu) * rs * gg.z + bb.z, o3 = (x[4 * k + 3] - mu) * rs * gg.w + bb.w;
        if (res != nullptr) {
            const int64_t ro = (int64_t)r * kFeat + c;
            if (res_bf16) {
                const __nv_bfloat16 *rb = reinterpret_cast<const __nv_bfloat16 *>(res) + ro;
                o0 += __bfloat162float(rb[0]); o1 += __bfloat162float(rb[1]); o2 += __bfloat162float(rb[2]); o3 += __bfloat162float(rb[3]);
            } else {
                const float4 rr = *reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(res) + ro);
                o0 += rr.x; o1 += rr.y; o2 += rr.z; o3 += rr.w;
            }
        }
        if (yn != nullptr) st_bf16x4(yn + (int64_t)r * kFeat + c, lo, o0, o1, o2, o3);
        if (y32 != nullptr) *reinterpret_cast<float4 *>(y32 + (int64_t)r * kFeat + c) = make_float4(o0, o1, o2, o3);
    }
}

__global__ void __launch_bounds__(ROW_WARPS * 32)
head_kernel(const float *__restrict__ h, const uint8_t *__restrict__ keep, const float *__restrict__ g,
            const float *__restrict__ b, float eps, const float *__restrict__ w2, const float *__restrict__ b2,
            int rows, float *__restrict__ scores, float *__restrict__ mean, float *__restrict__ rstd) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
    if (r >= rows) return;
    const float *row = h + (int64_t)r * kFeat;
    float x[32];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int c = lane * 4 + 128 * k;
        const float4 v = *reinterpret_cast<const float4 *>(row + c);
        x[4 * k] = v.x; x[4 * k + 1] = v.y; x[4 * k + 2] = v.z; x[4 * k + 3] = v.w;
        if (keep != nullptr) {
            const uchar4 kp = *reinterpret_cast<const uchar4 *>(keep + (int64_t)r * kFeat + c);
            x[4 * k] = kp.x ? 2.f * x[4 * k] : 0.f; x[4 * k + 1] = kp.y ? 2.f * x[4 * k + 1] : 0.f;
            x[4 * k + 2] = kp.z ? 2.f * x[4 * k + 2] : 0.f; x[4 * k + 3] = kp.w ? 2.f * x[4 * k + 3] : 0.f;
        }
        sum += (x[4 * k] + x[4 * k + 1]) + (x[4 * k + 2] + x[4 * k + 3]);
    }
    const float mu = warp_sum(sum) * (1.f / kFeat);
    float var = 0.f;
#pragma unroll
    for (int k = 0; k < 32; k++) { const float d = x[k] - mu; var += d * d; }
    const float rs = rsqrtf(warp_sum(var) * (1.f / kFeat) + eps);
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int c = lane * 4 + 128 * k;
        const float4 gg = *reinterpret_cast<const float4 *>(g + c);
        const float4 bb = *reinterpret_cast<const float4 *>(b + c);
        const float4 ww = *reinterpret_cast<const float4 *>(w2 + c);
        dot += ((x[4 * k] - mu) * rs * gg.x + bb.x) * ww.x + ((x[4 * k + 1] - mu) * rs * gg.y + bb.y) * ww.y +
               ((x[4 * k + 2] - mu) * rs * gg.z + bb.z) * ww.z + ((x[4 * k + 3] - mu) * rs * gg.w + bb.w) * ww.w;
    }
    dot = warp_sum(dot);
    if (lane == 0) {
        const float z = dot + __ldg(b2);
        scores[r] = 1.f / (1.f + __expf(-z));
        if (mean != nullptr) mean[r] = mu;
        if (rstd != nullptr) rstd[r] = rs;
    }
}


__global__ void head_from_stats_kernel(const float *__restrict__ stats, int slots, const float *__restrict__ c, float eps,
                                       int rows, float *__restrict__ scores) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float s1 = 0.f, s2 = 0.f, s3 = 0.f;
    for (int k = 0; k < slots; k++) {                         // fixed order: bitwise reproducible
        const float *p = stats + ((int64_t)r * slots + k) * 3;
        s1 += p[0]; s2 += p[1]; s3 += p[2];
    }
    const float mu = s1 * (1.f / kFeat);
    const float var = fmaxf(s2 * (1.f / kFeat) - mu * mu, 0.f);
    const float rs = rsqrtf(var + eps);
    const float z = rs * (s3 - mu * __ldg(c)) + __ldg(c + 1);
    scores[r] = 1.f / (1.f + __expf(-z));
}

// ---- backward row kernels -------------------------------------------------------------------------
// Column sums over rows (bias / LayerNorm-affine / k2 gradients) are accumulated per CTA in shared
// memory and flushed with one float atomic per column and CTA.
template <int NACC>
struct ColAcc {
    float *acc;   // [NACC][kFeat] in shared memory
    __device__ __forceinline__ void zero() {
        for (int i = threadIdx.x; i < NACC * kFeat; i += blockDim.x) acc[i] = 0.f;
        __syncthreads();
    }
    __device__ __forceinline__ void add(int a, int c, float v) { atomicAdd(acc + a * kFeat + c, v); }
    __device__ __forceinline__ void flush(int a, float *dst) {
        if (dst == nullptr) return;
        for (int c = threadIdx.x; c < kFeat; c += blockDim.x) atomicAdd(dst + c, acc[a * kFeat + c]);
    }
};

__global__ void __launch_bounds__(ROW_WARPS * 32)
head_bwd_kernel(const float *__restrict__ h, const uint8_t *__restrict__ keep, const float *__restrict__ g,
                const float *__restrict__ b, const float *__restrict__ w2, const float *__restrict__ mean,
                const float *__restrict__ rstd, const float *__restrict__ scores, const float *__restrict__ dscores,
                int rows, __nv_bfloat16 *__restrict__ dh, float *__restrict__ d_w2, float *__restrict__ d_b2,
                float *__restrict__ d_g, float *__restrict__ d_b, float *__restrict__ d_b1, int64_t lo) {
    extern __shared__ float s_acc[];
    ColAcc<4> A{s_acc};
    smz::pdl_trigger();
    A.zero();
    smz::pdl_wait();
    const int lane = threadIdx.x & 31;
    float db2 = 0.f;
    for (int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5); r < rows; r += gridDim.x * ROW_WARPS) {
        const float *row = h + (int64_t)r * kFeat;
        float xh[32], dx[32];
        uint32_t live = 0u;      // bit k: the unit passes gradient (ReLU active and kept by dropout)
        const float mu = mean[r], rs = rstd[r];
        const float sc = scores[r];
        const float dz = dscores[r] * sc * (1.f - sc);            // sigmoid'
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int c = lane * 4 + 128 * k;
            const float4 v = *reinterpret_cast<const float4 *>(row + c);
            float x[4] = {v.x, v.y, v.z, v.w};
            uint32_t kb = 0xfu;
            if (keep != nullptr) {
                const uchar4 kp = *reinterpret_cast<const uchar4 *>(keep + (int64_t)r * kFeat + c);
                kb = (kp.x ? 1u : 0u) | (kp.y ? 2u : 0u) | (kp.z ? 4u : 0u) | (kp.w ? 8u : 0u);
            }
            const float4 gg = *reinterpret_cast<const float4 *>(g + c);
            const float4 bb = *reinterpret_cast<const float4 *>(b + c);
            const float4 ww = *reinterpret_cast<const float4 *>(w2 + c);
            const float gv[4] = {gg.x, gg.y, gg.z, gg.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w}, wv[4] = {ww.x, ww.y, ww.z, ww.w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const bool kept = (kb >> t) & 1u;
                if (x[t] > 0.f && kept) live |= 1u << (4 * k + t);
                const float hd = keep != nullptr ? (kept ? 2.f * x[t] : 0.f) : x[t];
                const float xhat = (hd - mu) * rs;
                const float ln = xhat * gv[t] + bv[t];
                const float dln = dz * wv[t];
                A.add(0, c + t, dz * ln);        // d k2.weight
                A.add(1, c + t, dln * xhat);     // d layer_norm.weight
                A.add(2, c + t, dln);            // d layer_norm.bias
                const float dxh = dln * gv[t];
                xh[4 * k + t] = xhat; dx[4 * k + t] = dxh;
                s1 += dxh; s2 += dxh * xhat;
            }
        }
        const float c1 = warp_sum(s1) * (1.f / kFeat), c2 = warp_sum(s2) * (1.f / kFeat);
        const float dscale = keep != nullptr ? 2.f : 1.f;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int c = lane * 4 + 128 * k;
            float o[4];
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const float d = rs * (dx[4 * k + t] - c1 - xh[4 * k + t] * c2) * dscale;
                o[t] = ((live >> (4 * k + t)) & 1u) ? d : 0.f;
                A.add(3, c + t, o[t]);           // d k1.bias
            }
            st_bf16x4(dh + (int64_t)r * kFeat + c, lo, o[0], o[1], o[2], o[3]);
        }
        if (lane == 0) db2 += dz;
    }
    __syncthreads();
    A.flush(0, d_w2); A.flush(1, d_g); A.flush(2, d_b); A.flush(3, d_b1);
    if (lane == 0 && db2 != 0.f && d_b2 != nullptr) atomicAdd(d_b2, db2);
}

__global__ void __launch_bounds__(ROW_WARPS * 32)
layernorm_bwd_kernel(const float *__restrict__ dyn, const float *__restrict__ y, const uint8_t *__restrict__ keep,
                     const float *__restrict__ g, const float *__restrict__ mean, const float *__restrict__ rstd,
                     int rows, __nv_bfloat16 *__restrict__ dy, float *__restrict__ dy_f32, float *__restrict__ d_g,
                     float *__restrict__ d_b, int64_t lo) {
    extern __shared__ float s_acc[];
    ColAcc<2> A{s_acc};
    smz::pdl_trigger();
    A.zero();
    smz::pdl_wait();
    const int lane = threadIdx.x & 31;
    for (int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5); r < rows; r += gridDim.x * ROW_WARPS) {
        float xh[32], dx[32];
        uint32_t kept_bits = 0xffffffffu;
        const float mu = mean[r], rs = rstd[r];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int c = lane * 4 + 128 * k;
            const float4 v = *reinterpret_cast<const float4 *>(y + (int64_t)r * kFeat + c);
            const float4 d = *reinterpret_cast<const float4 *>(dyn + (int64_t)r * kFeat + c);
            const float4 gg = *reinterpret_cast<const float4 *>(g + c);
            float x[4] = {v.x, v.y, v.z, v.w};
            const float dv[4] = {d.x, d.y, d.z, d.w}, gv[4] = {gg.x, gg.y, gg.z, gg.w};
            if (keep != nullptr) {
                const uchar4 kp = *reinterpret_cast<const uchar4 *>(keep + (int64_t)r * kFeat + c);
                const uint32_t kb = (kp.x ? 1u : 0u) | (kp.y ? 2u : 0u) | (kp.z ? 4u : 0u) | (kp.w ? 8u : 0u);
                kept_bits = (kept_bits & ~(0xfu << (4 * k))) | (kb << (4 * k));
#pragma unroll
                for (int t = 0; t < 4; t++) x[t] = ((kb >> t) & 1u) ? 2.f * x[t] : 0.f;
            }
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const float xhat = (x[t] - mu) * rs;
                A.add(0, c + t, dv[t] * xhat);
                A.add(1, c + t, dv[t]);
                const float dxh = dv[t] * gv[t];
                xh[4 * k + t] = xhat; dx[4 * k + t] = dxh;
                s1 += dxh; s2 += dxh * xhat;
            }
        }
        const float c1 = warp_sum(s1) * (1.f / kFeat), c2 = warp_sum(s2) * (1.f / kFeat);
        const float dscale = keep != nullptr ? 2.f : 1.f;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int c = lane * 4 + 128 * k;
            float o[4];
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const float d = rs * (dx[4 * k + t] - c1 - xh[4 * k + t] * c2) * dscale;
                o[t] = ((kept_bits >> (4 * k + t)) & 1u) ? d : 0.f;
            }
            st_bf16x4(dy + (int64_t)r * kFeat + c, lo, o[0], o[1], o[2], o[3]);
            if (dy_f32 != nullptr)
                *reinterpret_cast<float4 *>(dy_f32 + (int64_t)r * kFeat + c) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
    __syncthreads();
    A.flush(0, d_g); A.flush(1, d_b);
}

__global__ void __launch_bounds__(ROW_WARPS * 32)
softmax_bwd_kernel(const float *__restrict__ dP, const __nv_bfloat16 *__restrict__ alpha,
                   const uint8_t *__restrict__ keep, int T, int ld, __nv_bfloat16 *__restrict__ dS, int64_t lo) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
    if (i >= T) return;
    const float *dp = dP + (int64_t)i * ld;
    const __nv_bfloat16 *al = alpha + (int64_t)i * ld;
    const uint8_t *kp = keep != nullptr ? keep + (int64_t)i * T : nullptr;
    float dot = 0.f;
    for (int j = lane; j < T; j += 32) {
        float da = dp[j];
        if (kp != nullptr) da = kp[j] ? 2.f * da : 0.f;
        dot += da * (__bfloat162float(al[j]) + (lo != 0 ? __bfloat162float(al[lo + j]) : 0.f));
    }
    dot = warp_sum(dot);
    const int W64 = (T + 63) & ~63;
    for (int j = lane; j < W64; j += 32) {
        float o = 0.f;
        if (j < T) {
            float da = dp[j];
            if (kp != nullptr) da = kp[j] ? 2.f * da : 0.f;
            o = (__bfloat162float(al[j]) + (lo != 0 ? __bfloat162float(al[lo + j]) : 0.f)) * (da - dot);
        }
        const __nv_bfloat16 hi = __float2bfloat16_rn(o);
        dS[(int64_t)i * ld + j] = hi;
        if (lo != 0) dS[lo + (int64_t)i * ld + j] = __float2bfloat16_rn(o - __bfloat162float(hi));
    }
}

}  // namespace

namespace smz {

int launch_head_from_stats(const float *stats, int slots, const float *c, float eps, int rows, float *scores,
                           cudaStream_t st) {
    if (rows <= 0) return SMZ_OK;
    SMZ_CUDA_CHECK(launch_pdl(head_from_stats_kernel, dim3((rows + 255) / 256), dim3(256), 0, st, stats, slots, c, eps, rows, scores));
    return SMZ_OK;
}

int launch_head_bwd(const float *h, const uint8_t *keep, const float *g, const float *b, const float *w2,
                    const float *mean, const float *rstd, const float *scores, const float *dscores, int rows,
                    __nv_bfloat16 *dh, float *d_w2, float *d_b2, float *d_g, float *d_b, float *d_b1, cudaStream_t st,
                    int64_t lo) {
    if (rows <= 0) return SMZ_OK;
    int grid = (rows + ROW_WARPS - 1) / ROW_WARPS;
    if (grid > 2 * sm_count()) grid = 2 * sm_count();
    SMZ_CUDA_CHECK(launch_pdl(head_bwd_kernel, dim3(grid), dim3(ROW_WARPS * 32), 4 * kFeat * sizeof(float), st, h, keep, g, b, w2, mean,
                             rstd, scores, dscores, rows, dh, d_w2, d_b2, d_g, d_b, d_b1, lo));
    return SMZ_OK;
}

int launch_layernorm_bwd(const float *dyn, const float *y, const uint8_t *keep, const float *g, const float *mean,
                         const float *rstd, int rows, __nv_bfloat16 *dy, float *dy_f32, float *d_g, float *d_b,
                         cudaStream_t st, int64_t lo) {
    if (rows <= 0) return SMZ_OK;
    int grid = (rows + ROW_WARPS - 1) / ROW_WARPS;
    if (grid > 2 * sm_count()) grid = 2 * sm_count();
    SMZ_CUDA_CHECK(launch_pdl(layernorm_bwd_kernel, dim3(grid), dim3(ROW_WARPS * 32), 2 * kFeat * sizeof(float), st, dyn, y, keep, g,
                             mean, rstd, rows, dy, dy_f32, d_g, d_b, lo));
    return SMZ_OK;
}

int launch_softmax_bwd(const float *dP, const __nv_bfloat16 *alpha, const uint8_t *keep, int T, int ld,
                       __nv_bfloat16 *dS, cudaStream_t st, int64_t lo) {
    if (T <= 0) return SMZ_OK;
    SMZ_CUDA_CHECK(launch_pdl(softmax_bwd_kernel, dim3((T + ROW_WARPS - 1) / ROW_WARPS), dim3(ROW_WARPS * 32), 0, st, dP, alpha, keep, T, ld,
                             dS, lo));
    return SMZ_OK;
}

}  // namespace smz

// float32 -> bfloat16 copies of up to 8 tensors in ONE launch: src[i] (n[i] floats, 16-byte aligned) -> dst[i].  What a
// training step uses to refresh the bf16 weight copies (replaces one torch cast kernel per parameter).
static int cvt_segments(const float *const *src, void *const *dst, void *const *lo, const int64_t *n, int count, void *stream) {
    SMZ_REQUIRE(src && dst && n && count >= 1 && count <= 8, "cvt_bf16_multi: 1..8 segments");
    CvtSegments seg = {};
    long long most = 0;
    for (int i = 0; i < count; i++) {
        SMZ_REQUIRE(src[i] && dst[i] && n[i] >= 0 && (lo == nullptr || lo[i]), "cvt_bf16_multi: bad segment %d", i);
        SMZ_REQUIRE(((uintptr_t)src[i] & 15) == 0 && ((uintptr_t)dst[i] & 15) == 0 && (lo == nullptr || ((uintptr_t)lo[i] & 15) == 0),
                    "cvt_bf16_multi: segment %d is not 16-byte aligned", i);
        seg.src[i] = src[i]; seg.dst[i] = reinterpret_cast<__nv_bfloat16 *>(dst[i]); seg.n[i] = n[i];
        seg.lo[i] = lo != nullptr ? reinterpret_cast<__nv_bfloat16 *>(lo[i]) : nullptr;
        most = n[i] > most ? n[i] : most;
    }
    if (most == 0) return SMZ_OK;
    long long blocks = (most + 8 * 256 - 1) / (8 * 256);
    if (blocks > 2048) blocks = 2048;
    SMZ_CUDA_CHECK(smz::launch_pdl(cvt_bf16_segments_kernel, dim3((unsigned)blocks, count), dim3(256), 0, (cudaStream_t)stream, seg));
    return SMZ_OK;
}

extern "C" int smz_cvt_bf16_multi(const float *const *src, void *const *dst, const int64_t *n, int count, void *stream) {
    return cvt_segments(src, dst, nullptr, n, count, stream);
}

// The same with hi + lo planes: hi[i] = bf16(src[i]), lo[i] = bf16(src[i] - hi[i]) — the operand form of the
// float32-accurate (split-bf16) GEMM mode.
extern "C" int smz_split_bf16_multi(const float *const *src, void *const *hi, void *const *lo, const int64_t *n, int count,
                                    void *stream) {
    SMZ_REQUIRE(lo != nullptr, "split_bf16_multi: lo is NULL");
    return cvt_segments(src, hi, lo, n, count, stream);
}

namespace smz {

int launch_cvt_bf16(const float *x, __nv_bfloat16 *y, int64_t n, cudaStream_t st, int64_t lo) {
    if (n <= 0) return SMZ_OK;
    const int64_t blocks = (n + 8 * 256 - 1) / (8 * 256);
    SMZ_CUDA_CHECK(launch_pdl(cvt_bf16_kernel, dim3((unsigned)blocks), dim3(256), 0, st, x, y, n, lo));
    return SMZ_OK;
}

int launch_cvt_f16(const float *x, void *y, int64_t n, int *guard, int bit, cudaStream_t st) {
    if (n <= 0) return SMZ_OK;
    const int64_t blocks = (n + 8 * 256 - 1) / (8 * 256);
    SMZ_CUDA_CHECK(launch_pdl(cvt_f16_kernel, dim3((unsigned)blocks), dim3(256), 0, st, x, reinterpret_cast<__half *>(y), n, guard, bit));
    return SMZ_OK;
}

int launch_softmax(const GemmProblem *d_probs, int n_probs, int total_rows, const float *S, __nv_bfloat16 *alpha,
                   __nv_bfloat16 *P, const uint8_t *drop, const int64_t *d_drop_off, int aperture, int ignore_self,
                   cudaStream_t st, const int *gate, float *sum_slots, int n_slots, int64_t lo) {
    if (total_rows <= 0) return SMZ_OK;
    SMZ_CUDA_CHECK(launch_pdl(softmax_kernel, dim3((total_rows + ROW_WARPS - 1) / ROW_WARPS), dim3(ROW_WARPS * 32), 0, st, d_probs, n_probs,
                             total_rows, S, alpha, P, drop, d_drop_off, aperture, ignore_self, gate, sum_slots, n_slots, lo));
    return SMZ_OK;
}

int launch_layernorm(const float *y, const uint8_t *keep, const float *g, const float *b, float eps, int rows,
                     __nv_bfloat16 *yn, float *mean, float *rstd, cudaStream_t st, int64_t lo, float *y32, const void *res,
                     bool res_bf16) {
    if (rows <= 0) return SMZ_OK;
    SMZ_CUDA_CHECK(launch_pdl(layernorm_kernel, dim3((rows + ROW_WARPS - 1) / ROW_WARPS), dim3(ROW_WARPS * 32), 0, st, y, keep, g, b, eps, rows,
                             yn, mean, rstd, lo, y32, res, (int)res_bf16));
    return SMZ_OK;
}

int launch_head(const float *h, const uint8_t *keep, const float *g, const float *b, float eps,
                const float *w2, const float *b2, int rows, float *scores, float *mean, float *rstd,
                cudaStream_t st) {
    if (rows <= 0) return SMZ_OK;
    SMZ_CUDA_CHECK(launch_pdl(head_kernel, dim3((rows + ROW_WARPS - 1) / ROW_WARPS), dim3(ROW_WARPS * 32), 0, st, h, keep, g, b, eps, w2, b2,
                             rows, scores, mean, rstd));
    return SMZ_OK;
}

}  // namespace smz

// ---------------------------------------------------------------------------------------------------
// Keep masks of nn.Dropout(0.5) (vasnet.py:130,136,142): n bytes, 1 = keep with probability 1/2, one Philox bit per
// byte.  `state` = three device uint64 words {seed, call number, 0}: the call number is advanced on the device by the
// last CTA to finish, so a captured training step draws fresh masks at every graph replay and no host-side generator
// (a process-wide object that cannot be drawn from while another thread captures a graph) is involved.
namespace {

__global__ void __launch_bounds__(256) keep_mask_kernel(unsigned long long *__restrict__ state, uint8_t *__restrict__ out, long long n) {
    smz::pdl_trigger();
    smz::pdl_wait();
    const unsigned long long seed = state[0], call = state[1];
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const long long n_blk = (n + 127) / 128;                   // 128 mask bytes per Philox call
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < n_blk; b += (long long)gridDim.x * blockDim.x) {
        const uint4 r = smz::philox4x32_10(make_uint4((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)call, (uint32_t)(call >> 32)), key);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
        uint8_t *dst = out + b * 128;
        if (b * 128 + 128 <= n && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
            for (int q = 0; q < 8; q++) {                      // 16 bits -> 16 bytes
                const uint32_t bits = w[q >> 1] >> ((q & 1) * 16);
                uint32_t o[4];
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    const uint32_t nib = (bits >> (4 * t)) & 0xfu;
                    o[t] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
                }
                reinterpret_cast<uint4 *>(dst)[q] = make_uint4(o[0], o[1], o[2], o[3]);
            }
        } else {
            for (int i = 0; i < 128 && b * 128 + i < n; i++) dst[i] = (w[i >> 5] >> (i & 31)) & 1u;
        }
    }
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned int *ticket = reinterpret_cast<unsigned int *>(state + 2);
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
        if (last) { *ticket = 0u; state[1] = call + 1ull; }    // every CTA has read the call number by now
    }
}

}  // namespace

extern "C" int smz_dropout_keep_masks(uint64_t *state, uint8_t *out, int64_t n, void *stream) {
    SMZ_REQUIRE(state && out && n >= 0, "dropout_keep_masks: bad argument");
    if (n == 0) return SMZ_OK;
    int rc = smz_device_check();
    if (rc != SMZ_OK) return rc;
    long long blocks = ((n + 127) / 128 + 255) / 256;
    if (blocks > 4 * smz::sm_count()) blocks = 4 * smz::sm_count();
    SMZ_CUDA_CHECK(smz::launch_pdl(keep_mask_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream,
                                   reinterpret_cast<unsigned long long *>(state), out, (long long)n));
    return SMZ_OK;
}
