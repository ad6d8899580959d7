// sm_100a device primitives used by the dense kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM allocation, UMMA issue/commit, TMEM loads) — thin inline-PTX wrappers, nothing else.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace smztc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier --------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) __trap();   // ~2 s at 1.9 GHz
    }
}

// ---- TMA -------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load: c0 = coordinate along the contiguous dimension, c1 = row.
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *m, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// ---- clusters / CTA pairs ----------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    __syncwarp();
    asm volatile("barrier.cluster.arrive.release;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t *bar, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
// PAIR: the load lands in THIS CTA's shared memory but completes its bytes on the LEADER CTA's barrier
// (shared::cluster address with the peer bit cleared), on which the pair's single MMA thread waits.
template <bool PAIR>
__device__ __forceinline__ void tma_load(void *smem_dst, const CUtensorMap *m, uint64_t *bar, int c0, int c1) {
    if (PAIR) {
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
            ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
            : "memory");
    } else {
        tma_load_2d(smem_dst, m, bar, c0, c1);
    }
}

// ---- tcgen05 ---------------------------------------------------------------------------------
// one lane of the (converged) warp: the tcgen05 / TMA issue idiom — the WHOLE warp runs the role's loop, so every loop
// variable is warp-uniform and lives in the uniform datapath; only the issue itself is predicated on the elected lane
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// whole warp; writes the TMEM base address to *smem_dst
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(NCOLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}

template <int NCOLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t *smem_dst) {     // same warp index in both CTAs of the pair
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(NCOLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}

// Shared-memory matrix descriptor, K-major operand tile stored as rows of 128 bytes with the
// 128-byte swizzle (what a TMA box of 64 bf16 x rows with CU_TENSOR_MAP_SWIZZLE_128B writes):
//   bits [0,14)  start address >> 4      bits [16,30) leading byte offset >> 4 (unused here)
//   bits [32,46) stride byte offset >> 4 = 1024 B between 8-row groups
//   bits [46,48) descriptor version = 1 (sm_100)     bits [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
    const uint64_t lo = (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    const uint64_t hi = (uint64_t)(1024u >> 4) | (1ull << 14) | (2ull << 29);
    return lo | (hi << 32);
}

// MN-major operand tile: 64x64 boxes ([64 k-rows][64 m/n] = 128-byte rows, 128-byte swizzle), one box
// per 64 m/n.  LBO = 8192 B (next 64-element m/n group = next box), SBO = 1024 B (next 8 k-rows).
__device__ __forceinline__ uint64_t make_mnmajor_sw128_desc(uint32_t smem_addr) {
    const uint64_t lo = (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)(8192u >> 4) << 16);
    const uint64_t hi = (uint64_t)(1024u >> 4) | (1ull << 14) | (2ull << 29);
    return lo | (hi << 32);
}

// Instruction descriptor, kind::f16, bf16 x bf16 -> fp32, both operands K-major.
//   [4,6) D format 1 = f32   [7,10) A format 1 = bf16   [10,13) B format 1 = bf16
//   [15] A major 0 = K   [16] B major 0 = K   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; one thread issues on behalf of the CTA (PAIR: of both CTAs, M = 256)
template <bool PAIR>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if (PAIR) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    }
}
// arrives on the mbarrier once every MMA issued so far by this thread has completed (PAIR: on the barrier at
// this offset in BOTH CTAs)
template <bool PAIR>
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    if (PAIR) {
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
    } else {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
    }
}

// TMEM -> registers: lane i of the warp reads TMEM lane (taddr.lane + i), 32 consecutive columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM, the inverse of tmem_ld32
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
          "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
          "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// generic-proxy shared-memory writes (st.shared) made visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&t);
}

__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    __half2 t = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&t);
}

}  // namespace smztc
