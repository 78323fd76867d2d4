// tc.cuh -- every PTX wrapper of the tcgen05 kernels of net.cu (inference) and train.cu (training): mbarrier (CTA and cluster scope),
// TMA (single CTA, multicast, CTA pair) and plain bulk copies, tcgen05 alloc / mma / commit / ld, cluster and distributed-shared-memory
// access, proxy fences, and the encodings of the shared-memory matrix and instruction descriptors.  Each hardware encoding is written
// here once (established on the hardware: scripts/desc_probe.cu, scripts/mma_rate_probe.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace szb {

constexpr long long TC_TIMEOUT_CYCLES = 4000000000ll;          // ~2 s: a stuck pipeline flags an error instead of hanging the GPU
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;                     // shared::cluster address of the same offset in the pair's even CTA

// =================================================================================================
// descriptor encodings
// =================================================================================================
// Shared-memory matrix descriptor, K-major, 128-byte swizzle, as (lo, hi) 32-bit halves.  lo: start address >> 4 and LBO = 1 (unused
// for swizzled K-major); hi: SBO (distance between 8-row groups) >> 4, version 1, layout type 2 (SWIZZLE_128B).
constexpr uint32_t DESC_LO_FLAGS = 1u << 16;
__host__ __device__ constexpr uint32_t desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29); }
// Instruction descriptor of tcgen05.mma.kind::f16: bf16 x bf16 -> fp32, M x N, A / B K-major (false) or MN-major (true).  N = 0 gives
// the base word a kernel ORs its run-time N into.
__host__ __device__ constexpr uint32_t idesc_bf16(int m, int n, bool a_mn = false, bool b_mn = false) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(m >> 4) << 24);
}

// =================================================================================================
// PTX wrappers
// =================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major SWIZZLE_128B descriptor of the operand at `addr` (see desc_hi)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t sbo_bytes = 1024) {
    return ((uint64_t)desc_hi(sbo_bytes) << 32) | (uint64_t)(((addr >> 4) & 0x3FFF) | DESC_LO_FLAGS);
}
// absolute-address 128-byte swizzle (what TMA and tcgen05.mma apply): address bits 4..6 ^= bits 7..9
__device__ __forceinline__ uint32_t swz128(uint32_t addr) { return addr ^ (((addr >> 7) & 7u) << 4); }

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// makes the barriers initialised above visible to the async proxy and to the other CTAs of the cluster
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// one arrival on the barrier at this offset in the pair's even (leader) CTA
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_MASK) : "memory");
}
// one arrival, release at cluster scope, on a barrier of any CTA of the cluster (address from mapa_u32)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t remote_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: returns false (and raises the flag) instead of spinning forever
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, volatile int* abort_flag) {
    if (mbar_try_wait(bar, parity)) return true;
    const long long t0 = clock64();
    for (;;) {
        if (mbar_try_wait(bar, parity)) return true;
        if (*abort_flag) return false;
        if (clock64() - t0 > TC_TIMEOUT_CYCLES) { *abort_flag = 1; return false; }
    }
}
// the same with cluster-scope acquire (the arrivals come from other CTAs after their distributed-shared-memory stores)
__device__ __forceinline__ bool mbar_wait_cluster(uint32_t bar, uint32_t parity, volatile int* abort_flag) {
    if (mbar_try_wait_cluster(bar, parity)) return true;
    const long long t0 = clock64();
    for (;;) {
        if (mbar_try_wait_cluster(bar, parity)) return true;
        if (*abort_flag) return false;
        if (clock64() - t0 > TC_TIMEOUT_CYCLES) { *abort_flag = 1; return false; }
    }
}
// all 32 lanes wait; the result is warp-uniform
__device__ __forceinline__ bool warp_mbar_wait(uint32_t bar, uint32_t parity, volatile int* abort_flag) {
    return __all_sync(0xFFFFFFFFu, mbar_wait(bar, parity, abort_flag));
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// ---- synchronisation and fences ----------------------------------------------------------------
// named barrier ID among COUNT threads (whole warps)
template <int ID, int COUNT>
__device__ __forceinline__ void named_bar_sync() { asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(COUNT) : "memory"); }
// generic-proxy accesses before it -> async-proxy (TMA, tcgen05) accesses after it: shared memory / global memory
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void red_release_gpu_add(int32_t* p, int v) {
    asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_gpu(const int32_t* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// ---- cluster and distributed shared memory -----------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// this CTA's shared::cta address -> the shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
// asynchronous 16-byte store into a peer's shared memory; the peer's mbarrier counts the bytes (complete_tx, release.cluster)
__device__ __forceinline__ void st_async_v4(uint32_t remote_addr, const uint4& v, uint32_t remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(remote_addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(remote_bar) : "memory");
}

// ---- TMA and bulk copies -----------------------------------------------------------------------
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1)
                 : "memory");
}
// multicast: the box lands at this offset in every CTA of the mask, each CTA's barrier at `bar` counts its bytes
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void tma_load_4d_mc(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(mask)
                 : "memory");
}
// 2-CTA TMA loads: data lands in THIS CTA's shared memory, the transaction bytes are counted on the LEADER's barrier
__device__ __forceinline__ void tma2_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar & PEER_MASK), "r"(c0), "r"(c1)
                 : "memory");
}
// one contiguous global -> shared bulk copy (no tensor map); the bytes are counted on `bar`
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// ---- tcgen05: tensor memory, MMA, commit, load -------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// TMEM allocation by one whole warp (the base column address is written to shared memory at `dst`), then this CTA gives up its
// right to allocate more; tc_* = cta_group::1, tc2_* = cta_group::2 (the pair allocates together)
__device__ __forceinline__ void tc_tmem_alloc(uint32_t dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc2_tmem_alloc(uint32_t dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc2_tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// MMA completion -> one arrival on the barrier at this offset in every CTA of the mask
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}
// MMA completion -> one arrival on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc2_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// tcgen05.mma with the 64-bit shared-memory descriptors given as (lo, hi) halves: hi is a constant of the operand's layout (desc_hi),
// lo = address field, advanced by plain 32-bit adds -- the single issuing thread's instruction stream is what bounds short MMAs
__device__ __forceinline__ void tc1_mma_bf16_split(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                                   uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same issued by the pair's leader for both CTAs (cta_group::2)
__device__ __forceinline__ void tc2_mma_bf16_split(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                                   uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace szb
