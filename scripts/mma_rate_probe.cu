// mma_rate_probe.cu -- hardware probe (not part of the library): what does ONE tcgen05.mma.kind::f16 cost when nothing else is in the
// way?  One CTA (or a cta_group::2 pair), operands resident in shared memory (no TMA, no pipeline), one thread issues `count` MMAs back to
// back and commits; the time from the first issue to the commit's arrival, divided by count, is the sustained cost per instruction.
// Varied: N (32..256), M (128 with cta_group::1, 256 with cta_group::2), one accumulator (dependent chain) vs two alternating ones,
// operands at one address vs walking over 8 stages, K-major 1024-byte groups vs the halo layout's 1280-byte groups.
// The arithmetic alone needs M x N x 16 x 2 / 8192 cycles on an SM (N = 128: 64, N = 256: 128).
//
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -I../sigma-zero_b200/csrc -o mma_rate_probe mma_rate_probe.cu     run: ./mma_rate_probe
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include "tc.cuh"

using namespace szb;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)

struct Args { int n; int count; int dual; int walk; int sbo; long long* out; const uint8_t* src; int copy_bytes; int commit_every; };

// cta_group::1, M = 128
__global__ void __launch_bounds__(128, 1) k_rate1(const Args a) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar, cbar[4], sbar;
    __shared__ uint32_t tmem_base_sh;
    __shared__ volatile int stop_sh;
    __shared__ long long copied_sh;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    for (uint32_t i = threadIdx.x; i < 160 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem_raw)[i] = 0x3c003c00u + (i & 3);   // any finite bf16
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&bar), 1);
        for (int i = 0; i < 4; i++) mbar_init(smem_u32(&cbar[i]), 1);
        mbar_init(smem_u32(&sbar), 1);
        stop_sh = 0;
        copied_sh = 0;
        fence_mbarrier_init();
    }
    if (threadIdx.x < 32) tc_tmem_alloc(smem_u32(&tmem_base_sh), 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = tmem_base_sh;
    if (threadIdx.x == 32 && a.copy_bytes) {
        // a stream of bulk copies global (L2-resident) -> shared memory into a region the MMAs do not read, four in flight
        const uint32_t cdst = base + 160 * 1024;
        uint32_t ph[4] = {0, 0, 0, 0};
        long long n = 0;
        for (int i = 0; i < 4; i++) { mbar_expect_tx(smem_u32(&cbar[i]), a.copy_bytes); bulk_load(cdst + i * 16384, a.src + (size_t)i * 16384, a.copy_bytes, smem_u32(&cbar[i])); }
        for (int i = 0; !stop_sh; i = (i + 1) & 3) {
            while (!mbar_try_wait(smem_u32(&cbar[i]), ph[i])) {}
            ph[i] ^= 1;
            n += a.copy_bytes;
            mbar_expect_tx(smem_u32(&cbar[i]), a.copy_bytes);
            bulk_load(cdst + i * 16384, a.src + (size_t)((n >> 14) & 63) * 16384, a.copy_bytes, smem_u32(&cbar[i]));
        }
        for (int i = 0; i < 4; i++) while (!mbar_try_wait(smem_u32(&cbar[i]), ph[i])) {}
        copied_sh = n;
    }
    if (threadIdx.x == 0) {
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(a.n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t hi = (uint32_t)(a.sbo >> 4) | (1u << 14) | (2u << 29), hib = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
        const uint32_t a_lo0 = ((base >> 4) & 0x3FFFu) | (1u << 16), b_lo0 = (((base + 32768) >> 4) & 0x3FFFu) | (1u << 16);
        const long long t0 = clock64();
        for (int i = 0; i < a.count; i += 4) {
            const uint32_t st = a.walk ? (uint32_t)((i >> 2) & 3) : 0u;                 // A stages of 32 KB / 4, B stages of 32 KB: 4 each inside 160 KB
            const uint32_t al = a_lo0 + st * (8192 >> 4), bl = b_lo0 + st * (32768 >> 4);
            const uint32_t d1 = tm + (a.dual ? 256u : 0u);
            tc1_mma_bf16_split(tm, al, hi, bl, hib, idesc, i != 0);
            tc1_mma_bf16_split(d1, al + 2, hi, bl + 2, hib, idesc, a.dual ? (i != 0) : 1u);
            tc1_mma_bf16_split(tm, al + 4, hi, bl + 4, hib, idesc, 1u);
            tc1_mma_bf16_split(d1, al + 6, hi, bl + 6, hib, idesc, 1u);
            if (a.commit_every && (i + 4) % a.commit_every == 0 && i + 4 < a.count) tc_commit(smem_u32(&sbar));      // a commit per stage, as a pipeline issues them (barrier nobody waits on)
        }
        tc_commit(smem_u32(&bar));
        const long long t1 = clock64();
        while (!mbar_try_wait(smem_u32(&bar), 0)) {}
        const long long t2 = clock64();
        stop_sh = 1;
        a.out[0] = t1 - t0;
        a.out[1] = t2 - t0;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x == 0) a.out[2] = copied_sh;
    if (threadIdx.x < 32) tc_tmem_dealloc(tm, 512);
}

// cta_group::2, M = 256 (128 rows per CTA), N split between the CTAs
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1) k_rate2(const Args a) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar, sbar;
    __shared__ uint32_t tmem_base_sh;
    const uint32_t rank = cluster_ctarank();
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    for (uint32_t i = threadIdx.x; i < 160 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem_raw)[i] = 0x3c003c00u + (i & 3);
    if (threadIdx.x == 0) { mbar_init(smem_u32(&bar), 1); mbar_init(smem_u32(&sbar), 1); fence_mbarrier_init(); }
    if (threadIdx.x < 32) tc2_tmem_alloc(smem_u32(&tmem_base_sh), 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tm = tmem_base_sh;
    if (rank == 0 && threadIdx.x == 0) {
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(a.n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
        const uint32_t hi = (uint32_t)(a.sbo >> 4) | (1u << 14) | (2u << 29), hib = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
        const uint32_t a_lo0 = ((base >> 4) & 0x3FFFu) | (1u << 16), b_lo0 = (((base + 32768) >> 4) & 0x3FFFu) | (1u << 16);
        const long long t0 = clock64();
        for (int i = 0; i < a.count; i += 4) {
            const uint32_t st = a.walk ? (uint32_t)((i >> 2) & 3) : 0u;
            const uint32_t al = a_lo0 + st * (8192 >> 4), bl = b_lo0 + st * (32768 >> 4);
            const uint32_t d1 = tm + (a.dual ? 256u : 0u);
            tc2_mma_bf16_split(tm, al, hi, bl, hib, idesc, i != 0);
            tc2_mma_bf16_split(d1, al + 2, hi, bl + 2, hib, idesc, a.dual ? (i != 0) : 1u);
            tc2_mma_bf16_split(tm, al + 4, hi, bl + 4, hib, idesc, 1u);
            tc2_mma_bf16_split(d1, al + 6, hi, bl + 6, hib, idesc, 1u);
            if (a.commit_every && (i + 4) % a.commit_every == 0 && i + 4 < a.count)        // stage release to BOTH CTAs, as k_tower_tc2 issues it
                tc2_commit(smem_u32(&sbar));
        }
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(&bar)), "h"((uint16_t)1) : "memory");
        const long long t1 = clock64();
        while (!mbar_try_wait(smem_u32(&bar), 0)) {}
        const long long t2 = clock64();
        a.out[0] = t1 - t0;
        a.out[1] = t2 - t0;
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    if (threadIdx.x < 32) tc2_tmem_dealloc(tm, 512);
}

int main() {
    long long* out;
    uint8_t* src;
    CK(cudaMalloc(&out, 32));
    CK(cudaMalloc(&src, 64 * 16384));
    CK(cudaMemset(src, 0x3c, 64 * 16384));
    const int smem = 226 * 1024;
    CK(cudaFuncSetAttribute(k_rate1, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CK(cudaFuncSetAttribute(k_rate2, cudaFuncAttributeMaxDynamicSharedMemorySize, 161 * 1024));
    const int count = 512;
    printf("part 1: MMAs alone (operands resident in shared memory), %d back-to-back instructions\n", count);
    printf("%-10s %4s %5s %5s %5s | %10s %10s | %8s\n", "group", "N", "dual", "walk", "SBO", "issue clk", "total clk", "clk/MMA");
    for (int group = 1; group <= 2; group++)
        for (int n : {32, 64, 128, 256})
            for (int variant = 0; variant < 3; variant++) {
                const int dual = variant == 1, walk = variant == 2, sbo = variant == 2 ? 1280 : 1024;
                Args a{n, count, dual, walk, sbo, out, src, 0, 0};
                for (int rep = 0; rep < 2; rep++) {          // second run: warm instruction cache
                    if (group == 1) k_rate1<<<1, 128, smem>>>(a); else k_rate2<<<2, 128, 161 * 1024>>>(a);
                    CK(cudaDeviceSynchronize());
                }
                long long h[3];
                CK(cudaMemcpy(h, out, 24, cudaMemcpyDeviceToHost));
                printf("%-10s %4d %5d %5d %5d | %10lld %10lld | %8.1f   (arithmetic %5.1f)\n", group == 1 ? "cta_group1" : "cta_group2", n, dual, walk, sbo, h[0], h[1],
                       (double)h[1] / count, 128.0 * n * 16 * 2 / 8192.0);
            }
    printf("\npart 2: the same MMAs (cta_group::1, M 128) while another warp streams bulk copies L2 -> shared memory (4 x copy_bytes in flight)\n");
    printf("%4s %10s | %8s %14s\n", "N", "copy_bytes", "clk/MMA", "copied B/clk");
    for (int n : {128, 256})
        for (int cb : {0, 4096, 16384}) {
            Args a{n, 2048, 0, 1, 1280, out, src, cb, 0};
            for (int rep = 0; rep < 2; rep++) { k_rate1<<<1, 128, smem>>>(a); CK(cudaDeviceSynchronize()); }
            long long h[3];
            CK(cudaMemcpy(h, out, 24, cudaMemcpyDeviceToHost));
            printf("%4d %10d | %8.1f %14.1f\n", n, cb, (double)h[1] / 2048, (double)h[2] / (double)h[1]);
        }
    printf("\npart 3: a tcgen05.commit after every `commit_every` MMAs (what a pipeline does to release a shared-memory stage); cta_group::2 commits are\n"
           "multicast to both CTAs\n");
    printf("%-10s %4s %12s | %8s %12s %16s\n", "group", "N", "commit_every", "clk/MMA", "arithmetic", "clk per commit");
    for (int group = 1; group <= 2; group++)
        for (int n : {64, 128, 256})
            for (int ce : {0, 4, 8, 12, 16, 36}) {
                Args a{n, 2304, 0, 1, 1280, out, src, 0, ce};
                for (int rep = 0; rep < 2; rep++) {
                    if (group == 1) k_rate1<<<1, 128, smem>>>(a); else k_rate2<<<2, 128, 161 * 1024>>>(a);
                    CK(cudaDeviceSynchronize());
                }
                long long h[3];
                CK(cudaMemcpy(h, out, 24, cudaMemcpyDeviceToHost));
                printf("%-10s %4d %12d | %8.1f %12.1f %16.1f\n", group == 1 ? "cta_group1" : "cta_group2", n, ce, (double)h[1] / 2304, 128.0 * n * 16 * 2 / 8192.0,
                       ce ? (double)h[1] / (2304.0 / ce) : 0.0);
            }
    return 0;
}
