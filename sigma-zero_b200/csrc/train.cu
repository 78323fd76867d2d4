// train.cu -- the trainer of the self-play loop (train_RL.py:77-154) as hand-written sm_100a kernels.
//
//   loss = mse_loss(v, z) + cross_entropy(logits, pi)   (train_RL.py:103-113; pi = soft visit-fraction target over all 4672 logits)
//   Adam(lr 1e-4, weight_decay 1e-4) (train_RL.py:187), StepLR(500, 0.95) stepped per batch (:199, :123-124)
//   network.py:100-192 in TRAINING mode: every BatchNorm normalises with the statistics of the batch and updates its running buffers.
//
// Mixed precision: fp32 master weights, Adam moments and BatchNorm arithmetic; bf16 operands on the tensor cores with fp32 accumulation
// in TMEM; activations and activation gradients are stored as bf16.  Three tcgen05 GEMM shapes do all the heavy work of a step:
//   forward   Y[pos][co]  = sum_{tap,ci} X[pos+tap][ci] * W[co][tap][ci]          k_tconv_pair  (A: a halo chunk of X resident in shared memory,
//                                                                                               every tap a shifted descriptor; cta_group::2)
//   dgrad     dX[pos][ci] = sum_{tap,co} dY[pos+tap][co] * W[co][8-tap][ci]       k_tconv_pair  (same kernel, transposed / tap-mirrored weights)
//   wgrad     dW[co][tap][ci] = sum_pos dY[pos][co] * X[pos+tap][ci]              k_wgrad       (both operands MN-major: the K dimension is the
//                                                                                               board square, exactly as the tensors lie in HBM)
// The convolution epilogues also produce the sums the BatchNorm kernels need (forward statistics; backward: residual join, ReLU mask,
// gradient sums).  The 38 tower layers' weight gradients run as one launch after the backward chain; the three odd-shaped layers split the
// batch into partial sums that a second kernel adds in a fixed order.  No value atomics anywhere: a step is deterministic.  The whole step
// is captured as one CUDA graph per (batch size, flags).
// Activations live in HBM as NHWC bf16 with a one-square zero halo, [B][10][10][C], like the inference tower (net.cu).
//
// Everything here is reached through szb_train_* (include/szb200.h); there is no CPU path.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include "engine.cuh"
#include "tc.cuh"

using namespace szb;

namespace szb {

typedef __nv_bfloat16 bf16;

constexpr int TH = 10;                       // halo board edge
constexpr int TPIX = TH * TH;
constexpr int TC = 256;                      // tower channels
constexpr int TCIN = 128;                    // 119 input planes padded
constexpr int T_LAYERS = 41;                 // stem, 38 tower convolutions, conv_p1, conv_p2
constexpr int T_BN = 40;                     // all of them but conv_p2 carry a BatchNorm
constexpr int L_P1 = 39, L_P2 = 40;
constexpr int T_ACTIONS = 4672;
constexpr int T_PLANES = 119;
constexpr int DL_C = 128;                    // channels of the logits-gradient buffer (73 policy planes padded)

constexpr int TR_THREADS = 192;              // k_wgrad: warp 0 TMA, warp 1 MMA + TMEM, warps 2..5 epilogue
constexpr int TC_CONV_THREADS = 320;         // k_tconv / k_tconv_pair: eight epilogue warps (two per TMEM lane group, 64 columns each)
constexpr int TR_A_CHUNKS = 2;
constexpr int TR_A_CHUNK_BYTES = 2 * TPIX * 128;      // two boards with their halo x 64 channels: 25600 = 25 * 1024
constexpr int TR_TPS = 3;                             // taps per weight stage of a 3x3 layer
constexpr int TR_B_STAGES = 3;
constexpr bool TR_DUAL_ACC = false;                   // A/B aid: even / odd K steps accumulate into two TMEM tiles (two independent MMA chains); measured: no change
constexpr int TR_CLUSTER = 4;                         // CTAs (neighbouring tiles) that share every weight tile through TMA multicast
constexpr int TR_B_BYTES = 128 * 64 * 2;              // 128 output channels x 64 k
constexpr int TR_B_STAGE_BYTES = TR_TPS * TR_B_BYTES;
constexpr int TR_SMEM = TR_A_CHUNKS * TR_A_CHUNK_BYTES + TR_B_STAGES * TR_B_STAGE_BYTES + 1024;

constexpr int WG_STAGES = 4;
constexpr int WG_BOX = 64 * 64 * 2;          // one board (64 squares) x 64 channels
constexpr int WG_MAX_SPLIT = 64;
constexpr int ROWS_RING = 8;

__device__ __forceinline__ int halo_pix(int sq) { return ((sq >> 3) + 1) * TH + (sq & 7) + 1; }

// =================================================================================================
// forward / dgrad convolution: one 128-square x 128-channel tile per CTA
// =================================================================================================
struct TConvArgs {
    int taps, kchunks;           // K = taps * kchunks * 64
    int n_boards;
    bf16* out;                   // MODE 0: halo NHWC, `ldc` channels per square
    int ldc;
    float* logits;               // MODE 1: [board][4672] plane-major (torch.flatten of conv_p2's output), + bias
    const float* bias;
    // MODE 0, optional: per-tile column sums [tile][2][ldc] of what this launch stores (after bf16 rounding), for the BatchNorm that follows:
    //   forward  (bn_o == null): sum(y), sum(y^2)                      -> batch statistics (k_bn_fwd)
    //   backward (bn_o != null): the accumulator is the gradient arriving at the OUTPUT of the BatchNorm below; the epilogue applies the
    //            residual join and the ReLU mask, g = (acc [+ bn_skip]) * [bn_o > 0], stores g, and sums g, g * xhat (k_bn_bwd)
    float* stat_part;
    const bf16* bn_skip; const bf16* bn_o; const bf16* bn_y;
    const float* bn_mean; const float* bn_invstd;
    int32_t* error;
    unsigned long long* trace;   // measurement aid (SZB_TRAIN_TRACE): %globaltimer stamps of CTA (0, 0), or null
};

// Column sums over the 32 lanes of a warp of 32 per-lane values: lane L returns the sum over all lanes of v[L].  Halving exchange
// (16 + 8 + 4 + 2 + 1 shuffles, no dynamic register indexing); the order of the additions is fixed.
__device__ __forceinline__ float warp_col_sum32(float (&v)[32], int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < s; i++) {
            const float send = up ? v[i] : v[i + s];
            const float keep = up ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, s);
        }
    }
    return v[0];
}

__device__ __forceinline__ void t_stamp(unsigned long long* tr, int k) {
    if (tr) tr[k] = global_ns();
}

// Epilogue of the training convolutions (the four epilogue warps of a CTA; `tile` = index of this CTA's two boards): TMEM -> registers ->
// [backward: + skip, ReLU mask] -> bf16 rows / fp32 logits, and the fused BatchNorm sums (see TConvArgs).
template <int MODE, bool DUAL = false>
__device__ __forceinline__ void tconv_epilogue(const TConvArgs& a, uint32_t tmem_base, int tile, int nh, int warp, int lane, uint32_t bar_acc_addr,
                                               volatile int* abort_flag, float (*st_sh)[4][128], float (*mi_sh)[128], unsigned long long* trace) {
    const int lane_group = warp & 3;                                   // TMEM lanes this warp may read
    const int col0 = ((warp - 2) >> 2) * 64;                           // ... and its half of the 128 columns
    const int e = (warp - 2) * 32 + lane;                              // 0..255 over the eight epilogue warps
    const bool stats = MODE == 0 && a.stat_part != nullptr, bwd = MODE == 0 && a.bn_o != nullptr;
    if (bwd) mi_sh[e >> 7][e & 127] = (e < 128 ? a.bn_mean : a.bn_invstd)[nh * 128 + (e & 127)];
    bool ok = mbar_wait(bar_acc_addr, 0, abort_flag);
    ok = __all_sync(0xFFFFFFFFu, ok);
    if (warp == 2 && lane == 0) t_stamp(trace, 5);
    if (ok) {
        tc_fence_after();
        if (bwd) named_bar_sync<1, 256>();
        const int m = lane_group * 32 + lane;                          // row (oy * 2 + board) * 8 + ox
        const int board = tile * 2 + ((m >> 3) & 1), sq = (m >> 4) * 8 + (m & 7);
        const bool live = board < a.n_boards;
        const uint32_t taddr = tmem_base + ((uint32_t)(lane_group * 32) << 16);
        const size_t pix = (size_t)board * TPIX + halo_pix(sq);
#pragma unroll 1
        for (int c0 = col0; c0 < col0 + 64; c0 += 32) {
            uint32_t v[32];
            tmem_ld_32x32b_x16(taddr + c0, v);
            tmem_ld_32x32b_x16(taddr + c0 + 16, v + 16);
            if (DUAL) {
                // two interleaved accumulation chains (even / odd K steps): their sum is the convolution
                uint32_t w[32];
                tmem_ld_32x32b_x16(taddr + 128 + c0, w);
                tmem_ld_32x32b_x16(taddr + 128 + c0 + 16, w + 16);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; j++) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(w[j]));
            } else {
                tmem_ld_wait();
            }
            if (MODE == 0) {
                const size_t off = pix * a.ldc + nh * 128 + c0;
                float f[32], xh[32];
#pragma unroll
                for (int j = 0; j < 32; j++) f[j] = live ? __uint_as_float(v[j]) : 0.f;
                if (bwd) {
                    if (live) {
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            const uint4 ov = *reinterpret_cast<const uint4*>(a.bn_o + off + q * 8), yv = *reinterpret_cast<const uint4*>(a.bn_y + off + q * 8);
                            const bf16* ob = reinterpret_cast<const bf16*>(&ov);
                            const bf16* yb = reinterpret_cast<const bf16*>(&yv);
                            if (a.bn_skip) {
                                const uint4 sv = *reinterpret_cast<const uint4*>(a.bn_skip + off + q * 8);
                                const bf16* sb = reinterpret_cast<const bf16*>(&sv);
#pragma unroll
                                for (int j = 0; j < 8; j++) f[q * 8 + j] += __bfloat162float(sb[j]);
                            }
#pragma unroll
                            for (int j = 0; j < 8; j++) {
                                if (!(__bfloat162float(ob[j]) > 0.f)) f[q * 8 + j] = 0.f;
                                xh[q * 8 + j] = (__bfloat162float(yb[j]) - mi_sh[0][c0 + q * 8 + j]) * mi_sh[1][c0 + q * 8 + j];
                            }
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++) xh[j] = 0.f;
                    }
                }
                uint4 o[4];
                __nv_bfloat162* ob2 = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
                for (int j = 0; j < 16; j++) ob2[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
                if (live) {
                    uint4* op = reinterpret_cast<uint4*>(a.out + off);
#pragma unroll
                    for (int j = 0; j < 4; j++) op[j] = o[j];
                }
                if (stats) {
                    // sums of the ROUNDED values: exactly what the BatchNorm kernel will read back
                    float s2[32];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        const float2 r = __bfloat1622float2(ob2[j]);
                        f[2 * j] = r.x;
                        f[2 * j + 1] = r.y;
                    }
#pragma unroll
                    for (int j = 0; j < 32; j++) s2[j] = bwd ? f[j] * xh[j] : f[j] * f[j];
                    const float c1 = warp_col_sum32(f, lane), c2 = warp_col_sum32(s2, lane);
                    st_sh[0][lane_group][c0 + lane] = c1;
                    st_sh[1][lane_group][c0 + lane] = c2;
                }
            } else if (live) {
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    const int c = nh * 128 + c0 + j;
                    if (c < 73) a.logits[(size_t)board * T_ACTIONS + c * 64 + sq] = __uint_as_float(v[j]) + a.bias[c];
                }
            }
        }
        if (stats) {
            named_bar_sync<1, 256>();
            if (tile * 2 < a.n_boards) {
                const int which = e >> 7, c = e & 127;
                a.stat_part[((size_t)tile * 2 + which) * a.ldc + nh * 128 + c] = ((st_sh[which][0][c] + st_sh[which][1][c]) + st_sh[which][2][c]) + st_sh[which][3][c];
            }
        }
    }
}

// Shared memory: a ring of TR_A_CHUNKS activation chunks and a ring of TR_B_STAGES weight tiles.  An activation chunk is one 64-channel
// slice of the tile's two boards INCLUDING the halo, 200 rows of 128 bytes in the order [y][board][x] (one TMA box through a tensor map
// with dims (c, x, board, y)); all nine taps read it in place: the A descriptor of tap (ky, kx) starts (ky * 20 + kx) rows into the chunk
// and strides 10 rows between 8-row groups, so MMA row m = (oy * 2 + board) * 8 + ox reads halo square (oy + ky, ox + kx) -- the layout
// k_tower_tc2 (net.cu) uses.  An activation byte enters the SM once per layer instead of once per tap.
// Weights: the TR_CLUSTER CTAs of a cluster work on neighbouring tiles with the SAME weights; each loads a quarter of every weight tile and
// multicasts it into all four shared memories, and a stage is refilled only when all four CTAs' MMAs have released it (their commits arrive
// on every CTA's barrier).  The kernel is bound by L2 -> SM traffic (measured: 6.8 TB/s with one L2 read per CTA and tile); multicast cuts
// the weight reads four-fold.
template <int MODE>
__global__ void __cluster_dims__(TR_CLUSTER, 1, 1) __launch_bounds__(TC_CONV_THREADS, 1)
k_tconv(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, const TConvArgs a) {
    constexpr uint32_t IDESC = idesc_bf16(128, 128);
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_af[TR_A_CHUNKS], bar_ae[TR_A_CHUNKS], bar_bf[TR_B_STAGES], bar_be[TR_B_STAGES], bar_acc;
    __shared__ uint32_t tmem_base_sh;
    __shared__ int abort_sh;
    __shared__ float st_sh[2][4][128], mi_sh[2][128];                  // fused BatchNorm sums of the four epilogue warps; mean / invstd

    const uint32_t smem_a = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_b = smem_a + TR_A_CHUNKS * TR_A_CHUNK_BYTES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x, nh = blockIdx.y;
    volatile int* abort_flag = &abort_sh;
    unsigned long long* trace = (blockIdx.x == 0 && blockIdx.y == 0) ? a.trace : nullptr;
    if (threadIdx.x == 0) t_stamp(trace, 0);

    if (threadIdx.x == 0) {
        abort_sh = 0;
        for (int s = 0; s < TR_A_CHUNKS; s++) { mbar_init(smem_u32(&bar_af[s]), 1); mbar_init(smem_u32(&bar_ae[s]), 1); }
        for (int s = 0; s < TR_B_STAGES; s++) { mbar_init(smem_u32(&bar_bf[s]), 1); mbar_init(smem_u32(&bar_be[s]), TR_CLUSTER); }
        mbar_init(smem_u32(&bar_acc), 1);
        fence_mbarrier_init();
    }
    if (warp == 1) tc_tmem_alloc(smem_u32(&tmem_base_sh), TR_DUAL_ACC ? 256 : 128);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                             // every CTA's barriers exist before a peer's multicast or commit can reach them
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;
    const uint32_t crank = cluster_ctarank();
    constexpr uint16_t CMASK = (uint16_t)((1u << TR_CLUSTER) - 1);
    if (threadIdx.x == 0) t_stamp(trace, 1);
    pdl_trigger();                                  // programmatic dependent launch: everything above overlapped the predecessor's tail
    pdl_wait();
    if (threadIdx.x == 0) t_stamp(trace, 2);

    if (warp == 0) {
        if (lane == 0) {
            int ac = 0, bs = 0;
            uint32_t a_phase = 0, b_phase = 0;
            bool ok = true;
            for (int kc = 0; kc < a.kchunks && ok; kc++) {
                if (!(ok = mbar_wait(smem_u32(&bar_ae[ac]), a_phase ^ 1, abort_flag))) break;
                const uint32_t af = smem_u32(&bar_af[ac]);
                mbar_expect_tx(af, TR_A_CHUNK_BYTES);
                tma_load_4d(smem_a + ac * TR_A_CHUNK_BYTES, &tm_a, af, kc * 64, 0, tile * 2, 0);
                if (++ac == TR_A_CHUNKS) { ac = 0; a_phase ^= 1; }
                // weight stages: TR_TPS consecutive taps of this K chunk per stage (3x3 layers), one tile for a 1x1 layer
                const int per = a.taps == 9 ? TR_TPS : 1;
                for (int tap0 = 0; tap0 < a.taps; tap0 += per) {
                    if (!(ok = mbar_wait(smem_u32(&bar_be[bs]), b_phase ^ 1, abort_flag))) break;
                    const uint32_t bf = smem_u32(&bar_bf[bs]);
                    mbar_expect_tx(bf, (uint32_t)per * TR_B_BYTES);          // four quarters of every tile, one from each CTA of the cluster
                    for (int u = 0; u < per; u++)
                        tma_load_2d_mc(smem_b + bs * TR_B_STAGE_BYTES + u * TR_B_BYTES + crank * (TR_B_BYTES / TR_CLUSTER), &tm_w, bf,
                                       ((tap0 + u) * a.kchunks + kc) * 64, nh * 128 + (int)crank * (128 / TR_CLUSTER), CMASK);
                    if (++bs == TR_B_STAGES) { bs = 0; b_phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // The whole warp runs the loop convergently (descriptors and barrier addresses stay in uniform registers), one elected lane issues;
        // the nine taps of a K chunk are straight-line code with immediate descriptor offsets (a generic tap loop costs the issuing
        // thread ~100 cycles per MMA -- more than the 64 cycles a 128 x 128 x 16 MMA takes).
        const uint32_t a_lo0 = ((smem_a >> 4) & 0x3FFFu) | DESC_LO_FLAGS, b_lo0 = ((smem_b >> 4) & 0x3FFFu) | DESC_LO_FLAGS;
        const uint32_t bar_af0 = smem_u32(&bar_af[0]), bar_ae0 = smem_u32(&bar_ae[0]), bar_bf0 = smem_u32(&bar_bf[0]), bar_be0 = smem_u32(&bar_be[0]);
        uint32_t ac = 0, bs = 0, a_phase = 0, b_phase = 0, accumulate = 0;
        bool ok = true;
        for (int kc = 0; kc < a.kchunks && ok; kc++) {
            if (!(ok = warp_mbar_wait(bar_af0 + ac * 8, a_phase, abort_flag))) break;
            tc_fence_after();
            if (kc == 0 && lane == 0) t_stamp(trace, 3);
            const uint32_t chunk_lo = a_lo0 + ac * (TR_A_CHUNK_BYTES >> 4);
            if (a.taps == 9) {
                // One wait / elect / commit per TR_TPS taps: the issuing warp's own instruction stream costs ~450 cycles per stage whatever the
                // stage holds (scripts/mma_rate_probe.cu) -- more than the 256 cycles four 128 x 128 x 16 MMAs take, less than the 768 of twelve.
#pragma unroll
                for (int s0 = 0; s0 < 9; s0 += TR_TPS) {
                    if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t d1 = tmem_base + (TR_DUAL_ACC ? 128u : 0u);
#pragma unroll
                        for (int u = 0; u < TR_TPS; u++) {
                            const int tap = s0 + u;
                            const uint32_t a_lo = chunk_lo + (uint32_t)((tap / 3) * 2 * TH + tap % 3) * (128 >> 4);
                            const uint32_t b_lo = b_lo0 + bs * (TR_B_STAGE_BYTES >> 4) + u * (TR_B_BYTES >> 4);
                            const uint32_t first = tap == 0 ? accumulate : 1u;
                            tc1_mma_bf16_split(tmem_base, a_lo, desc_hi(TH * 128), b_lo, desc_hi(1024), IDESC, first);
                            tc1_mma_bf16_split(d1, a_lo + 2, desc_hi(TH * 128), b_lo + 2, desc_hi(1024), IDESC, TR_DUAL_ACC ? first : 1u);
                            tc1_mma_bf16_split(tmem_base, a_lo + 4, desc_hi(TH * 128), b_lo + 4, desc_hi(1024), IDESC, 1u);
                            tc1_mma_bf16_split(d1, a_lo + 6, desc_hi(TH * 128), b_lo + 6, desc_hi(1024), IDESC, 1u);
                        }
                        tc_commit_mc(bar_be0 + bs * 8, CMASK);
                    }
                    __syncwarp();
                    if (++bs == TR_B_STAGES) { bs = 0; b_phase ^= 1; }
                }
            } else {
                if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_lo = chunk_lo + (uint32_t)(2 * TH + 1) * (128 >> 4);            // centre tap
                    const uint32_t b_lo = b_lo0 + bs * (TR_B_STAGE_BYTES >> 4);
                    const uint32_t d1 = tmem_base + (TR_DUAL_ACC ? 128u : 0u);
                    tc1_mma_bf16_split(tmem_base, a_lo, desc_hi(TH * 128), b_lo, desc_hi(1024), IDESC, accumulate);
                    tc1_mma_bf16_split(d1, a_lo + 2, desc_hi(TH * 128), b_lo + 2, desc_hi(1024), IDESC, TR_DUAL_ACC ? accumulate : 1u);
                    tc1_mma_bf16_split(tmem_base, a_lo + 4, desc_hi(TH * 128), b_lo + 4, desc_hi(1024), IDESC, 1u);
                    tc1_mma_bf16_split(d1, a_lo + 6, desc_hi(TH * 128), b_lo + 6, desc_hi(1024), IDESC, 1u);
                    tc_commit_mc(bar_be0 + bs * 8, CMASK);
                }
                __syncwarp();
                if (++bs == TR_B_STAGES) { bs = 0; b_phase ^= 1; }
            }
            accumulate = 1;
            if (ok && elect_one()) tc_commit(bar_ae0 + ac * 8);
            __syncwarp();
            if (++ac == TR_A_CHUNKS) { ac = 0; a_phase ^= 1; }
        }
        if (ok && elect_one()) { tc_commit(smem_u32(&bar_acc)); t_stamp(trace, 4); }
        __syncwarp();
    } else {
        tconv_epilogue<MODE, TR_DUAL_ACC>(a, tmem_base, tile, nh, warp, lane, smem_u32(&bar_acc), abort_flag, st_sh, mi_sh, trace);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tc_tmem_dealloc(tmem_base, TR_DUAL_ACC ? 256 : 128);
    cluster_sync_all();                             // no CTA leaves while a peer's commit may still arrive on its barriers
    if (threadIdx.x == 0) t_stamp(trace, 6);
    if (threadIdx.x == 0 && abort_sh) atomicExch(a.error, 1);
}


// -------------------------------------------------------------------------------------------------
// The same convolution as a CTA PAIR (cta_group::2): M 256 (four boards, 128 rows per CTA) x N 128 x K 16 per MMA, issued by the leader for
// both SMs.  Each CTA stages its own activation chunk and HALF of every weight tile (64 rows); per 64-cycle MMA an SM then reads 4 KB of A
// and 2 KB of B from shared memory instead of 4 + 4 KB.  A/B aid (SZB_TRAIN_CONV=2): it measured no faster than k_tconv (9.4 vs 8.6 us main
// loop at 128 boards), which rules shared-memory operand bandwidth out as the bound of the 64-cycle MMAs (DESIGN 3.5).  Barriers live on the
// leader for "data landed" (both CTAs' TMA bytes are counted there) and in both CTAs for "stage free" / "accumulator ready" (the leader's
// commits are multicast) -- the protocol of k_tower_tc2 (net.cu).
constexpr int TP_B_STAGES = 6;
constexpr int TP_B_BYTES = 64 * 64 * 2;               // this CTA's half of a 128-channel x 64-k weight tile
constexpr int TP_B_STAGE_BYTES = TR_TPS * TP_B_BYTES;
constexpr int TP_SMEM = TR_A_CHUNKS * TR_A_CHUNK_BYTES + TP_B_STAGES * TP_B_STAGE_BYTES + 1024;

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_CONV_THREADS, 1)
k_tconv_pair(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, const TConvArgs a) {
    constexpr uint32_t IDESC = idesc_bf16(256, 128);
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_af[TR_A_CHUNKS], bar_ae[TR_A_CHUNKS], bar_bf[TP_B_STAGES], bar_be[TP_B_STAGES], bar_acc;
    __shared__ uint32_t tmem_base_sh;
    __shared__ int abort_sh;
    __shared__ float st_sh[2][4][128], mi_sh[2][128];

    const uint32_t smem_a = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_b = smem_a + TR_A_CHUNKS * TR_A_CHUNK_BYTES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int tile = blockIdx.x, nh = blockIdx.y;          // tile = this CTA's two boards; the pair = tiles (2p, 2p + 1)
    volatile int* abort_flag = &abort_sh;
    unsigned long long* trace = (blockIdx.x == 0 && blockIdx.y == 0) ? a.trace : nullptr;
    if (threadIdx.x == 0) t_stamp(trace, 0);

    if (threadIdx.x == 0) {
        abort_sh = 0;
        for (int s = 0; s < TR_A_CHUNKS; s++) { mbar_init(smem_u32(&bar_af[s]), 1); mbar_init(smem_u32(&bar_ae[s]), 1); }
        for (int s = 0; s < TP_B_STAGES; s++) { mbar_init(smem_u32(&bar_bf[s]), 1); mbar_init(smem_u32(&bar_be[s]), 1); }
        mbar_init(smem_u32(&bar_acc), 1);
        fence_mbarrier_init();
    }
    if (warp == 1) tc2_tmem_alloc(smem_u32(&tmem_base_sh), 128);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                             // both CTAs' barriers and TMEM exist from here on
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;
    if (threadIdx.x == 0) t_stamp(trace, 1);
    pdl_trigger();
    pdl_wait();
    if (threadIdx.x == 0) t_stamp(trace, 2);

    if (warp == 0) {
        if (lane == 0) {
            int ac = 0, bs = 0;
            uint32_t a_phase = 0, b_phase = 0;
            bool ok = true;
            for (int kc = 0; kc < a.kchunks && ok; kc++) {
                if (!(ok = mbar_wait(smem_u32(&bar_ae[ac]), a_phase ^ 1, abort_flag))) break;
                const uint32_t af = smem_u32(&bar_af[ac]);
                if (rank == 0) mbar_expect_tx(af, 2u * TR_A_CHUNK_BYTES);      // both CTAs' bytes land on the leader's barrier
                tma2_load_4d(smem_a + ac * TR_A_CHUNK_BYTES, &tm_a, af, kc * 64, 0, tile * 2, 0);
                if (++ac == TR_A_CHUNKS) { ac = 0; a_phase ^= 1; }
                const int per = a.taps == 9 ? TR_TPS : 1;
                for (int tap0 = 0; tap0 < a.taps; tap0 += per) {
                    if (!(ok = mbar_wait(smem_u32(&bar_be[bs]), b_phase ^ 1, abort_flag))) break;
                    const uint32_t bf = smem_u32(&bar_bf[bs]);
                    if (rank == 0) mbar_expect_tx(bf, 2u * (uint32_t)per * TP_B_BYTES);
                    for (int u = 0; u < per; u++)
                        tma2_load_2d(smem_b + bs * TP_B_STAGE_BYTES + u * TP_B_BYTES, &tm_w, bf, ((tap0 + u) * a.kchunks + kc) * 64, nh * 128 + (int)rank * 64);
                    if (++bs == TP_B_STAGES) { bs = 0; b_phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            const uint32_t a_lo0 = ((smem_a >> 4) & 0x3FFFu) | DESC_LO_FLAGS, b_lo0 = ((smem_b >> 4) & 0x3FFFu) | DESC_LO_FLAGS;
            const uint32_t bar_af0 = smem_u32(&bar_af[0]), bar_ae0 = smem_u32(&bar_ae[0]), bar_bf0 = smem_u32(&bar_bf[0]), bar_be0 = smem_u32(&bar_be[0]);
            uint32_t ac = 0, bs = 0, a_phase = 0, b_phase = 0, accumulate = 0;
            bool ok = true;
            for (int kc = 0; kc < a.kchunks && ok; kc++) {
                if (!(ok = warp_mbar_wait(bar_af0 + ac * 8, a_phase, abort_flag))) break;
                tc_fence_after();
                if (kc == 0 && lane == 0) t_stamp(trace, 3);
                const uint32_t chunk_lo = a_lo0 + ac * (TR_A_CHUNK_BYTES >> 4);
                if (a.taps == 9) {
#pragma unroll
                    for (int s0 = 0; s0 < 9; s0 += TR_TPS) {
                        if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                        tc_fence_after();
                        if (elect_one()) {
#pragma unroll
                            for (int u = 0; u < TR_TPS; u++) {
                                const int tap = s0 + u;
                                const uint32_t a_lo = chunk_lo + (uint32_t)((tap / 3) * 2 * TH + tap % 3) * (128 >> 4);
                                const uint32_t b_lo = b_lo0 + bs * (TP_B_STAGE_BYTES >> 4) + u * (TP_B_BYTES >> 4);
                                tc2_mma_bf16_split(tmem_base, a_lo, desc_hi(TH * 128), b_lo, desc_hi(1024), IDESC, tap == 0 ? accumulate : 1u);
                                tc2_mma_bf16_split(tmem_base, a_lo + 2, desc_hi(TH * 128), b_lo + 2, desc_hi(1024), IDESC, 1u);
                                tc2_mma_bf16_split(tmem_base, a_lo + 4, desc_hi(TH * 128), b_lo + 4, desc_hi(1024), IDESC, 1u);
                                tc2_mma_bf16_split(tmem_base, a_lo + 6, desc_hi(TH * 128), b_lo + 6, desc_hi(1024), IDESC, 1u);
                            }
                            tc2_commit(bar_be0 + bs * 8);
                        }
                        __syncwarp();
                        if (++bs == TP_B_STAGES) { bs = 0; b_phase ^= 1; }
                    }
                } else {
                    if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t a_lo = chunk_lo + (uint32_t)(2 * TH + 1) * (128 >> 4);
                        const uint32_t b_lo = b_lo0 + bs * (TP_B_STAGE_BYTES >> 4);
                        tc2_mma_bf16_split(tmem_base, a_lo, desc_hi(TH * 128), b_lo, desc_hi(1024), IDESC, accumulate);
                        tc2_mma_bf16_split(tmem_base, a_lo + 2, desc_hi(TH * 128), b_lo + 2, desc_hi(1024), IDESC, 1u);
                        tc2_mma_bf16_split(tmem_base, a_lo + 4, desc_hi(TH * 128), b_lo + 4, desc_hi(1024), IDESC, 1u);
                        tc2_mma_bf16_split(tmem_base, a_lo + 6, desc_hi(TH * 128), b_lo + 6, desc_hi(1024), IDESC, 1u);
                        tc2_commit(bar_be0 + bs * 8);
                    }
                    __syncwarp();
                    if (++bs == TP_B_STAGES) { bs = 0; b_phase ^= 1; }
                }
                accumulate = 1;
                if (ok && elect_one()) tc2_commit(bar_ae0 + ac * 8);
                __syncwarp();
                if (++ac == TR_A_CHUNKS) { ac = 0; a_phase ^= 1; }
            }
            if (ok && elect_one()) { tc2_commit(smem_u32(&bar_acc)); t_stamp(trace, 4); }
            __syncwarp();
        }
    } else {
        tconv_epilogue<MODE>(a, tmem_base, tile, nh, warp, lane, smem_u32(&bar_acc), abort_flag, st_sh, mi_sh, trace);
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    if (warp == 1) tc2_tmem_dealloc(tmem_base, 128);
    if (threadIdx.x == 0) t_stamp(trace, 6);
    if (threadIdx.x == 0 && abort_sh) atomicExch(a.error, 1);
}

// =================================================================================================
// wgrad: D[co 128][ci N] (+)= sum over the squares of this CTA's boards of dY[sq][co] * X[sq + tap][ci]
// =================================================================================================
struct alignas(64) WgLayer {     // one entry per layer, in device memory: k_wgrad reads its tensor maps straight from here
    CUtensorMap tm_dy;           // gradient of the layer's convolution output, 1-board boxes
    CUtensorMap tm_x;            // the layer's input, 1-board boxes
    float* out;                  // the layer's slot in the flat gradient buffer [cout_pad][ldw]
    unsigned char pad[56];
};

static_assert(sizeof(WgLayer) == 320, "WgLayer: two tensor maps and a pointer, padded to a multiple of 64 bytes");

struct WgArgs {
    int taps, m_halves, n_boards, ksplit;
    int layer0;                  // blockIdx.z + layer0 = entry of the layer table
    float* partial;              // ksplit > 1: [ksplit][cout_pad][ldw] partial sums (one layer per launch); else null: write the layer's `out`
    int ldw;                     // taps * cin_pad
    int cin_pad;
    size_t split_stride;         // cout_pad * ldw
    int32_t* error;
    uint32_t lbo, sbo;           // descriptor strides (probe aid; 8192 / 1024)
};

// CS = 2: the two CTAs that compute the two halves of the output channels of one (layer, tap, batch split) form a cluster and share the
// input tile X -- each loads half of its 64-channel boxes and multicasts them into both shared memories (a third less L2 -> SM traffic,
// which is what bounds this kernel); a stage is refilled when both CTAs' MMAs have released it.
template <int NB, int CS>        // NB: 64-channel boxes of X (N = NB * 64 input channels); CS: cluster size (1 when there is one half only)
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(TR_THREADS, 1)
k_wgrad(const WgLayer* __restrict__ layers, const WgArgs a) {
    const WgLayer* wl = layers + a.layer0 + blockIdx.z;
    const CUtensorMap* tm_dy = &wl->tm_dy;
    const CUtensorMap* tm_x = &wl->tm_x;
    constexpr int N = NB * 64;
    constexpr int STAGE = (2 + NB) * WG_BOX;
    constexpr uint32_t IDESC = idesc_bf16(128, N, true, true);          // both operands MN-major
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[WG_STAGES], bar_empty[WG_STAGES], bar_acc;
    __shared__ uint32_t tmem_base_sh;
    __shared__ int abort_sh;

    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tap = blockIdx.x / a.m_halves, mh = blockIdx.x - tap * a.m_halves;
    const int ks = blockIdx.y;
    const int b_lo = (int)((long long)ks * a.n_boards / a.ksplit), b_hi = (int)((long long)(ks + 1) * a.n_boards / a.ksplit);
    const int ky = a.taps == 9 ? tap / 3 : 1, kx = a.taps == 9 ? tap - (tap / 3) * 3 : 1;
    volatile int* abort_flag = &abort_sh;

    if (threadIdx.x == 0) {
        abort_sh = 0;
        for (int s = 0; s < WG_STAGES; s++) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), CS); }
        mbar_init(smem_u32(&bar_acc), 1);
        fence_mbarrier_init();
    }
    if (warp == 1) tc_tmem_alloc(smem_u32(&tmem_base_sh), 256);
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();                // the peer's barriers exist before a multicast or a commit can reach them
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;
    const uint32_t crank = CS > 1 ? cluster_ctarank() : 0u;
    constexpr uint16_t CMASK = (uint16_t)((1u << CS) - 1);
    pdl_trigger();
    pdl_wait();

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int b = b_lo; b < b_hi; b++) {
                if (!mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1, abort_flag)) break;
                const uint32_t full = smem_u32(&bar_full[stage]);
                const uint32_t sa = smem_base + stage * STAGE;
                mbar_expect_tx(full, STAGE);
                tma_load_4d(sa, tm_dy, full, mh * 128, 1, 1, b);
                tma_load_4d(sa + WG_BOX, tm_dy, full, mh * 128 + 64, 1, 1, b);
#pragma unroll
                for (int j = 0; j < NB; j++) {
                    if (CS == 1) tma_load_4d(sa + (2 + j) * WG_BOX, tm_x, full, j * 64, kx, ky, b);
                    else if ((uint32_t)(j % CS) == crank) tma_load_4d_mc(sa + (2 + j) * WG_BOX, tm_x, full, j * 64, kx, ky, b, CMASK);
                }
                if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // warp-convergent loop, one elected lane issues; descriptors as (lo, hi) halves advanced with 32-bit adds (see k_tconv)
        const uint32_t lo_flags = ((a.lbo >> 4) & 0x3FFFu) << 16, hi = desc_hi(a.sbo);
        const uint32_t s_lo0 = ((smem_base >> 4) & 0x3FFFu) | lo_flags;
        const uint32_t bar_f0 = smem_u32(&bar_full[0]), bar_e0 = smem_u32(&bar_empty[0]);
        uint32_t stage = 0, phase = 0, accumulate = 0;
        bool ok = true;
        for (int b = b_lo; b < b_hi; b++) {
            if (!(ok = warp_mbar_wait(bar_f0 + stage * 8, phase, abort_flag))) break;
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a_lo = s_lo0 + stage * (STAGE >> 4), b_lo2 = a_lo + ((2 * WG_BOX) >> 4);
                tc1_mma_bf16_split(tmem_base, a_lo, hi, b_lo2, hi, IDESC, accumulate);
                tc1_mma_bf16_split(tmem_base, a_lo + 128, hi, b_lo2 + 128, hi, IDESC, 1u);
                tc1_mma_bf16_split(tmem_base, a_lo + 256, hi, b_lo2 + 256, hi, IDESC, 1u);
                tc1_mma_bf16_split(tmem_base, a_lo + 384, hi, b_lo2 + 384, hi, IDESC, 1u);
                if (CS > 1) tc_commit_mc(bar_e0 + stage * 8, CMASK); else tc_commit(bar_e0 + stage * 8);
            }
            __syncwarp();
            accumulate = 1;
            if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
        }
        if (ok && elect_one()) tc_commit(smem_u32(&bar_acc));
        __syncwarp();
    } else {
        const int lane_group = warp & 3;
        bool ok = mbar_wait(smem_u32(&bar_acc), 0, abort_flag);
        ok = __all_sync(0xFFFFFFFFu, ok);
        if (ok) {
            tc_fence_after();
            const int co = mh * 128 + lane_group * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(lane_group * 32) << 16);
            float* dst = (a.partial ? a.partial + (size_t)ks * a.split_stride : wl->out) + (size_t)co * a.ldw + (size_t)tap * a.cin_pad;
#pragma unroll 1
            for (int c0 = 0; c0 < N; c0 += 32) {
                uint32_t v[32];
                tmem_ld_32x32b_x16(taddr + c0, v);
                tmem_ld_32x32b_x16(taddr + c0 + 16, v + 16);
                tmem_ld_wait();
                uint4* op = reinterpret_cast<uint4*>(dst + c0);
#pragma unroll
                for (int j = 0; j < 8; j++) op[j] = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tc_tmem_dealloc(tmem_base, 256);
    if (CS > 1) cluster_sync_all();                // no CTA leaves while the peer's commit may still arrive on its barriers
    if (threadIdx.x == 0 && abort_sh) atomicExch(a.error, 1);
}

// grad[i] = sum_s partial[s][i], s ascending (deterministic)
__global__ void k_reduce_partials(const float* partial, size_t stride, int ksplit, float* grad, size_t n) {
    pdl_trigger();
    pdl_wait();
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n) return;
    float4 acc = *reinterpret_cast<const float4*>(partial + i);
    for (int s = 1; s < ksplit; s++) {
        const float4 p = *reinterpret_cast<const float4*>(partial + (size_t)s * stride + i);
        acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
    }
    *reinterpret_cast<float4*>(grad + i) = acc;
}

// =================================================================================================
// input: gather packed records -> bf16 NHWC halo planes
// =================================================================================================
__global__ void k_gather_input(const uint64_t* states, long long n_records, int32_t* rows, int n, bf16* out, int32_t* error) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;        // (board, square, 8-channel group)
    if (i >= (size_t)n * 64 * 16) return;
    const int cg = (int)(i & 15), sq = (int)((i >> 4) & 63);
    const size_t b = i >> 10;
    int row = rows[b];
    if (row < 0 || row >= n_records) {                                     // reported by szb_train_step; the later kernels read row 0 instead
        if ((i & 1023) == 0) { atomicExch(error, 2); rows[b] = 0; }
        row = 0;
    }
    const uint64_t* p = states + (size_t)row * T_PLANES;
    uint4 o;
    __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int c = cg * 8 + 2 * j;
        const float f0 = c < T_PLANES ? (float)((p[c] >> sq) & 1ull) : 0.f;
        const float f1 = c + 1 < T_PLANES ? (float)((p[c + 1] >> sq) & 1ull) : 0.f;
        ob[j] = __floats2bfloat162_rn(f0, f1);
    }
    *reinterpret_cast<uint4*>(out + (b * TPIX + halo_pix(sq)) * TCIN + cg * 8) = o;
}

// =================================================================================================
// BatchNorm (training mode), 256 channels
// =================================================================================================
constexpr int BN_SLICES = 8;                 // blocks own 32 channels ...
constexpr int BN_GROUPS = 64;                // ... of one group of boards (few boards per thread = few dependent round trips)

// Every block first folds the per-tile column sums the convolution's epilogue left (k_tconv: stat_part [tile][2][256]) for its 32
// channels -- 8 strided partial sums, then one thread per channel adds those in a fixed order, in double.  Returns (sum 0, sum 1) to
// threads 0..31 (channel slice * 32 + t).
__device__ __forceinline__ void bn_fold_tile_sums(const float* part, int n_tiles, int slice, double (*red)[8][32], double& S1, double& S2) {
    const int t = threadIdx.x, c = t & 31, pr = t >> 5;
    double a1 = 0, a2 = 0;
    for (int tile = pr; tile < n_tiles; tile += 8) {
        a1 += (double)part[((size_t)tile * 2) * 256 + slice * 32 + c];
        a2 += (double)part[((size_t)tile * 2 + 1) * 256 + slice * 32 + c];
    }
    red[0][pr][c] = a1;
    red[1][pr][c] = a2;
    __syncthreads();
    S1 = S2 = 0;
    if (t < 32) {
#pragma unroll
        for (int i = 0; i < 8; i++) { S1 += red[0][i][t]; S2 += red[1][i][t]; }
    }
}

struct BnFwd {
    const bf16* y; const bf16* residual; bf16* out;
    const float* gamma; const float* beta;
    float* running_mean; float* running_var;
    float* mean; float* invstd;          // saved for the backward pass
    const float* part;                   // [tiles][2][256]: sum(y), sum(y^2) per tile, from the convolution's epilogue
    int n_tiles, n;
    float momentum, eps;
};

// Training-mode BatchNorm + ReLU (+ residual): batch statistics from the convolution's per-tile sums, then normalise this block's boards.
__global__ void __launch_bounds__(256) k_bn_fwd(BnFwd p) {
    __shared__ double red[2][8][32];
    __shared__ float sc_sh[32], sh_sh[32];
    pdl_trigger();
    pdl_wait();
    const int slice = blockIdx.x, grp = blockIdx.y, G = gridDim.y;
    const int t = threadIdx.x, cq = t & 3, pos = t >> 2;
    const int b_lo = (int)((long long)grp * p.n / G), b_hi = (int)((long long)(grp + 1) * p.n / G);
    double S1, S2;
    bn_fold_tile_sums(p.part, p.n_tiles, slice, red, S1, S2);
    if (t < 32) {
        const int c = slice * 32 + t;
        const double cnt = (double)p.n * 64.0, mean = S1 / cnt;
        double var = S2 / cnt - mean * mean;
        if (var < 0) var = 0;
        const float invstd = (float)(1.0 / sqrt(var + (double)p.eps));
        const float sc = p.gamma[c] * invstd;
        sc_sh[t] = sc;
        sh_sh[t] = p.beta[c] - (float)mean * sc;
        if (grp == 0) {
            p.mean[c] = (float)mean;
            p.invstd[c] = invstd;
            p.running_mean[c] = (1.f - p.momentum) * p.running_mean[c] + p.momentum * (float)mean;
            p.running_var[c] = (1.f - p.momentum) * p.running_var[c] + p.momentum * (float)(var * cnt / (cnt - 1.0));
        }
    }
    __syncthreads();
    const size_t coff = (size_t)halo_pix(pos) * TC + slice * 32 + cq * 8;
    float sc[8], sh[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { sc[j] = sc_sh[cq * 8 + j]; sh[j] = sh_sh[cq * 8 + j]; }
#pragma unroll 2
    for (int b = b_lo; b < b_hi; b++) {
        const size_t off = (size_t)b * TPIX * TC + coff;
        const uint4 v = *reinterpret_cast<const uint4*>(p.y + off);
        const bf16* vb = reinterpret_cast<const bf16*>(&v);
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; j++) f[j] = __bfloat162float(vb[j]) * sc[j] + sh[j];
        if (p.residual) {
            const uint4 rv = *reinterpret_cast<const uint4*>(p.residual + off);
            const bf16* rb = reinterpret_cast<const bf16*>(&rv);
#pragma unroll
            for (int j = 0; j < 8; j++) f[j] += __bfloat162float(rb[j]);
        }
        uint4 o;
        __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
        for (int j = 0; j < 4; j++) ob[j] = __floats2bfloat162_rn(fmaxf(f[2 * j], 0.f), fmaxf(f[2 * j + 1], 0.f));
        *reinterpret_cast<uint4*>(p.out + off) = o;
    }
}

struct BnBwd {
    const bf16* gm;                      // (d_out [+ skip]) * [out > 0], written by the dgrad convolution's epilogue
    const bf16* y;
    bf16* dy;                            // gradient of the convolution output
    const float* gamma; const float* mean; const float* invstd;
    float* g_gamma; float* g_beta;       // gradient slots of the flat gradient buffer
    const float* part;                   // [tiles][2][256]: sum(g), sum(g * xhat) per tile
    int n_tiles, n;
};

// BatchNorm backward: dy = gamma * invstd * (g - mean(g) - xhat * mean(g * xhat)); d_gamma, d_beta by the first board group.
__global__ void __launch_bounds__(256) k_bn_bwd(BnBwd p) {
    __shared__ double red[2][8][32];
    __shared__ float ca_sh[32], cb_sh[32], cc_sh[32];
    pdl_trigger();
    pdl_wait();
    const int slice = blockIdx.x, grp = blockIdx.y, G = gridDim.y;
    const int t = threadIdx.x, cq = t & 3, pos = t >> 2;
    const int b_lo = (int)((long long)grp * p.n / G), b_hi = (int)((long long)(grp + 1) * p.n / G);
    double S1, S2;
    bn_fold_tile_sums(p.part, p.n_tiles, slice, red, S1, S2);
    if (t < 32) {
        const int c = slice * 32 + t;
        const double cnt = (double)p.n * 64.0;
        ca_sh[t] = p.gamma[c] * p.invstd[c];
        cb_sh[t] = (float)(S1 / cnt);
        cc_sh[t] = (float)(S2 / cnt);
        if (grp == 0) { p.g_beta[c] = (float)S1; p.g_gamma[c] = (float)S2; }
    }
    __syncthreads();
    const int c0 = slice * 32 + cq * 8;
    const size_t coff = (size_t)halo_pix(pos) * TC + c0;
    float mean[8], invstd[8], ca[8], cb[8], cc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        mean[j] = p.mean[c0 + j]; invstd[j] = p.invstd[c0 + j];
        ca[j] = ca_sh[cq * 8 + j]; cb[j] = cb_sh[cq * 8 + j]; cc[j] = cc_sh[cq * 8 + j];
    }
#pragma unroll 2
    for (int b = b_lo; b < b_hi; b++) {
        const size_t off = (size_t)b * TPIX * TC + coff;
        const uint4 gv = *reinterpret_cast<const uint4*>(p.gm + off), yv = *reinterpret_cast<const uint4*>(p.y + off);
        const bf16* gb = reinterpret_cast<const bf16*>(&gv);
        const bf16* yb = reinterpret_cast<const bf16*>(&yv);
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; j++) f[j] = ca[j] * (__bfloat162float(gb[j]) - cb[j] - (__bfloat162float(yb[j]) - mean[j]) * invstd[j] * cc[j]);
        uint4 o;
        __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
        for (int j = 0; j < 4; j++) ob[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
        *reinterpret_cast<uint4*>(p.dy + off) = o;
    }
}

// =================================================================================================
// value head (network.py:156-174) forward + backward, fp32 SIMT (0.02 % of the step's FLOP)
// =================================================================================================
// yv[b][sq] = sum_c T[b][sq][c] * wv[c]: one warp per square
__global__ void __launch_bounds__(256) k_vconv(const bf16* T, const float* wv, float* yv, int n) {
    const int w = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= n * 64) return;
    const int b = w >> 6, sq = w & 63;
    const uint4 tv = *reinterpret_cast<const uint4*>(T + ((size_t)b * TPIX + halo_pix(sq)) * TC + lane * 8);
    const bf16* tb = reinterpret_cast<const bf16*>(&tv);
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 8; j++) acc += __bfloat162float(tb[j]) * wv[lane * 8 + j];
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    if (lane == 0) yv[w] = acc;
}

__device__ __forceinline__ double block_sum_1024(double v, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double t = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += sh[i];
    return t;
}

struct VStat { float mean, invstd; };

// one-channel BatchNorm statistics over all n*64 values (single block)
__global__ void __launch_bounds__(1024) k_vbn_stats(const float* yv, int n, float* running_mean, float* running_var, VStat* st, float momentum, float eps) {
    __shared__ double sh[32];
    double s1 = 0, s2 = 0;
    for (int i = threadIdx.x; i < n * 64; i += blockDim.x) { const double v = yv[i]; s1 += v; s2 += v * v; }
    s1 = block_sum_1024(s1, sh);
    s2 = block_sum_1024(s2, sh);
    if (threadIdx.x == 0) {
        const double cnt = (double)n * 64.0, mean = s1 / cnt;
        double var = s2 / cnt - mean * mean;
        if (var < 0) var = 0;
        st->mean = (float)mean;
        st->invstd = (float)(1.0 / sqrt(var + (double)eps));
        *running_mean = (1.f - momentum) * *running_mean + momentum * (float)mean;
        *running_var = (1.f - momentum) * *running_var + momentum * (float)(var * cnt / (cnt - 1.0));
    }
}

struct VHead {
    const float* yv; const VStat* st;
    const float* gamma; const float* beta;               // v_norm
    const float* fc1_w; const float* fc1_b;              // [256][64], [256]
    const float* fc2_w; const float* fc2_b;              // [256], [1]
    const int8_t* z; const int32_t* rows;
    float* value; float* se;                             // [n]: tanh output, squared error
    float* r; float* dh1; float* h1r; float* du; float* gr;    // saved for the gradient kernels: [n][64], [n][256], [n][256], [n], [n][64]
    int n;
};

// per board: BN -> ReLU -> fc1 -> ReLU -> fc2 -> tanh, squared error, and the backward pass down to the gradient of the BN output
__global__ void __launch_bounds__(256) k_vhead(VHead p) {
    __shared__ float r_sh[64], dh_sh[256], red[8];
    const int b = blockIdx.x, t = threadIdx.x;
    const float mean = p.st->mean, invstd = p.st->invstd;
    if (t < 64) {
        const float xh = (p.yv[b * 64 + t] - mean) * invstd;
        const float r = fmaxf(xh * p.gamma[0] + p.beta[0], 0.f);
        r_sh[t] = r;
        p.r[b * 64 + t] = r;
    }
    __syncthreads();
    float h = p.fc1_b[t];
    const float* w1 = p.fc1_w + t * 64;
#pragma unroll 8
    for (int s = 0; s < 64; s++) h += w1[s] * r_sh[s];
    const float hr = fmaxf(h, 0.f);
    float acc = hr * p.fc2_w[t];
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    if ((t & 31) == 0) red[t >> 5] = acc;
    __syncthreads();
    float u = p.fc2_b[0];
#pragma unroll
    for (int i = 0; i < 8; i++) u += red[i];
    const float v = tanhf(u);
    const float zt = (float)p.z[p.rows[b]];
    const float du = 2.f * (v - zt) / (float)p.n * (1.f - v * v);
    if (t == 0) { p.value[b] = v; p.se[b] = (v - zt) * (v - zt); p.du[b] = du; }
    const float dh = h > 0.f ? du * p.fc2_w[t] : 0.f;
    dh_sh[t] = dh;
    p.dh1[b * 256 + t] = dh;
    p.h1r[b * 256 + t] = hr;
    __syncthreads();
    if (t < 64) {
        float dr = 0.f;
        for (int j = 0; j < 256; j++) dr += dh_sh[j] * p.fc1_w[j * 64 + t];
        p.gr[b * 64 + t] = r_sh[t] > 0.f ? dr : 0.f;
    }
}

// one-channel BatchNorm backward over all n*64 values (single block): dyv, d_gamma, d_beta
__global__ void __launch_bounds__(1024) k_vbn_bwd(const float* yv, const float* gr, const VStat* st, const float* gamma, float* g_gamma, float* g_beta,
                                                  float* dyv, int n) {
    __shared__ double sh[32];
    const float mean = st->mean, invstd = st->invstd;
    double s1 = 0, s2 = 0;
    for (int i = threadIdx.x; i < n * 64; i += blockDim.x) { const double g = gr[i]; s1 += g; s2 += g * (double)((yv[i] - mean) * invstd); }
    s1 = block_sum_1024(s1, sh);
    s2 = block_sum_1024(s2, sh);
    const double cnt = (double)n * 64.0;
    if (threadIdx.x == 0) { *g_beta = (float)s1; *g_gamma = (float)s2; }
    const float ca = gamma[0] * invstd, cb = (float)(s1 / cnt), cc = (float)(s2 / cnt);
    for (int i = threadIdx.x; i < n * 64; i += blockDim.x) dyv[i] = ca * (gr[i] - cb - (yv[i] - mean) * invstd * cc);
}

// per board: the value branch's share of the tower-output gradient (bf16, added as the "skip" term of the last block) and this board's
// partial of d conv_v1.weight
__global__ void __launch_bounds__(256) k_vconv_bwd(const bf16* T, const float* wv, const float* dyv, bf16* skip, float* part) {
    const int b = blockIdx.x, c = threadIdx.x;
    const float w = wv[c];
    float acc = 0.f;
    for (int sq = 0; sq < 64; sq++) {
        const size_t o = ((size_t)b * TPIX + halo_pix(sq)) * TC + c;
        const float d = dyv[b * 64 + sq];
        acc += d * __bfloat162float(T[o]);
        skip[o] = __float2bfloat16(d * w);
    }
    part[(size_t)b * 256 + c] = acc;
}

// out[j] = sum_i part[i][j], i ascending
__global__ void k_colsum(const float* part, int rows, int cols, int ld, float* out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cols) return;
    float acc = 0.f;
    for (int i = 0; i < rows; i++) acc += part[(size_t)i * ld + j];
    out[j] = acc;
}

// d fc_v1.weight[j][sq] = sum_b dh1[b][j] * r[b][sq];  d fc_v1.bias[j] = sum_b dh1[b][j];  d fc_v2.weight[j] = sum_b du[b] * h1r[b][j];  d fc_v2.bias
__global__ void __launch_bounds__(256) k_vhead_grads(const float* dh1, const float* r, const float* h1r, const float* du, int n, float* g_fc1w, float* g_fc1b,
                                                     float* g_fc2w, float* g_fc2b) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 256 * 64) {
        const int j = i >> 6, sq = i & 63;
        float acc = 0.f;
        for (int b = 0; b < n; b++) acc += dh1[b * 256 + j] * r[b * 64 + sq];
        g_fc1w[i] = acc;
    } else if (i < 256 * 64 + 256) {
        const int j = i - 256 * 64;
        float a1 = 0.f, a2 = 0.f;
        for (int b = 0; b < n; b++) { a1 += dh1[b * 256 + j]; a2 += du[b] * h1r[b * 256 + j]; }
        g_fc1b[j] = a1;
        g_fc2w[j] = a2;
    } else if (i == 256 * 64 + 256) {
        float a = 0.f;
        for (int b = 0; b < n; b++) a += du[b];
        g_fc2b[0] = a;
    }
}

// =================================================================================================
// policy loss: cross entropy with a soft target over all 4672 logits (torch.nn.functional.cross_entropy with probabilities)
// =================================================================================================
struct LossArgs {
    const float* logits;                 // [n][4672]
    const int32_t* rows;                 // record row of each batch slot
    const long long* pi_off; const uint16_t* pi_index; const float* pi_prob;   // CSR over ALL records
    bf16* dl;                            // [n][10][10][128] halo NHWC gradient of the logits (x 1/n)
    float* ce;                           // [n]
    float* db_part;                      // [n][128] per-board sums of the gradient per policy plane (conv_p2.bias)
    int n;
};

__global__ void __launch_bounds__(256) k_policy_loss(LossArgs a) {
    __shared__ float dl[73 * 65];
    __shared__ float red[8];
    __shared__ float bc;
    const int b = blockIdx.x, t = threadIdx.x;
    const float* lg = a.logits + (size_t)b * T_ACTIONS;
    float m = -INFINITY;
    for (int j = t; j < T_ACTIONS; j += 256) m = fmaxf(m, lg[j]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((t & 31) == 0) red[t >> 5] = m;
    __syncthreads();
    if (t == 0) { float x = red[0]; for (int i = 1; i < 8; i++) x = fmaxf(x, red[i]); bc = x; }
    __syncthreads();
    m = bc;
    float s = 0.f;
    for (int j = t; j < T_ACTIONS; j += 256) s += expf(lg[j] - m);
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    __syncthreads();
    if ((t & 31) == 0) red[t >> 5] = s;
    __syncthreads();
    if (t == 0) { float x = 0.f; for (int i = 0; i < 8; i++) x += red[i]; bc = m + logf(x); }
    __syncthreads();
    const float lse = bc;
    // target mass and cross entropy over the sparse target
    const int row = a.rows[b];
    const long long lo = a.pi_off[row], hi = a.pi_off[row + 1];
    float mass = 0.f, ce = 0.f;
    for (long long e = lo + t; e < hi; e += 256) {
        const float p = a.pi_prob[e];
        mass += p;
        ce -= p * (lg[a.pi_index[e]] - lse);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { mass += __shfl_xor_sync(0xFFFFFFFFu, mass, o); ce += __shfl_xor_sync(0xFFFFFFFFu, ce, o); }
    __syncthreads();
    if ((t & 31) == 0) red[t >> 5] = mass;
    __syncthreads();
    if (t == 0) { float x = 0.f; for (int i = 0; i < 8; i++) x += red[i]; bc = x; }
    __syncthreads();
    mass = bc;
    __syncthreads();
    if ((t & 31) == 0) red[t >> 5] = ce;
    __syncthreads();
    if (t == 0) { float x = 0.f; for (int i = 0; i < 8; i++) x += red[i]; a.ce[b] = x; }
    const float inv_n = 1.f / (float)a.n;
    for (int j = t; j < T_ACTIONS; j += 256) dl[(j >> 6) * 65 + (j & 63)] = expf(lg[j] - lse) * mass * inv_n;
    __syncthreads();
    for (long long e = lo + t; e < hi; e += 256) {
        const int j = a.pi_index[e];
        dl[(j >> 6) * 65 + (j & 63)] -= a.pi_prob[e] * inv_n;       // indices of one position are distinct
    }
    __syncthreads();
    if (t < DL_C) {
        float acc = 0.f;
        if (t < 73) for (int sq = 0; sq < 64; sq++) acc += dl[t * 65 + sq];
        a.db_part[(size_t)b * DL_C + t] = acc;
    }
    for (int e = t; e < 64 * DL_C; e += 256) {
        const int sq = e >> 7, c = e & (DL_C - 1);
        a.dl[((size_t)b * TPIX + halo_pix(sq)) * DL_C + c] = __float2bfloat16(c < 73 ? dl[c * 65 + sq] : 0.f);
    }
}

// losses[0] = mean squared error, losses[1] = mean cross entropy (sequential sums: deterministic)
// ... and appended to a ring of the last LOSS_HIST steps' losses, so that a training loop can queue steps without a host round trip each
// and read the history back in bulk (szb_train_loss_history)
constexpr int LOSS_HIST = 1 << 16;
__global__ void k_loss_reduce(const float* se, const float* ce, int n, float* losses, float* hist, unsigned long long* hist_count) {
    if (threadIdx.x == 0) {
        double a = 0, c = 0;
        for (int i = 0; i < n; i++) { a += se[i]; c += ce[i]; }
        losses[0] = (float)(a / n);
        losses[1] = (float)(c / n);
        const unsigned long long k = (*hist_count)++ % LOSS_HIST;
        hist[2 * k] = losses[0];
        hist[2 * k + 1] = losses[1];
    }
}

// =================================================================================================
// optimiser + weight packs
// =================================================================================================
// torch.optim.Adam (weight decay added to the gradient, bias-corrected moments), one thread per parameter of the flat buffer
// advances the optimiser step counter ON THE DEVICE and derives what k_adam needs from it (StepLR learning rate over Adam's first bias
// correction, square root of the second): a captured step replays without any host-side parameter
__global__ void k_hyper(long long* step, float lr0, float lr_gamma, int lr_step, float beta1, float beta2, float* hyper) {
    const long long t = ++*step;
    const double lr = (double)lr0 * pow((double)lr_gamma, (double)((t - 1) / (lr_step > 0 ? lr_step : 1)));
    hyper[0] = (float)(lr / (1.0 - pow((double)beta1, (double)t)));
    hyper[1] = (float)sqrt(1.0 - pow((double)beta2, (double)t));
}

__global__ void k_adam(float* w, const float* g, float* m, float* v, size_t n, const float* hyper, float beta1, float beta2, float eps, float wd) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float step_size = hyper[0], bc2_sqrt = hyper[1];
    const float p = w[i];
    const float gg = g[i] + wd * p;
    const float mm = m[i] + (gg - m[i]) * (1.f - beta1);
    const float vv = beta2 * v[i] + (1.f - beta2) * gg * gg;
    m[i] = mm;
    v[i] = vv;
    w[i] = p - step_size * (mm / (sqrtf(vv) / bc2_sqrt + eps));
}

// torch.optim.SGD (_single_tensor_sgd): the same device step counter and StepLR learning rate, no bias correction.  hyper[1] records
// whether the momentum buffers existed BEFORE this step (torch's first step clones the gradient instead of blending it in); the flag is
// then raised for the steps after, all on the device, so a captured step replays the first and the later steps alike
__global__ void k_hyper_sgd(long long* step, float lr0, float lr_gamma, int lr_step, int32_t* have_buf, float* hyper) {
    const long long t = ++*step;
    hyper[0] = (float)((double)lr0 * pow((double)lr_gamma, (double)((t - 1) / (lr_step > 0 ? lr_step : 1))));
    hyper[1] = *have_buf ? 1.f : 0.f;
    *have_buf = 1;
}

__global__ void k_sgd(float* w, const float* g, float* buf, size_t n, const float* hyper, float momentum, float dampening, int nesterov, float wd) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float lr = hyper[0];
    const float p = w[i];
    float d = g[i] + wd * p;
    if (momentum != 0.f) {
        const float b = hyper[1] != 0.f ? momentum * buf[i] + (1.f - dampening) * d : d;
        buf[i] = b;
        d = nesterov ? d + momentum * b : b;
    }
    w[i] = p - lr * d;
}

struct PackDesc {
    const float* w;      // master [cout_pad][taps][cin_pad]
    bf16* wf;            // forward pack, same layout
    bf16* wd;            // dgrad pack [cin_pad][taps][cout_pad] with the taps mirrored, or null
    int cout_pad, taps, cin_pad;
};

// 32 x 32 (co, ci) tiles of one tap through shared memory: the master is read once, both packs are written in 64-byte runs
__global__ void __launch_bounds__(256) k_pack(const PackDesc* descs) {
    __shared__ float tile[32][33];
    const PackDesc d = descs[blockIdx.y];
    const int tiles_ci = d.cin_pad / 32, tiles_co = d.cout_pad / 32;
    const int n_tiles = d.taps * tiles_co * tiles_ci;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
        const int tci = tl % tiles_ci, tco = (tl / tiles_ci) % tiles_co, tap = tl / (tiles_ci * tiles_co);
#pragma unroll
        for (int r = ty; r < 32; r += 8) {
            const size_t i = ((size_t)(tco * 32 + r) * d.taps + tap) * d.cin_pad + tci * 32 + tx;
            const float x = d.w[i];
            d.wf[i] = __float2bfloat16(x);
            tile[r][tx] = x;
        }
        __syncthreads();
        if (d.wd) {
#pragma unroll
            for (int r = ty; r < 32; r += 8)
                d.wd[((size_t)(tci * 32 + r) * d.taps + (d.taps - 1 - tap)) * d.cout_pad + tco * 32 + tx] = __float2bfloat16(tile[tx][r]);
        }
        __syncthreads();
    }
}

// torch [cout][cin][taps] <-> packed [cout_pad][taps][cin_pad]
__global__ void k_conv_to_packed(const float* src, float* dst, int cout, int cin, int taps, int cout_pad, int cin_pad) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)cout_pad * taps * cin_pad) return;
    const int ci = (int)(i % cin_pad), tap = (int)((i / cin_pad) % taps), co = (int)(i / ((size_t)cin_pad * taps));
    dst[i] = (co < cout && ci < cin) ? src[((size_t)co * cin + ci) * taps + tap] : 0.f;
}
__global__ void k_packed_to_conv(const float* src, float* dst, int cout, int cin, int taps, int cin_pad) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)cout * cin * taps) return;
    const int tap = (int)(i % taps), ci = (int)((i / taps) % cin), co = (int)(i / ((size_t)taps * cin));
    dst[i] = src[((size_t)co * taps + tap) * cin_pad + ci];
}

// =================================================================================================
// host side
// =================================================================================================
struct TParam {
    std::string name;
    int kind = 0;                // 0: vector (stored as torch has it), 1: convolution weight (stored packed)
    int64_t numel = 0;           // torch element count
    size_t off = 0, n = 0;       // slot in the flat buffers
    int cout = 0, cin = 0, taps = 0, cout_pad = 0, cin_pad = 0;
};
struct TBuffer { std::string name; int64_t numel; float* ptr; };

struct TLayer {
    int taps = 9, cin_pad = 256, cout_pad = 256;
    int param = -1, gamma = -1, beta = -1;       // indices into Trainer::params
    bf16* wf = nullptr; bf16* wd = nullptr;
    CUtensorMap tm_wf[2], tm_wd[2];              // box rows: [0] 32 (k_tconv: a quarter tile per CTA of the cluster), [1] 64 (k_tconv_pair: half a tile)
    bf16* y = nullptr; bf16* o = nullptr;        // pre-BatchNorm convolution output, layer output
    bf16* dy = nullptr;                          // gradient of the convolution output (kept per layer: every tower wgrad runs in ONE launch at the end)
    CUtensorMap tm_dy2, tm_dy1;
    CUtensorMap tm_o2, tm_o1;                    // layer output as the next layer's operand: 2-board boxes (forward), 1-board boxes (wgrad)
    float* bn = nullptr;                         // running_mean, running_var, mean, invstd: 4 x 256
};

struct Trainer {
    szb_train_config cfg{};
    int cap = 0;                                 // boards (even)
    std::vector<TParam> params;
    std::map<std::string, int> index;
    std::vector<TBuffer> buffers;
    size_t total = 0;
    float *w = nullptr, *g = nullptr, *m = nullptr, *v = nullptr;
    TLayer L[T_LAYERS];
    bf16* x_in = nullptr; CUtensorMap tm_in2, tm_in1;
    bf16 *dl = nullptr, *gm1 = nullptr, *skip[2] = {nullptr, nullptr};
    CUtensorMap tm_dl2, tm_dl1;
    WgLayer* wg_layers = nullptr;                // [T_LAYERS] device table of k_wgrad
    unsigned long long* trace = nullptr;         // SZB_TRAIN_TRACE=1: stamps of the forward convolution of layer 20
    float* logits = nullptr;
    float* partial = nullptr; size_t partial_floats = 0;
    float* bn_part = nullptr;                    // [tiles][2][256] per-tile sums from the convolution epilogues
    // value head
    float *yv = nullptr, *vr = nullptr, *dh1 = nullptr, *h1r = nullptr, *du = nullptr, *gr = nullptr, *dyv = nullptr, *value = nullptr, *se = nullptr, *ce = nullptr;
    float *vpart = nullptr, *db_part = nullptr, *v_running = nullptr;
    VStat* vstat = nullptr;
    float* losses = nullptr;
    float* loss_hist = nullptr; unsigned long long* hist_count = nullptr;      // device ring of per-step losses and its step counter
    int64_t steps_run = 0;                                                     // host mirror of *hist_count
    PackDesc* pack_descs = nullptr;
    int32_t* error = nullptr;
    int32_t* rows = nullptr;
    // records on the device
    uint64_t* rec_states = nullptr; long long* rec_off = nullptr; uint16_t* rec_index = nullptr; float* rec_prob = nullptr; int8_t* rec_z = nullptr;
    int64_t rec_n = 0;
    int64_t step = 0;                            // host mirror of *d_step
    long long* d_step = nullptr; float* hyper = nullptr;
    // optimiser (szb_train_set_optimizer): fixed before the first step, so no captured step depends on it.  SGD keeps its momentum
    // buffers in `m` (Adam's first moment, unused under SGD); *d_have_buf: they hold a value (torch's "momentum_buffer" state exists)
    int32_t opt_kind = SZB_TRAIN_ADAM;
    float momentum = 0.f, dampening = 0.f;
    int32_t nesterov = 0;
    int32_t* d_have_buf = nullptr;
    int32_t* rows_host = nullptr;                // [ROWS_RING][cap] pinned staging of the steps' row numbers
    cudaEvent_t rows_ev[8] = {};
    bool rows_used[8] = {};
    uint64_t steps_queued = 0;
    std::map<std::pair<int, int>, cudaGraphExec_t> graphs;     // (boards, flags) -> the captured step
    bool use_graph = true;
    bool conv_pair = true;                       // convolutions as CTA pairs (k_tconv_pair); SZB_TRAIN_CONV=1: the single-CTA kernel with multicast weights
    bool pdl = true;                             // programmatic dependent launch along the convolution / BatchNorm chain (SZB_TRAIN_NO_PDL=1: off)
    std::map<std::pair<int, int>, uint64_t> launches_per_step;
    int last_n = 0;
    bool loaded = false, attr_set = false;
    std::vector<bool> have_param, have_buffer;   // set at least once through szb_train_set(SZB_TRAIN_PARAMS)
    std::vector<void*> allocs;
};

template <class T>
static int t_alloc(szb_ctx* ctx, Trainer* tr, T** p, size_t count) {
    SZB_CUDA(ctx, cudaMalloc((void**)p, count * sizeof(T)));
    tr->allocs.push_back(*p);
    SZB_CUDA(ctx, cudaMemsetAsync(*p, 0, count * sizeof(T), ctx->stream));
    return 0;
}

void trainer_destroy(szb_ctx* ctx) {
    Trainer* tr = ctx->trainer;
    if (!tr) return;
    cudaStreamSynchronize(ctx->stream);
    for (void* p : tr->allocs) cudaFree(p);
    for (auto& kv : tr->graphs) cudaGraphExecDestroy(kv.second);
    if (tr->rows_host) cudaFreeHost(tr->rows_host);
    for (int i = 0; i < ROWS_RING; i++) if (tr->rows_ev[i]) cudaEventDestroy(tr->rows_ev[i]);
    void* rec[5] = {tr->rec_states, tr->rec_off, tr->rec_index, tr->rec_prob, tr->rec_z};
    for (void* p : rec) if (p) cudaFree(p);
    delete tr;
    ctx->trainer = nullptr;
}

static void t_add_vec(Trainer* tr, const std::string& name, int64_t n) {
    TParam p;
    p.name = name; p.kind = 0; p.numel = n; p.n = (size_t)((n + 3) & ~3LL);
    tr->index[name] = (int)tr->params.size();
    tr->params.push_back(p);
}
static void t_add_conv(Trainer* tr, const std::string& name, int cout, int cin, int taps, int cout_pad, int cin_pad) {
    TParam p;
    p.name = name; p.kind = 1; p.numel = (int64_t)cout * cin * taps;
    p.cout = cout; p.cin = cin; p.taps = taps; p.cout_pad = cout_pad; p.cin_pad = cin_pad;
    p.n = (size_t)cout_pad * taps * cin_pad;
    tr->index[name] = (int)tr->params.size();
    tr->params.push_back(p);
}

// the parameters in the order network.py registers them (torch.optim.Adam's state is numbered in this order)
static void t_build_params(Trainer* tr) {
    auto bn = [&](const std::string& p, int c) { t_add_vec(tr, p + ".weight", c); t_add_vec(tr, p + ".bias", c); };
    t_add_conv(tr, "conv1.weight", 256, 119, 9, 256, TCIN);
    bn("norm_layer", 256);
    t_add_conv(tr, "conv_p1.weight", 256, 256, 1, 256, 256);
    bn("p_norm1", 256);
    t_add_conv(tr, "conv_p2.weight", 73, 256, 1, 128, 256);
    t_add_vec(tr, "conv_p2.bias", 73);
    t_add_vec(tr, "conv_v1.weight", 256);
    bn("v_norm", 1);
    t_add_vec(tr, "fc_v1.weight", 256 * 64); t_add_vec(tr, "fc_v1.bias", 256);
    t_add_vec(tr, "fc_v2.weight", 256); t_add_vec(tr, "fc_v2.bias", 1);
    for (int b = 0; b < 19; b++)
        for (int j = 1; j <= 2; j++) {
            const std::string pfx = "resnet_blocks." + std::to_string(b);
            t_add_conv(tr, pfx + ".conv" + std::to_string(j) + ".weight", 256, 256, 9, 256, 256);
            bn(pfx + ".bn" + std::to_string(j), 256);
        }
    size_t off = 0;
    for (auto& p : tr->params) { p.off = off; off += p.n; }
    tr->total = off;
}

static std::string t_layer_conv_name(int l) {
    if (l == 0) return "conv1";
    if (l == L_P1) return "conv_p1";
    if (l == L_P2) return "conv_p2";
    return "resnet_blocks." + std::to_string((l - 1) / 2) + ".conv" + std::to_string((l - 1) % 2 + 1);
}
static std::string t_layer_bn_name(int l) {
    if (l == 0) return "norm_layer";
    if (l == L_P1) return "p_norm1";
    return "resnet_blocks." + std::to_string((l - 1) / 2) + ".bn" + std::to_string((l - 1) % 2 + 1);
}

static int t_create(szb_ctx* ctx, const szb_train_config* cfg) {
    int rc;
    if ((rc = net_tmap_init(ctx))) return rc;
    trainer_destroy(ctx);
    Trainer* tr = new Trainer();
    ctx->trainer = tr;
    tr->cfg = *cfg;
    tr->cap = (cfg->batch + 1) & ~1;
    tr->step = cfg->step0;
    t_build_params(tr);
    const int cap = tr->cap;
    const size_t act = (size_t)cap * TPIX * TC;
    // the two tensor maps of an activation buffer (2-board halo chunks, 1-board boxes) and of a weight pack (32 / 64 rows): see TLayer
    auto act_maps = [&](CUtensorMap* chunk, CUtensorMap* board, void* base, int channels) {
        const int r = net_tmap_halo(ctx, chunk, base, channels, cap, 2, "training halo activations");
        return r ? r : net_tmap_act(ctx, board, base, channels, cap, 1, "training activations");
    };
    auto w_maps = [&](CUtensorMap* tm, void* base, int k_total, int rows) {
        const int r = net_tmap_rows(ctx, &tm[0], base, k_total, rows, 128 / TR_CLUSTER, "training weights");
        return r ? r : net_tmap_rows(ctx, &tm[1], base, k_total, rows, 64, "training weights");
    };
    if ((rc = t_alloc(ctx, tr, &tr->w, tr->total)) || (rc = t_alloc(ctx, tr, &tr->g, tr->total)) || (rc = t_alloc(ctx, tr, &tr->m, tr->total)) ||
        (rc = t_alloc(ctx, tr, &tr->v, tr->total)))
        return rc;
    if ((rc = t_alloc(ctx, tr, &tr->x_in, (size_t)cap * TPIX * TCIN))) return rc;
    if ((rc = act_maps(&tr->tm_in2, &tr->tm_in1, tr->x_in, TCIN))) return rc;
    for (int l = 0; l < T_LAYERS; l++) {
        TLayer& L = tr->L[l];
        L.taps = (l == L_P1 || l == L_P2) ? 1 : 9;
        L.cin_pad = l == 0 ? TCIN : 256;
        L.cout_pad = l == L_P2 ? 128 : 256;
        L.param = tr->index.at(t_layer_conv_name(l) + ".weight");
        const size_t wn = (size_t)L.cout_pad * L.taps * L.cin_pad;
        if ((rc = t_alloc(ctx, tr, &L.wf, wn))) return rc;
        if ((rc = w_maps(L.tm_wf, L.wf, L.taps * L.cin_pad, L.cout_pad))) return rc;
        if (l != 0) {
            if ((rc = t_alloc(ctx, tr, &L.wd, wn))) return rc;
            if ((rc = w_maps(L.tm_wd, L.wd, L.taps * L.cout_pad, L.cin_pad))) return rc;
        }
        if (l < T_BN) {
            L.gamma = tr->index.at(t_layer_bn_name(l) + ".weight");
            L.beta = tr->index.at(t_layer_bn_name(l) + ".bias");
            if ((rc = t_alloc(ctx, tr, &L.y, act)) || (rc = t_alloc(ctx, tr, &L.o, act)) || (rc = t_alloc(ctx, tr, &L.dy, act)) ||
                (rc = t_alloc(ctx, tr, &L.bn, 4 * 256)))
                return rc;
            if ((rc = act_maps(&L.tm_o2, &L.tm_o1, L.o, TC)) || (rc = act_maps(&L.tm_dy2, &L.tm_dy1, L.dy, TC))) return rc;
            tr->buffers.push_back({t_layer_bn_name(l) + ".running_mean", 256, L.bn});
            tr->buffers.push_back({t_layer_bn_name(l) + ".running_var", 256, L.bn + 256});
        }
    }
    if (        (rc = t_alloc(ctx, tr, &tr->gm1, act)) || (rc = t_alloc(ctx, tr, &tr->skip[0], act)) || (rc = t_alloc(ctx, tr, &tr->skip[1], act)) ||
        (rc = t_alloc(ctx, tr, &tr->dl, (size_t)cap * TPIX * DL_C)))
        return rc;
    if ((rc = act_maps(&tr->tm_dl2, &tr->tm_dl1, tr->dl, DL_C))) return rc;
    tr->partial_floats = (size_t)WG_MAX_SPLIT * 256 * 256;                      // 1x1 layers: up to 64 splits of 256 x 256
    if (tr->partial_floats < (size_t)8 * 256 * 2304) tr->partial_floats = (size_t)8 * 256 * 2304;
    if ((rc = t_alloc(ctx, tr, &tr->partial, tr->partial_floats)) || (rc = t_alloc(ctx, tr, &tr->logits, (size_t)cap * T_ACTIONS)) ||
        (rc = t_alloc(ctx, tr, &tr->bn_part, (size_t)(cap / 2) * 512)) ||
        (rc = t_alloc(ctx, tr, &tr->yv, (size_t)cap * 64)) || (rc = t_alloc(ctx, tr, &tr->vr, (size_t)cap * 64)) ||
        (rc = t_alloc(ctx, tr, &tr->dh1, (size_t)cap * 256)) || (rc = t_alloc(ctx, tr, &tr->h1r, (size_t)cap * 256)) ||
        (rc = t_alloc(ctx, tr, &tr->du, (size_t)cap)) || (rc = t_alloc(ctx, tr, &tr->gr, (size_t)cap * 64)) ||
        (rc = t_alloc(ctx, tr, &tr->dyv, (size_t)cap * 64)) || (rc = t_alloc(ctx, tr, &tr->value, (size_t)cap)) ||
        (rc = t_alloc(ctx, tr, &tr->se, (size_t)cap)) || (rc = t_alloc(ctx, tr, &tr->ce, (size_t)cap)) ||
        (rc = t_alloc(ctx, tr, &tr->vpart, (size_t)cap * 256)) || (rc = t_alloc(ctx, tr, &tr->db_part, (size_t)cap * DL_C)) ||
        (rc = t_alloc(ctx, tr, &tr->v_running, 4)) || (rc = t_alloc(ctx, tr, &tr->vstat, 1)) || (rc = t_alloc(ctx, tr, &tr->losses, 2)) ||
        (rc = t_alloc(ctx, tr, &tr->error, 1)) || (rc = t_alloc(ctx, tr, &tr->rows, (size_t)cap)) ||
        (rc = t_alloc(ctx, tr, &tr->pack_descs, (size_t)T_LAYERS)) || (rc = t_alloc(ctx, tr, &tr->d_step, 1)) || (rc = t_alloc(ctx, tr, &tr->hyper, 2)) ||
        (rc = t_alloc(ctx, tr, &tr->d_have_buf, 1)) ||
        (rc = t_alloc(ctx, tr, &tr->loss_hist, (size_t)2 * LOSS_HIST)) || (rc = t_alloc(ctx, tr, &tr->hist_count, 1)))
        return rc;
    SZB_CUDA(ctx, cudaMallocHost((void**)&tr->rows_host, (size_t)ROWS_RING * cap * 4));
    for (int i = 0; i < ROWS_RING; i++) SZB_CUDA(ctx, cudaEventCreateWithFlags(&tr->rows_ev[i], cudaEventDisableTiming));
    {
        const long long s0 = cfg->step0;
        SZB_CUDA(ctx, cudaMemcpyAsync(tr->d_step, &s0, 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    tr->have_param.assign(tr->params.size(), false);
    tr->have_buffer.assign(tr->buffers.size(), false);
    if (const char* e = getenv("SZB_TRAIN_NO_GRAPH")) tr->use_graph = atoi(e) == 0;
    if (const char* e = getenv("SZB_TRAIN_NO_PDL")) tr->pdl = atoi(e) == 0;
    if (const char* e = getenv("SZB_TRAIN_CONV")) tr->conv_pair = atoi(e) != 1;
    if (const char* e = getenv("SZB_TRAIN_TRACE")) {
        if (atoi(e) && (rc = t_alloc(ctx, tr, &tr->trace, 8))) return rc;
    }
    tr->buffers.push_back({"v_norm.running_mean", 1, tr->v_running});
    tr->buffers.push_back({"v_norm.running_var", 1, tr->v_running + 1});
    std::vector<PackDesc> pd(T_LAYERS);
    for (int l = 0; l < T_LAYERS; l++) {
        const TLayer& L = tr->L[l];
        pd[l] = PackDesc{tr->w + tr->params[L.param].off, L.wf, L.wd, L.cout_pad, L.taps, L.cin_pad};
    }
    SZB_CUDA(ctx, cudaMemcpyAsync(tr->pack_descs, pd.data(), sizeof(PackDesc) * T_LAYERS, cudaMemcpyHostToDevice, ctx->stream));
    std::vector<WgLayer> wl(T_LAYERS);
    for (int l = 0; l < T_LAYERS; l++) {
        memset(&wl[l], 0, sizeof(WgLayer));
        wl[l].tm_dy = l == L_P2 ? tr->tm_dl1 : tr->L[l].tm_dy1;
        wl[l].tm_x = l == 0 ? tr->tm_in1 : l == L_P1 ? tr->L[38].tm_o1 : l == L_P2 ? tr->L[L_P1].tm_o1 : tr->L[l - 1].tm_o1;
        wl[l].out = tr->g + tr->params[tr->L[l].param].off;
    }
    if ((rc = t_alloc(ctx, tr, &tr->wg_layers, (size_t)T_LAYERS))) return rc;
    SZB_CUDA(ctx, cudaMemcpyAsync(tr->wg_layers, wl.data(), sizeof(WgLayer) * T_LAYERS, cudaMemcpyHostToDevice, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!tr->attr_set) {
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_tconv<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, TR_SMEM));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_tconv<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TR_SMEM));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_tconv_pair<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_tconv_pair<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_wgrad<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_STAGES * 6 * WG_BOX + 1024));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_wgrad<4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_STAGES * 6 * WG_BOX + 1024));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_wgrad<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_STAGES * 4 * WG_BOX + 1024));
        tr->attr_set = true;
    }
    return 0;
}

static int t_pack(szb_ctx* ctx, Trainer* tr) {
    k_pack<<<dim3(144, T_LAYERS), 256, 0, ctx->stream>>>(tr->pack_descs);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

static float* t_kind_base(Trainer* tr, int kind) {
    return kind == 0 ? tr->w : kind == 1 ? tr->g : (kind == 2 || kind == SZB_TRAIN_MOMENTUM_BUFFER) ? tr->m : kind == 3 ? tr->v : nullptr;
}

// copy tensors by name between caller memory (host or device, torch layout) and the flat buffers
static int t_transfer(szb_ctx* ctx, int kind, int32_t n_tensors, const char* const* names, float* const* data, const int64_t* numel, bool to_trainer) {
    Trainer* tr = ctx->trainer;
    if (!tr) return fail(ctx, SZB_ERR_ARG, "no trainer: call szb_train_create first");
    if (kind < 0 || kind > SZB_TRAIN_MOMENTUM_BUFFER || n_tensors < 0 || (n_tensors && (!names || !data || !numel)))
        return fail(ctx, SZB_ERR_ARG, "szb_train_get/set: bad arguments");
    const bool sgd = tr->opt_kind == SZB_TRAIN_SGD;
    if ((kind == SZB_TRAIN_EXP_AVG || kind == SZB_TRAIN_EXP_AVG_SQ) && sgd) return fail(ctx, SZB_ERR_STATE, "the trainer runs SGD: it has no Adam moments");
    if (kind == SZB_TRAIN_MOMENTUM_BUFFER && !(sgd && tr->momentum != 0.f))
        return fail(ctx, SZB_ERR_STATE, "momentum buffers exist only under SGD with momentum (szb_train_set_optimizer)");
    float* scratch = nullptr;
    int rc = 0;
    for (int i = 0; i < n_tensors && !rc; i++) {
        const std::string name = names[i];
        if (kind == 4) {
            if (to_trainer) { rc = fail(ctx, SZB_ERR_ARG, "activations are read-only"); break; }
            const float* src = nullptr;
            int64_t cnt = 0;
            if (name == "logits") { src = tr->logits; cnt = (int64_t)tr->last_n * T_ACTIONS; }
            else if (name == "value") { src = tr->value; cnt = tr->last_n; }
            else { rc = fail(ctx, SZB_ERR_ARG, "unknown activation '%s'", name.c_str()); break; }
            if (numel[i] != cnt) { rc = fail(ctx, SZB_ERR_ARG, "'%s' has %lld elements, caller expects %lld", name.c_str(), (long long)cnt, (long long)numel[i]); break; }
            cudaError_t e = cudaMemcpyAsync(data[i], src, (size_t)cnt * 4, cudaMemcpyDefault, ctx->stream);
            if (e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaMemcpyAsync(activation)");
            continue;
        }
        auto it = tr->index.find(name);
        if (it == tr->index.end()) {
            const TBuffer* bf = nullptr;
            for (auto& b : tr->buffers) if (b.name == name) bf = &b;
            if (!bf || kind != 0) { rc = fail(ctx, SZB_ERR_ARG, "unknown tensor '%s' (kind %d)", name.c_str(), kind); break; }
            if (numel[i] != bf->numel) { rc = fail(ctx, SZB_ERR_ARG, "'%s' has %lld elements, expected %lld", name.c_str(), (long long)numel[i], (long long)bf->numel); break; }
            if (to_trainer) tr->have_buffer[(size_t)(bf - tr->buffers.data())] = true;
            cudaError_t e = to_trainer ? cudaMemcpyAsync(bf->ptr, data[i], (size_t)bf->numel * 4, cudaMemcpyDefault, ctx->stream)
                                       : cudaMemcpyAsync(data[i], bf->ptr, (size_t)bf->numel * 4, cudaMemcpyDefault, ctx->stream);
            if (e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaMemcpyAsync(buffer)");
            continue;
        }
        const TParam& p = tr->params[it->second];
        if (numel[i] != p.numel) { rc = fail(ctx, SZB_ERR_ARG, "'%s' has %lld elements, expected %lld", name.c_str(), (long long)numel[i], (long long)p.numel); break; }
        float* slot = t_kind_base(tr, kind) + p.off;
        if (to_trainer && kind == 0) tr->have_param[(size_t)it->second] = true;
        if (p.kind == 0) {
            cudaError_t e = to_trainer ? cudaMemcpyAsync(slot, data[i], (size_t)p.numel * 4, cudaMemcpyDefault, ctx->stream)
                                       : cudaMemcpyAsync(data[i], slot, (size_t)p.numel * 4, cudaMemcpyDefault, ctx->stream);
            if (e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaMemcpyAsync(parameter)");
            continue;
        }
        // convolution weight: permute through a device scratch tensor in torch layout
        if (!scratch) {
            cudaError_t e = cudaMalloc((void**)&scratch, (size_t)256 * 256 * 9 * 4);
            if (e != cudaSuccess) { rc = cuda_fail(ctx, e, "cudaMalloc(scratch)"); break; }
        }
        const int threads = 256;
        if (to_trainer) {
            cudaError_t e = cudaMemcpyAsync(scratch, data[i], (size_t)p.numel * 4, cudaMemcpyDefault, ctx->stream);
            if (e != cudaSuccess) { rc = cuda_fail(ctx, e, "cudaMemcpyAsync(weight)"); break; }
            k_conv_to_packed<<<(unsigned)((p.n + threads - 1) / threads), threads, 0, ctx->stream>>>(scratch, slot, p.cout, p.cin, p.taps, p.cout_pad, p.cin_pad);
        } else {
            k_packed_to_conv<<<(unsigned)((p.numel + threads - 1) / threads), threads, 0, ctx->stream>>>(slot, scratch, p.cout, p.cin, p.taps, p.cin_pad);
            cudaError_t e = cudaMemcpyAsync(data[i], scratch, (size_t)p.numel * 4, cudaMemcpyDefault, ctx->stream);
            if (e != cudaSuccess) { rc = cuda_fail(ctx, e, "cudaMemcpyAsync(weight)"); break; }
        }
        ctx->launches++;
        // the scratch tensor is reused by the next convolution weight: stream order keeps that safe
    }
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (scratch) cudaFree(scratch);
    if (!rc && e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaStreamSynchronize");
    if (!rc && (e = cudaGetLastError()) != cudaSuccess) rc = cuda_fail(ctx, e, "szb_train_get/set");
    if (!rc && to_trainer && kind == 0) {
        tr->loaded = true;
        for (bool b : tr->have_param) tr->loaded = tr->loaded && b;
        for (bool b : tr->have_buffer) tr->loaded = tr->loaded && b;
        rc = t_pack(ctx, tr);
    }
    if (!rc && to_trainer && kind == SZB_TRAIN_MOMENTUM_BUFFER && n_tensors > 0) {
        const int32_t one = 1;                   // a resumed torch state: the next step blends into these buffers instead of starting them
        SZB_CUDA(ctx, cudaMemcpyAsync(tr->d_have_buf, &one, 4, cudaMemcpyHostToDevice, ctx->stream));
        SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return rc;
}

struct TConvFuse {               // what the epilogue adds for the BatchNorm that follows (see TConvArgs)
    bool stats = false;
    const bf16* skip = nullptr; const bf16* o = nullptr; const bf16* y = nullptr;
    const float* mean = nullptr; const float* invstd = nullptr;
};

static int t_conv(szb_ctx* ctx, Trainer* tr, const CUtensorMap& tm_a, const CUtensorMap* tm_w2, int taps, int kchunks, int n_out, int n, bf16* out, int mode,
                  const float* bias, unsigned long long* trace = nullptr, const TConvFuse& fuse = TConvFuse()) {
    const CUtensorMap& tm_w = tm_w2[tr->conv_pair ? 1 : 0];
    TConvArgs a{};
    a.trace = trace;
    a.stat_part = fuse.stats ? tr->bn_part : nullptr;
    a.bn_skip = fuse.skip; a.bn_o = fuse.o; a.bn_y = fuse.y; a.bn_mean = fuse.mean; a.bn_invstd = fuse.invstd;
    a.taps = taps; a.kchunks = kchunks; a.n_boards = n; a.out = out; a.ldc = TC; a.logits = tr->logits; a.bias = bias; a.error = tr->error;
    if (tr->conv_pair) {
        const dim3 grid2((unsigned)(((n + 3) / 4) * 2), n_out / 128);                       // whole pairs: a surplus CTA computes on zero fill, stores nothing
        if (mode == 0) SZB_CUDA(ctx, launch_kernel(k_tconv_pair<0>, grid2, dim3(TC_CONV_THREADS), TP_SMEM, ctx->stream, tr->pdl, tm_a, tm_w, a));
        else SZB_CUDA(ctx, launch_kernel(k_tconv_pair<1>, grid2, dim3(TC_CONV_THREADS), TP_SMEM, ctx->stream, tr->pdl, tm_a, tm_w, a));
        ctx->launches++;
        return 0;
    }
    const dim3 grid((unsigned)((((n + 1) / 2 + TR_CLUSTER - 1) / TR_CLUSTER) * TR_CLUSTER), n_out / 128);      // whole clusters: surplus CTAs compute on zero fill, store nothing
    if (mode == 0) SZB_CUDA(ctx, launch_kernel(k_tconv<0>, grid, dim3(TC_CONV_THREADS), TR_SMEM, ctx->stream, tr->pdl, tm_a, tm_w, a));
    else SZB_CUDA(ctx, launch_kernel(k_tconv<1>, grid, dim3(TC_CONV_THREADS), TR_SMEM, ctx->stream, tr->pdl, tm_a, tm_w, a));
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

static int t_ksplit(int n, int tiles_x) {
    int k = 144 / tiles_x;
    if (k > WG_MAX_SPLIT) k = WG_MAX_SPLIT;
    if (k > n) k = n;
    if (k < 1) k = 1;
    return k;
}

// dW of `count` layers from `l0` on, all of one shape.  One layer: split over the batch into partial sums that k_reduce_partials adds in
// a fixed order (the GPU is filled by taps x halves x splits).  Several layers (the 38 tower convolutions, at the end of the backward
// pass): one CTA per (layer, tap, half) sums over the whole batch and writes the gradient itself -- no partials, no second kernel.
static int t_wgrad(szb_ctx* ctx, Trainer* tr, int l0, int count, int n) {
    const TLayer& L = tr->L[l0];
    const TParam& p = tr->params[L.param];
    WgArgs a{};
    a.taps = L.taps; a.m_halves = L.cout_pad / 128; a.n_boards = n; a.layer0 = l0;
    a.ksplit = count > 1 ? 1 : t_ksplit(n, L.taps * a.m_halves);
    a.partial = a.ksplit > 1 ? tr->partial : nullptr;
    a.ldw = L.taps * L.cin_pad; a.cin_pad = L.cin_pad; a.split_stride = (size_t)L.cout_pad * a.ldw; a.error = tr->error;
    a.lbo = tr->cfg.probe_lbo ? (uint32_t)tr->cfg.probe_lbo : WG_BOX;
    a.sbo = tr->cfg.probe_sbo ? (uint32_t)tr->cfg.probe_sbo : 1024;
    if ((size_t)a.ksplit * a.split_stride > tr->partial_floats) return fail(ctx, SZB_ERR_INTERNAL, "wgrad scratch too small");
    const dim3 grid(L.taps * a.m_halves, a.ksplit, count);
    const size_t smem4 = (size_t)(WG_STAGES * 6 * WG_BOX + 1024), smem2 = (size_t)(WG_STAGES * 4 * WG_BOX + 1024);
    if (L.cin_pad == 256 && a.m_halves == 2) SZB_CUDA(ctx, launch_kernel(k_wgrad<4, 2>, grid, dim3(TR_THREADS), smem4, ctx->stream, tr->pdl, (const WgLayer*)tr->wg_layers, a));
    else if (L.cin_pad == 256) SZB_CUDA(ctx, launch_kernel(k_wgrad<4, 1>, grid, dim3(TR_THREADS), smem4, ctx->stream, tr->pdl, (const WgLayer*)tr->wg_layers, a));
    else SZB_CUDA(ctx, launch_kernel(k_wgrad<2, 2>, grid, dim3(TR_THREADS), smem2, ctx->stream, tr->pdl, (const WgLayer*)tr->wg_layers, a));
    ctx->launches++;
    if (a.ksplit > 1) {
        const size_t cnt = a.split_stride;
        SZB_CUDA(ctx, launch_kernel(k_reduce_partials, dim3((unsigned)((cnt / 4 + 255) / 256)), dim3(256), 0, ctx->stream, tr->pdl, (const float*)tr->partial,
                                    a.split_stride, a.ksplit, tr->g + p.off, cnt));
        ctx->launches++;
    }
    return 0;
}

static float* t_slot(Trainer* tr, float* base, const std::string& name) { return base + tr->params[tr->index.at(name)].off; }

// every launch of one step on the context's stream (no synchronisation: this is what a CUDA graph captures)
static int t_step_launches(szb_ctx* ctx, Trainer* tr, int n, int flags) {
    cudaStream_t st = ctx->stream;
    int rc;
    // an odd batch leaves a phantom board in the last 2-board tile: GEMM rows are independent, its rows are computed and never stored
    k_gather_input<<<(unsigned)(((size_t)n * 64 * 16 + 255) / 256), 256, 0, st>>>(tr->rec_states, (long long)tr->rec_n, tr->rows, n, tr->x_in, tr->error);
    ctx->launches++;
    const int bn_groups = n / 2 < BN_GROUPS ? (n / 2 > 0 ? n / 2 : 1) : BN_GROUPS;
    const int n_tiles = (n + 1) / 2;
    TConvFuse fwd_stats;
    fwd_stats.stats = true;
    // ---------------- forward ----------------
    for (int l = 0; l < T_BN; l++) {
        TLayer& L = tr->L[l];
        const CUtensorMap& tm_a = l == 0 ? tr->tm_in2 : l == L_P1 ? tr->L[38].tm_o2 : tr->L[l - 1].tm_o2;
        if ((rc = t_conv(ctx, tr, tm_a, L.tm_wf, L.taps, L.cin_pad / 64, 256, n, L.y, 0, nullptr, l == 20 ? tr->trace : nullptr, fwd_stats))) return rc;
        const bf16* res = (l >= 2 && l <= 38 && ((l - 1) & 1)) ? tr->L[l - 2].o : nullptr;
        BnFwd bp{L.y, res, L.o, tr->w + tr->params[L.gamma].off, tr->w + tr->params[L.beta].off, L.bn, L.bn + 256, L.bn + 512, L.bn + 768,
                 tr->bn_part, n_tiles, n, tr->cfg.bn_momentum, tr->cfg.bn_eps};
        SZB_CUDA(ctx, launch_kernel(k_bn_fwd, dim3(BN_SLICES, bn_groups), dim3(256), 0, st, tr->pdl, bp));
        ctx->launches++;
    }
    if ((rc = t_conv(ctx, tr, tr->L[L_P1].tm_o2, tr->L[L_P2].tm_wf, 1, 4, 128, n, nullptr, 1, t_slot(tr, tr->w, "conv_p2.bias")))) return rc;
    const bf16* T = tr->L[38].o;
    k_vconv<<<(unsigned)(((size_t)n * 64 * 32 + 255) / 256), 256, 0, st>>>(T, t_slot(tr, tr->w, "conv_v1.weight"), tr->yv, n);
    k_vbn_stats<<<1, 1024, 0, st>>>(tr->yv, n, tr->v_running, tr->v_running + 1, tr->vstat, tr->cfg.bn_momentum, tr->cfg.bn_eps);
    VHead vh{tr->yv, tr->vstat, t_slot(tr, tr->w, "v_norm.weight"), t_slot(tr, tr->w, "v_norm.bias"), t_slot(tr, tr->w, "fc_v1.weight"),
             t_slot(tr, tr->w, "fc_v1.bias"), t_slot(tr, tr->w, "fc_v2.weight"), t_slot(tr, tr->w, "fc_v2.bias"), tr->rec_z, tr->rows, tr->value, tr->se,
             tr->vr, tr->dh1, tr->h1r, tr->du, tr->gr, n};
    k_vhead<<<n, 256, 0, st>>>(vh);
    LossArgs la{tr->logits, tr->rows, tr->rec_off, tr->rec_index, tr->rec_prob, tr->dl, tr->ce, tr->db_part, n};
    k_policy_loss<<<n, 256, 0, st>>>(la);
    k_loss_reduce<<<1, 32, 0, st>>>(tr->se, tr->ce, n, tr->losses, tr->loss_hist, tr->hist_count);
    ctx->launches += 5;
    SZB_CUDA(ctx, cudaGetLastError());
    if (!(flags & SZB_TRAIN_FORWARD_ONLY)) {
        // ---------------- backward: heads ----------------
        k_colsum<<<1, 128, 0, st>>>(tr->db_part, n, 73, DL_C, t_slot(tr, tr->g, "conv_p2.bias"));
        k_vbn_bwd<<<1, 1024, 0, st>>>(tr->yv, tr->gr, tr->vstat, t_slot(tr, tr->w, "v_norm.weight"), t_slot(tr, tr->g, "v_norm.weight"),
                                      t_slot(tr, tr->g, "v_norm.bias"), tr->dyv, n);
        k_vconv_bwd<<<n, 256, 0, st>>>(T, t_slot(tr, tr->w, "conv_v1.weight"), tr->dyv, tr->skip[0], tr->vpart);
        k_colsum<<<1, 256, 0, st>>>(tr->vpart, n, 256, 256, t_slot(tr, tr->g, "conv_v1.weight"));
        k_vhead_grads<<<(256 * 64 + 256 + 1 + 255) / 256, 256, 0, st>>>(tr->dh1, tr->vr, tr->h1r, tr->du, n, t_slot(tr, tr->g, "fc_v1.weight"),
                                                                       t_slot(tr, tr->g, "fc_v1.bias"), t_slot(tr, tr->g, "fc_v2.weight"),
                                                                       t_slot(tr, tr->g, "fc_v2.bias"));
        ctx->launches += 5;
        // conv_p2: weight gradient, then the gradient of its input (conv_p1's output after BN + ReLU)
        if ((rc = t_wgrad(ctx, tr, L_P2, 1, n))) return rc;
        // Every dgrad convolution's epilogue finishes the layer BELOW it: residual join, ReLU mask, the masked gradient `gm` and the two
        // per-tile sums its BatchNorm backward needs.  below(l) = the layer whose output convolution l reads.
        int sk = 0;                                             // skip[sk] holds the skip-path gradient for the next residual join
        bf16* gm_next = nullptr;                                // where the running dgrad left gm for the layer being processed
        auto fuse_for = [&](int lb, bf16** gm_out) {
            const TLayer& B = tr->L[lb];
            const bool join = lb == 0 || (lb <= 38 && ((lb - 1) & 1));   // layers whose output feeds a residual add as well (or both heads)
            TConvFuse f;
            f.stats = true;
            f.skip = join ? tr->skip[sk] : nullptr;
            f.o = B.o; f.y = B.y; f.mean = B.bn + 512; f.invstd = B.bn + 768;
            *gm_out = join ? tr->skip[sk ^ 1] : tr->gm1;
            if (join) sk ^= 1;
            return f;
        };
        {
            const TConvFuse f = fuse_for(L_P1, &gm_next);
            if ((rc = t_conv(ctx, tr, tr->tm_dl2, tr->L[L_P2].tm_wd, 1, DL_C / 64, 256, n, gm_next, 0, nullptr, nullptr, f))) return rc;
        }
        for (int l = L_P1; l >= 0; l--) {
            TLayer& L = tr->L[l];
            BnBwd bp{gm_next, L.y, L.dy, tr->w + tr->params[L.gamma].off, L.bn + 512, L.bn + 768, tr->g + tr->params[L.gamma].off,
                     tr->g + tr->params[L.beta].off, tr->bn_part, n_tiles, n};
            SZB_CUDA(ctx, launch_kernel(k_bn_bwd, dim3(BN_SLICES, bn_groups), dim3(256), 0, st, tr->pdl, bp));
            ctx->launches++;
            if (l == 0 || l == L_P1) {
                if ((rc = t_wgrad(ctx, tr, l, 1, n))) return rc;
            }
            if (l > 0) {
                const int lb = l == L_P1 ? 38 : l - 1;
                const TConvFuse f = fuse_for(lb, &gm_next);
                if ((rc = t_conv(ctx, tr, L.tm_dy2, L.tm_wd, L.taps, 4, 256, n, gm_next, 0, nullptr, nullptr, f))) return rc;
            }
        }
        if ((rc = t_wgrad(ctx, tr, 1, 38, n))) return rc;         // every tower convolution's weight gradient
        if (!(flags & SZB_TRAIN_NO_UPDATE)) {
            const szb_train_config& c = tr->cfg;
            if (tr->opt_kind == SZB_TRAIN_SGD) {
                k_hyper_sgd<<<1, 1, 0, st>>>(tr->d_step, c.lr, c.lr_gamma, c.lr_step, tr->d_have_buf, tr->hyper);
                k_sgd<<<(unsigned)((tr->total + 255) / 256), 256, 0, st>>>(tr->w, tr->g, tr->m, tr->total, tr->hyper, tr->momentum, tr->dampening,
                                                                          tr->nesterov, c.weight_decay);
            } else {
                k_hyper<<<1, 1, 0, st>>>(tr->d_step, c.lr, c.lr_gamma, c.lr_step, c.beta1, c.beta2, tr->hyper);
                k_adam<<<(unsigned)((tr->total + 255) / 256), 256, 0, st>>>(tr->w, tr->g, tr->m, tr->v, tr->total, tr->hyper, c.beta1, c.beta2, c.eps, c.weight_decay);
            }
            ctx->launches += 2;
            if ((rc = t_pack(ctx, tr))) return rc;
        }
    }
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

static int t_step(szb_ctx* ctx, int32_t n, const int32_t* rows, int32_t flags, float* losses_out) {
    Trainer* tr = ctx->trainer;
    if (!tr) return fail(ctx, SZB_ERR_STATE, "no trainer: szb_train_create first");
    if (!tr->loaded) {
        for (size_t i = 0; i < tr->params.size(); i++)
            if (!tr->have_param[i]) return fail(ctx, SZB_ERR_STATE, "trainer weights incomplete: '%s' was never set (szb_train_set, SZB_TRAIN_PARAMS)", tr->params[i].name.c_str());
        for (size_t i = 0; i < tr->buffers.size(); i++)
            if (!tr->have_buffer[i]) return fail(ctx, SZB_ERR_STATE, "trainer weights incomplete: '%s' was never set (szb_train_set, SZB_TRAIN_PARAMS)", tr->buffers[i].name.c_str());
        return fail(ctx, SZB_ERR_STATE, "trainer has no weights: szb_train_set(SZB_TRAIN_PARAMS) first");
    }
    if (!tr->rec_states) return fail(ctx, SZB_ERR_STATE, "no records: szb_train_records first");
    if (n < 2 || n > tr->cfg.batch || !rows) return fail(ctx, SZB_ERR_ARG, "szb_train_step: 2 <= n <= %d boards (BatchNorm needs more than one)", tr->cfg.batch);
    cudaStream_t st = ctx->stream;
    int rc;
    // row numbers: through a ring of pinned staging slots, so that the host can queue several steps ahead of the GPU
    {
        const int slot = (int)(tr->steps_queued++ % ROWS_RING);
        int32_t* stage = tr->rows_host + (size_t)slot * tr->cap;
        if (tr->rows_used[slot]) SZB_CUDA(ctx, cudaEventSynchronize(tr->rows_ev[slot]));
        SZB_CUDA(ctx, cudaMemcpy(stage, rows, (size_t)n * 4, cudaMemcpyDefault));
        SZB_CUDA(ctx, cudaMemcpyAsync(tr->rows, stage, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        SZB_CUDA(ctx, cudaEventRecord(tr->rows_ev[slot], st));
        tr->rows_used[slot] = true;
    }
    tr->last_n = n;
    const uint64_t launches0 = ctx->launches;
    bool done = false;
    if (tr->use_graph) {
        // one graph per (boards, flags): ~210 launches become one submission
        const std::pair<int, int> key(n, flags);
        auto it = tr->graphs.find(key);
        if (it == tr->graphs.end()) {
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                rc = t_step_launches(ctx, tr, n, flags);
                cudaError_t e = cudaStreamEndCapture(st, &graph);
                if (!rc && e == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) it = tr->graphs.emplace(key, exec).first;
                if (graph) cudaGraphDestroy(graph);
            }
            if (it == tr->graphs.end()) { cudaGetLastError(); tr->use_graph = false; }       // capture unavailable: plain launches from here on
            tr->launches_per_step[key] = ctx->launches - launches0;
        }
        if (it != tr->graphs.end()) {
            SZB_CUDA(ctx, cudaGraphLaunch(it->second, st));
            ctx->launches = launches0 + tr->launches_per_step[key];
            done = true;
        }
    }
    if (!done && (rc = t_step_launches(ctx, tr, n, flags))) return rc;
    if (!(flags & (SZB_TRAIN_NO_UPDATE | SZB_TRAIN_FORWARD_ONLY))) tr->step++;
    tr->steps_run++;
    if (losses_out) {
        int32_t err = 0;
        SZB_CUDA(ctx, cudaMemcpyAsync(losses_out, tr->losses, 8, cudaMemcpyDefault, st));
        SZB_CUDA(ctx, cudaMemcpyAsync(&err, tr->error, 4, cudaMemcpyDeviceToHost, st));
        SZB_CUDA(ctx, cudaStreamSynchronize(st));
        if (tr->trace) {
            unsigned long long t[8];
            SZB_CUDA(ctx, cudaMemcpy(t, tr->trace, sizeof(t), cudaMemcpyDeviceToHost));
            fprintf(stderr, "[szb train trace] layer-20 forward convolution, CTA (0,0), us since entry: prologue %.2f, dependency wait %.2f, first chunk landed %.2f, "
                            "last MMA issued %.2f, accumulator ready %.2f, exit %.2f\n", (t[1] - t[0]) * 1e-3, (t[2] - t[0]) * 1e-3, (t[3] - t[0]) * 1e-3,
                    (t[4] - t[0]) * 1e-3, (t[5] - t[0]) * 1e-3, (t[6] - t[0]) * 1e-3);
        }
        if (err) {
            cudaMemsetAsync(tr->error, 0, 4, st);
            return err == 2 ? fail(ctx, SZB_ERR_ARG, "szb_train_step: a row index is outside the %lld records", (long long)tr->rec_n)
                            : fail(ctx, SZB_ERR_INTERNAL, "a training kernel's pipeline timed out");
        }
    }
    return 0;
}

}  // namespace szb

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int szb_train_create(szb_ctx* ctx, const szb_train_config* cfg) {
    if (!ctx || !cfg) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    if (cfg->batch < 2 || cfg->batch > 4096) return fail(ctx, SZB_ERR_ARG, "szb_train_create: batch must be 2..4096");
    return t_create(ctx, cfg);
}

int szb_train_set_optimizer(szb_ctx* ctx, int32_t kind, float momentum, float dampening, int32_t nesterov) {
    if (!ctx) return SZB_ERR_ARG;
    Trainer* tr = ctx->trainer;
    if (!tr) return fail(ctx, SZB_ERR_STATE, "no trainer: call szb_train_create first");
    if (tr->steps_run > 0) return fail(ctx, SZB_ERR_STATE, "szb_train_set_optimizer: a step has already run");
    if (kind != SZB_TRAIN_ADAM && kind != SZB_TRAIN_SGD) return fail(ctx, SZB_ERR_ARG, "szb_train_set_optimizer: unknown optimiser %d", (int)kind);
    if (kind == SZB_TRAIN_SGD) {
        // torch.optim.SGD's constructor rules (and a dampening that is a number, not negative)
        if (!(momentum >= 0.f) || !(dampening >= 0.f)) return fail(ctx, SZB_ERR_ARG, "szb_train_set_optimizer: negative momentum or dampening");
        if (nesterov && (momentum <= 0.f || dampening != 0.f))
            return fail(ctx, SZB_ERR_ARG, "szb_train_set_optimizer: Nesterov momentum requires a momentum and zero dampening");
    }
    tr->opt_kind = kind;
    tr->momentum = kind == SZB_TRAIN_SGD ? momentum : 0.f;
    tr->dampening = kind == SZB_TRAIN_SGD ? dampening : 0.f;
    tr->nesterov = kind == SZB_TRAIN_SGD && nesterov ? 1 : 0;
    return 0;
}

int szb_train_destroy(szb_ctx* ctx) {
    if (!ctx) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    trainer_destroy(ctx);
    return 0;
}

int szb_train_set(szb_ctx* ctx, int32_t kind, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel) {
    if (!ctx) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    return t_transfer(ctx, kind, n_tensors, names, const_cast<float* const*>(data), numel, true);
}

int szb_train_get(szb_ctx* ctx, int32_t kind, int32_t n_tensors, const char* const* names, float* const* data, const int64_t* numel) {
    if (!ctx) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    return t_transfer(ctx, kind, n_tensors, names, data, numel, false);
}

int szb_train_records(szb_ctx* ctx, int64_t n, const uint64_t* states, const int64_t* pi_off, const uint16_t* pi_index, const float* pi_prob, const int8_t* z) {
    if (!ctx) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    Trainer* tr = ctx->trainer;
    if (!tr) return fail(ctx, SZB_ERR_STATE, "no trainer: call szb_train_create first");
    if (n < 1 || !states || !pi_off || !pi_index || !pi_prob || !z) return fail(ctx, SZB_ERR_ARG, "szb_train_records: bad arguments");
    cudaStreamSynchronize(ctx->stream);
    // the captured steps carry the old buffers' addresses as kernel parameters: drop them, the next step captures afresh
    for (auto& kv : tr->graphs) cudaGraphExecDestroy(kv.second);
    tr->graphs.clear();
    void* old[5] = {tr->rec_states, tr->rec_off, tr->rec_index, tr->rec_prob, tr->rec_z};
    for (void* p : old) if (p) cudaFree(p);
    tr->rec_states = nullptr; tr->rec_off = nullptr; tr->rec_index = nullptr; tr->rec_prob = nullptr; tr->rec_z = nullptr;
    int64_t first = 0, last = 0;
    SZB_CUDA(ctx, cudaMemcpy(&first, pi_off, 8, cudaMemcpyDefault));
    SZB_CUDA(ctx, cudaMemcpy(&last, pi_off + n, 8, cudaMemcpyDefault));
    if (first != 0 || last < 0) return fail(ctx, SZB_ERR_ARG, "szb_train_records: pi_off must start at 0 and ascend");
    const size_t m = (size_t)last;
    SZB_CUDA(ctx, cudaMalloc((void**)&tr->rec_states, (size_t)n * T_PLANES * 8));
    SZB_CUDA(ctx, cudaMalloc((void**)&tr->rec_off, (size_t)(n + 1) * 8));
    SZB_CUDA(ctx, cudaMalloc((void**)&tr->rec_index, (m ? m : 1) * 2));
    SZB_CUDA(ctx, cudaMalloc((void**)&tr->rec_prob, (m ? m : 1) * 4));
    SZB_CUDA(ctx, cudaMalloc((void**)&tr->rec_z, (size_t)n));
    SZB_CUDA(ctx, cudaMemcpyAsync(tr->rec_states, states, (size_t)n * T_PLANES * 8, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaMemcpyAsync(tr->rec_off, pi_off, (size_t)(n + 1) * 8, cudaMemcpyDefault, ctx->stream));
    if (m) {
        SZB_CUDA(ctx, cudaMemcpyAsync(tr->rec_index, pi_index, m * 2, cudaMemcpyDefault, ctx->stream));
        SZB_CUDA(ctx, cudaMemcpyAsync(tr->rec_prob, pi_prob, m * 4, cudaMemcpyDefault, ctx->stream));
    }
    SZB_CUDA(ctx, cudaMemcpyAsync(tr->rec_z, z, (size_t)n, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    tr->rec_n = n;
    return 0;
}

int szb_train_step(szb_ctx* ctx, int32_t n, const int32_t* rows, int32_t flags, float* losses_out) {
    if (!ctx) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    return t_step(ctx, n, rows, flags, losses_out);
}

int szb_train_loss_history(szb_ctx* ctx, int64_t first, int32_t count, float* out) {
    if (!ctx) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    Trainer* tr = ctx->trainer;
    if (!tr) return fail(ctx, SZB_ERR_STATE, "no trainer");
    if (count < 0 || first < 0 || first + count > tr->steps_run || (count && !out))
        return fail(ctx, SZB_ERR_ARG, "szb_train_loss_history: steps [%lld, %lld) of %lld run", (long long)first, (long long)(first + count), (long long)tr->steps_run);
    if (tr->steps_run - first > LOSS_HIST) return fail(ctx, SZB_ERR_ARG, "szb_train_loss_history: only the last %d steps are kept", LOSS_HIST);
    int32_t err = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(&err, tr->error, 4, cudaMemcpyDeviceToHost, ctx->stream));
    for (int32_t done = 0; done < count;) {
        const int64_t k = (first + done) % LOSS_HIST;
        const int32_t run = (int32_t)((LOSS_HIST - k) < (count - done) ? (LOSS_HIST - k) : (count - done));
        SZB_CUDA(ctx, cudaMemcpyAsync(out + 2 * (size_t)done, tr->loss_hist + 2 * k, (size_t)run * 8, cudaMemcpyDefault, ctx->stream));
        done += run;
    }
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (err) {
        cudaMemsetAsync(tr->error, 0, 4, ctx->stream);
        return err == 2 ? fail(ctx, SZB_ERR_ARG, "a step's row index was outside the %lld records", (long long)tr->rec_n)
                        : fail(ctx, SZB_ERR_INTERNAL, "a training kernel's pipeline timed out");
    }
    return 0;
}

int szb_train_state(szb_ctx* ctx, int64_t* step_inout, int32_t set) {
    if (!ctx || !step_inout) return SZB_ERR_ARG;
    if (!ctx->trainer) return fail(ctx, SZB_ERR_STATE, "no trainer");
    if (set) {
        cudaSetDevice(ctx->device);
        ctx->trainer->step = *step_inout;
        const long long v = *step_inout;
        SZB_CUDA(ctx, cudaMemcpyAsync(ctx->trainer->d_step, &v, 8, cudaMemcpyHostToDevice, ctx->stream));
        SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    } else {
        *step_inout = ctx->trainer->step;
    }
    return 0;
}

}  // extern "C"
