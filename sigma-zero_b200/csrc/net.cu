// net.cu -- the policy/value network (network.py:89-192) as hand-written sm_100a kernels.
//
//   bf16 path : every convolution is an implicit GEMM on the 5th-gen tensor cores (GEMM view: M = 64*B board squares,
//               N = C_out, K = taps*C_in; bf16 in, fp32 accumulate in TMEM, epilogue +bias(BN folded) [+residual] -> ReLU
//               -> bf16 fused after tcgen05.ld).
//               k_tower_tc2  (the product path): ONE persistent launch over all 41 layers; CTA pairs with
//                            tcgen05.mma.cta_group::2 (256 x 256 x 16), weight tiles split between the two CTAs, a whole
//                            halo tile of activations resident in shared memory per 64-channel K chunk (all nine taps read
//                            it in place through shifted descriptors), per-item dependency counters between layers.
//               k_conv_tc    (first version, kept for A/B and the bit-identity test): single CTA, 128 x N x 16, one launch per
//                            layer, one TMA box per tap.
//   fp32 path : SIMT FFMA implicit GEMM with the same folded weights (parity mode, <= 1e-5 abs vs torch CPU).
//
// Activations live in HBM as NHWC bf16 with a one-square zero halo: [B][10][10][C]; a tap is a shifted window of it.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <array>
#include <map>
#include <string>
#include "engine.cuh"
#include "tc.cuh"

using namespace szb;

namespace szb {

constexpr int HALO = 10;
constexpr int C_TOWER = 256;
constexpr int C_IN_PAD = 128;            // 119 input planes padded to 128 channels
constexpr int N_BLOCKS = 19;
constexpr int POLICY_PLANES = 73;
constexpr int POLICY_PAD = 80;           // N of the last policy GEMM (multiple of 16)
// algorithmic FLOP (2 x MAC, no credit for channel padding) per board: one 3x3 256->256 layer; stem + 38 tower layers + policy 1x1 + policy out
constexpr uint64_t FLOP_TOWER_LAYER = 2ull * 64 * 256 * 2304;
constexpr uint64_t FLOP_TOWER_ALL = 2ull * 64 * (256 * (119 * 9 + 38 * 2304 + 256) + 73 * 256);

// ---- tcgen05 conv kernel geometry ---------------------------------------------------------------
constexpr int TC_BLOCK_M = 128;          // two boards per tile
constexpr int TC_BLOCK_K = 64;           // one 128-byte swizzle atom of bf16
constexpr int TC_STAGES = 4;
constexpr int TC_A_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;       // 16 KiB
constexpr int TC_THREADS = 192;          // warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2..5 epilogue

struct ConvLayer {
    int taps = 9, cin = 256, cout = 256, cout_pad = 256;
    float* w32 = nullptr;                // [taps][cin][cout_pad]
    float* bias = nullptr;               // [cout_pad]  (BatchNorm folded)
    __nv_bfloat16* w16 = nullptr;        // [cout_pad][taps*cin]  K-major
    CUtensorMap tm_w;
};

struct TowerMaps;
struct TowerArgs;
constexpr int CL_MAX_BOARDS_DEFAULT = 18;   // k_tower_cl: one 8-CTA cluster per board, 18 clusters = 144 of 148 SMs

struct Net {
    bool loaded = false;
    bool allocated = false;              // buffers, tensor maps and layer table exist (net_ensure_allocated)
    unsigned long long* digest = nullptr;
    int cap = 0;                         // boards the activation buffers hold (even)
    ConvLayer stem, tower[2 * N_BLOCKS], p1, p2;
    // value head (fp32 everywhere)
    float* v_w = nullptr;                // [256] conv_v1 * bn scale
    float* head_scalars = nullptr;       // device: {v_norm shift (conv_v1 BN folded), fc_v2.bias}
    float* fc1_w = nullptr;              // [64][256] (fc_v1.weight transposed)
    float* fc1_b = nullptr;              // [256]
    float* fc2_w = nullptr;              // [256]
    // activations
    __nv_bfloat16* in16 = nullptr;       // [cap][10][10][128]
    __nv_bfloat16* act16[3] = {nullptr, nullptr, nullptr};     // [cap][10][10][256]
    float* in32 = nullptr;
    float* act32[3] = {nullptr, nullptr, nullptr};
    float* logits = nullptr;             // [cap][4672]
    CUtensorMap tm_in16, tm_act16[3];
    int32_t* tc_error = nullptr;
    // CTA-pair tower kernel (k_tower_tc2): all 40 N=256 layers in one weight / bias buffer + per-item completion counters
    __nv_bfloat16* w16_all = nullptr;    // [MAX_TOWER_LAYERS * 256][2304]
    __nv_bfloat16* w16_cl[2] = {nullptr, nullptr};   // k_tower_cl<8> / <16> weight streams: [layer][rank][K chunk][tap][rows x 128 B], pre-swizzled smem images
    float* bias_all = nullptr;           // [MAX_TOWER_LAYERS][256]
    int32_t* ready = nullptr;            // [MAX_TOWER_LAYERS][ceil(cap / 4)]
    struct TowerMaps* tower_maps = nullptr;   // host copies, passed by value at launch
    struct TowerArgs* tower_args = nullptr;
    int final_x = 0, final_y = 0;        // activation buffers holding the tower output / the policy-head hidden layer
    int tower_mode = 2;                  // 0: single-CTA kernel per layer, 1: pair kernel per layer, 2: pair kernel, one launch
    int tower_nsplit = 0;                // 0: automatic (launch_tower), else forced 1 / 2 / 4 / 8
    int tower_tps1 = 1;                  // taps per weight stage of large-batch launches (SZB_TOWER_TPS=2: three 32 KiB stages)
    int last_nsplit = 1;                 // what the last multi-layer launch used (trace aid)
    int chunk = 512;                     // boards per tower launch of a large evaluation (net_forward_chunked); 0 = unlimited
    int tower_pairs = 74;                // CTA pairs of an exclusive launch (SZB_TOWER_PAIRS)
    bool tower_exclusive = false;        // SZB_TOWER_EXCLUSIVE: experiment, see launch_tower
    bool no_fuse = false;                // SZB_NO_FUSE=1: A/B aid, search steps use the separate head kernels
    int cluster_max = CL_MAX_BOARDS_DEFAULT;   // batches up to this many boards run the cluster-resident tower (SZB_TOWER_CLUSTER=<n>, 0 = off)
    int cluster_force = 0;                     // SZB_TOWER_CLUSTER_SIZE=8|16: A/B aid, use only that cluster size
    bool attr_set_cl = false;
    int clusters_resident[2] = {0, 0};         // clusters of 8 / 16 CTAs of k_tower_cl this device holds at once
    unsigned long long* cl_trace = nullptr;
    unsigned long long* span = nullptr;  // [SPAN_CAP][4] device stamps of whole-tower launches (szb_tower_spans_record / SZB_TOWER_SPAN)
    bool span_on = false;
    std::vector<int> span_boards, span_b0;
    std::string span_path;
    // SZB_TOWER_TRACE inside searches: per-item stamps of the last TRACE_RING large-batch whole-tower launches (ring, dumped at destroy)
    unsigned long long* trace_ring = nullptr;
    std::string trace_path;
    std::vector<std::array<long long, 5>> trace_meta;   // per ring slot: {launch ordinal, boards, tiles, pairs, span index or -1}
    long long trace_launches = 0;
    int num_sms = 148;
    int pairs_resident = 74;             // CTA pairs of k_tower_tc2 this device holds at once (cudaOccupancyMaxActiveClusters)
    bool attr_set = false;               // per context (= per device): dynamic shared memory opt-ins done
    bool attr_set_tc[2] = {false, false};
    int smem_exclusive = 0;
    std::vector<void*> allocs;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

int net_tmap_init(szb_ctx* ctx) {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) return fail(ctx, SZB_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    g_encode = (EncodeTiledFn)fn;
    return 0;
}

static int encode_bf16(szb_ctx* ctx, CUtensorMap* tm, int rank, void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                       const cuuint32_t* box, const char* what) {
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, SZB_ERR_CUDA, "cuTensorMapEncodeTiled(%s) failed: %d", what, (int)r);
    return 0;
}
int net_tmap_act(szb_ctx* ctx, CUtensorMap* tm, void* base, int channels, int boards, int box_boards, const char* what) {
    const cuuint64_t dims[4] = {(cuuint64_t)channels, HALO, HALO, (cuuint64_t)boards};
    const cuuint64_t strides[3] = {(cuuint64_t)channels * 2, (cuuint64_t)channels * 2 * HALO, (cuuint64_t)channels * 2 * HALO * HALO};
    const cuuint32_t box[4] = {TC_BLOCK_K, 8, 8, (cuuint32_t)box_boards};
    return encode_bf16(ctx, tm, 4, base, dims, strides, box, what);
}
int net_tmap_halo(szb_ctx* ctx, CUtensorMap* tm, void* base, int channels, int boards, int box_boards, const char* what) {
    const cuuint64_t dims[4] = {(cuuint64_t)channels, HALO, (cuuint64_t)boards, HALO};
    const cuuint64_t strides[3] = {(cuuint64_t)channels * 2, (cuuint64_t)channels * 2 * HALO * HALO, (cuuint64_t)channels * 2 * HALO};
    const cuuint32_t box[4] = {TC_BLOCK_K, HALO, (cuuint32_t)box_boards, HALO};
    return encode_bf16(ctx, tm, 4, base, dims, strides, box, what);
}
int net_tmap_rows(szb_ctx* ctx, CUtensorMap* tm, void* base, int k_total, int rows, int box_rows, const char* what) {
    const cuuint64_t dims[2] = {(cuuint64_t)k_total, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)k_total * 2};
    const cuuint32_t box[2] = {TC_BLOCK_K, (cuuint32_t)box_rows};
    return encode_bf16(ctx, tm, 2, base, dims, strides, box, what);
}


// =================================================================================================
// tcgen05 implicit-GEMM convolution
// =================================================================================================
struct TcArgs {
    int n_tiles;                 // ceil(B / 2)
    int taps;                    // 9 or 1
    int kchunks;                 // C_in / 64
    const float* bias;           // [N]
    const __nv_bfloat16* residual;   // halo NHWC [.][10][10][256] or null
    __nv_bfloat16* out;          // halo NHWC (mode 0)
    float* logits;               // [B][4672] (mode 1)
    int n_boards;                // boards beyond board0 + n_boards are not stored
    int board0;                  // first board of this launch inside the activation buffers (cohort offset, even)
    int relu;
    int32_t* error;
};

template <int N_TILE, int MODE>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_conv_tc(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, const TcArgs a) {
    constexpr int B_BYTES = N_TILE * TC_BLOCK_K * 2;
    constexpr int STAGE_BYTES = TC_A_BYTES + B_BYTES;
    constexpr uint32_t IDESC = idesc_bf16(TC_BLOCK_M, N_TILE);
    constexpr int ACC_COLS = 256;                                // column stride between the two accumulator stages

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[TC_STAGES], bar_empty[TC_STAGES], bar_acc_full[2], bar_acc_empty[2];
    __shared__ uint32_t tmem_base_sh;
    __shared__ int abort_sh;
    __shared__ float bias_sh[N_TILE];

    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    volatile int* abort_flag = &abort_sh;

    if (threadIdx.x == 0) {
        abort_sh = 0;
        for (int s = 0; s < TC_STAGES; s++) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), 1); }
        for (int s = 0; s < 2; s++) { mbar_init(smem_u32(&bar_acc_full[s]), 1); mbar_init(smem_u32(&bar_acc_empty[s]), 4); }
        fence_mbarrier_init();
    }
    for (int i = threadIdx.x; i < N_TILE; i += blockDim.x) bias_sh[i] = a.bias[i];
    if (warp == 1) tc_tmem_alloc(smem_u32(&tmem_base_sh), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;
    const int k_iters = a.taps * a.kchunks;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            bool ok = true;
            for (int tile = blockIdx.x; tile < a.n_tiles && ok; tile += gridDim.x) {
                for (int it = 0; it < k_iters; it++) {
                    const int kc = it / a.taps, tap = it - kc * a.taps;          // K chunk outer, tap inner: the order k_tower_tc2 accumulates in
                    const int ky = a.taps == 9 ? tap / 3 : 1, kx = a.taps == 9 ? tap - (tap / 3) * 3 : 1;
                    if (!(ok = mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1, abort_flag))) break;
                    const uint32_t full = smem_u32(&bar_full[stage]);
                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                    mbar_expect_tx(full, STAGE_BYTES);
                    tma_load_4d(sa, &tm_a, full, kc * TC_BLOCK_K, kx, ky, a.board0 + tile * 2);
                    tma_load_2d(sa + TC_A_BYTES, &tm_w, full, (tap * a.kchunks + kc) * TC_BLOCK_K, 0);
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int local = 0;
            bool ok = true;
            for (int tile = blockIdx.x; tile < a.n_tiles && ok; tile += gridDim.x, local++) {
                const int acc = local & 1;
                const uint32_t acc_phase = (local >> 1) & 1;
                if (!(ok = mbar_wait(smem_u32(&bar_acc_empty[acc]), acc_phase ^ 1, abort_flag))) break;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * ACC_COLS;
                for (int it = 0; it < k_iters; it++) {
                    if (!(ok = mbar_wait(smem_u32(&bar_full[stage]), phase, abort_flag))) break;
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                    const uint32_t sb = sa + TC_A_BYTES;
#pragma unroll
                    for (int k = 0; k < TC_BLOCK_K / 16; k++) {
                        tc_mma_bf16(d_tmem, make_smem_desc(sa + k * 32), make_smem_desc(sb + k * 32), IDESC, (it | k) != 0);
                    }
                    tc_commit(smem_u32(&bar_empty[stage]));        // frees the smem stage once these MMAs retire
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
                if (ok) tc_commit(smem_u32(&bar_acc_full[acc]));
            }
        }
    } else {
        // ===== epilogue: TMEM -> registers -> +bias [+residual] -> ReLU -> global =====
        const int lane_group = warp & 3;                          // TMEM lanes this warp may read
        int local = 0;
        bool ok = true;
        for (int tile = blockIdx.x; tile < a.n_tiles && ok; tile += gridDim.x, local++) {
            const int acc = local & 1;
            const uint32_t acc_phase = (local >> 1) & 1;
            ok = mbar_wait(smem_u32(&bar_acc_full[acc]), acc_phase, abort_flag);
            ok = __all_sync(0xFFFFFFFFu, ok);
            if (!ok) break;
            tc_fence_after();
            const int row = lane_group * 32 + lane;
            const int m = tile * TC_BLOCK_M + row;
            const int board = a.board0 + (m >> 6), sq = m & 63;
            const bool live = board < a.board0 + a.n_boards;
            const uint32_t taddr = tmem_base + ((uint32_t)(lane_group * 32) << 16) + acc * ACC_COLS;
            const size_t pix = ((size_t)board * HALO + (sq >> 3) + 1) * HALO + (sq & 7) + 1;
#pragma unroll 1
            for (int c0 = 0; c0 < N_TILE; c0 += 16) {
                uint32_t v[16];
                tmem_ld_32x32b_x16(taddr + c0, v);
                tmem_ld_wait();
                if (MODE == 0) {
                    float f[16];
#pragma unroll
                    for (int j = 0; j < 16; j++) f[j] = __uint_as_float(v[j]) + bias_sh[c0 + j];
                    if (live) {
                        if (a.residual) {
                            const uint4* rp = reinterpret_cast<const uint4*>(a.residual + pix * C_TOWER + c0);
                            uint4 r0 = rp[0], r1 = rp[1];
                            const __nv_bfloat16* rb0 = reinterpret_cast<const __nv_bfloat16*>(&r0);
                            const __nv_bfloat16* rb1 = reinterpret_cast<const __nv_bfloat16*>(&r1);
#pragma unroll
                            for (int j = 0; j < 8; j++) { f[j] += __bfloat162float(rb0[j]); f[8 + j] += __bfloat162float(rb1[j]); }
                        }
                        uint4 o[2];
                        __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            float x0 = f[2 * j], x1 = f[2 * j + 1];
                            if (a.relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
                            ob[j] = __floats2bfloat162_rn(x0, x1);
                        }
                        uint4* op = reinterpret_cast<uint4*>(a.out + pix * C_TOWER + c0);
                        op[0] = o[0];
                        op[1] = o[1];
                    }
                } else {
                    // policy logits, plane-major like torch.flatten(conv_p2(x)): index = plane*64 + row*8 + col
                    if (live) {
#pragma unroll
                        for (int j = 0; j < 16; j++) {
                            const int c = c0 + j;
                            if (c < POLICY_PLANES) a.logits[(size_t)board * N_ACTIONS + c * 64 + sq] = __uint_as_float(v[j]) + bias_sh[c];
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&bar_acc_empty[acc]));
        }
    }
    // ===== teardown =====
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tc_tmem_dealloc(tmem_base, 512);
    if (threadIdx.x == 0 && abort_sh) atomicExch(a.error, 1);
}

// =================================================================================================
// tower kernel: CTA-pair (cta_group::2) implicit GEMM over a RANGE OF LAYERS in one persistent launch
// =================================================================================================
// The single-CTA kernel above is shared-memory-bandwidth bound (ncu, profiles/r01a_*): per 64-wide K step it
// writes 48 KiB by TMA and reads 48 KiB by UTCHMMA in the 512 cycles the MMAs need -> 192 B/cycle against the
// 128 B/cycle the SM has -> tensor pipe 68 % busy.  Here two CTAs of a cluster form one 256 x 256 tile
// (4 boards x 256 channels): each CTA stages its own 128 rows of A and HALF of the weight tile, the leader
// issues tcgen05.mma.cta_group::2, and both SMs read the two weight halves -> 64 KiB per 512 cycles.
//
// The launch is persistent over (layer, tile) work items in layer-major order, statically dealt round-robin to
// the CTA pairs.  A 3x3 convolution of a board needs only that board of the previous layer, so item (l, t)
// depends on item (l-1, t) alone: the producer acquires a per-item completion counter before its first
// activation load, the epilogue warps release it after their last store.  Items are taken in increasing order
// by every pair, so the wait chain always ends at the first layer: no deadlock, no grid-wide barrier, no wave
// quantisation between layers (10240 items over 74 pairs instead of 40 launches of 3.46 waves).
// Shared memory of one CTA: a ring of T2_A_CHUNKS activation chunks and a ring of T2_B_STAGES weight stages.
// An activation chunk is ONE 64-channel slice of this CTA's two boards INCLUDING the halo, 200 pixel rows of 128 bytes
// in the order [y 0..9][board 0..1][x 0..9] (one TMA box through a tensor map with dims (c, x, board, y)).  All nine
// taps of a 3x3 convolution read it in place: the A descriptor of tap (ky, kx) starts (ky * 20 + kx) rows into the
// chunk and strides 10 rows (1280 B) between 8-row groups, so MMA row m = (oy * 2 + board) * 8 + ox reads halo pixel
// (oy + ky, ox + kx).  tcgen05.mma applies the 128-byte swizzle to absolute shared-memory address bits, exactly like
// TMA, so starts and strides that are not multiples of 1024 B are fine (probed on hardware: scripts/desc_probe.cu).
// => an activation byte is loaded from L2 once per layer instead of once per tap.
constexpr int T2_A_CHUNKS = 4;
constexpr int T2_A_ROWS = 2 * HALO * HALO;                // 200
constexpr int T2_A_CHUNK_BYTES = T2_A_ROWS * 128;         // 25600 = 25 * 1024
constexpr int T2_A_SBO = HALO * 128;                      // 1280: one halo row of one board
constexpr int T2_B_STAGES = 7;
constexpr int T2_B_BYTES = 128 * TC_BLOCK_K * 2;          // this CTA's half (128 output channels) of a 64-wide weight tile
constexpr int T2_BIG_STAGES = 3;                          // tps1 == 2: the same ring seen as three stages of two tiles
constexpr int T2_BIG_BYTES = 2 * T2_B_BYTES;
constexpr int T2_SMEM = T2_A_CHUNKS * T2_A_CHUNK_BYTES + T2_B_STAGES * T2_B_BYTES + 1024;
constexpr int MAX_TOWER_LAYERS = 41;                      // stem + 38 tower convolutions + policy 1x1 + policy output (256 -> 73)
constexpr int POLICY_LAYER = MAX_TOWER_LAYERS - 1;
constexpr int READY_PER_ITEM = 8;                         // 4 epilogue warps x 2 CTAs
constexpr int SPAN_CAP = 1 << 17;                         // launches recorded by szb_tower_spans_record / SZB_TOWER_SPAN (a c2 bench run: 32,000)
constexpr int TRACE_STAMPS = 5;                           // SZB_TOWER_TRACE stamps per item (TowerArgs::trace)
constexpr int TRACE_RING = 64;                            // large-batch launches inside searches kept by SZB_TOWER_TRACE
constexpr int TRACE_MAX_TILES = 128;                      // ... of at most 512 boards

struct TowerLayer {
    uint8_t a_map;       // 0: input planes (128 ch), 1..3: activation buffer 0..2
    uint8_t taps;        // 9 or 1
    uint8_t kchunks;     // C_in / 64
    uint8_t res;         // activation buffer of the residual, 255 = none
    uint8_t out;         // activation buffer written
    uint8_t relu;
    uint8_t mode;        // 0: bf16 NHWC activations, 1: fp32 policy logits [board][4672] (plane-major)
    uint8_t n_half;      // output channels per CTA of the pair: 128 (N = 256) or 64 (N = 128, the 73 policy planes padded)
};

struct alignas(64) TowerMaps {
    CUtensorMap a[4];    // input planes, activation buffers 0..2 with dims (c, x, board, y): box 64 ch x 10 x 2 boards x 10
    CUtensorMap w;       // all layers' folded weights [MAX_TOWER_LAYERS * 256][2304]: box 64 k x 128 rows
    CUtensorMap w64;     // same buffer, box 64 k x 64 rows (policy output layer; N-split launches)
    CUtensorMap w32;     // box 64 k x 32 rows
    CUtensorMap w16;     // box 64 k x 16 rows
    CUtensorMap w8;      // box 64 k x 8 rows
    CUtensorMap in1;     // input planes, box 64 ch x 10 x ONE board x 10 (k_tower_cl)
};

// Search mode (mcts.py:72-79 fused into the last layer's epilogue): instead of fp32 logits the policy-output layer emits, for every
// board that needs an evaluation, softmax(logits)[i] for the LEGAL move indices i only (bit-identical to k_softmax over the full
// row: same maximum, same exp, same summation order) straight into the rows k_finish reads, and the value head
// (network.py:156-174) of the tile's boards.  mask == null: plain logits output (szb_net_forward*).
struct TowerHeads {
    const uint64_t* mask;              // [row][MASK_STRIDE] legal-move bitsets; row = board + row_delta
    const uint8_t* need_eval;          // [row]
    float* policy;                     // [row][4672]
    float* value;                      // [row]
    const __nv_bfloat16* tower_out;    // activation buffer holding the last residual block's output
    const float *v_w, *fc1_wT, *fc1_b, *fc2_w;
    const float* scalars;              // {value-conv BN shift, fc_v2 bias}
    int row_delta;
    // Evaluation cache (engine.cu, szb_set_eval_cache): the tree kernel compacts the leaves that missed the cache into the first
    // *n_live rows of its cohort and records each row's slot in row_slot.  The launch then serves min(n_boards, *n_live - live_off)
    // boards, read after griddepcontrol.wait; mask, need_eval, policy and value stay addressed by slot.  n_live == null: the host's
    // count, row = slot.
    const int32_t* row_slot;
    const int32_t* n_live;
    int live_off;                      // rows of the cohort before this launch's first board (chunked launches)
};
// boards of this launch the tree kernel filled, and the slot of an input row (see TowerHeads)
__device__ __forceinline__ int heads_live_boards(const TowerHeads& h, int n_boards) { return max(0, min(n_boards, *h.n_live - h.live_off)); }
__device__ __forceinline__ long heads_slot(const TowerHeads& h, long row) { return h.row_slot ? (long)h.row_slot[row] : row; }

struct TowerArgs {
    int n_pair_tiles;    // ceil(boards / 4)
    int n_boards;
    int board0;          // first board of this launch inside the activation buffers (cohort offset, multiple of 4)
    int in_delta;        // the input planes of board b are row b + in_delta of the NHWC input buffer (rows written by k_tree_step)
    int layer_begin, layer_end;
    int nsplit;          // 1, 2, 4 or 8: a (layer, tile) is cut into nsplit work items of N / nsplit output channels each (small batches)
    int tps1;            // nsplit == 1 launches: taps per weight stage, 1 (seven 16 KiB stages) or 2 (three 32 KiB stages: half as many waits /
                         // commits on the MMA-issuing warp per MMA; SZB_TOWER_TPS=2, scripts/mma_rate_probe.cu)
    int n_main;          // work items of the layers cut nsplit ways; the items after them are whole tiles of the LAST layer (fused heads
                         // need all 73 planes of a board in one accumulator)
    int n_items;
    TowerHeads heads;
    int32_t* ready;      // [MAX_TOWER_LAYERS][n_pair_tiles] completion counters, zeroed before the launch
    const float* bias;   // [MAX_TOWER_LAYERS][256]
    __nv_bfloat16* act[3];
    float* logits;       // [boards][4672]
    int32_t* error;
    unsigned long long* trace;   // measurement aid (SZB_TOWER_TRACE): [item][TRACE_STAMPS] %globaltimer stamps of the leader CTA, or null:
                                 // 0 dependency resolved, 1 first chunk in shared memory, 2 accumulator complete, 3 stored and released,
                                 // 4 last MMA of the item issued
    unsigned long long* span;    // measurement aid (SZB_TOWER_SPAN): {first CTA start, last CTA end (%globaltimer), CTA 0's SM cycles, CTA 0's ns}, or null
    TowerLayer L[MAX_TOWER_LAYERS];
};

struct TowerItem { int l, t, q, ns; };
// tiles / n_main: a.n_pair_tiles / a.n_main, or their values for the tiles the device count leaves (TowerHeads::n_live)
__device__ __forceinline__ TowerItem tower_item(const TowerArgs& a, int item, int tiles, int n_main) {
    TowerItem it;
    if (item < n_main) {
        const int ti = item / a.nsplit;
        it.q = item - ti * a.nsplit;
        it.l = a.layer_begin + ti / tiles;
        it.t = ti % tiles;
        it.ns = a.nsplit;
    } else {
        it.l = a.layer_end - 1;
        it.t = item - n_main;
        it.q = 0;
        it.ns = 1;
    }
    return it;
}

// 256-bit global accesses (sm_100): 16 bf16 channels of one pixel per instruction.  The tower epilogue's lanes hold different
// pixels, so every instruction touches 32 lines whatever its width; twice the width is half the instructions and L1 wavefronts.
// p must be 32-byte aligned.
__device__ __forceinline__ void ldcg_256(const void* p, uint4& a, uint4& b) {
    asm volatile("ld.global.cg.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_256(void* p, const uint4& a, const uint4& b) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}

// one definition for every kernel that must agree bit for bit (k_softmax, the fused heads, k_value_head)
__device__ __noinline__ float sm_exp(float x, float mx) { return expf(__fsub_rn(x, mx)); }
__device__ __noinline__ float vh_tanh(float x) { return tanhf(x); }

// small-batch MMA issue of one K chunk of a 3x3 layer: nine taps in weight stages of TPS taps (4 + 4 + 1 or 2 + 2 + 2 + 2 + 1),
// each tap four K = 16 MMAs; straight-line, all descriptor offsets immediates.  Called warp-convergently by the leader's MMA warp.
template <int TPS>
__device__ __forceinline__ bool mma_chunk_3x3(uint32_t d_tmem, uint32_t chunk_lo, uint32_t b_lo0, uint32_t bar_bf0, uint32_t bar_be0,
                                              uint32_t& bs, uint32_t& b_phase, uint32_t idesc, uint32_t accumulate, volatile int* abort_flag) {
    constexpr uint32_t TILE_LO = (uint32_t)((128 / TPS) * TC_BLOCK_K * 2) >> 4;      // one tap's weight tile: 128 / TPS rows per CTA
#pragma unroll
    for (int s0 = 0; s0 < 9; s0 += TPS) {
        if (!warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag)) return false;
        tc_fence_after();
        const uint32_t b_base = b_lo0 + bs * (T2_B_BYTES >> 4);
        if (elect_one()) {
#pragma unroll
            for (int u = 0; u < TPS; u++) {
                const int tap = s0 + u;
                if (tap < 9) {
                    const uint32_t a_lo = chunk_lo + (uint32_t)((tap / 3) * 2 * HALO + tap % 3) * (128 >> 4);     // halo pixel (ky, board 0, kx)
                    const uint32_t b_lo = b_base + u * TILE_LO;
                    tc2_mma_bf16_split(d_tmem, a_lo, desc_hi(T2_A_SBO), b_lo, desc_hi(1024), idesc, tap == 0 ? accumulate : 1u);
                    tc2_mma_bf16_split(d_tmem, a_lo + 2, desc_hi(T2_A_SBO), b_lo + 2, desc_hi(1024), idesc, 1u);
                    tc2_mma_bf16_split(d_tmem, a_lo + 4, desc_hi(T2_A_SBO), b_lo + 4, desc_hi(1024), idesc, 1u);
                    tc2_mma_bf16_split(d_tmem, a_lo + 6, desc_hi(T2_A_SBO), b_lo + 6, desc_hi(1024), idesc, 1u);
                }
            }
            tc2_commit(bar_be0 + bs * 8);
        }
        __syncwarp();
        if (++bs == T2_B_STAGES) { bs = 0; b_phase ^= 1; }
    }
    return true;
}

// the same for whole 128-row tiles, two taps per 32 KiB stage (2 + 2 + 2 + 2 + 1): large-batch launches with TowerArgs::tps1 == 2
__device__ __forceinline__ bool mma_chunk_3x3_big(uint32_t d_tmem, uint32_t chunk_lo, uint32_t b_lo0, uint32_t bar_bf0, uint32_t bar_be0, uint32_t& bs,
                                                  uint32_t& b_phase, uint32_t idesc, uint32_t accumulate, volatile int* abort_flag) {
#pragma unroll
    for (int s0 = 0; s0 < 9; s0 += 2) {
        if (!warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag)) return false;
        tc_fence_after();
        const uint32_t b_base = b_lo0 + bs * (T2_BIG_BYTES >> 4);
        if (elect_one()) {
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int tap = s0 + u;
                if (tap < 9) {
                    const uint32_t a_lo = chunk_lo + (uint32_t)((tap / 3) * 2 * HALO + tap % 3) * (128 >> 4);
                    const uint32_t b_lo = b_base + u * (T2_B_BYTES >> 4);
                    tc2_mma_bf16_split(d_tmem, a_lo, desc_hi(T2_A_SBO), b_lo, desc_hi(1024), idesc, tap == 0 ? accumulate : 1u);
                    tc2_mma_bf16_split(d_tmem, a_lo + 2, desc_hi(T2_A_SBO), b_lo + 2, desc_hi(1024), idesc, 1u);
                    tc2_mma_bf16_split(d_tmem, a_lo + 4, desc_hi(T2_A_SBO), b_lo + 4, desc_hi(1024), idesc, 1u);
                    tc2_mma_bf16_split(d_tmem, a_lo + 6, desc_hi(T2_A_SBO), b_lo + 6, desc_hi(1024), idesc, 1u);
                }
            }
            tc2_commit(bar_be0 + bs * 8);
        }
        __syncwarp();
        if (++bs == T2_BIG_STAGES) { bs = 0; b_phase ^= 1; }
    }
    return true;
}

// DEV_COUNT: the launch serves the evaluation cache's compacted rows (TowerHeads::n_live / row_slot).  A template parameter, so that
// the launch without it is the same kernel as before.
template <bool DEV_COUNT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
k_tower_tc2(const __grid_constant__ TowerMaps maps, const __grid_constant__ TowerArgs a) {
    constexpr uint32_t IDESC_BASE = idesc_bf16(256, 0);                    // M = 256, N per layer
    constexpr int ACC_COLS = 256;

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_a_full[T2_A_CHUNKS], bar_a_empty[T2_A_CHUNKS], bar_b_full[T2_B_STAGES], bar_b_empty[T2_B_STAGES],
        bar_acc_full[2], bar_acc_empty[2];
    __shared__ uint32_t tmem_base_sh;
    __shared__ int abort_sh;
    __shared__ float bias_sh[2][C_TOWER];
    // fused heads (this CTA's two boards)
    __shared__ uint64_t hd_mask[2][MASK_WORDS];
    __shared__ float hd_red[2][2][4], hd_plane[2][64], hd_vw[C_TOWER], hd_fc[2][8];

    const uint32_t smem_a = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_b = smem_a + T2_A_CHUNKS * T2_A_CHUNK_BYTES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    int n_items = a.n_items, n_main = a.n_main, tiles = a.n_pair_tiles, n_live = a.n_boards;
    volatile int* abort_flag = &abort_sh;

    pdl_trigger();                                                // the next tree kernel may start its set-up; it waits for my completion
    auto slot_of = [&](long row) -> long { return DEV_COUNT ? heads_slot(a.heads, row) : row; };
    if (DEV_COUNT) {
        // evaluation cache: only the first n_live boards were filled (the cache misses).  The count is the tree kernel's, so every
        // thread waits for it first; the items of the tiles past it are dropped from the round-robin, which stays the same in every role.
        pdl_wait();
        n_live = heads_live_boards(a.heads, a.n_boards);
        tiles = (n_live + 3) / 4;
        n_main = a.n_main / a.n_pair_tiles * tiles;
        n_items = n_main + (a.n_items - a.n_main) / a.n_pair_tiles * tiles;
    }
    if (threadIdx.x == 0) {
        if (a.span) {
            atomicMin(a.span, global_ns());
            if (blockIdx.x == 0) { a.span[3] = global_ns(); a.span[2] = (unsigned long long)clock64(); }
        }
        abort_sh = 0;
        for (int s = 0; s < T2_A_CHUNKS; s++) { mbar_init(smem_u32(&bar_a_full[s]), 1); mbar_init(smem_u32(&bar_a_empty[s]), 1); }
        for (int s = 0; s < T2_B_STAGES; s++) { mbar_init(smem_u32(&bar_b_full[s]), 1); mbar_init(smem_u32(&bar_b_empty[s]), 1); }
        for (int s = 0; s < 2; s++) { mbar_init(smem_u32(&bar_acc_full[s]), 1); mbar_init(smem_u32(&bar_acc_empty[s]), READY_PER_ITEM); }
        fence_mbarrier_init();
    }
    if (warp == 1) tc2_tmem_alloc(smem_u32(&tmem_base_sh), 512);
    tc_fence_before();
    cluster_sync_all();                                           // both CTAs' barriers and TMEM exist from here on
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;

    if (warp == 0) {
        // ===== TMA producer (warp 0 of each CTA, convergent; one elected lane issues) =====
        // One blocking in-order stream (a polled two-stream variant was measured: the 32-lane mbarrier polling competes with
        // the MMAs for shared-memory cycles, +5 % tower time at 1024 boards).
        const uint32_t bar_af0 = smem_u32(&bar_a_full[0]), bar_ae0 = smem_u32(&bar_a_empty[0]);
        const uint32_t bar_bf0 = smem_u32(&bar_b_full[0]), bar_be0 = smem_u32(&bar_b_empty[0]);
        const int need = READY_PER_ITEM * a.nsplit;
        uint32_t ac = 0, bs = 0, a_phase = 0, b_phase = 0;
        bool ok = true;
        // tile (l-1, t) must be complete: all 8 epilogue warps of every pair that ran one of its nsplit items have stored and
        // released.  Every lane acquires (one transaction) so that whichever lane is elected afterwards has done so.
        auto wait_dependency = [&](int l, int t) -> bool {
            const int32_t* flag = a.ready + (size_t)(l - 1) * a.n_pair_tiles + t;
            if (!__all_sync(0xFFFFFFFFu, ld_acquire_gpu(flag) >= need)) {
                const long long t0 = clock64();
                for (;;) {
                    if (__all_sync(0xFFFFFFFFu, ld_acquire_gpu(flag) >= need)) break;
                    bool give_up = *abort_flag != 0;
                    if (clock64() - t0 > TC_TIMEOUT_CYCLES) { *abort_flag = 1; give_up = true; }
                    if (__any_sync(0xFFFFFFFFu, give_up)) return false;
                }
            }
            fence_proxy_async_global();     // generic-proxy stores -> this thread's TMA reads
            return true;
        };
        if (a.nsplit == 1) {
            // large batches: per K chunk the activation chunk, then its weight tiles (one per stage) -- in steady state the rings
            // keep the loads ~7 taps ahead of the MMAs
            pdl_wait();                                           // input rows and cleared counters come from the kernel before me
            for (int item = pair; item < n_items && ok; item += n_pairs) {
                const int l = a.layer_begin + item / tiles, t = item % tiles;
                const TowerLayer L = a.L[l];
                if (l > a.layer_begin && !(ok = wait_dependency(l, t))) break;
                if (a.trace && rank == 0 && lane == 0) a.trace[(size_t)item * TRACE_STAMPS + 0] = global_ns();      // dependency resolved
                const CUtensorMap* tm_a = &maps.a[L.a_map];
                const int board0 = a.board0 + (t * 2 + (int)rank) * 2 + (L.a_map == 0 ? a.in_delta : 0);
                const int wrow = l * C_TOWER + (int)rank * L.n_half;
                const CUtensorMap* tm_w = L.n_half == 128 ? &maps.w : &maps.w64;
                const uint32_t b_tx = 2u * (uint32_t)L.n_half * TC_BLOCK_K * 2;
                for (int kc = 0; kc < L.kchunks && ok; kc++) {
                    // one 64-channel slice of both boards' halo tiles: read by all taps of this K chunk
                    if (!(ok = warp_mbar_wait(bar_ae0 + ac * 8, a_phase ^ 1, abort_flag))) break;
                    if (elect_one()) {
                        const uint32_t a_full = bar_af0 + ac * 8;
                        if (rank == 0) mbar_expect_tx(a_full, 2u * T2_A_CHUNK_BYTES);     // both CTAs' bytes land on the leader's barrier
                        tma2_load_4d(smem_a + ac * T2_A_CHUNK_BYTES, tm_a, a_full, kc * TC_BLOCK_K, 0, board0, 0);
                    }
                    __syncwarp();
                    if (++ac == T2_A_CHUNKS) { ac = 0; a_phase ^= 1; }
                    int kcol = kc * TC_BLOCK_K;                                           // weight column of (tap 0, kc); taps are C_in apart
                    if (a.tps1 == 2) {
                        // two taps per stage, three 32 KiB stages (a 1x1 layer: one tile per stage)
                        for (int tap = 0; tap < L.taps; tap += 2) {
                            const int cnt = min(2, L.taps - tap);
                            if (!(ok = warp_mbar_wait(bar_be0 + bs * 8, b_phase ^ 1, abort_flag))) break;
                            if (elect_one()) {
                                const uint32_t b_full = bar_bf0 + bs * 8;
                                if (rank == 0) mbar_expect_tx(b_full, b_tx * (uint32_t)cnt);
                                for (int u = 0; u < cnt; u++)
                                    tma2_load_2d(smem_b + bs * T2_BIG_BYTES + u * T2_B_BYTES, tm_w, b_full, kcol + (tap + u) * L.kchunks * TC_BLOCK_K, wrow);
                            }
                            __syncwarp();
                            if (++bs == T2_BIG_STAGES) { bs = 0; b_phase ^= 1; }
                        }
                        continue;
                    }
                    for (int tap = 0; tap < L.taps; tap++, kcol += L.kchunks * TC_BLOCK_K) {
                        if (!(ok = warp_mbar_wait(bar_be0 + bs * 8, b_phase ^ 1, abort_flag))) break;
                        if (elect_one()) {
                            const uint32_t b_full = bar_bf0 + bs * 8;
                            if (rank == 0) mbar_expect_tx(b_full, b_tx);
                            tma2_load_2d(smem_b + bs * T2_B_BYTES, tm_w, b_full, kcol, wrow);
                        }
                        __syncwarp();
                        if (++bs == T2_B_STAGES) { bs = 0; b_phase ^= 1; }
                    }
                }
            }
        } else {
            // small batches (at most one item per pair and layer; every item really waits for its dependency).  An item's weight
            // tiles are only 128 / nsplit rows per CTA, so a 16 KiB stage takes `tps` consecutive tiles (one barrier, several
            // boxes): with one small tile per stage the 7-stage ring covers ~0.5 us of MMAs, less than one L2 -> SM latency, and
            // the item runs at TMA latency (traced: 9 us per 3x3 layer for 2.4 us of MMAs).  The first stages are issued BEFORE
            // the dependency wait (weights do not depend on the previous layer), then all activation chunks at once, then the
            // remaining weight stages.
            for (int item = pair; item < n_items && ok; item += n_pairs) {
                const TowerItem it = tower_item(a, item, tiles, n_main);
                const int l = it.l, t = it.t, q = it.q;
                const TowerLayer L = a.L[l];
                const CUtensorMap* tm_a = &maps.a[L.a_map];
                const int board0 = a.board0 + (t * 2 + (int)rank) * 2 + (L.a_map == 0 ? a.in_delta : 0);
                const int nh = L.n_half / it.ns;                                  // weight rows per CTA of this item
                const int tps = L.taps == 9 ? it.ns : 1;                          // weight tiles per stage (3x3 layers: 128 / nh)
                const int wrow = l * C_TOWER + q * 2 * nh + (int)rank * nh;
                const CUtensorMap* tm_w = nh == 64 ? &maps.w64 : nh == 32 ? &maps.w32 : nh == 16 ? &maps.w16 : &maps.w8;
                const uint32_t tile_bytes = (uint32_t)nh * TC_BLOCK_K * 2;
                const int n_b = L.taps * L.kchunks;
                int jb = 0, kc_b = 0, tap_b = 0;
                // next stage of weight tiles in MMA order (K chunk outer, tap inner; stages do not straddle K chunks, so the MMA
                // warp's per-chunk code is straight-line); weight column of (tap, kc): taps are C_in apart
                auto issue_b_stage = [&]() -> bool {
                    if (!warp_mbar_wait(bar_be0 + bs * 8, b_phase ^ 1, abort_flag)) return false;
                    const int cnt = min(tps, L.taps - tap_b);
                    if (elect_one()) {
                        const uint32_t b_full = bar_bf0 + bs * 8;
                        if (rank == 0) mbar_expect_tx(b_full, 2u * tile_bytes * (uint32_t)cnt);
                        for (int u = 0; u < cnt; u++)
                            tma2_load_2d(smem_b + bs * T2_B_BYTES + u * tile_bytes, tm_w, b_full, ((tap_b + u) * L.kchunks + kc_b) * TC_BLOCK_K, wrow);
                    }
                    __syncwarp();
                    if (++bs == T2_B_STAGES) { bs = 0; b_phase ^= 1; }
                    tap_b += cnt;
                    if (tap_b == L.taps) { tap_b = 0; kc_b++; }
                    jb += cnt;
                    return true;
                };
                for (int k = 0; k < T2_B_STAGES && jb < n_b && ok; k++) ok = issue_b_stage();
                if (!ok) break;
                pdl_wait();                                       // (weights above do not depend on the kernel before me; everything below does)
                if (l > a.layer_begin && !(ok = wait_dependency(l, t))) break;
                if (a.trace && rank == 0 && lane == 0) a.trace[(size_t)item * TRACE_STAMPS + 0] = global_ns();      // dependency resolved
                for (int kc = 0; kc < L.kchunks && ok; kc++) {
                    if (!(ok = warp_mbar_wait(bar_ae0 + ac * 8, a_phase ^ 1, abort_flag))) break;
                    if (elect_one()) {
                        const uint32_t a_full = bar_af0 + ac * 8;
                        if (rank == 0) mbar_expect_tx(a_full, 2u * T2_A_CHUNK_BYTES);
                        tma2_load_4d(smem_a + ac * T2_A_CHUNK_BYTES, tm_a, a_full, kc * TC_BLOCK_K, 0, board0, 0);
                    }
                    __syncwarp();
                    if (++ac == T2_A_CHUNKS) { ac = 0; a_phase ^= 1; }
                }
                while (jb < n_b && ok) ok = issue_b_stage();
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (leader CTA only) =====
        // One thread feeds the tensor cores of both SMs; its instruction stream is the limit once loads are ahead (ncu: no
        // barrier stalls, ~1100 cycles of issue per 512 cycles of MMA with naive descriptor code).  So: descriptors are
        // kept as (lo, hi) halves with constant hi and an incrementally advanced lo, barrier addresses are computed once,
        // the 3x3 tap loop has no division.
        // The whole warp runs the loop convergently (so the compiler keeps descriptors and barrier addresses in uniform
        // registers instead of broadcasting them per MMA); one elected lane issues.
        if (rank == 0) {
            const uint32_t a_lo0 = ((smem_a >> 4) & 0x3FFFu) | DESC_LO_FLAGS, b_lo0 = ((smem_b >> 4) & 0x3FFFu) | DESC_LO_FLAGS;
            const uint32_t bar_af0 = smem_u32(&bar_a_full[0]), bar_ae0 = smem_u32(&bar_a_empty[0]);
            const uint32_t bar_bf0 = smem_u32(&bar_b_full[0]), bar_be0 = smem_u32(&bar_b_empty[0]);
            const uint32_t bar_cf0 = smem_u32(&bar_acc_full[0]), bar_ce0 = smem_u32(&bar_acc_empty[0]);
            uint32_t ac = 0, bs = 0, a_phase = 0, b_phase = 0;
            int local = 0;
            bool ok = true;
            const bool big = a.nsplit == 1 && a.tps1 == 2;
            for (int item = pair; item < n_items && ok; item += n_pairs, local++) {
                const TowerItem it = tower_item(a, item, tiles, n_main);
                const TowerLayer L = a.L[it.l];
                const uint32_t idesc = IDESC_BASE | ((uint32_t)(2 * L.n_half / it.ns >> 3) << 17);
                const uint32_t acc = local & 1;
                const uint32_t acc_phase = (local >> 1) & 1;
                if (!(ok = warp_mbar_wait(bar_ce0 + acc * 8, acc_phase ^ 1, abort_flag))) break;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * ACC_COLS;
                uint32_t accumulate = 0;
                // One MMA costs this warp ~100 cycles of instructions in a generic tap loop (traced: 210 ns per tap of four MMAs
                // whatever N) -- as long as the four N = 256 MMAs of a tap themselves (512 cycles), and far longer than the
                // N <= 128 MMAs of small-batch items -- so the nine taps of a K chunk are straight-line code (mma_chunk_3x3).
                for (int kc = 0; kc < L.kchunks && ok; kc++) {
                    if (!(ok = warp_mbar_wait(bar_af0 + ac * 8, a_phase, abort_flag))) break;
                    if (a.trace && kc == 0 && lane == 0) a.trace[(size_t)item * TRACE_STAMPS + 1] = global_ns();     // first activation chunk in shared memory
                    const uint32_t chunk_lo = a_lo0 + ac * (T2_A_CHUNK_BYTES >> 4);
                    if (L.taps == 9) {
                        // a weight stage holds nsplit consecutive taps of 128 / nsplit rows per CTA (see the producer)
                        ok = big          ? mma_chunk_3x3_big(d_tmem, chunk_lo, b_lo0, bar_bf0, bar_be0, bs, b_phase, idesc, accumulate, abort_flag)
                             : it.ns == 1 ? mma_chunk_3x3<1>(d_tmem, chunk_lo, b_lo0, bar_bf0, bar_be0, bs, b_phase, idesc, accumulate, abort_flag)
                             : it.ns == 2 ? mma_chunk_3x3<2>(d_tmem, chunk_lo, b_lo0, bar_bf0, bar_be0, bs, b_phase, idesc, accumulate, abort_flag)
                             : it.ns == 8 ? mma_chunk_3x3<8>(d_tmem, chunk_lo, b_lo0, bar_bf0, bar_be0, bs, b_phase, idesc, accumulate, abort_flag)
                                             : mma_chunk_3x3<4>(d_tmem, chunk_lo, b_lo0, bar_bf0, bar_be0, bs, b_phase, idesc, accumulate, abort_flag);
                    } else {
                        // 1x1 convolution = centre tap, one weight tile per stage
                        if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                        tc_fence_after();
                        const uint32_t a_lo = chunk_lo + (uint32_t)(2 * HALO + 1) * (128 >> 4);
                        const uint32_t b_lo = b_lo0 + bs * ((big ? T2_BIG_BYTES : T2_B_BYTES) >> 4);
                        if (elect_one()) {
                            tc2_mma_bf16_split(d_tmem, a_lo, desc_hi(T2_A_SBO), b_lo, desc_hi(1024), idesc, accumulate);
                            tc2_mma_bf16_split(d_tmem, a_lo + 2, desc_hi(T2_A_SBO), b_lo + 2, desc_hi(1024), idesc, 1u);
                            tc2_mma_bf16_split(d_tmem, a_lo + 4, desc_hi(T2_A_SBO), b_lo + 4, desc_hi(1024), idesc, 1u);
                            tc2_mma_bf16_split(d_tmem, a_lo + 6, desc_hi(T2_A_SBO), b_lo + 6, desc_hi(1024), idesc, 1u);
                            tc2_commit(bar_be0 + bs * 8);
                        }
                        __syncwarp();
                        if (++bs == (uint32_t)(big ? T2_BIG_STAGES : T2_B_STAGES)) { bs = 0; b_phase ^= 1; }
                    }
                    accumulate = 1;
                    if (ok && elect_one()) tc2_commit(bar_ae0 + ac * 8);                              // chunk free once its last tap's MMAs retire
                    __syncwarp();
                    if (++ac == T2_A_CHUNKS) { ac = 0; a_phase ^= 1; }
                }
                if (a.trace && lane == 0) a.trace[(size_t)item * TRACE_STAMPS + 4] = global_ns();        // last MMA of the item issued
                if (ok && elect_one()) tc2_commit(bar_cf0 + acc * 8);
                __syncwarp();
            }
        }
    } else {
        // ===== epilogue (4 warps in each CTA): TMEM -> +bias [+residual] -> ReLU -> bf16 NHWC store =====
        pdl_wait();
        const int lane_group = warp & 3;
        const int etid = threadIdx.x - 64;                         // 0..127
        int local = 0;
        bool ok = true;
        for (int item = pair; item < n_items && ok; item += n_pairs, local++) {
            const TowerItem it = tower_item(a, item, tiles, n_main);
            const int l = it.l, t = it.t, q = it.q;
            const TowerLayer L = a.L[l];
            const int n_item = 2 * L.n_half / it.ns, cb = q * n_item;         // this item's output channels: [cb, cb + n_item)
            const int acc = local & 1;
            const uint32_t acc_phase = (local >> 1) & 1;
            bias_sh[acc][etid] = a.bias[l * C_TOWER + etid];
            bias_sh[acc][etid + 128] = a.bias[l * C_TOWER + etid + 128];
            named_bar_sync<1, 128>();
            // accumulator row (TMEM lane) = (oy * 2 + board-in-CTA) * 8 + ox
            const int row = lane_group * 32 + lane;
            const int board = a.board0 + (t * 2 + (int)rank) * 2 + ((row >> 3) & 1);
            const int sq = (row >> 4) * 8 + (row & 7);
            const bool live = board < a.board0 + n_live;
            const uint32_t taddr = tmem_base + ((uint32_t)(lane_group * 32) << 16) + acc * ACC_COLS;
            const size_t pix = ((size_t)board * HALO + (sq >> 3) + 1) * HALO + (sq & 7) + 1;
            // The residual (output of layer l - 2) starts its way from L2 before the accumulator wait -- but only once this warp
            // has itself acquired the completion counter of tile (l-1, t), which implies (l-2, t): before the accumulator
            // barrier nothing else orders this warp after the other pairs' stores.  One poll; if the tile is not complete
            // yet the loads are issued after the wait as before.
            const __nv_bfloat16* resp = (L.mode == 0 && L.res != 255 && live) ? a.act[L.res] + pix * C_TOWER + cb : nullptr;
            uint4 rnext[4];
            const bool early = l == a.layer_begin || ld_acquire_gpu(a.ready + (size_t)(l - 1) * a.n_pair_tiles + t) >= READY_PER_ITEM * a.nsplit;
            if (resp && early) {                                                                  // written by another SM: bypass L1
                ldcg_256(resp, rnext[0], rnext[1]);
                ldcg_256(resp + 16, rnext[2], rnext[3]);
            }
            ok = mbar_wait(smem_u32(&bar_acc_full[acc]), acc_phase, abort_flag);
            ok = __all_sync(0xFFFFFFFFu, ok);
            if (!ok) break;
            tc_fence_after();
            if (resp && !early) {
                ldcg_256(resp, rnext[0], rnext[1]);
                ldcg_256(resp + 16, rnext[2], rnext[3]);
            }
            const bool tracer = a.trace && rank == 0 && warp == 2 && lane == 0;
            if (tracer) a.trace[(size_t)item * TRACE_STAMPS + 2] = global_ns();                    // accumulator complete
            if (L.mode == 1 && a.heads.mask != nullptr) {
                // ===== fused heads (an unsplit item: all 73 planes of this CTA's two boards sit in this accumulator) =====
                // Thread = (board, square) row with its 73 logits in TMEM.  softmax over the board's 4672 logits in the order
                // k_softmax uses (per square over the planes, then a fixed tree over the squares), so that the priors are
                // bit-identical to the unfused path's; only the legal moves' entries are written.
                const int rb = (row >> 3) & 1;                                        // board within this CTA
                const int cta_board0 = a.board0 + (t * 2 + (int)rank) * 2;
                const long row_slot = DEV_COUNT ? (live ? heads_slot(a.heads, (long)board + a.heads.row_delta) : 0) : (long)board + a.heads.row_delta;
                const bool want = live && a.heads.need_eval[row_slot] != 0;
                for (int i = etid; i < 2 * MASK_WORDS; i += 128) {
                    const int bb = i >= MASK_WORDS, w = i - bb * MASK_WORDS, brd = cta_board0 + bb;
                    hd_mask[bb][w] = brd < a.board0 + n_live ? a.heads.mask[(size_t)slot_of(brd + a.heads.row_delta) * MASK_STRIDE + w] : 0ull;
                }
                hd_vw[etid] = a.heads.v_w[etid];
                hd_vw[etid + 128] = a.heads.v_w[etid + 128];
                const float* bias = bias_sh[acc];
                float mx = -INFINITY;
#pragma unroll 1
                for (int c0 = 0; c0 < 96; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(taddr + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j++)
                        if (c0 + j < POLICY_PLANES) mx = fmaxf(mx, __fadd_rn(__uint_as_float(v[j]), bias[c0 + j]));
                }
                // the 16 squares of this board held by this warp: lane bits 0-2 (file) and 4 (rank parity); lane bit 3 is the board
                mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, 1));
                mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, 2));
                mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, 4));
                mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, 16));
                if ((lane & 0x17) == 0) hd_red[0][rb][lane_group] = mx;
                named_bar_sync<1, 128>();
                mx = fmaxf(fmaxf(hd_red[0][rb][0], hd_red[0][rb][1]), fmaxf(hd_red[0][rb][2], hd_red[0][rb][3]));
                float ssum = 0.f;
#pragma unroll 1
                for (int c0 = 0; c0 < 96; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(taddr + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j++)
                        if (c0 + j < POLICY_PLANES) ssum = __fadd_rn(ssum, sm_exp(__fadd_rn(__uint_as_float(v[j]), bias[c0 + j]), mx));
                }
                ssum = __fadd_rn(ssum, __shfl_xor_sync(0xFFFFFFFFu, ssum, 1));
                ssum = __fadd_rn(ssum, __shfl_xor_sync(0xFFFFFFFFu, ssum, 2));
                ssum = __fadd_rn(ssum, __shfl_xor_sync(0xFFFFFFFFu, ssum, 4));
                ssum = __fadd_rn(ssum, __shfl_xor_sync(0xFFFFFFFFu, ssum, 16));
                if ((lane & 0x17) == 0) hd_red[1][rb][lane_group] = ssum;           // squares [16 g, 16 g + 16), g = lane_group
                named_bar_sync<1, 128>();
                const float tot = __fadd_rn(__fadd_rn(__fadd_rn(hd_red[1][rb][0], hd_red[1][rb][1]), hd_red[1][rb][2]), hd_red[1][rb][3]);
                float* prow = a.heads.policy + (size_t)row_slot * N_ACTIONS + sq;
#pragma unroll 1
                for (int c0 = 0; c0 < 96; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(taddr + c0, v);
                    tmem_ld_wait();
                    if (want) {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (c0 + j < POLICY_PLANES && ((hd_mask[rb][c0 + j] >> sq) & 1ull))
                                prow[(c0 + j) * 64] = __fdiv_rn(sm_exp(__fadd_rn(__uint_as_float(v[j]), bias[c0 + j]), mx), tot);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(smem_u32(&bar_acc_empty[acc]));      // accumulator free; nothing waits on this layer's counter
                // ---- value head (network.py:156-174) on the tower output of this thread's pixel, same arithmetic as k_value_head ----
                float p4[4] = {0.f, 0.f, 0.f, 0.f};
                if (live) {
                    const __nv_bfloat16* tp = a.heads.tower_out + pix * C_TOWER;
#pragma unroll
                    for (int part = 0; part < 4; part++) {
#pragma unroll
                        for (int qq = 0; qq < 8; qq += 2) {
                            uint4 u[2];
                            ldcg_256(tp + part * 64 + qq * 8, u[0], u[1]);              // written by other SMs during this launch
                            const __nv_bfloat16* h8 = reinterpret_cast<const __nv_bfloat16*>(u);
#pragma unroll
                            for (int j = 0; j < 16; j++) p4[part] = fmaf(__bfloat162float(h8[j]), hd_vw[part * 64 + qq * 8 + j], p4[part]);
                        }
                    }
                }
                hd_plane[rb][sq] = fmaxf(__fadd_rn(__fadd_rn(__fadd_rn(p4[0], p4[1]), __fadd_rn(p4[2], p4[3])), a.heads.scalars[0]), 0.f);
                named_bar_sync<1, 128>();
#pragma unroll 1
                for (int k2 = 0; k2 < 4; k2++) {
                    const int bb = k2 >> 1, o = etid + 128 * (k2 & 1);
                    float h = a.heads.fc1_b[o];
#pragma unroll 8
                    for (int k = 0; k < 64; k++) h = fmaf(hd_plane[bb][k], a.heads.fc1_wT[k * 256 + o], h);
                    h = __fmul_rn(fmaxf(h, 0.f), a.heads.fc2_w[o]);
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) h = __fadd_rn(h, __shfl_xor_sync(0xFFFFFFFFu, h, off));
                    if (lane == 0) hd_fc[bb][(k2 & 1) * 4 + (etid >> 5)] = h;
                }
                named_bar_sync<1, 128>();
                if (etid < 2) {
                    const int brd = cta_board0 + etid;
                    const long bslot = DEV_COUNT ? (brd < a.board0 + n_live ? heads_slot(a.heads, brd + a.heads.row_delta) : 0) : brd + a.heads.row_delta;
                    if (brd < a.board0 + n_live && a.heads.need_eval[bslot]) {
                        float tt = a.heads.scalars[1];
#pragma unroll
                        for (int w = 0; w < 8; w++) tt = __fadd_rn(tt, hd_fc[etid][w]);
                        a.heads.value[bslot] = vh_tanh(tt);
                    }
                }
                continue;
            }
            if (L.mode == 1) {
                // policy logits, plane-major like torch.flatten(conv_p2(x)): index = plane * 64 + row * 8 + col
                float* lg = a.logits + (size_t)board * N_ACTIONS + sq;
#pragma unroll 1
                for (int c0 = 0; c0 < n_item && cb + c0 < POLICY_PLANES; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(taddr + c0, v);
                    tmem_ld_wait();
                    if (live) {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (c0 + j < n_item && cb + c0 + j < POLICY_PLANES)
                                lg[(cb + c0 + j) * 64] = __fadd_rn(__uint_as_float(v[j]), bias_sh[acc][cb + c0 + j]);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(smem_u32(&bar_acc_empty[acc]));      // last layer: nothing waits on its counter
                continue;
            }
            __nv_bfloat16* outp = a.act[L.out] + pix * C_TOWER + cb;
            const float* bias = bias_sh[acc] + cb;
#pragma unroll 1
            for (int c0 = 0; c0 < n_item; c0 += 32) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + c0, v);
                uint4 rcur[4];
                if (resp) {
#pragma unroll
                    for (int u = 0; u < 4; u++) rcur[u] = rnext[u];
                    if (c0 + 32 < n_item) {
                        ldcg_256(resp + c0 + 32, rnext[0], rnext[1]);
                        ldcg_256(resp + c0 + 48, rnext[2], rnext[3]);
                    }
                }
                tmem_ld_wait();
                if (live) {
                    uint4 o[4];
                    __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(o);
                    const __nv_bfloat162* rb = reinterpret_cast<const __nv_bfloat162*>(rcur);
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        float x0 = __uint_as_float(v[2 * j]) + bias[c0 + 2 * j];
                        float x1 = __uint_as_float(v[2 * j + 1]) + bias[c0 + 2 * j + 1];
                        if (resp) {
                            const float2 r = __bfloat1622float2(rb[j]);
                            x0 += r.x;
                            x1 += r.y;
                        }
                        if (L.relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
                        ob[j] = __floats2bfloat162_rn(x0, x1);
                    }
                    st_256(outp + c0, o[0], o[1]);
                    st_256(outp + c0 + 16, o[2], o[3]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive_leader(smem_u32(&bar_acc_empty[acc]));            // accumulator stage free again (leader's barrier)
                // the warp's stores happen-before this lane's release (__syncwarp above; release is cumulative); the reader
                // orders its TMA (async-proxy) loads after its acquire with fence.proxy.async
                fence_proxy_async_global();
                red_release_gpu_add(a.ready + (size_t)l * a.n_pair_tiles + t, 1);
                if (tracer) a.trace[(size_t)item * TRACE_STAMPS + 3] = global_ns();                // outputs stored and released
            }
        }
    }
    // ===== teardown =====
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    if (warp == 1) tc2_tmem_dealloc(tmem_base, 512);
    if (threadIdx.x == 0 && abort_sh) atomicExch(a.error, 1);
    if (threadIdx.x == 0 && a.span) {
        if (blockIdx.x == 0) { a.span[2] = (unsigned long long)clock64() - a.span[2]; a.span[3] = global_ns() - a.span[3]; }   // SM clocks per ns inside this launch
        atomicMax(a.span + 1, global_ns());
    }
}

// =================================================================================================
// cluster-resident tower for very small batches: ONE BOARD PER 8-CTA CLUSTER, activations never leave shared memory
// =================================================================================================
// k_tower_tc2 at <= 72 boards is a chain of 41 dependent layers at ~6.7-8 us each: every layer hands its output to the next through
// L2 (epilogue stores -> red.release -> ld.acquire -> TMA reload, ~2.5 us of round trips) and every tensor-core instruction re-reads
// 128 activation rows per CTA from shared memory whatever the batch (144 x ~40 clk, ~3 us).  For a handful of boards -- a single game
// (play.py, the reference's real API), an arena pair, the tail of a self-play iteration -- this kernel keeps a board inside one
// cluster of 8 SMs for the whole tower:
//   * CTA r of the cluster computes output channels [32 r, 32 r + 32) of every layer: tcgen05.mma.cta_group::1, M = 64 (the board's
//     squares: half the shared-memory operand traffic of M = 128), N = 32, accumulator in 32 TMEM columns;
//   * every CTA holds the board's full activation tile (256 channels x 100 halo pixels, bf16, the same 128-byte-swizzled halo layout
//     k_tower_tc2 stages per K chunk, so all nine taps read it in place through shifted descriptors) TWICE (layer l reads buffer l & 1
//     and the cluster writes buffer (l + 1) & 1);
//   * the epilogue (TMEM -> +bias [+residual, kept in registers: a CTA only ever needs its own 32 channels of it] -> ReLU -> bf16)
//     stores its 64 x 32 slice straight into all eight CTAs' next-layer buffers (st.shared::cluster, distributed shared memory) and
//     arrives on each CTA's mbarrier (release.cluster); a layer starts when its CTA has collected all 32 arrivals -- no global memory,
//     no TMA reload, no cluster-wide hardware barrier, the weight producer warp runs ahead freely (7 x 16 KiB ring);
//   * the heads run inside the same launch: CTA 0 gathers the 73 logit planes (fp32, distributed shared memory) and does the softmax
//     in k_softmax's order (full logits, or just the priors of the legal moves in search mode), CTA 1 the value head on the tower
//     output still sitting in its shared memory.
// Same MMAs per output element in the same K order (K chunk outer, tap inner) -> bit-identical to k_tower_tc2
// (test_cluster_tower_bit_identical).
// Two cluster sizes: 8 CTAs (N = 32 channels per CTA; the default) and 16 CTAs (N = 16, non-portable cluster size, A/B aid).
// What a layer costs (device timestamps, scripts/cluster_trace.py, one board): 3.6 us from "input complete" to "last MMA issued",
// 0.1 us to the accumulator, 1.4 us of distributed-shared-memory stores (32 KiB out of every CTA at ~12 B/clk), 1.3 us until the
// slowest CTA's bytes have landed and the MMA warp is awake.  The 3.6 us are the ISSUE of the layer's 144 dependent tcgen05.mma by
// one thread (~28 clk each; per weight stage: 106-152 clk barrier wait + 16 x 28 clk) -- not the tensor core (issuing half of the
// MMAs: -0.5 us), not the weight stream (16 CTAs per board = a whole layer prefetched, or the contiguous pre-swizzled stream below:
// no change).  K = 16 per instruction and one accumulation chain per output (bit-identity with the large-batch kernel) fix the
// count; a shorter chain needs split-K, i.e. other roundings than k_tower_tc2's.
constexpr int CL_CHUNK_BYTES = 13 * 1024;                     // 100 halo pixels x 128 B = 12800, padded to the 1024-byte swizzle period
constexpr int CL_BUF_BYTES = 4 * CL_CHUNK_BYTES;              // 256 channels
constexpr int CL_RING_BYTES = 7 * 16384;                      // weight ring
constexpr int CL_SMEM = 2 * CL_BUF_BYTES + CL_RING_BYTES + 1024;
constexpr int CL_MAX_STAGES = 14;
template <int CS> struct ClCfg {
    static constexpr int N = C_TOWER / CS;                    // output channels per CTA: 32 | 16
    static constexpr int TILE_BYTES = N * TC_BLOCK_K * 2;     // one tap's N x 64 weights
    static constexpr int STAGE_BYTES = 4 * TILE_BYTES;        // four taps per stage (a K chunk of a 3x3 layer = 4 + 4 + 1)
    static constexpr int STAGES = CL_RING_BYTES / STAGE_BYTES;   // 7 | 14
    static constexpr int NP = 128 / CS;                       // policy planes per CTA (73 padded to 128): 16 | 8
};
constexpr uint32_t CL_LAYER_BYTES = 64 * C_TOWER * 2;         // a layer's output for one board
constexpr int CL_MAX_BOARDS = 18;                             // 18 clusters x 8 = 144 of 148 SMs

// Weight stream of k_tower_cl.  Through a tensor map a 32-row weight tile arrives as 32 separate 128-byte rows (4608 B apart in
// w16_all) and a CTA ingests only ~44 GB/s that way -- measured: issuing HALF of a layer's MMAs left the layer's MMA phase at
// 3.3 of 3.6 us, the phase waits for weights, not for the tensor core.  So the folded weights are stored once more in exactly the
// order and byte image a CTA consumes them: per (layer, rank) one contiguous run of [K chunk][tap] tiles, each tile the
// 128-byte-swizzled shared-memory image of its (rows x 64) block; a ring stage is then ONE contiguous bulk copy of up to 16 KiB.
constexpr size_t CL_W_LAYER_ELEMS = (size_t)C_TOWER * 9 * C_TOWER;          // 2304 x 256: stride of a layer in the stream
// one thread per 16-byte piece: (layer l, rank, tile = kc * taps + tap, row, piece)
__global__ void k_pack_cluster_weights(const __nv_bfloat16* w16_all, __nv_bfloat16* out, int l, int taps, int kchunks, int n, int cs) {
    const int tiles = taps * kchunks;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)cs * tiles * n * 8;
    if (i >= total) return;
    const int j = (int)(i & 7), r = (int)((i >> 3) % n), tile = (int)((i / (8 * (size_t)n)) % tiles), rank = (int)(i / (8 * (size_t)n * tiles));
    const int kc = tile / taps, tap = tile - kc * taps;
    const uint4 v = *reinterpret_cast<const uint4*>(w16_all + ((size_t)l * C_TOWER + rank * n + r) * (9 * C_TOWER) + (size_t)(tap * kchunks + kc) * TC_BLOCK_K + j * 8);
    __nv_bfloat16* dst = out + (size_t)l * CL_W_LAYER_ELEMS + (size_t)rank * (CL_W_LAYER_ELEMS / cs) + (size_t)tile * n * TC_BLOCK_K + (size_t)r * TC_BLOCK_K + (size_t)((j ^ (r & 7)) * 8);
    *reinterpret_cast<uint4*>(dst) = v;
}

struct ClusterArgs {
    int n_boards;
    int board0;                  // first board (row of the NHWC input buffer, before in_delta)
    int in_delta;
    const float* bias;           // [MAX_TOWER_LAYERS][256]
    const __nv_bfloat16* w_stream;   // Net::w16_cl
    TowerHeads heads;            // mask == null: full fp32 logits to `logits`; value always written (heads.value)
    float* logits;               // [row][4672], row = board + heads.row_delta
    int32_t* error;
    unsigned long long* trace;   // measurement aid (SZB_TOWER_TRACE with szb_time_kernel(6)): [layer][8] %globaltimer stamps of cluster 0, CTA 0
    TowerLayer L[MAX_TOWER_LAYERS];
};

template <int CS>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(TC_THREADS, 1)
k_tower_cl(const __grid_constant__ TowerMaps maps, const __grid_constant__ ClusterArgs a) {
    constexpr int CL_SIZE = CS, CL_N = ClCfg<CS>::N, CL_B_STAGES = ClCfg<CS>::STAGES, CL_TILE_BYTES = ClCfg<CS>::TILE_BYTES,
                  CL_STAGE_BYTES = ClCfg<CS>::STAGE_BYTES, CL_NP = ClCfg<CS>::NP;
    constexpr size_t CL_W_RANK_ELEMS = CL_W_LAYER_ELEMS / CS;
    constexpr uint32_t IDESC_M64 = idesc_bf16(64, 0);                     // M = 64, N per layer

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_b_full[CL_MAX_STAGES], bar_b_empty[CL_MAX_STAGES], bar_acc_full, bar_act[2], bar_in, bar_lg;
    __shared__ uint32_t tmem_base_sh;
    __shared__ int abort_sh;
    __shared__ float bias_sh[2][32];
    __shared__ uint64_t hd_mask[MASK_WORDS];
    __shared__ float hd_red[2][4], hd_plane[64], hd_vw[C_TOWER], hd_fc[8];

    const uint32_t smem_act = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_b = smem_act + 2 * CL_BUF_BYTES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int board = a.board0 + (int)(blockIdx.x / CL_SIZE);            // this cluster's board
    volatile int* abort_flag = &abort_sh;

    pdl_trigger();
    // evaluation cache: a cluster whose board lies past the tree kernel's count of filled rows has nothing to do (all its CTAs see
    // the same board and leave together, before any cluster barrier)
    if (a.heads.n_live) {
        pdl_wait();
        if (board - a.board0 >= heads_live_boards(a.heads, a.n_boards)) return;
    }
    if (threadIdx.x == 0) {
        abort_sh = 0;
        for (int s = 0; s < CL_B_STAGES; s++) { mbar_init(smem_u32(&bar_b_full[s]), 1); mbar_init(smem_u32(&bar_b_empty[s]), 1); }
        mbar_init(smem_u32(&bar_acc_full), 1);
        // layer l's output (32 KiB: 64 squares x 256 channels, from the eight CTAs' asynchronous stores) is counted in BYTES on
        // bar_act[l & 1]; its one arrival is this CTA's own expect_tx, posted two layers ahead
        mbar_init(smem_u32(&bar_act[0]), 1);
        mbar_init(smem_u32(&bar_act[1]), 1);
        mbar_init(smem_u32(&bar_in), 1);
        mbar_init(smem_u32(&bar_lg), 4 * CL_SIZE);
        fence_mbarrier_init();
        mbar_expect_tx(smem_u32(&bar_act[0]), CL_LAYER_BYTES);            // layer 0's and layer 1's outputs
        mbar_expect_tx(smem_u32(&bar_act[1]), CL_LAYER_BYTES);
    }
    // both activation buffers start as zeros: the halo pixels are never written afterwards
    {
        uint4* z = reinterpret_cast<uint4*>(smem_raw + (smem_act - smem_u32(smem_raw)));
        for (int i = threadIdx.x; i < 2 * CL_BUF_BYTES / 16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
    }
    if (warp == 1) tc_tmem_alloc(smem_u32(&tmem_base_sh), 32);
    fence_proxy_async();                      // the zeros (generic proxy) -> TMA writes / tensor-core reads
    tc_fence_before();
    cluster_sync_all();                                                   // every CTA's barriers and zeroed buffers exist from here on
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_sh;

    if (warp == 0) {
        // ===== producer: the board's input planes once, then this CTA's weight slices of all 41 layers, as far ahead as the ring allows =====
        const uint32_t bar_bf0 = smem_u32(&bar_b_full[0]), bar_be0 = smem_u32(&bar_b_empty[0]);
        // the weight ring is primed first (weights do not depend on the kernel before this one: with programmatic dependent launch
        // they stream in while the tree kernel still runs); then the dependency wait, then the board's input planes
        int issued = 0;
        auto send_input = [&]() {
            pdl_wait();
            if (elect_one()) {
                const uint32_t in_full = smem_u32(&bar_in);
                mbar_expect_tx(in_full, 2u * 12800u);
                for (int kc = 0; kc < C_IN_PAD / TC_BLOCK_K; kc++)
                    tma_load_4d(smem_act + kc * CL_CHUNK_BYTES, &maps.in1, in_full, kc * TC_BLOCK_K, 0, board + a.in_delta, 0);
            }
            __syncwarp();
        };
        uint32_t bs = 0, b_phase = 0;
        bool ok = true;
        for (int l = 0; l < MAX_TOWER_LAYERS && ok; l++) {
            const TowerLayer L = a.L[l];
            const int n = L.mode == 1 ? CL_NP : CL_N;
            const uint32_t tile_bytes = (uint32_t)n * TC_BLOCK_K * 2;
            // this CTA's tiles of the layer, contiguous in consumption order (K chunk outer, tap inner)
            const __nv_bfloat16* wl = a.w_stream + (size_t)l * CL_W_LAYER_ELEMS + (size_t)rank * CL_W_RANK_ELEMS;
            // a stage = four consecutive tiles of the layer's (K chunk, tap) sequence (stages straddle K chunks: a 3x3 layer is nine
            // full stages, a 1x1 layer one), one contiguous bulk copy
            const int T = L.taps * L.kchunks;
            for (int s0 = 0; s0 < T && ok; s0 += 4) {
                const int cnt = min(4, T - s0);
                if (issued++ == CL_B_STAGES) send_input();
                if (!(ok = warp_mbar_wait(bar_be0 + bs * 8, b_phase ^ 1, abort_flag))) break;
                if (elect_one()) {
                    const uint32_t full = bar_bf0 + bs * 8;
                    mbar_expect_tx(full, tile_bytes * (uint32_t)cnt);
                    bulk_load(smem_b + bs * CL_STAGE_BYTES, wl + (size_t)s0 * n * TC_BLOCK_K, tile_bytes * (uint32_t)cnt, full);
                }
                __syncwarp();
                if (++bs == CL_B_STAGES) { bs = 0; b_phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: warp-convergent loop, one elected lane issues (straight-line taps, see k_tower_tc2) =====
        const uint32_t a_lo0 = ((smem_act >> 4) & 0x3FFFu) | DESC_LO_FLAGS, b_lo0 = ((smem_b >> 4) & 0x3FFFu) | DESC_LO_FLAGS;
        const uint32_t bar_bf0 = smem_u32(&bar_b_full[0]), bar_be0 = smem_u32(&bar_b_empty[0]);
        uint32_t bs = 0, b_phase = 0;
        bool ok = true;
        for (int l = 0; l < MAX_TOWER_LAYERS && ok; l++) {
            const TowerLayer L = a.L[l];
            const int n = L.mode == 1 ? CL_NP : CL_N;
            const uint32_t idesc = IDESC_M64 | ((uint32_t)(n >> 3) << 17);
            // this layer's input: the TMA-loaded planes, or the 32 arrivals of the previous layer's epilogues
            if (l == 0) ok = warp_mbar_wait(smem_u32(&bar_in), 0, abort_flag);
            else ok = __all_sync(0xFFFFFFFFu, mbar_wait_cluster(smem_u32(&bar_act[(l - 1) & 1]), (uint32_t)(((l - 1) >> 1) & 1), abort_flag));
            if (!ok) break;
            // re-arm that barrier for the output of layer l + 1 (bytes of it cannot be sent before this CTA has finished layer l)
            if (l >= 1 && l + 1 <= POLICY_LAYER - 1 && elect_one()) mbar_expect_tx(smem_u32(&bar_act[(l - 1) & 1]), CL_LAYER_BYTES);
            __syncwarp();
            fence_proxy_async();                  // peers' generic-proxy stores -> tensor-core reads
            tc_fence_after();
            if (a.trace && blockIdx.x == 0 && lane == 0) a.trace[l * 8 + 0] = global_ns();
            const uint32_t buf_lo = a_lo0 + (uint32_t)(l & 1) * (CL_BUF_BYTES >> 4);
            if (L.taps == 9) {
                // straight-line issue: stage s holds tiles 4 s .. 4 s + 3 of the layer's (K chunk outer, tap inner) sequence; every
                // descriptor offset below is an immediate
                const int T = 9 * L.kchunks;                               // 36, or 18 for the stem
#pragma unroll
                for (int s = 0; s < 9; s++) {
                    if (4 * s >= T) break;
                    if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                    tc_fence_after();
                    const uint32_t b_base = b_lo0 + bs * (CL_STAGE_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            const int t = 4 * s + u, kc = t / 9, tap = t % 9;
                            if (t < T) {
                                const uint32_t a_lo = buf_lo + (uint32_t)kc * (CL_CHUNK_BYTES >> 4) + (uint32_t)((tap / 3) * HALO + tap % 3) * (128 >> 4);   // halo pixel (ky, kx)
                                const uint32_t b_lo = b_base + u * (CL_TILE_BYTES >> 4);
                                tc1_mma_bf16_split(tmem_base, a_lo, desc_hi(T2_A_SBO), b_lo, desc_hi(1024), idesc, t == 0 ? 0u : 1u);
                                tc1_mma_bf16_split(tmem_base, a_lo + 2, desc_hi(T2_A_SBO), b_lo + 2, desc_hi(1024), idesc, 1u);
                                tc1_mma_bf16_split(tmem_base, a_lo + 4, desc_hi(T2_A_SBO), b_lo + 4, desc_hi(1024), idesc, 1u);
                                tc1_mma_bf16_split(tmem_base, a_lo + 6, desc_hi(T2_A_SBO), b_lo + 6, desc_hi(1024), idesc, 1u);
                            }
                        }
                        tc_commit(bar_be0 + bs * 8);
                    }
                    __syncwarp();
                    if (++bs == CL_B_STAGES) { bs = 0; b_phase ^= 1; }
                }
            } else {
                // 1x1 convolution = centre tap of the four K chunks: one stage of four tiles
                if (!(ok = warp_mbar_wait(bar_bf0 + bs * 8, b_phase, abort_flag))) break;
                tc_fence_after();
                const uint32_t b_base = b_lo0 + bs * (CL_STAGE_BYTES >> 4);
                const uint32_t tile_lo = (uint32_t)(n * TC_BLOCK_K * 2) >> 4;
                if (elect_one()) {
#pragma unroll
                    for (int kc = 0; kc < C_TOWER / TC_BLOCK_K; kc++) {
                        const uint32_t a_lo = buf_lo + (uint32_t)kc * (CL_CHUNK_BYTES >> 4) + (uint32_t)(HALO + 1) * (128 >> 4);
                        const uint32_t b_lo = b_base + kc * tile_lo;
                        tc1_mma_bf16_split(tmem_base, a_lo, desc_hi(T2_A_SBO), b_lo, desc_hi(1024), idesc, kc == 0 ? 0u : 1u);
                        tc1_mma_bf16_split(tmem_base, a_lo + 2, desc_hi(T2_A_SBO), b_lo + 2, desc_hi(1024), idesc, 1u);
                        tc1_mma_bf16_split(tmem_base, a_lo + 4, desc_hi(T2_A_SBO), b_lo + 4, desc_hi(1024), idesc, 1u);
                        tc1_mma_bf16_split(tmem_base, a_lo + 6, desc_hi(T2_A_SBO), b_lo + 6, desc_hi(1024), idesc, 1u);
                    }
                    tc_commit(bar_be0 + bs * 8);
                }
                __syncwarp();
                if (++bs == CL_B_STAGES) { bs = 0; b_phase ^= 1; }
            }
            if (ok && elect_one()) tc_commit(smem_u32(&bar_acc_full));
            __syncwarp();
            if (a.trace && blockIdx.x == 0 && lane == 0) a.trace[l * 8 + 1] = global_ns();
        }
    } else {
        // ===== epilogue warps: accumulator rows 16 w .. 16 w + 15 sit in lanes 0..15 of TMEM quarter w (M = 64 layout) =====
        pdl_wait();
        const int lane_group = warp & 3;
        const int etid = threadIdx.x - 64;
        const bool has_row = lane < 16;
        const int m = lane_group * 16 + (lane & 15);                       // board square: oy = m >> 3, ox = m & 7
        const int prow = ((m >> 3) + 1) * HALO + (m & 7) + 1;              // its pixel row in the halo tile
        const uint32_t taddr = tmem_base + ((uint32_t)(lane_group * 32) << 16);
        uint32_t xin[CL_N / 2];                                            // this CTA's channels of the current residual block's input
#pragma unroll
        for (int j = 0; j < CL_N / 2; j++) xin[j] = 0;
        bool ok = true;
        const uint32_t lg_base = smem_act + CL_BUF_BYTES;                  // CTA 0's buffer 1: fp32 logits [plane][64], see the head section
        for (int l = 0; l < MAX_TOWER_LAYERS && ok; l++) {
            const TowerLayer L = a.L[l];
            const int n = L.mode == 1 ? CL_NP : CL_N;
            if (etid < n) bias_sh[l & 1][etid] = a.bias[l * C_TOWER + (int)rank * n + etid];
            named_bar_sync<1, 128>();
            ok = __all_sync(0xFFFFFFFFu, mbar_wait(smem_u32(&bar_acc_full), (uint32_t)(l & 1), abort_flag));
            if (!ok) break;
            tc_fence_after();
            const bool tracer = a.trace && blockIdx.x == 0 && warp == 2 && lane == 0;
            if (tracer) a.trace[l * 8 + 2] = global_ns();
            uint32_t v[CL_N];
            if constexpr (CL_N == 32) tmem_ld_32x32b_x32(taddr, v); else tmem_ld_32x32b_x16(taddr, v);      // (the last layer fills fewer columns)
            tmem_ld_wait();
            tc_fence_before();
            if (tracer) a.trace[l * 8 + 3] = global_ns();
            const float* bias = bias_sh[l & 1];
            if (L.mode == 1) {
                // policy logits of this CTA's 16 planes -> CTA 0 (fp32, plane-major like torch.flatten(conv_p2(x)))
                if (has_row) {
#pragma unroll
                    for (int j = 0; j < CL_NP; j++) {
                        const int plane = (int)rank * CL_NP + j;
                        if (plane < POLICY_PLANES) st_cluster_f32(mapa_u32(lg_base + (uint32_t)(plane * 64 + m) * 4, 0), __fadd_rn(__uint_as_float(v[j]), bias[j]));
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&bar_lg), 0));
                break;
            }
            constexpr int PIECES = CL_N / 8;                                // 16-byte pieces of this CTA's slice of a pixel row
            uint4 o[PIECES];
            {
                __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(o);
                const __nv_bfloat162* rb = reinterpret_cast<const __nv_bfloat162*>(xin);
#pragma unroll
                for (int j = 0; j < CL_N / 2; j++) {
                    float x0 = __uint_as_float(v[2 * j]) + bias[2 * j];
                    float x1 = __uint_as_float(v[2 * j + 1]) + bias[2 * j + 1];
                    if (L.res != 255) {
                        const float2 r2 = __bfloat1622float2(rb[j]);
                        x0 += r2.x;
                        x1 += r2.y;
                    }
                    if (L.relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
                    ob[j] = __floats2bfloat162_rn(x0, x1);
                }
            }
            if (l == 0 || L.res != 255) {                                   // the stem's and every block's output is the next block's input
                const uint32_t* ow = reinterpret_cast<const uint32_t*>(o);
#pragma unroll
                for (int j = 0; j < CL_N / 2; j++) xin[j] = ow[j];
            }
            {
                // this CTA's channels of pixel prow.  Lanes 0..15 hold the rows; lanes 16..31 take a copy and serve the upper half of the
                // peers, so every lane issues 16 asynchronous 16-byte stores.
#pragma unroll
                for (int u = 0; u < PIECES; u++) {
                    o[u].x = __shfl_sync(0xFFFFFFFFu, o[u].x, lane & 15);
                    o[u].y = __shfl_sync(0xFFFFFFFFu, o[u].y, lane & 15);
                    o[u].z = __shfl_sync(0xFFFFFFFFu, o[u].z, lane & 15);
                    o[u].w = __shfl_sync(0xFFFFFFFFu, o[u].w, lane & 15);
                }
                const uint32_t ch0 = rank * CL_N;                            // first channel of the slice: K chunk ch0 / 64, byte (ch0 % 64) * 2 of the row
                const uint32_t row_addr = smem_act + (uint32_t)((l + 1) & 1) * CL_BUF_BYTES + (ch0 >> 6) * CL_CHUNK_BYTES + (uint32_t)prow * 128 + (ch0 & 63) * 2;
                const uint32_t bar_local = smem_u32(&bar_act[l & 1]);
#pragma unroll
                for (int k = 0; k < CL_SIZE / 2; k++) {
                    const uint32_t dst = (uint32_t)(lane >> 4) * (CL_SIZE / 2) + k;
                    const uint32_t rbar = mapa_u32(bar_local, dst);
#pragma unroll
                    for (int u = 0; u < PIECES; u++) st_async_v4(mapa_u32(swz128(row_addr + u * 16), dst), o[u], rbar);
                }
            }
            if (tracer) a.trace[l * 8 + 4] = global_ns();
            if (tracer) a.trace[l * 8 + 5] = global_ns();
        }
        // ===== heads =====
        if (ok && rank == 0) {
            // softmax over the board's 73 x 64 logits gathered in this CTA's buffer 1, in k_softmax's order; thread = square (64 threads)
            ok = __all_sync(0xFFFFFFFFu, mbar_wait_cluster(smem_u32(&bar_lg), 0, abort_flag));
            const float* lg = reinterpret_cast<const float*>(smem_raw + (lg_base - smem_u32(smem_raw)));
            const long row_slot = heads_slot(a.heads, (long)board + a.heads.row_delta);
            const bool search = a.heads.mask != nullptr;
            const bool want = ok && (!search || a.heads.need_eval[row_slot] != 0);
            if (search)
                for (int i = etid; i < MASK_WORDS; i += 128) hd_mask[i] = a.heads.mask[(size_t)row_slot * MASK_STRIDE + i];
            const int sq = etid & 63;
            float mx = -INFINITY, ssum = 0.f;
            if (etid < 64) {
                for (int c = 0; c < POLICY_PLANES; c++) mx = fmaxf(mx, lg[c * 64 + sq]);
#pragma unroll
                for (int off = 1; off < 16; off <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, off));
                if ((lane & 15) == 0) hd_red[0][sq >> 4] = mx;
            }
            named_bar_sync<1, 128>();
            mx = fmaxf(fmaxf(hd_red[0][0], hd_red[0][1]), fmaxf(hd_red[0][2], hd_red[0][3]));
            if (etid < 64) {
#pragma unroll 1
                for (int c = 0; c < POLICY_PLANES; c++) ssum = __fadd_rn(ssum, sm_exp(lg[c * 64 + sq], mx));
#pragma unroll
                for (int off = 1; off < 16; off <<= 1) ssum = __fadd_rn(ssum, __shfl_xor_sync(0xFFFFFFFFu, ssum, off));
                if ((lane & 15) == 0) hd_red[1][sq >> 4] = ssum;
            }
            named_bar_sync<1, 128>();
            const float tot = __fadd_rn(__fadd_rn(__fadd_rn(hd_red[1][0], hd_red[1][1]), hd_red[1][2]), hd_red[1][3]);
            if (want) {
                // two threads per square: planes of equal parity
                if (search) {
                    float* prw = a.heads.policy + (size_t)row_slot * N_ACTIONS + sq;
#pragma unroll 1
                    for (int c = etid >> 6; c < POLICY_PLANES; c += 2)
                        if ((hd_mask[c] >> sq) & 1ull) prw[c * 64] = __fdiv_rn(sm_exp(lg[c * 64 + sq], mx), tot);
                } else {
                    float* out = a.logits + (size_t)row_slot * N_ACTIONS + sq;
#pragma unroll 1
                    for (int c = etid >> 6; c < POLICY_PLANES; c += 2) out[c * 64] = lg[c * 64 + sq];
                }
            }
        } else if (ok && rank == 1) {
            // value head (network.py:156-174) on the tower output = the input of layer 39, still in this CTA's buffer 1; same arithmetic
            // as k_value_head.  Two threads per square: channel quarters {0, 1} and {2, 3}.
            // (complete and visible: this warp's accumulator waits of layers 39 / 40 are ordered after the MMA warp's acquire of it)
            hd_vw[etid] = a.heads.v_w[etid];
            hd_vw[etid + 128] = a.heads.v_w[etid + 128];
            named_bar_sync<1, 128>();
            const int sq = etid >> 1, half = etid & 1;
            const uint32_t px = smem_act + CL_BUF_BYTES + (uint32_t)(((sq >> 3) + 1) * HALO + (sq & 7) + 1) * 128;
            float p2[2] = {0.f, 0.f};
#pragma unroll
            for (int pp = 0; pp < 2; pp++) {
                const int part = half * 2 + pp;                             // channels [64 part, 64 part + 64) = K chunk `part`
#pragma unroll
                for (int qq = 0; qq < 8; qq++) {
                    const uint32_t ad = swz128(px + (uint32_t)part * CL_CHUNK_BYTES + qq * 16);
                    const uint4 u = *reinterpret_cast<const uint4*>(smem_raw + (ad - smem_u32(smem_raw)));
                    const __nv_bfloat16* h8 = reinterpret_cast<const __nv_bfloat16*>(&u);
#pragma unroll
                    for (int j = 0; j < 8; j++) p2[pp] = fmaf(__bfloat162float(h8[j]), hd_vw[part * 64 + qq * 8 + j], p2[pp]);
                }
            }
            float s = __fadd_rn(p2[0], p2[1]);                               // (p0 + p1) | (p2 + p3)
            s = __fadd_rn(s, __shfl_xor_sync(0xFFFFFFFFu, s, 1));
            if (half == 0) hd_plane[sq] = fmaxf(__fadd_rn(s, a.heads.scalars[0]), 0.f);
            named_bar_sync<1, 128>();
#pragma unroll 1
            for (int k2 = 0; k2 < 2; k2++) {
                const int o = etid + 128 * k2;
                float h = a.heads.fc1_b[o];
#pragma unroll 8
                for (int k = 0; k < 64; k++) h = fmaf(hd_plane[k], a.heads.fc1_wT[k * 256 + o], h);
                h = __fmul_rn(fmaxf(h, 0.f), a.heads.fc2_w[o]);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) h = __fadd_rn(h, __shfl_xor_sync(0xFFFFFFFFu, h, off));
                if (lane == 0) hd_fc[k2 * 4 + (etid >> 5)] = h;
            }
            named_bar_sync<1, 128>();
            if (etid == 0 && ok) {
                const long row_slot = heads_slot(a.heads, (long)board + a.heads.row_delta);
                if (a.heads.mask == nullptr || a.heads.need_eval[row_slot]) {
                    float tt = a.heads.scalars[1];
#pragma unroll
                    for (int w = 0; w < 8; w++) tt = __fadd_rn(tt, hd_fc[w]);
                    a.heads.value[row_slot] = vh_tanh(tt);
                }
            }
        }
    }
    // ===== teardown: nobody leaves while a peer may still store into this CTA's shared memory or arrive on its barriers =====
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    if (warp == 1) tc_tmem_dealloc(tmem_base, 32);
    if (threadIdx.x == 0 && abort_sh) atomicExch(a.error, 1);
}

// =================================================================================================
// fp32 SIMT convolution (parity path)
// =================================================================================================
struct F32Args {
    const float* in;             // halo NHWC [B][10][10][cin]
    const float* w;              // [taps][cin][cout_pad]
    const float* bias;
    const float* residual;       // halo NHWC [.][256] or null
    float* out;                  // halo NHWC [.][256] (mode 0) / logits [B][4672] (mode 1)
    int cin, cout_pad, taps, relu, mode;
};

// grid (B, cout_pad/64), 256 threads: thread = 4 squares x 4 output channels
__global__ void __launch_bounds__(256) k_conv_f32(const F32Args a) {
    __shared__ float in_s[HALO * HALO][33];
    __shared__ __align__(16) float w_s[32][64];
    const int b = blockIdx.x, co0 = blockIdx.y * 64;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int y = ty >> 1, x0 = (ty & 1) * 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
    const float* inb = a.in + (size_t)b * HALO * HALO * a.cin;
    for (int c0 = 0; c0 < a.cin; c0 += 32) {
        __syncthreads();
        for (int i = tid; i < HALO * HALO * 32; i += 256) {
            const int pos = i >> 5, c = i & 31;
            in_s[pos][c] = inb[(size_t)pos * a.cin + c0 + c];
        }
        for (int tap = 0; tap < a.taps; tap++) {
            const int ky = a.taps == 9 ? tap / 3 : 1, kx = a.taps == 9 ? tap % 3 : 1;
            __syncthreads();
            for (int i = tid; i < 32 * 64; i += 256) {
                const int c = i >> 6, co = i & 63;
                w_s[c][co] = a.w[((size_t)tap * a.cin + c0 + c) * a.cout_pad + co0 + co];
            }
            __syncthreads();
            const int p0 = (y + ky) * HALO + x0 + kx;
#pragma unroll 8
            for (int c = 0; c < 32; c++) {
                const float4 w = *reinterpret_cast<const float4*>(&w_s[c][tx * 4]);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const float v = in_s[p0 + i][c];
                    acc[i][0] = fmaf(v, w.x, acc[i][0]);
                    acc[i][1] = fmaf(v, w.y, acc[i][1]);
                    acc[i][2] = fmaf(v, w.z, acc[i][2]);
                    acc[i][3] = fmaf(v, w.w, acc[i][3]);
                }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = x0 + i;
        const size_t pix = ((size_t)b * HALO + y + 1) * HALO + x + 1;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int co = co0 + tx * 4 + j;
            float v = acc[i][j] + a.bias[co];
            if (a.mode == 0) {
                if (a.residual) v += a.residual[pix * C_TOWER + co];
                if (a.relu) v = fmaxf(v, 0.f);
                a.out[pix * C_TOWER + co] = v;
            } else if (co < POLICY_PLANES) {
                a.out[(size_t)b * N_ACTIONS + co * 64 + y * 8 + x] = v;
            }
        }
    }
}

// =================================================================================================
// small fused kernels
// =================================================================================================
// bit-packed planes [B][stride] -> halo NHWC [B][10][10][128] (interior only; the halo stays zero)
template <class T>
__global__ void k_planes_to_nhwc(const uint64_t* planes, int stride, int n, T* out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;        // (board, square, 8-channel group)
    if (i >= (size_t)n * 64 * 16) return;
    const int cg = (int)(i & 15), sq = (int)((i >> 4) & 63);
    const size_t b = i >> 10;
    const uint64_t* p = planes + b * stride;
    T v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int c = cg * 8 + j;
        const float f = c < N_PLANES ? (float)((p[c] >> sq) & 1ull) : 0.f;
        if constexpr (sizeof(T) == 2) v[j] = __float2bfloat16(f); else v[j] = f;
    }
    T* o = out + (((size_t)b * HALO + (sq >> 3) + 1) * HALO + (sq & 7) + 1) * C_IN_PAD + cg * 8;
#pragma unroll
    for (int j = 0; j < 8; j++) o[j] = v[j];
}

// value head (network.py:156-174): conv1x1 256->1 (+BN, ReLU) -> fc 64->256 (ReLU) -> fc 256->1 -> tanh.  Block per board.
// fc1_wT is fc_v1.weight transposed to [64][256] so that the 256 threads read consecutive floats.  Every rounding is explicit and in
// the order the fused heads of k_tower_tc2 use, so the two agree bit for bit (test_tower_kernel_variants_bit_identical).
template <class T>
__global__ void __launch_bounds__(256) k_value_head(const T* act, const float* v_w, const float* scalars, const float* fc1_wT, const float* fc1_b,
                                                    const float* fc2_w, float* value, int n) {
    const float v_b = scalars[0], fc2_b = scalars[1];
    __shared__ float plane[64];
    __shared__ float red[8];
    __shared__ float vw_sh[C_TOWER];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int sq = tid >> 2, part = tid & 3;
    vw_sh[tid] = v_w[tid];
    __syncthreads();
    const T* row = act + (((size_t)b * HALO + (sq >> 3) + 1) * HALO + (sq & 7) + 1) * C_TOWER + part * 64;
    const float* vw = vw_sh + part * 64;
    float s = 0.f;
    if constexpr (sizeof(T) == 2) {
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const uint4 u = reinterpret_cast<const uint4*>(row)[q];
            const __nv_bfloat16* h8 = reinterpret_cast<const __nv_bfloat16*>(&u);
#pragma unroll
            for (int j = 0; j < 8; j++) s = fmaf(__bfloat162float(h8[j]), vw[q * 8 + j], s);
        }
    } else {
#pragma unroll
        for (int q = 0; q < 16; q++) {
            const float4 u = reinterpret_cast<const float4*>(row)[q];
            s = fmaf(u.x, vw[q * 4], s);
            s = fmaf(u.y, vw[q * 4 + 1], s);
            s = fmaf(u.z, vw[q * 4 + 2], s);
            s = fmaf(u.w, vw[q * 4 + 3], s);
        }
    }
    s = __fadd_rn(s, __shfl_xor_sync(0xFFFFFFFFu, s, 1));              // (p0 + p1), (p2 + p3)
    s = __fadd_rn(s, __shfl_xor_sync(0xFFFFFFFFu, s, 2));              // (p0 + p1) + (p2 + p3)
    if (part == 0) plane[sq] = fmaxf(__fadd_rn(s, v_b), 0.f);
    __syncthreads();
    float h = fc1_b[tid];
#pragma unroll 8
    for (int k = 0; k < 64; k++) h = fmaf(plane[k], fc1_wT[k * 256 + tid], h);
    h = __fmul_rn(fmaxf(h, 0.f), fc2_w[tid]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) h = __fadd_rn(h, __shfl_xor_sync(0xFFFFFFFFu, h, off));
    if ((tid & 31) == 0) red[tid >> 5] = h;
    __syncthreads();
    if (tid == 0) {
        float t = fc2_b;
#pragma unroll
        for (int w = 0; w < 8; w++) t = __fadd_rn(t, red[w]);
        value[b] = vh_tanh(t);
    }
}

// nn.Softmax(dim=1) over the 4672 logits of every board (network.py:190).  Four boards per block, thread = (board, square).
// Fixed order, shared with the fused heads of k_tower_tc2 (whose epilogue threads own one square's 73 logits each): maximum (order-free);
// per square the sum of exp(l - max) over the planes 0..72 in turn; a balanced tree over each group of 16 squares (bits 0..3 of the
// square index); the four groups in turn.  Batch invariant by construction.
__global__ void __launch_bounds__(256) k_softmax(const float* logits, float* policy, int n) {
    __shared__ float red[2][4][4];
    const int tid = threadIdx.x, bl = tid >> 6, sq = tid & 63, lane = tid & 31;
    const int b = blockIdx.x * 4 + bl;
    const bool live = b < n;
    const float* l = logits + (size_t)(live ? b : 0) * N_ACTIONS + sq;
    float* p = policy + (size_t)(live ? b : 0) * N_ACTIONS + sq;
    float mx = -INFINITY;
    if (live)
        for (int c = 0; c < POLICY_PLANES; c++) mx = fmaxf(mx, l[c * 64]);
#pragma unroll
    for (int off = 1; off < 16; off <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, off));
    if ((lane & 15) == 0) red[0][bl][sq >> 4] = mx;
    __syncthreads();
    mx = fmaxf(fmaxf(red[0][bl][0], red[0][bl][1]), fmaxf(red[0][bl][2], red[0][bl][3]));
    float s = 0.f;
    if (live) {
#pragma unroll 1
        for (int c = 0; c < POLICY_PLANES; c++) s = __fadd_rn(s, sm_exp(l[c * 64], mx));
    }
#pragma unroll
    for (int off = 1; off < 16; off <<= 1) s = __fadd_rn(s, __shfl_xor_sync(0xFFFFFFFFu, s, off));
    if ((lane & 15) == 0) red[1][bl][sq >> 4] = s;
    __syncthreads();
    const float tot = __fadd_rn(__fadd_rn(__fadd_rn(red[1][bl][0], red[1][bl][1]), red[1][bl][2]), red[1][bl][3]);
    if (live) {
#pragma unroll 1
        for (int c = 0; c < POLICY_PLANES; c++) p[c * 64] = __fdiv_rn(sm_exp(l[c * 64], mx), tot);
    }
}

// =================================================================================================
// host: weights
// =================================================================================================
template <class T>
static int net_alloc(szb_ctx* ctx, Net* net, T** out, size_t count, bool zero = true) {
    void* p = nullptr;
    SZB_CUDA(ctx, cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
    if (zero) SZB_CUDA(ctx, cudaMemsetAsync(p, 0, std::max<size_t>(count, 1) * sizeof(T), ctx->stream));
    net->allocs.push_back(p);
    *out = (T*)p;
    return 0;
}

struct BN { const float *g, *b, *m, *v; };          // DEVICE pointers

// BatchNorm folding and packing ON THE GPU (eval mode, eps 1e-5; the arithmetic of the former host loop: double precision, one
// rounding to fp32): conv weight [cout][cin_src][taps] (+ BN | + conv bias) -> fp32 [tap][cin][cout_pad] (SIMT path), bf16 K-major
// [cout_pad][taps * cin] (tensor-core paths), bias [cout_pad].  One thread per (co, ci, tap) of the padded pack.
__global__ void k_fold_conv(const float* w, BN bn, int has_bn, const float* conv_bias, int cout, int cin_src, int cin, int taps, int cout_pad,
                            float* w32, float* bias, __nv_bfloat16* w16) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)cout_pad * cin * taps;
    if (i >= total) return;
    const int t = (int)(i % taps), ci = (int)((i / taps) % cin), co = (int)(i / ((size_t)taps * cin));
    double scale = 1.0;
    if (co < cout && has_bn) scale = (double)bn.g[co] / sqrt((double)bn.v[co] + 1e-5);
    float f = 0.f;
    if (co < cout && ci < cin_src) f = (float)((double)w[((size_t)co * cin_src + ci) * taps + t] * scale);
    w32[((size_t)t * cin + ci) * cout_pad + co] = f;
    w16[(size_t)co * taps * cin + (size_t)t * cin + ci] = __float2bfloat16_rn(f);
    if (ci == 0 && t == 0) {
        double shift = 0.0;
        if (co < cout) shift = has_bn ? (double)bn.b[co] - (double)bn.m[co] * scale : (conv_bias ? (double)conv_bias[co] : 0.0);
        bias[co] = (float)shift;
    }
}
// value head packs: conv_v1 x BN scale, {BN shift, fc_v2.bias}, fc_v1.weight transposed to [64][256]
__global__ void k_fold_value_head(const float* vw, BN bn, const float* f1w, const float* f1b, const float* f2w, const float* f2b,
                                  float* v_w, float* scalars, float* fc1_wT, float* fc1_b, float* fc2_w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;                  // 0 .. 256 * 64
    const double scale = (double)bn.g[0] / sqrt((double)bn.v[0] + 1e-5);
    if (i < 256) {
        v_w[i] = (float)((double)vw[i] * scale);
        fc1_b[i] = f1b[i];
        fc2_w[i] = f2w[i];
    }
    if (i == 0) {
        scalars[0] = (float)((double)bn.b[0] - (double)bn.m[0] * scale);
        scalars[1] = f2b[0];
    }
    if (i < 256 * 64) {
        const int o = i / 64, k = i % 64;
        fc1_wT[k * 256 + o] = f1w[o * 64 + k];
    }
}
// 64-bit digest of a device buffer (order-independent sum of mixed words): szb_net_checksum
__global__ void k_digest(const uint32_t* p, size_t n_words, uint64_t salt, unsigned long long* out) {
    unsigned long long acc = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (size_t)gridDim.x * blockDim.x)
        acc += mix64(((uint64_t)p[i] << 20) ^ (uint64_t)i ^ salt);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, off);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

static int alloc_conv(szb_ctx* ctx, Net* net, ConvLayer& L, int cin, int taps, int cout, int cout_pad) {
    L.taps = taps; L.cin = cin; L.cout = cout; L.cout_pad = cout_pad;
    const size_t K = (size_t)taps * cin;
    int rc;
    if ((rc = net_alloc(ctx, net, &L.w32, K * cout_pad, false))) return rc;
    if ((rc = net_alloc(ctx, net, &L.bias, (size_t)cout_pad, false))) return rc;
    if ((rc = net_alloc(ctx, net, &L.w16, K * cout_pad, false))) return rc;
    return net_tmap_rows(ctx, &L.tm_w, L.w16, (int)K, cout_pad, cout_pad, "weights");
}
static int fold_conv(szb_ctx* ctx, ConvLayer& L, const float* w, int cin_src, const BN* bn, const float* conv_bias) {
    const size_t total = (size_t)L.cout_pad * L.cin * L.taps;
    BN z = {nullptr, nullptr, nullptr, nullptr};
    k_fold_conv<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(w, bn ? *bn : z, bn != nullptr, conv_bias, L.cout, cin_src, L.cin, L.taps,
                                                                         L.cout_pad, L.w32, L.bias, L.w16);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

void net_destroy(szb_ctx* ctx) {
    if (!ctx->net) return;
    if (ctx->net->span && !ctx->net->span_path.empty() && !ctx->net->span_boards.empty()) {
        Net* net = ctx->net;
        std::vector<unsigned long long> h(4 * net->span_boards.size());
        cudaDeviceSynchronize();
        if (cudaMemcpy(h.data(), net->span, h.size() * 8, cudaMemcpyDeviceToHost) == cudaSuccess) {
            if (FILE* f = fopen(net->span_path.c_str(), "w")) {
                fprintf(f, "launch,board0,boards,start_ns,end_ns\n");
                const unsigned long long t0 = h[0];
                for (size_t i = 0; i < net->span_boards.size(); i++)
                    fprintf(f, "%zu,%d,%d,%lld,%lld\n", i, net->span_b0[i], net->span_boards[i], (long long)(h[4 * i] - t0), (long long)(h[4 * i + 1] - t0));
                fclose(f);
            }
        }
    }
    if (ctx->net->trace_ring && ctx->net->trace_launches > 0) {
        // the last TRACE_RING large-batch launches of the searches, oldest first; times relative to each launch's first stamp (or its
        // first CTA's start when SZB_TOWER_SPAN records it too)
        Net* net = ctx->net;
        const size_t per = (size_t)MAX_TOWER_LAYERS * TRACE_MAX_TILES * TRACE_STAMPS;
        std::vector<unsigned long long> h(per * TRACE_RING), sp(4 * net->span_boards.size());
        cudaDeviceSynchronize();
        if (cudaMemcpy(h.data(), net->trace_ring, h.size() * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
            (sp.empty() || cudaMemcpy(sp.data(), net->span, sp.size() * 8, cudaMemcpyDeviceToHost) == cudaSuccess)) {
            if (FILE* f = fopen(net->trace_path.c_str(), "a")) {
                fprintf(f, "launch,boards,pairs,start_ns,end_ns,item,layer,tile,dep_ns,operands_ns,acc_ns,released_ns,last_mma_ns\n");
                for (long long k = std::max(0ll, net->trace_launches - TRACE_RING); k < net->trace_launches; k++) {
                    const std::array<long long, 5>& m = net->trace_meta[k % TRACE_RING];
                    const unsigned long long* tr = h.data() + (size_t)(k % TRACE_RING) * per;
                    const int tiles = (int)m[2];
                    const size_t n_st = (size_t)MAX_TOWER_LAYERS * tiles * TRACE_STAMPS;
                    unsigned long long t0 = ~0ull, s0 = 0, s1 = 0;
                    if (m[4] >= 0) { s0 = sp[4 * m[4]]; s1 = sp[4 * m[4] + 1]; t0 = s0; }
                    else for (size_t i = 0; i < n_st; i++) if (tr[i] && tr[i] < t0) t0 = tr[i];
                    for (int item = 0; item < MAX_TOWER_LAYERS * tiles; item++) {
                        fprintf(f, "%lld,%lld,%lld,%lld,%lld,%d,%d,%d", m[0], m[1], m[3], s0 ? 0ll : -1ll, s1 ? (long long)(s1 - t0) : -1ll,
                                item, item / tiles, item % tiles);
                        for (int j = 0; j < TRACE_STAMPS; j++) {
                            const unsigned long long v = tr[(size_t)item * TRACE_STAMPS + j];
                            fprintf(f, ",%lld", v ? (long long)(v - t0) : -1ll);
                        }
                        fprintf(f, "\n");
                    }
                }
                fclose(f);
            }
        }
    }
    for (void* p : ctx->net->allocs) cudaFree(p);
    delete ctx->net->tower_maps;
    delete ctx->net->tower_args;
    delete ctx->net;
    ctx->net = nullptr;
}

static int net_alloc_activations(szb_ctx* ctx, Net* net) {
    int rc;
    const size_t cap = (size_t)net->cap;
    if ((rc = net_alloc(ctx, net, &net->in16, cap * HALO * HALO * C_IN_PAD))) return rc;
    if ((rc = net_alloc(ctx, net, &net->in32, cap * HALO * HALO * C_IN_PAD))) return rc;
    for (int i = 0; i < 3; i++) {
        if ((rc = net_alloc(ctx, net, &net->act16[i], cap * HALO * HALO * C_TOWER))) return rc;
        if ((rc = net_alloc(ctx, net, &net->act32[i], cap * HALO * HALO * C_TOWER))) return rc;
        if ((rc = net_tmap_act(ctx, &net->tm_act16[i], net->act16[i], C_TOWER, net->cap, 2, "activations"))) return rc;
    }
    if ((rc = net_tmap_act(ctx, &net->tm_in16, net->in16, C_IN_PAD, net->cap, 2, "activations"))) return rc;
    if ((rc = net_alloc(ctx, net, &net->logits, cap * N_ACTIONS))) return rc;
    if ((rc = net_alloc(ctx, net, &net->tc_error, 1))) return rc;
    return 0;
}

static int net_span_reset(szb_ctx* ctx, Net* net) {
    std::vector<unsigned long long> init((size_t)SPAN_CAP * 4, 0ull);
    for (int i = 0; i < SPAN_CAP; i++) init[4 * (size_t)i] = ~0ull;
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SZB_CUDA(ctx, cudaMemcpy(net->span, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
    net->span_boards.clear();
    net->span_b0.clear();
    return 0;
}

// combined weight / bias buffers, layer table and tensor maps of the CTA-pair tower kernel
static int net_setup_tower(szb_ctx* ctx, Net* net) {
    int rc;
    constexpr int KMAX = 9 * C_TOWER;
    if ((rc = net_alloc(ctx, net, &net->w16_all, (size_t)MAX_TOWER_LAYERS * C_TOWER * KMAX))) return rc;
    if ((rc = net_alloc(ctx, net, &net->bias_all, (size_t)MAX_TOWER_LAYERS * C_TOWER))) return rc;
    for (int v = 0; v < 2; v++)
        if ((rc = net_alloc(ctx, net, &net->w16_cl[v], (size_t)MAX_TOWER_LAYERS * CL_W_LAYER_ELEMS))) return rc;
    if ((rc = net_alloc(ctx, net, &net->ready, (size_t)MAX_TOWER_LAYERS * ((net->cap + 3) / 4)))) return rc;
    delete net->tower_maps;
    delete net->tower_args;
    net->tower_maps = new TowerMaps();
    net->tower_args = new TowerArgs();
    TowerArgs& a = *net->tower_args;
    memset(&a, 0, sizeof a);
    auto layer = [&](int l, int a_map, int taps, int kchunks, int res, int out) {
        TowerLayer& T = a.L[l];
        T.a_map = (uint8_t)a_map; T.taps = (uint8_t)taps; T.kchunks = (uint8_t)kchunks;
        T.res = (uint8_t)res; T.out = (uint8_t)out; T.relu = 1; T.mode = 0; T.n_half = 128;
    };
    layer(0, 0, 9, C_IN_PAD / TC_BLOCK_K, 255, 0);
    int x = 0;
    for (int blk = 0; blk < N_BLOCKS; blk++) {
        const int y = (x + 1) % 3, o = (x + 2) % 3;
        layer(1 + 2 * blk, 1 + x, 9, C_TOWER / TC_BLOCK_K, 255, y);
        layer(2 + 2 * blk, 1 + y, 9, C_TOWER / TC_BLOCK_K, x, o);
        x = o;
    }
    const int y = (x + 1) % 3;
    layer(POLICY_LAYER - 1, 1 + x, 1, C_TOWER / TC_BLOCK_K, 255, y);
    // policy output 256 -> 73 (+ conv bias): N = 128 (two halves of 64 rows, the 73 planes zero-padded), fp32 logits epilogue
    layer(POLICY_LAYER, 1 + y, 1, C_TOWER / TC_BLOCK_K, 255, 0);
    a.L[POLICY_LAYER].relu = 0; a.L[POLICY_LAYER].mode = 1; a.L[POLICY_LAYER].n_half = 64;
    a.logits = net->logits;
    net->final_x = x;
    net->final_y = y;
    a.ready = net->ready;
    a.bias = net->bias_all;
    for (int i = 0; i < 3; i++) a.act[i] = net->act16[i];
    a.error = net->tc_error;
    if ((rc = net_tmap_halo(ctx, &net->tower_maps->a[0], net->in16, C_IN_PAD, net->cap, 2, "halo activations"))) return rc;
    for (int i = 0; i < 3; i++)
        if ((rc = net_tmap_halo(ctx, &net->tower_maps->a[1 + i], net->act16[i], C_TOWER, net->cap, 2, "halo activations"))) return rc;
    // one board's halo tile of the input planes (k_tower_cl): box 64 x 10 x 1 x 10
    if ((rc = net_tmap_halo(ctx, &net->tower_maps->in1, net->in16, C_IN_PAD, net->cap, 1, "single-board input"))) return rc;
    {
        TowerMaps& m = *net->tower_maps;
        const int rows = MAX_TOWER_LAYERS * C_TOWER;
        if ((rc = net_tmap_rows(ctx, &m.w, net->w16_all, KMAX, rows, 128, "tower weights")) ||
            (rc = net_tmap_rows(ctx, &m.w64, net->w16_all, KMAX, rows, 64, "policy weights")) ||
            (rc = net_tmap_rows(ctx, &m.w32, net->w16_all, KMAX, rows, 32, "N-split weights")) ||
            (rc = net_tmap_rows(ctx, &m.w16, net->w16_all, KMAX, rows, 16, "N-split weights")) ||
            (rc = net_tmap_rows(ctx, &m.w8, net->w16_all, KMAX, rows, 8, "N-split weights")))
            return rc;
    }
    const char* mode = getenv("SZB_TOWER_MODE");             // measurement aid: 0 single-CTA per layer, 1 pair per layer, 2 one launch
    if (mode && mode[0] >= '0' && mode[0] <= '2') net->tower_mode = mode[0] - '0';
    // start / end device time of whole-tower launches: szb_tower_spans_record, or SZB_TOWER_SPAN=<csv> (every launch, dumped at destroy)
    if ((rc = net_alloc(ctx, net, &net->span, (size_t)SPAN_CAP * 4, false))) return rc;
    if ((rc = net_span_reset(ctx, net))) return rc;
    if (const char* sp = getenv("SZB_TOWER_SPAN")) {
        if (sp[0]) { net->span_path = sp; net->span_on = true; }
    }
    if (const char* tp = getenv("SZB_TOWER_TRACE")) {
        if (tp[0]) {
            net->trace_path = tp;
            if ((rc = net_alloc(ctx, net, &net->trace_ring, (size_t)TRACE_RING * MAX_TOWER_LAYERS * TRACE_MAX_TILES * TRACE_STAMPS))) return rc;
            net->trace_meta.assign(TRACE_RING, std::array<long long, 5>{-1, 0, 0, 0, -1});
        }
    }
    net->tower_pairs = net->num_sms / 2;
    if (const char* e = getenv("SZB_TOWER_PAIRS")) { if (atoi(e) > 0) net->tower_pairs = std::min(atoi(e), net->num_sms / 2); }
    if (const char* e = getenv("SZB_TOWER_EXCLUSIVE")) net->tower_exclusive = e[0] == '1';
    if (const char* e = getenv("SZB_NO_FUSE")) net->no_fuse = e[0] == '1';
    if (const char* e = getenv("SZB_TOWER_CLUSTER")) net->cluster_max = std::max(0, std::min(atoi(e), CL_MAX_BOARDS));
    if (const char* e = getenv("SZB_TOWER_CLUSTER_SIZE")) net->cluster_force = atoi(e);
    const char* ck = getenv("SZB_TOWER_CHUNK");              // measurement aid: boards per tower launch (0 = whole batch)
    if (ck && ck[0]) net->chunk = std::max(0, atoi(ck)) & ~3;
    if (const char* e = getenv("SZB_TOWER_TPS")) net->tower_tps1 = atoi(e) == 2 ? 2 : 1;
    const char* ns = getenv("SZB_TOWER_NSPLIT");             // measurement aid: force the N split of small batches (1, 2, 4); default automatic
    if (ns && (ns[0] == '1' || ns[0] == '2' || ns[0] == '4' || ns[0] == '8')) net->tower_nsplit = ns[0] - '0';
    ctx->net_tower_mode = net->tower_mode;
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// the folded per-layer packs -> the one [41 * 256][2304] bf16 weight buffer and [41][256] bias table the tower kernels read
// (device-to-device, asynchronous on the context's stream: part of every weight load)
static int net_assemble_tower(szb_ctx* ctx, Net* net) {
    constexpr int KMAX = 9 * C_TOWER;
    auto put = [&](int l, const ConvLayer& L, int rows) -> int {
        const int K = L.taps * L.cin;
        SZB_CUDA(ctx, cudaMemcpy2DAsync(net->w16_all + (size_t)l * C_TOWER * KMAX, (size_t)KMAX * 2, L.w16, (size_t)K * 2, (size_t)K * 2,
                                        rows, cudaMemcpyDeviceToDevice, ctx->stream));
        SZB_CUDA(ctx, cudaMemcpyAsync(net->bias_all + (size_t)l * C_TOWER, L.bias, (size_t)rows * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        return 0;
    };
    int rc;
    if ((rc = put(0, net->stem, C_TOWER))) return rc;
    for (int i = 0; i < 2 * N_BLOCKS; i++)
        if ((rc = put(1 + i, net->tower[i], C_TOWER))) return rc;
    if ((rc = put(POLICY_LAYER - 1, net->p1, C_TOWER))) return rc;
    if ((rc = put(POLICY_LAYER, net->p2, 128))) return rc;
    // the same weights once more as k_tower_cl's per-CTA streams
    for (int v = 0; v < 2; v++) {
        const int cs = 8 << v;
        if (cs == 16 && net->cluster_force != 16) continue;      // the 16-CTA variant only runs when it is asked for (A/B aid)
        for (int l = 0; l < MAX_TOWER_LAYERS; l++) {
            const TowerLayer& T = net->tower_args->L[l];
            const int n = (T.mode == 1 ? 128 : C_TOWER) / cs;
            const size_t total = (size_t)cs * T.taps * T.kchunks * n * 8;
            k_pack_cluster_weights<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(net->w16_all, net->w16_cl[v], l, T.taps, T.kchunks, n, cs);
            ctx->launches++;
        }
    }
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// =================================================================================================
// host: forward
// =================================================================================================
// how a whole-tower launch is wired into a search step
struct TowerRun {
    bool heads = false;          // fused policy / value heads into d.mask / d.policy / d.value rows (else fp32 logits)
    bool in16_rows = false;      // the input planes of board b0 + i already sit in NHWC input row out_row + i (written by k_tree_step)
    bool ready_zeroed = false;   // the launch's completion counters were cleared by the kernel before it on the stream
    bool pdl = false;            // programmatic dependent launch behind the step's tree kernel
    const int32_t* n_live = nullptr;     // evaluation cache: device count of the rows the tree kernel filled (TowerHeads::n_live)
    const int32_t* row_slot = nullptr;
    int live_off = 0;
};

// layers [layer_begin, layer_end) of the tower for n boards in one persistent CTA-pair launch
static int launch_tower(szb_ctx* ctx, Net* net, int b0, int n, int layer_begin, int layer_end, int out_row = -1, TowerRun run = TowerRun()) {
    if (!net->attr_set) {
        // "exclusive" launches ask for all the shared memory a block can have, so that no other block fits on an SM next to a
        // tower CTA (every block also reserves 1 KiB of system shared memory): see Net::tower_pairs
        cudaFuncAttributes fa;
        SZB_CUDA(ctx, cudaFuncGetAttributes(&fa, k_tower_tc2<false>));
        net->smem_exclusive = std::max(T2_SMEM, 232448 - (int)fa.sharedSizeBytes);
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_tower_tc2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, net->smem_exclusive));
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_tower_tc2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, net->smem_exclusive));
        // The pairs of a launch wait on one another (per-item completion counters), so every pair must be able to become
        // resident while the others spin: never launch more pairs than this device can hold at once.
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(net->num_sms);
        cfg.blockDim = dim3(TC_THREADS);
        cfg.dynamicSmemBytes = T2_SMEM;
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, k_tower_tc2<false>, &cfg) == cudaSuccess && clusters > 0)
            net->pairs_resident = std::min(net->num_sms / 2, clusters);
        else
            cudaGetLastError();
        net->attr_set = true;
    }
    TowerArgs a = *net->tower_args;
    a.n_pair_tiles = (n + 3) / 4;
    a.n_boards = n;
    a.board0 = b0;
    a.in_delta = run.in16_rows && out_row >= 0 ? out_row - b0 : 0;
    a.layer_begin = layer_begin;
    a.layer_end = layer_end;
    if (out_row >= 0) a.logits = net->logits + (size_t)(out_row - b0) * N_ACTIONS;      // board b0 + i -> logits row out_row + i
    a.ready = net->ready + (size_t)MAX_TOWER_LAYERS * (b0 / 4);      // cohorts (disjoint board ranges) get disjoint counter regions
    if (layer_end - layer_begin > 1 && !run.ready_zeroed)
        SZB_CUDA(ctx, cudaMemsetAsync(a.ready, 0, sizeof(int32_t) * (size_t)MAX_TOWER_LAYERS * a.n_pair_tiles, ctx->work));
    const bool heads = run.heads && layer_end == MAX_TOWER_LAYERS;
    if (heads) {
        const Dev& d = ctx->d;
        TowerHeads& h = a.heads;
        h.mask = d.mask; h.need_eval = d.need_eval; h.policy = d.policy; h.value = d.value;
        h.tower_out = net->act16[net->final_x];
        h.v_w = net->v_w; h.fc1_wT = net->fc1_w; h.fc1_b = net->fc1_b; h.fc2_w = net->fc2_w; h.scalars = net->head_scalars;
        h.row_delta = (out_row >= 0 ? out_row : b0) - b0;
        h.row_slot = run.row_slot; h.n_live = run.n_live; h.live_off = run.live_off;
    } else {
        a.heads.mask = nullptr;
        a.heads.row_slot = nullptr; a.heads.n_live = nullptr;
    }
    // Small batches leave most CTA pairs idle and the launch becomes a chain of 41 dependent layers: cut every (layer, tile)
    // into 2 or 4 items of N / nsplit output channels so that up to all pairs work on one layer.  Same MMAs per output, same K
    // order: bit-identical results.  Measured (scripts/small_batch.py, ms per launch, split 1 / 2 / 4): 64 boards 0.75 / - / 0.33,
    // 148 boards 0.79 / 0.44 / -, 200 boards 0.72 / 0.49 / -, 296 boards 0.73 / 0.70 / -, 512 boards 0.89 / 1.24 / -.
    const bool exclusive = net->tower_exclusive && (n + 3) / 4 > net->tower_pairs;      // large launches only
    const int pairs = std::min(exclusive ? net->tower_pairs : net->num_sms / 2, net->pairs_resident);
    a.nsplit = 1;
    a.tps1 = net->tower_tps1;
    if (layer_end - layer_begin > 1) {
        if (net->tower_nsplit) a.nsplit = net->tower_nsplit;
        else if (a.n_pair_tiles * 8 <= pairs) a.nsplit = 8;
        else if (a.n_pair_tiles * 4 <= pairs) a.nsplit = 4;
        else if (a.n_pair_tiles <= pairs) a.nsplit = 2;
    }
    net->last_nsplit = a.nsplit;
    // with fused heads the last layer's items are whole tiles (a board's 73 planes in one accumulator) whatever the split
    const int layers = layer_end - layer_begin;
    const int main_layers = heads && a.nsplit > 1 ? layers - 1 : layers;
    a.n_main = main_layers * a.n_pair_tiles * a.nsplit;
    a.n_items = a.n_main + (layers - main_layers) * a.n_pair_tiles;
    if (net->span_on && (int)net->span_boards.size() < SPAN_CAP && layer_end - layer_begin > 1) {
        a.span = net->span + 4 * net->span_boards.size();
        net->span_boards.push_back(n);
        net->span_b0.push_back(b0);
    }
    const int grid = 2 * std::min(a.n_pair_tiles * a.nsplit, pairs);
    if (net->trace_ring && !a.trace && a.nsplit == 1 && !a.heads.n_live && layers == MAX_TOWER_LAYERS && a.n_pair_tiles <= TRACE_MAX_TILES) {
        const int slot = (int)(net->trace_launches % TRACE_RING);
        a.trace = net->trace_ring + (size_t)slot * MAX_TOWER_LAYERS * TRACE_MAX_TILES * TRACE_STAMPS;
        net->trace_meta[slot] = {net->trace_launches, n, a.n_pair_tiles, grid / 2, a.span ? (long long)net->span_boards.size() - 1 : -1};
        net->trace_launches++;
    }
    SZB_CUDA(ctx, launch_kernel(a.heads.mask && a.heads.n_live ? k_tower_tc2<true> : k_tower_tc2<false>, dim3(grid), dim3(TC_THREADS), (size_t)(exclusive ? net->smem_exclusive : T2_SMEM), ctx->work,
                                run.pdl, *net->tower_maps, a));
    ctx->launches++;
    return 0;
}

// the whole forward (tower + both heads) of n <= cluster_max boards with one 8-CTA cluster per board; value_out[i] belongs to board b0 + i
// unless the heads are fused (then d.policy / d.value rows, as in launch_tower)
template <int CS>
static int cluster_setup_one(szb_ctx* ctx, Net* net, int v) {
    SZB_CUDA(ctx, cudaFuncSetAttribute(k_tower_cl<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, CL_SMEM));
    if (CS > 8) SZB_CUDA(ctx, cudaFuncSetAttribute(k_tower_cl<CS>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(CS * CL_MAX_BOARDS);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = CL_SMEM;
    int clusters = 0;
    if (cudaOccupancyMaxActiveClusters(&clusters, k_tower_cl<CS>, &cfg) == cudaSuccess) net->clusters_resident[v] = clusters;
    else cudaGetLastError();
    return 0;
}
static int cluster_setup(szb_ctx* ctx, Net* net) {
    if (net->attr_set_cl) return 0;
    int rc;
    if ((rc = cluster_setup_one<8>(ctx, net, 0)) || (rc = cluster_setup_one<16>(ctx, net, 1))) return rc;
    if (const char* e = getenv("SZB_TOWER_CLUSTER_VERBOSE")) {
        if (e[0] == '1') fprintf(stderr, "[szb200] k_tower_cl: %d clusters of 8 CTAs, %d clusters of 16 CTAs resident\n", net->clusters_resident[0], net->clusters_resident[1]);
    }
    net->attr_set_cl = true;
    return 0;
}
// cluster size that serves n boards in one wave (more boards than clusters fit at once would run in waves: then the pair kernel is
// the faster one), or 0
static int cluster_size_for(szb_ctx* ctx, Net* net, int n) {
    if (cluster_setup(ctx, net) || n > net->cluster_max) return 0;
    // clusters of 8 by default: with 16 CTAs per board a layer's weights fit the ring whole, but the MMA phase is bound by the
    // issue of its 144 tcgen05.mma (~28 clk each from one thread), not by weights, and the 16-way exchange costs 0.15 us more per
    // layer (measured 6.54 vs 6.39 us per layer); SZB_TOWER_CLUSTER_SIZE=16 keeps the variant reachable for A/B runs
    if (net->cluster_force == 16) return n <= net->clusters_resident[1] ? 16 : 0;
    return n <= net->clusters_resident[0] ? 8 : 0;
}

// the whole forward (tower + both heads) of n boards with one cluster of cs CTAs per board; value_out[i] belongs to board b0 + i
// unless the heads are fused (then d.policy / d.value rows, as in launch_tower)
static int launch_tower_cluster(szb_ctx* ctx, Net* net, int cs, int b0, int n, int out_row, float* value_out, TowerRun run) {
    int rc = cluster_setup(ctx, net);
    if (rc) return rc;
    if (out_row < 0) out_row = b0;
    ClusterArgs a;
    memset(&a, 0, sizeof a);
    a.n_boards = n;
    a.board0 = b0;
    a.in_delta = run.in16_rows ? out_row - b0 : 0;
    a.bias = net->bias_all;
    a.w_stream = net->w16_cl[cs == 16];
    a.error = net->tc_error;
    a.logits = net->logits;
    a.trace = net->cl_trace;
    memcpy(a.L, net->tower_args->L, sizeof a.L);
    TowerHeads& h = a.heads;
    h.row_delta = out_row - b0;
    h.v_w = net->v_w; h.fc1_wT = net->fc1_w; h.fc1_b = net->fc1_b; h.fc2_w = net->fc2_w; h.scalars = net->head_scalars;
    h.tower_out = nullptr;                                    // (the tower output never leaves shared memory)
    if (run.heads) {
        const Dev& d = ctx->d;
        h.mask = d.mask; h.need_eval = d.need_eval; h.policy = d.policy; h.value = d.value;
        h.row_slot = run.row_slot; h.n_live = run.n_live; h.live_off = run.live_off;
    } else {
        h.mask = nullptr; h.need_eval = nullptr; h.policy = nullptr;
        h.value = value_out - (ptrdiff_t)out_row;             // value[board + row_delta] == value_out[board - b0]
    }
    if (cs == 16) SZB_CUDA(ctx, launch_kernel(k_tower_cl<16>, dim3(16 * n), dim3(TC_THREADS), (size_t)CL_SMEM, ctx->work, run.pdl, *net->tower_maps, a));
    else SZB_CUDA(ctx, launch_kernel(k_tower_cl<8>, dim3(8 * n), dim3(TC_THREADS), (size_t)CL_SMEM, ctx->work, run.pdl, *net->tower_maps, a));
    ctx->launches++;
    return 0;
}

template <int N_TILE, int MODE>
static int launch_tc(szb_ctx* ctx, Net* net, const CUtensorMap& tm_a, const ConvLayer& L, const __nv_bfloat16* residual,
                     __nv_bfloat16* out, float* logits, int n, int relu, int b0 = 0) {
    constexpr int smem = TC_STAGES * (TC_A_BYTES + N_TILE * TC_BLOCK_K * 2) + 1024;
    if (!net->attr_set_tc[MODE]) {
        SZB_CUDA(ctx, cudaFuncSetAttribute(k_conv_tc<N_TILE, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        net->attr_set_tc[MODE] = true;
    }
    TcArgs a;
    a.n_tiles = (n + 1) / 2;
    a.taps = L.taps;
    a.kchunks = L.cin / TC_BLOCK_K;
    a.bias = L.bias;
    a.residual = residual;
    a.out = out;
    a.logits = logits;
    a.n_boards = n;
    a.board0 = b0;
    a.relu = relu;
    a.error = net->tc_error;
    const int grid = std::min(a.n_tiles, net->num_sms);
    k_conv_tc<N_TILE, MODE><<<grid, TC_THREADS, smem, ctx->work>>>(tm_a, L.tm_w, a);
    ctx->launches++;
    return 0;
}

static void launch_f32(szb_ctx* ctx, const float* in, const ConvLayer& L, const float* residual, float* out, int n, int relu, int mode) {
    F32Args a;
    a.in = in; a.w = L.w32; a.bias = L.bias; a.residual = residual; a.out = out;
    a.cin = L.cin; a.cout_pad = L.cout_pad; a.taps = L.taps; a.relu = relu; a.mode = mode;
    k_conv_f32<<<dim3(n, L.cout_pad / 64), 256, 0, ctx->work>>>(a);
    ctx->launches++;
}

// next unused (start, stop) event pair for the conv timing hook; null if events cannot be created
static cudaEvent_t* conv_event_pair(szb_ctx* ctx) {
    if (ctx->conv_events_used + 2 > ctx->conv_events.size()) {
        cudaEvent_t a, b;
        if (cudaEventCreate(&a) != cudaSuccess) return nullptr;
        if (cudaEventCreate(&b) != cudaSuccess) { cudaEventDestroy(a); return nullptr; }
        ctx->conv_events.push_back(a);
        ctx->conv_events.push_back(b);
    }
    cudaEvent_t* p = &ctx->conv_events[ctx->conv_events_used];
    ctx->conv_events_used += 2;
    return p;
}

void net_collect_conv_times(szb_ctx* ctx) {
    for (size_t i = 0; i + 1 < ctx->conv_events_used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ctx->conv_events[i], ctx->conv_events[i + 1]) == cudaSuccess) {
            ctx->conv_ms += ms;
            ctx->conv_launches++;
        }
    }
    ctx->conv_events_used = 0;
}

// planes (device, row stride `stride` uint64; row 0 = board b0) -> net->logits[b0..] + value_out[0..n) (device).
// b0 is the first board inside the activation buffers (a multiple of 4): cohorts of one search use disjoint ranges.
// All launches go to ctx->work.
static int net_forward_device(szb_ctx* ctx, int evaluator, int b0, int n, const uint64_t* planes, int stride, float* value_out, int out_row = -1,
                              TowerRun run = TowerRun()) {
    Net* net = ctx->net;
    if (out_row < 0) out_row = b0;
    if ((run.heads || run.in16_rows) && !(evaluator == SZB_EVAL_NET_BF16 && net && net->tower_mode == 2))
        return fail(ctx, SZB_ERR_ARG, "only the one-launch bf16 tower has fused heads");
    if (out_row != b0 && !(evaluator == SZB_EVAL_NET_BF16 && net && net->tower_mode == 2))
        return fail(ctx, SZB_ERR_ARG, "only the one-launch bf16 tower writes logits rows apart from its activation rows");
    if (!net || !net->loaded) return fail(ctx, SZB_ERR_STATE, "network weights not loaded (szb_net_load)");
    if (b0 + n > net->cap || (b0 & 3)) return fail(ctx, SZB_ERR_ARG, "batch [%d, %d) outside capacity %d", b0, b0 + n, net->cap);
    cudaStream_t st = ctx->work;
    const unsigned up_blocks = (unsigned)(((size_t)n * 64 * 16 + 255) / 256);
    const size_t in_off = (size_t)b0 * HALO * HALO * C_IN_PAD, act_off = (size_t)b0 * HALO * HALO * C_TOWER;
    if (evaluator == SZB_EVAL_NET_BF16) {
        if (!run.in16_rows) {
            k_planes_to_nhwc<__nv_bfloat16><<<up_blocks, 256, 0, st>>>(planes, stride, n, net->in16 + in_off);
            ctx->launches++;
        }
        int rc;
        int x, y;
        if (net->tower_mode == 0) {
            // single-CTA kernel, one launch per layer (kept as the A/B reference of the pair kernel)
            if ((rc = launch_tc<256, 0>(ctx, net, net->tm_in16, net->stem, nullptr, net->act16[0], nullptr, n, 1, b0))) return rc;
            x = 0;
            for (int blk = 0; blk < N_BLOCKS; blk++) {
                const int yy = (x + 1) % 3, o = (x + 2) % 3;
                if ((rc = launch_tc<256, 0>(ctx, net, net->tm_act16[x], net->tower[2 * blk], nullptr, net->act16[yy], nullptr, n, 1, b0))) return rc;
                cudaEvent_t* cev = (ctx->profiling && blk == 9) ? conv_event_pair(ctx) : nullptr;
                if (cev) cudaEventRecord(cev[0], st);
                if ((rc = launch_tc<256, 0>(ctx, net, net->tm_act16[yy], net->tower[2 * blk + 1], net->act16[x], net->act16[o], nullptr, n, 1, b0))) return rc;
                if (cev) { cudaEventRecord(cev[1], st); ctx->conv_recorded++; ctx->conv_boards += n; ctx->conv_flop += FLOP_TOWER_LAYER * (uint64_t)n; }
                x = o;
            }
            y = (x + 1) % 3;
            if ((rc = launch_tc<256, 0>(ctx, net, net->tm_act16[x], net->p1, nullptr, net->act16[y], nullptr, n, 1, b0))) return rc;
        } else if (net->tower_mode == 1) {
            for (int l = 0; l < POLICY_LAYER; l++) {
                cudaEvent_t* cev = (ctx->profiling && l == 20) ? conv_event_pair(ctx) : nullptr;
                if (cev) cudaEventRecord(cev[0], st);
                if ((rc = launch_tower(ctx, net, b0, n, l, l + 1))) return rc;
                if (cev) { cudaEventRecord(cev[1], st); ctx->conv_recorded++; ctx->conv_boards += n; ctx->conv_flop += FLOP_TOWER_LAYER * (uint64_t)n; }
            }
            x = net->final_x; y = net->final_y;
        } else if (const int cs = cluster_size_for(ctx, net, n)) {
            // a handful of boards: the cluster-resident kernel does the whole forward, heads included (fused or not)
            cudaEvent_t* cev = ctx->profiling ? conv_event_pair(ctx) : nullptr;
            if (cev) cudaEventRecord(cev[0], st);
            if ((rc = launch_tower_cluster(ctx, net, cs, b0, n, out_row, value_out, run))) return rc;
            if (cev) { cudaEventRecord(cev[1], st); ctx->conv_recorded++; ctx->conv_boards += n; ctx->conv_flop += FLOP_TOWER_ALL * (uint64_t)n; }
            SZB_CUDA(ctx, cudaGetLastError());
            return 0;
        } else {
            // stem + 38 tower convolutions + both policy 1x1 layers in ONE persistent launch; the measurement hook brackets exactly that launch
            cudaEvent_t* cev = ctx->profiling ? conv_event_pair(ctx) : nullptr;
            if (cev) cudaEventRecord(cev[0], st);
            if ((rc = launch_tower(ctx, net, b0, n, 0, MAX_TOWER_LAYERS, out_row, run))) return rc;
            if (cev) { cudaEventRecord(cev[1], st); ctx->conv_recorded++; ctx->conv_boards += n; ctx->conv_flop += FLOP_TOWER_ALL * (uint64_t)n; }
            x = net->final_x; y = net->final_y;
            if (run.heads) {                                      // priors and values were written by the tower's last epilogue
                SZB_CUDA(ctx, cudaGetLastError());
                return 0;
            }
        }
        // (the one-launch tower ends with the policy output layer; the per-layer modes use the single-CTA kernel for it)
        if (net->tower_mode != 2 && (rc = launch_tc<POLICY_PAD, 1>(ctx, net, net->tm_act16[y], net->p2, nullptr, nullptr, net->logits, n, 0, b0))) return rc;
        k_value_head<__nv_bfloat16><<<n, 256, 0, st>>>(net->act16[x] + act_off, net->v_w, net->head_scalars, net->fc1_w, net->fc1_b, net->fc2_w,
                                                       value_out, n);
        ctx->launches++;
    } else if (evaluator == SZB_EVAL_NET_FP32) {
        float* a32[3] = {net->act32[0] + act_off, net->act32[1] + act_off, net->act32[2] + act_off};
        k_planes_to_nhwc<float><<<up_blocks, 256, 0, st>>>(planes, stride, n, net->in32 + in_off);
        ctx->launches++;
        launch_f32(ctx, net->in32 + in_off, net->stem, nullptr, a32[0], n, 1, 0);
        int x = 0;
        for (int blk = 0; blk < N_BLOCKS; blk++) {
            const int y = (x + 1) % 3, o = (x + 2) % 3;
            launch_f32(ctx, a32[x], net->tower[2 * blk], nullptr, a32[y], n, 1, 0);
            launch_f32(ctx, a32[y], net->tower[2 * blk + 1], a32[x], a32[o], n, 1, 0);
            x = o;
        }
        const int y = (x + 1) % 3;
        launch_f32(ctx, a32[x], net->p1, nullptr, a32[y], n, 1, 0);
        launch_f32(ctx, a32[y], net->p2, nullptr, net->logits + (size_t)b0 * N_ACTIONS, n, 0, 1);
        k_value_head<float><<<n, 256, 0, st>>>(a32[x], net->v_w, net->head_scalars, net->fc1_w, net->fc1_b, net->fc2_w, value_out, n);
        ctx->launches++;
    } else {
        return fail(ctx, SZB_ERR_ARG, "unknown evaluator %d", evaluator);
    }
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// The bf16 tower of a large batch runs as a sequence of launches of at most `chunk` boards that all use the SAME activation rows
// [b0, b0 + chunk): three activation buffers of 512 boards (79 MB) + the weights stay in the 126 MB L2, those of 1024+ boards do
// not (ncu: 0.42 GB of DRAM traffic per 512-board launch, 2.68 GB per 1024-board launch), and under the 1 kW power cap DRAM
// traffic costs clock.  Planes in, logits / values out keep their own rows.
static int net_forward_chunked(szb_ctx* ctx, int evaluator, int b0, int n, const uint64_t* planes, int stride, float* value_out,
                               TowerRun run = TowerRun()) {
    Net* net = ctx->net;
    if (!net || !net->loaded) return fail(ctx, SZB_ERR_STATE, "network weights not loaded (szb_net_load)");
    const int chunk = (evaluator == SZB_EVAL_NET_BF16 && net->tower_mode == 2 && net->chunk > 0) ? net->chunk : n;
    for (int off = 0; off < n; off += chunk) {
        const int m = std::min(chunk, n - off);
        run.live_off = off;                                       // (evaluation cache: each chunk clamps itself to the device count)
        int rc = net_forward_device(ctx, evaluator, b0, m, planes + (size_t)off * stride, stride, value_out + off, b0 + off, run);
        if (rc) return rc;
        run.ready_zeroed = false;                                 // later chunks reuse the first chunk's counters: clear them again
        run.pdl = false;
    }
    return 0;
}

// does a search step with this evaluator run as k_tree_step + one tower launch with fused heads?
bool net_fused_step(szb_ctx* ctx, int evaluator) {
    return evaluator == SZB_EVAL_NET_BF16 && ctx->net && ctx->net->loaded && ctx->net->tower_mode == 2 && !ctx->net->no_fuse;
}

// what k_tree_step hands to the tower launch that evaluates slots [g0, g0 + n): the NHWC input rows it fills and the completion
// counters (of the first chunk's launch) it clears
void net_handover(szb_ctx* ctx, int g0, int n, unsigned short** in16, int32_t** ready, int* ready_n) {
    Net* net = ctx->net;
    const int first = net->chunk > 0 ? std::min(n, net->chunk) : n;
    *in16 = reinterpret_cast<unsigned short*>(net->in16);
    *ready = net->ready + (size_t)MAX_TOWER_LAYERS * (g0 / 4);
    *ready_n = MAX_TOWER_LAYERS * ((first + 3) / 4);
}

// evaluate slots [g0, g0 + n) of the search batch (g0 a multiple of 4): d.planes -> d.policy (softmax; the legal entries only when the
// heads are fused) / d.value, on ctx->work.  fused: the step's k_tree_step filled the input rows and cleared the counters.  n_live
// (fused only; evaluation cache): the step's device count of compacted input rows, whose slots are d.row_slot[g0 ..].
int net_evaluate_batch(szb_ctx* ctx, int evaluator, int g0, int n, bool fused, const int32_t* n_live) {
    TowerRun run;
    run.heads = run.in16_rows = run.ready_zeroed = fused;
    run.pdl = fused && ctx->pdl;
    if (fused && n_live) { run.n_live = n_live; run.row_slot = ctx->d.row_slot; }
    int rc = net_forward_chunked(ctx, evaluator, g0, n, ctx->d.planes + (size_t)g0 * PLANE_STRIDE, PLANE_STRIDE, ctx->d.value + g0, run);
    if (rc || fused) return rc;
    k_softmax<<<(n + 3) / 4, 256, 0, ctx->work>>>(ctx->net->logits + (size_t)g0 * N_ACTIONS, ctx->d.policy + (size_t)g0 * N_ACTIONS, n);
    ctx->launches++;
    return 0;
}

// a search starts with a clean pipeline-error flag (a timed-out launch must not poison the context for good)
int net_reset_error(szb_ctx* ctx) {
    if (ctx->net && ctx->net->tc_error) SZB_CUDA(ctx, cudaMemsetAsync(ctx->net->tc_error, 0, sizeof(int32_t), ctx->stream));
    return 0;
}

int net_check_error(szb_ctx* ctx) {
    int32_t flag = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->net->tc_error, 4, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (flag) return fail(ctx, SZB_ERR_CUDA, "tcgen05 convolution pipeline timed out (mbarrier wait exceeded its bound)");
    return 0;
}

}  // namespace szb

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

// expected tensors of network.py's state_dict (name -> element count), in the order the loader reads them
static void net_expected_tensors(std::vector<std::pair<std::string, int64_t>>& out) {
    auto bn = [&](const std::string& p, int c) {
        out.push_back({p + ".weight", c}); out.push_back({p + ".bias", c}); out.push_back({p + ".running_mean", c}); out.push_back({p + ".running_var", c});
    };
    out.push_back({"conv1.weight", 256LL * 119 * 9});
    bn("norm_layer", 256);
    for (int b = 0; b < N_BLOCKS; b++)
        for (int j = 1; j <= 2; j++) {
            const std::string pfx = "resnet_blocks." + std::to_string(b);
            out.push_back({pfx + ".conv" + std::to_string(j) + ".weight", 256LL * 256 * 9});
            bn(pfx + ".bn" + std::to_string(j), 256);
        }
    out.push_back({"conv_p1.weight", 256LL * 256});
    bn("p_norm1", 256);
    out.push_back({"conv_p2.weight", 73LL * 256}); out.push_back({"conv_p2.bias", 73});
    out.push_back({"conv_v1.weight", 256});
    bn("v_norm", 1);
    out.push_back({"fc_v1.weight", 256LL * 64}); out.push_back({"fc_v1.bias", 256});
    out.push_back({"fc_v2.weight", 256}); out.push_back({"fc_v2.bias", 1});
}

// device buffers, tensor maps and layer table of the network: once per context (and again only if the capacity changes)
static int net_ensure_allocated(szb_ctx* ctx) {
    const int cap = (ctx->cfg.max_games * ctx->d.K + 1) & ~1;           // one activation row per path slot
    if (ctx->net && ctx->net->cap == cap && ctx->net->allocated) return 0;
    int rc;
    if ((rc = net_tmap_init(ctx))) return rc;
    net_destroy(ctx);
    Net* net = new Net();
    ctx->net = net;
    cudaDeviceProp prop;
    SZB_CUDA(ctx, cudaGetDeviceProperties(&prop, ctx->device));
    net->num_sms = prop.multiProcessorCount;
    net->cap = cap;
    if ((rc = alloc_conv(ctx, net, net->stem, C_IN_PAD, 9, 256, 256))) return rc;
    for (int i = 0; i < 2 * N_BLOCKS; i++)
        if ((rc = alloc_conv(ctx, net, net->tower[i], 256, 9, 256, 256))) return rc;
    if ((rc = alloc_conv(ctx, net, net->p1, 256, 1, 256, 256))) return rc;
    // the fp32 kernel wants cout_pad % 64 == 0, the tcgen05 kernel reads POLICY_PAD rows: pad to 128 and map the first 80
    if ((rc = alloc_conv(ctx, net, net->p2, 256, 1, 73, 128))) return rc;
    if ((rc = net_tmap_rows(ctx, &net->p2.tm_w, net->p2.w16, 256, POLICY_PAD, POLICY_PAD, "weights"))) return rc;
    if ((rc = net_alloc(ctx, net, &net->v_w, 256, false)) || (rc = net_alloc(ctx, net, &net->fc1_w, 256 * 64, false)) ||
        (rc = net_alloc(ctx, net, &net->fc1_b, 256, false)) || (rc = net_alloc(ctx, net, &net->fc2_w, 256, false)) ||
        (rc = net_alloc(ctx, net, &net->head_scalars, 2, false)) || (rc = net_alloc(ctx, net, &net->digest, 1)))
        return rc;
    if ((rc = net_alloc_activations(ctx, net))) return rc;
    if ((rc = net_setup_tower(ctx, net))) return rc;
    net->allocated = true;
    return 0;
}

// fold + pack all tensors (DEVICE pointers) into the network's buffers; asynchronous on the context's stream, no host round trip
static int net_fill_from_device(szb_ctx* ctx, const std::map<std::string, const float*>& sd) {
    Net* net = ctx->net;
    ctx->d.ec_epoch++;                  // the one place the packed weights change: every evaluation cache entry is dead from here on
    auto at = [&](const std::string& k) { return sd.at(k); };
    auto bn_of = [&](const std::string& p) { return BN{at(p + ".weight"), at(p + ".bias"), at(p + ".running_mean"), at(p + ".running_var")}; };
    int rc;
    BN bn = bn_of("norm_layer");
    if ((rc = fold_conv(ctx, net->stem, at("conv1.weight"), 119, &bn, nullptr))) return rc;
    for (int b = 0; b < N_BLOCKS; b++)
        for (int j = 0; j < 2; j++) {
            const std::string p = "resnet_blocks." + std::to_string(b);
            bn = bn_of(p + ".bn" + std::to_string(j + 1));
            if ((rc = fold_conv(ctx, net->tower[2 * b + j], at(p + ".conv" + std::to_string(j + 1) + ".weight"), 256, &bn, nullptr))) return rc;
        }
    bn = bn_of("p_norm1");
    if ((rc = fold_conv(ctx, net->p1, at("conv_p1.weight"), 256, &bn, nullptr))) return rc;
    if ((rc = fold_conv(ctx, net->p2, at("conv_p2.weight"), 256, nullptr, at("conv_p2.bias")))) return rc;
    bn = bn_of("v_norm");
    k_fold_value_head<<<64, 256, 0, ctx->stream>>>(at("conv_v1.weight"), bn, at("fc_v1.weight"), at("fc_v1.bias"), at("fc_v2.weight"), at("fc_v2.bias"),
                                                   net->v_w, net->head_scalars, net->fc1_w, net->fc1_b, net->fc2_w);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    if ((rc = net_assemble_tower(ctx, net))) return rc;
    net->loaded = true;
    return 0;
}

static int net_load_common(szb_ctx* ctx, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel, bool on_device) {
    if (!ctx || n_tensors <= 0 || !names || !data || !numel) return fail(ctx, SZB_ERR_ARG, "szb_net_load: bad arguments");
    // validate the whole state_dict BEFORE touching the network that is loaded and working: a bad checkpoint leaves it in place
    std::map<std::string, std::pair<const float*, int64_t>> given;
    for (int i = 0; i < n_tensors; i++) given[names[i]] = {data[i], numel[i]};
    std::vector<std::pair<std::string, int64_t>> want;
    net_expected_tensors(want);
    size_t total = 0;
    for (auto& w : want) {
        auto it = given.find(w.first);
        if (it == given.end()) return fail(ctx, SZB_ERR_ARG, "state_dict is missing '%s'", w.first.c_str());
        if (it->second.second != w.second)
            return fail(ctx, SZB_ERR_ARG, "'%s' has %lld elements, expected %lld", w.first.c_str(), (long long)it->second.second, (long long)w.second);
        if (!it->second.first) return fail(ctx, SZB_ERR_ARG, "'%s' has a null data pointer", w.first.c_str());
        total += (size_t)w.second;
    }
    int rc;
    if ((rc = net_ensure_allocated(ctx))) return rc;
    std::map<std::string, const float*> sd;
    float* staging = nullptr;
    if (on_device) {
        for (auto& w : want) sd[w.first] = given[w.first].first;
    } else {
        // host tensors: one staging buffer on the device, then the same GPU fold as szb_net_load_device
        SZB_CUDA(ctx, cudaMalloc((void**)&staging, total * sizeof(float)));
        size_t off = 0;
        for (auto& w : want) {
            cudaError_t e = cudaMemcpyAsync(staging + off, given[w.first].first, (size_t)w.second * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
            if (e != cudaSuccess) { cudaFree(staging); return cuda_fail(ctx, e, "cudaMemcpyAsync(state_dict tensor)"); }
            sd[w.first] = staging + off;
            off += (size_t)w.second;
        }
    }
    rc = net_fill_from_device(ctx, sd);
    if (staging) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(staging);
    }
    return rc;
}

int szb_net_load(szb_ctx* ctx, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    return net_load_common(ctx, n_tensors, names, data, numel, false);
}

int szb_net_load_device(szb_ctx* ctx, int32_t n_tensors, const char* const* names, const float* const* data_dev, const int64_t* numel) {
    if (ctx) cudaSetDevice(ctx->device);
    return net_load_common(ctx, n_tensors, names, data_dev, numel, true);
}

int szb_net_checksum(szb_ctx* ctx, uint64_t* out) {
    if (!ctx || !out) return SZB_ERR_ARG;
    cudaSetDevice(ctx->device);
    Net* net = ctx->net;
    if (!net || !net->loaded) return fail(ctx, SZB_ERR_STATE, "network weights not loaded (szb_net_load)");
    SZB_CUDA(ctx, cudaMemsetAsync(net->digest, 0, sizeof(unsigned long long), ctx->stream));
    struct { const void* p; size_t bytes; } parts[] = {
        {net->w16_all, (size_t)MAX_TOWER_LAYERS * C_TOWER * 9 * C_TOWER * 2}, {net->bias_all, (size_t)MAX_TOWER_LAYERS * C_TOWER * 4},
        {net->v_w, 256 * 4}, {net->fc1_w, 256 * 64 * 4}, {net->fc1_b, 256 * 4}, {net->fc2_w, 256 * 4}, {net->head_scalars, 8}};
    uint64_t salt = 1;
    for (auto& part : parts) {
        const size_t words = part.bytes / 4;
        k_digest<<<(unsigned)std::min<size_t>((words + 255) / 256, 1184), 256, 0, ctx->stream>>>((const uint32_t*)part.p, words, salt++ * 0x9E3779B97F4A7C15ull, net->digest);
        ctx->launches++;
    }
    unsigned long long h = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(&h, net->digest, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out = h;
    return 0;
}

static int net_forward_common(szb_ctx* ctx, int32_t n, const uint64_t* planes, int32_t evaluator, float* policy_out, float* value_out, bool softmax) {
    if (!ctx || n <= 0 || !planes) return fail(ctx, SZB_ERR_ARG, "szb_net_forward: bad arguments");
    if (!ctx->net || !ctx->net->loaded) return fail(ctx, SZB_ERR_STATE, "network weights not loaded (szb_net_load)");
    Net* net = ctx->net;
    // process in chunks of the activation capacity; staging: planes + value (+ policy)
    const int cap = net->cap;
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t b_pl = up((size_t)cap * N_PLANES * 8), b_v = up((size_t)cap * 4), b_p = up((size_t)cap * N_ACTIONS * 4);
    char* st = (char*)ctx_stage(ctx, b_pl + b_v + b_p);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    uint64_t* d_pl = (uint64_t*)st;
    float* d_v = (float*)(st + b_pl);
    float* d_p = (float*)(st + b_pl + b_v);
    for (int lo = 0; lo < n; lo += cap) {
        const int m = std::min(cap, n - lo);
        SZB_CUDA(ctx, cudaMemcpyAsync(d_pl, planes + (size_t)lo * N_PLANES, (size_t)m * N_PLANES * 8, cudaMemcpyDefault, ctx->stream));
        int rc = net_forward_chunked(ctx, evaluator, 0, m, d_pl, N_PLANES, d_v);
        if (rc) return rc;
        const float* src = net->logits;
        if (softmax) {
            k_softmax<<<(m + 3) / 4, 256, 0, ctx->work>>>(net->logits, d_p, m);
            ctx->launches++;
            src = d_p;
        }
        if (policy_out) SZB_CUDA(ctx, cudaMemcpyAsync(policy_out + (size_t)lo * N_ACTIONS, src, (size_t)m * N_ACTIONS * 4, cudaMemcpyDefault, ctx->stream));
        if (value_out) SZB_CUDA(ctx, cudaMemcpyAsync(value_out + lo, d_v, (size_t)m * 4, cudaMemcpyDefault, ctx->stream));
        SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    SZB_CUDA(ctx, cudaGetLastError());
    if (evaluator == SZB_EVAL_NET_BF16) return net_check_error(ctx);
    return 0;
}

int szb_time_kernel(szb_ctx* ctx, int32_t which, int32_t n, int32_t iters, float* ms_avg_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !ms_avg_out || n <= 0 || iters <= 0) return fail(ctx, SZB_ERR_ARG, "szb_time_kernel: bad arguments");
    Net* net = ctx->net;
    if (!net || !net->loaded) return fail(ctx, SZB_ERR_STATE, "network weights not loaded (szb_net_load)");
    if (n > net->cap) return fail(ctx, SZB_ERR_ARG, "batch %d exceeds capacity %d", n, net->cap);
    cudaEvent_t e0, e1;
    SZB_CUDA(ctx, cudaEventCreate(&e0));
    SZB_CUDA(ctx, cudaEventCreate(&e1));
    int rc = 0;
    for (int pass = 0; pass < 2 && !rc; pass++) {          // pass 0 warms up
        const int reps = pass == 0 ? 3 : iters;
        SZB_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
        for (int i = 0; i < reps && !rc; i++) {
            switch (which) {
            case 0: rc = launch_tc<256, 0>(ctx, net, net->tm_act16[i & 1], net->tower[1], net->act16[2], net->act16[(i + 1) & 1], nullptr, n, 1); break;
            case 1: rc = net_forward_chunked(ctx, SZB_EVAL_NET_BF16, 0, n, ctx->d.planes, PLANE_STRIDE, ctx->d.value); break;
            case 2: rc = net_forward_device(ctx, SZB_EVAL_NET_FP32, 0, n, ctx->d.planes, PLANE_STRIDE, ctx->d.value); break;
            case 3: launch_f32(ctx, net->act32[i & 1], net->tower[1], net->act32[2], net->act32[(i + 1) & 1], n, 1, 0); break;
            case 4: rc = launch_tower(ctx, net, 0, n, 20, 21); break;                       // one tower layer, CTA-pair kernel
            case 5: rc = launch_tower(ctx, net, 0, n, 0, MAX_TOWER_LAYERS); break;          // whole tower, one launch
            case 6:                                                                         // whole forward, cluster-resident kernel
                if (const int cs = cluster_size_for(ctx, net, n)) rc = launch_tower_cluster(ctx, net, cs, 0, n, 0, ctx->d.value, TowerRun());
                else rc = fail(ctx, SZB_ERR_ARG, "no cluster-resident configuration holds %d boards at once on this device", n);
                break;
            default: rc = fail(ctx, SZB_ERR_ARG, "unknown kernel selector %d", which);
            }
        }
        SZB_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
        SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    float ms = 0;
    if (!rc) { cudaEventElapsedTime(&ms, e0, e1); *ms_avg_out = ms / iters; }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc) return rc;
    const char* trace_path = getenv("SZB_TOWER_TRACE");      // measurement aid: per-item device timestamps of one more launch as CSV
    if (which == 6 && trace_path && trace_path[0]) {
        unsigned long long* d_tr = nullptr;
        const size_t slots = (size_t)MAX_TOWER_LAYERS * 8;
        SZB_CUDA(ctx, cudaMalloc((void**)&d_tr, slots * 8));
        SZB_CUDA(ctx, cudaMemsetAsync(d_tr, 0, slots * 8, ctx->stream));
        net->cl_trace = d_tr;
        rc = launch_tower_cluster(ctx, net, cluster_size_for(ctx, net, n), 0, n, 0, ctx->d.value, TowerRun());
        net->cl_trace = nullptr;
        std::vector<unsigned long long> h(slots);
        cudaMemcpyAsync(h.data(), d_tr, slots * 8, cudaMemcpyDeviceToHost, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        cudaFree(d_tr);
        if (rc) return rc;
        if (FILE* f = fopen(trace_path, "a")) {
            fprintf(f, "boards,layer,input_ready_ns,mma_issued_ns,acc_ready_ns,tmem_read_ns,stores_issued_ns,arrived_ns\n");
            const unsigned long long t0 = h[0];
            for (int l = 0; l < MAX_TOWER_LAYERS; l++) {
                fprintf(f, "%d,%d", n, l);
                for (int k = 0; k < 6; k++) fprintf(f, ",%lld", h[(size_t)l * 8 + k] ? (long long)(h[(size_t)l * 8 + k] - t0) : -1ll);
                fprintf(f, "\n");
            }
            fclose(f);
        }
    }
    if (which == 5 && trace_path && trace_path[0]) {
        const int tiles = (n + 3) / 4;
        const size_t slots = (size_t)MAX_TOWER_LAYERS * tiles * 8 * TRACE_STAMPS;
        unsigned long long* d_tr = nullptr;
        SZB_CUDA(ctx, cudaMalloc((void**)&d_tr, slots * 8));
        SZB_CUDA(ctx, cudaMemsetAsync(d_tr, 0, slots * 8, ctx->stream));
        net->tower_args->trace = d_tr;
        rc = launch_tower(ctx, net, 0, n, 0, MAX_TOWER_LAYERS);
        net->tower_args->trace = nullptr;
        std::vector<unsigned long long> h(slots);
        cudaMemcpyAsync(h.data(), d_tr, slots * 8, cudaMemcpyDeviceToHost, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        cudaFree(d_tr);
        if (rc) return rc;
        unsigned long long t0 = ~0ull;
        for (unsigned long long v : h) if (v && v < t0) t0 = v;
        if (FILE* f = fopen(trace_path, "a")) {
            fprintf(f, "boards,nsplit,item,layer,tile,q,dep_ns,operands_ns,acc_ns,released_ns,last_mma_ns\n");
            const int nsplit = net->last_nsplit;
            for (int item = 0; item < MAX_TOWER_LAYERS * tiles * nsplit; item++) {
                const int ti = item / nsplit;
                fprintf(f, "%d,%d,%d,%d,%d,%d", n, nsplit, item, ti / tiles, ti % tiles, item % nsplit);
                for (int k = 0; k < TRACE_STAMPS; k++)
                    fprintf(f, ",%lld", h[(size_t)item * TRACE_STAMPS + k] ? (long long)(h[(size_t)item * TRACE_STAMPS + k] - t0) : -1ll);
                fprintf(f, "\n");
            }
            fclose(f);
        }
    }
    SZB_CUDA(ctx, cudaGetLastError());
    return net_check_error(ctx);
}

int szb_tower_spans_record(szb_ctx* ctx, int32_t on, szb_tower_spans* out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    Net* net = ctx->net;
    if (!net || !net->loaded) return fail(ctx, SZB_ERR_STATE, "network weights not loaded (szb_net_load)");
    SZB_CUDA(ctx, cudaDeviceSynchronize());
    if (on) {
        int rc = net_span_reset(ctx, net);
        if (rc) return rc;
        net->span_on = true;
        return 0;
    }
    net->span_on = !net->span_path.empty();
    if (!out) return 0;
    memset(out, 0, sizeof *out);
    const size_t n = net->span_boards.size();
    if (n == 0) return 0;
    std::vector<unsigned long long> h(4 * n);
    SZB_CUDA(ctx, cudaMemcpy(h.data(), net->span, h.size() * 8, cudaMemcpyDeviceToHost));
    unsigned long long first = ~0ull, last = 0;
    for (size_t i = 0; i < n; i++) {
        if (h[4 * i] == ~0ull || h[4 * i + 1] == 0) continue;                 // launch not run (cannot happen after the sync above)
        out->launches++;
        out->boards += (uint64_t)net->span_boards[i];
        out->busy_ns += h[4 * i + 1] - h[4 * i];
        out->flop += FLOP_TOWER_ALL * (uint64_t)net->span_boards[i];
        out->sm_cycles += h[4 * i + 2];
        out->sm_ns += h[4 * i + 3];
        first = std::min(first, h[4 * i]);
        last = std::max(last, h[4 * i + 1]);
    }
    if (out->launches) out->wall_ns = last - first;
    return 0;
}

int szb_net_forward(szb_ctx* ctx, int32_t n, const uint64_t* planes, int32_t evaluator, float* policy_out, float* value_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    return net_forward_common(ctx, n, planes, evaluator, policy_out, value_out, true);
}

int szb_net_forward_logits(szb_ctx* ctx, int32_t n, const uint64_t* planes, int32_t evaluator, float* logits_out, float* value_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    return net_forward_common(ctx, n, planes, evaluator, logits_out, value_out, false);
}

}  // extern "C"
