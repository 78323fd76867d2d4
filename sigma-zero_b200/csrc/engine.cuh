// engine.cuh -- context layout shared by engine.cu (games, tree, search, perft) and net.cu (network).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <utility>
#include <vector>
#include "../../include/szb200.h"
#include "chess.cuh"
#include "tree.cuh"

namespace szb {

constexpr int RING = 256;                  // real-game positions kept per game (repetition walk <= 150 plies)
constexpr int PLANE_STRIDE = 120;          // uint64 per packed plane row (119 + 1 pad, 16-byte aligned rows)
constexpr int MASK_STRIDE = 80;            // uint64 per legal-mask row (73 + pad)
constexpr uint16_t NO_CHILD = 0xFFFF;
constexpr uint16_t CHILD_PENDING = 0xFFFE;  // multi-leaf mode: the edge's node is being created by an earlier path of this step
constexpr int PATH_DROPPED = -2;           // multi-leaf mode, sel_edge: this path slot carries no simulation in this step
constexpr int MAX_LEAVES = 8;              // szb_config.leaves_per_tree <= 8 (one warp per path in k_finish_vl)
constexpr int PATH_CAP = 64;               // edges of the selected path k_select records per tree (deeper paths: backup walks node_pedge)

// What an edge knows about the node behind it: {first child edge (int32) | child count << 32 | visited-node index << 48}.  PUCT
// selection reads it next to N / W / P, so the header of the next level arrives with the scan that picks it (one dependent memory
// round trip per tree level instead of two).
__host__ __device__ __forceinline__ unsigned long long link_pack(int32_t edge0, uint32_t nchild, uint32_t child) {
    return (unsigned long long)(uint32_t)edge0 | ((unsigned long long)(nchild & 0xFFFFu) << 32) | ((unsigned long long)(child & 0xFFFFu) << 48);
}
__host__ __device__ __forceinline__ int32_t link_edge0(unsigned long long l) { return (int32_t)(uint32_t)l; }
__host__ __device__ __forceinline__ int link_nchild(unsigned long long l) { return (int)((l >> 32) & 0xFFFFu); }
__host__ __device__ __forceinline__ uint16_t link_child(unsigned long long l) { return (uint16_t)(l >> 48); }

// One entry of the evaluation cache (32 bytes); its priors live in a parallel array of EC_PRI_STRIDE floats.
struct alignas(32) EcMeta {
    uint64_t k0, k1;         // 128-bit key: input planes, legal mask, evaluator id
    uint32_t epoch;          // Dev::ec_epoch when written
    uint32_t gen;            // Dev::ec_gen of the last search that wrote or hit it
    uint32_t n_legal;
    float value;
};
constexpr int EC_PRI_STRIDE = 224;         // 218 legal moves at most, padded
constexpr int EC_MIN_SLOTS = 64, EC_MAX_SLOTS = 65536;

struct Net;                                // net.cu
struct Trainer;                            // train.cu

// Device pointers of one context.  Passed to kernels by value.
struct Dev {
    // ---- games --------------------------------------------------------------------------------
    Pos* pool;               // [max_games][pool_stride]: slots [0,RING) real game ring, RING+i = tree node i
    int32_t* cur;            // [max_games] ring slot of the current position
    uint16_t* anc;           // [max_games][pool_stride][8] pool slots of a position's 8 predecessors, nearest first (0xFFFF: none), recorded
                             // when the position is made: the history planes load them side by side instead of walking Pos::prev
    const Tables* tables;
    const uint4* lut_bf16;   // [256] byte -> eight bf16 (0 / 1.0)
    int pool_stride;
    int n_games;
    int K;                   // leaves (in-flight simulations) per tree and step: 1 = the reference's algorithm
    int g_begin, g_end;      // SLOT range the step kernels of this launch work on (a cohort of the search batch)
    int32_t* order;          // [max_games] slot -> game: the games whose root is not terminal, ascending (k_active_list).  Finished
                             // games take no slot: no step kernel, no network row (the reference never searches a finished game,
                             // sim.py:46; a search on a terminal root only backs up its constant value, mcts.py:49-70,104-109)
    int32_t* n_active;       // device: number of slots
    // ---- tree: visited nodes (one per simulation) -------------------------------------------------
    int nodes_per_game;      // max_searches + 1
    int32_t* node_edge0;     // first child edge (global index)
    uint16_t* node_nchild;
    int32_t* node_pedge;     // edge that leads here, -1 for the root
    uint16_t* node_pnode;
    uint8_t* node_term;      // terminal position
    float* node_tval;        // its value: -1 mated, 0 draw
    int32_t* node_count;     // [max_games] last node index in use
    int32_t* root_n;         // [max_games] root.visit_count (starts at 1, mcts.py:46)
    double* root_w;
    // ---- tree: edges (one per child of every expanded node), structure of arrays ---------------
    int32_t* e_n;            // child.visit_count
    double* e_w;             // child.value_sum
    float* e_p;              // child.prior
    uint16_t* e_move;        // policy index of child.action_taken
    unsigned long long* e_link;   // link_pack(first edge, child count, visited-node index | NO_CHILD) of the node behind the edge
    unsigned long long edge_cap;
    unsigned long long* edge_top;
    int32_t* error_flag;
    // ---- per simulation step ------------------------------------------------------------------
    // (indexed by PATH slot = slot * K + j; the network reads contiguous rows of planes / writes contiguous rows of policy)
    int32_t* sel_node;       // leaf (or, before expansion, its parent)
    int32_t* sel_edge;       // edge to create a node for, -1 when the leaf already exists, PATH_DROPPED
    int32_t* sel_new;        // multi-leaf mode: node index the expansion must use
    int32_t* path;           // [slot][PATH_CAP] edges of the path k_select walked, root first (reference-exact mode)
    int32_t* path_len;       // [slot] its length (backup is one parallel read-modify-write per edge while it fits PATH_CAP)
    uint8_t* need_eval;
    float* leaf_value;
    int32_t* sims_done;      // [max_games] multi-leaf mode: simulations completed in this search
    uint64_t* planes;        // [path slot][PLANE_STRIDE]
    uint64_t* mask;          // [path slot][MASK_STRIDE]
    float* policy;           // [path slot][4672] evaluator output ("softmax over everything")
    float* value;            // [path slot]
    float* root_val;         // [max_games] evaluator value of the root position
    unsigned long long* stats;   // totals: 0 simulations, 1 evaluations, 2 terminal visits, 3 max depth,
                                 // 4 select edges, 5 select levels, 6 backup levels, 7 edges written
    // ---- hand-over to the network (net.cu), set per launch by run_search ----------------------------
    unsigned short* net_in16;    // bf16 NHWC input rows [path slot][10][10][128] the expansion writes directly, or null
    int32_t* net_ready;          // per-item completion counters of the tower launch that follows: zeroed by the tree kernel
    int net_ready_n;
    unsigned long long* step_trace;  // measurement aid (SZB_STEP_TRACE): %globaltimer stamps of the first tree's warp through k_tree_step, or null
    unsigned long long* gstats;  // [max_games][8] the same counters per game: the step kernels bump their own game's row
                                 // (no same-address atomics on the hot path), k_fold_stats folds the rows into `stats`
    // ---- keys and opt-in exploration (szb_set_game_id_base, szb_set_exploration) --------------------
    uint64_t game_id_base;       // global id of game 0 of this context (RNG keys; sharding)
    float dir_alpha;             // > 0: searches with learning != 0 put Dirichlet(dir_alpha) noise on the root's priors
    float dir_eps;
    uint64_t dir_seed;
    // ---- opt-in evaluation cache (szb_set_eval_cache): per game an open-addressed table keyed on the exact evaluator input ---------
    int ec_slots;                // entries per game (a power of two), 0 = off
    uint32_t ec_epoch;           // bumped whenever the weights change or the table is resized: older entries are dead
    uint32_t ec_gen;             // this search's generation; entries of this search and the previous one are live
    uint32_t ec_eval;            // evaluator id, part of the key
    EcMeta* ec_meta;             // [max_games][ec_slots]
    float* ec_pri;               // [max_games][ec_slots][EC_PRI_STRIDE] evaluator output of the legal moves, ascending policy index
    uint64_t* ec_key;            // [slot][2] key of the slot's leaf (lookup -> finish of the next step)
    int32_t* ec_ent;             // [slot] entry the leaf hit (hit) or reserved (miss), -1: none
    uint8_t* ec_hit;             // [slot]
    int32_t* row_slot;           // [row] slot whose leaf the evaluator's compacted input row `row` holds
    int32_t* ec_cnt;             // this cohort's two per-step-parity row counters (set per launch)
    unsigned long long* ec_boards;   // [2] per cohort: boards the evaluator ran on in searches that consulted the cache (cumulative;
                                     // this launch's cohort entry while a search runs)
    int ec_par;                  // parity of this launch's step
    unsigned long long* ec_gstats;   // [max_games][4] lookups, hits, inserts, dropped inserts (cumulative)
    uint32_t* ec_ghits;          // [max_games] hits of the last search
};

}  // namespace szb

struct szb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t work = nullptr;               // stream the launch helpers use: `stream`, or a cohort stream inside a search
    cudaStream_t cohort_stream[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    int cohorts = 0;                           // 0 = automatic
    std::string err;
    szb_config cfg{};
    szb::Dev d{};
    szb::Tables host_tables;
    std::vector<void*> allocs;
    uint64_t launches = 0;
    uint64_t edges_high_water = 0;
    // perft scratch (lazy)
    std::vector<szb::Pos*> perft_levels;
    size_t perft_cap = 0;
    unsigned long long* perft_counter = nullptr;
    // staging (lazy, grown on demand)
    void* stage = nullptr;
    size_t stage_bytes = 0;
    // network (net.cu)
    szb::Net* net = nullptr;
    // trainer (train.cu)
    szb::Trainer* trainer = nullptr;
    // self-play records
    int32_t* d_moves = nullptr;
    int32_t sample_plies = 0;                  // szb_exploration.sample_plies: sampled moves only while the root's ply is below it
    // evaluation cache (szb_set_eval_cache): one allocation for the tables, freed when the cache is resized or switched off
    void* ec_mem = nullptr;
    uint64_t ec_bytes = 0;
    // profiling
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;
    float phase_ms[4] = {0, 0, 0, 0};
    int phase_steps = 0;
    std::vector<cudaEvent_t> conv_events;      // pairs around the timed tower convolution (net.cu)
    size_t conv_events_used = 0;
    float conv_ms = 0;
    int conv_launches = 0;                     // launches folded into conv_ms
    int conv_recorded = 0;                     // launches bracketed by events since profiling was switched on
    uint64_t conv_boards = 0;                  // boards of the bracketed launches (sum)
    uint64_t conv_flop = 0;                    // algorithmic FLOP of the bracketed launches (sum)
    int net_tower_mode = 2;                    // which bf16 tower kernel runs (net.cu: Net::tower_mode)
    bool pdl = false;                          // the launches of the search step in flight use programmatic dependent launch
};

namespace szb {
// Programmatic dependent launch (one-cohort searches): a kernel launched with this attribute may start while its predecessor on the
// stream is still running; it does its set-up, then griddepcontrol.wait blocks until the predecessor has completed and flushed.
// Both kernels of a search step call pdl_trigger() first (let the successor's set-up overlap me) and pdl_wait() before they touch
// anything the predecessor wrote.  Without the attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// device time in ns (%globaltimer): the stamps of the measurement aids (SZB_STEP_TRACE, SZB_TOWER_TRACE, SZB_TRAIN_TRACE, ...)
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
template <class... KArgs, class... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
int fail(szb_ctx* ctx, int code, const char* fmt, ...);
int cuda_fail(szb_ctx* ctx, cudaError_t e, const char* what);
void* ctx_stage(szb_ctx* ctx, size_t bytes);
// net.cu: evaluate games [g0, g0 + n) of d.planes -> d.policy / d.value (softmax policy) on ctx->work.
int net_evaluate_batch(szb_ctx* ctx, int evaluator, int g0, int n, bool fused, const int32_t* n_live = nullptr);
bool net_fused_step(szb_ctx* ctx, int evaluator);
void net_handover(szb_ctx* ctx, int g0, int n, unsigned short** in16, int32_t** ready, int* ready_n);
int net_reset_error(szb_ctx* ctx);
void net_destroy(szb_ctx* ctx);
void trainer_destroy(szb_ctx* ctx);
int net_check_error(szb_ctx* ctx);
// net.cu: fold the recorded conv event pairs into ctx->conv_ms (call after the stream is synchronised)
void net_collect_conv_times(szb_ctx* ctx);
// net.cu: bf16 tensor maps with 128-byte swizzle (net.cu and train.cu).  net_tmap_init looks cuTensorMapEncodeTiled up once; a builder
// that fails reports "cuTensorMapEncodeTiled(<what>) failed".
int net_tmap_init(szb_ctx* ctx);
// halo activations [boards][10][10][channels]: box = 64 channels x 8 x 8 x box_boards (the interior of a board's halo tile)
int net_tmap_act(szb_ctx* ctx, CUtensorMap* tm, void* base, int channels, int boards, int box_boards, const char* what);
// the same seen as (c, x, board, y): box = 64 channels x 10 x box_boards x 10 -> shared-memory rows [y][board][x], a whole halo chunk
// (strides need not ascend: probed, scripts/desc_probe.cu)
int net_tmap_halo(szb_ctx* ctx, CUtensorMap* tm, void* base, int channels, int boards, int box_boards, const char* what);
// K-major rows [rows][k_total]: box = 64 k x box_rows rows
int net_tmap_rows(szb_ctx* ctx, CUtensorMap* tm, void* base, int k_total, int rows, int box_rows, const char* what);
}  // namespace szb

#define SZB_CUDA(ctx, call)                                             \
    do {                                                                \
        cudaError_t _e = (call);                                        \
        if (_e != cudaSuccess) return szb::cuda_fail(ctx, _e, #call);   \
    } while (0)
