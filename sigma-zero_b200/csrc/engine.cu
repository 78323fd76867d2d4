// engine.cu -- games, flat SoA search tree, batched MCTS step kernels, perft, and the C ABI around them.
//
// One simulation step of mcts.py:49-109 runs for ALL running games at once (finished games take no slot: k_search_begin closes
// terminal roots, k_active_list numbers the rest), a warp per tree through every phase:
//   select    : PUCT descent, one warp arg-max per level (puct_pick)                 (mctsnode.py:23-37, mcts.py:54-55)
//   expand    : make-move + legality + terminal + legal mask + planes (expand_warp)  (mcts.py:57-70, chess_tensor.py:88-172)
//   evaluator : hash kernel or the network (net.cu)                                   (mcts.py:72-75)
//   finish    : mask/normalise/noise, child allocation, backup (finish_block)         (mcts.py:77-109, mctsnode.py:39-63)
// A search runs select, expand and finish in one kernel, k_tree_step, between evaluator launches.  Profiled searches (and
// SZB_NO_FUSE) run the same code as the phase kernels k_select / k_expand / k_finish, and the opt-in multi-leaf mode
// (szb_config.leaves_per_tree > 1, not the reference's algorithm) as k_select_vl / k_expand / k_finish_vl.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include "engine.cuh"

using namespace szb;

// ------------------------------------------------------------------------------------------------
// host helpers
// ------------------------------------------------------------------------------------------------
namespace szb {
int fail(szb_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}
int cuda_fail(szb_ctx* ctx, cudaError_t e, const char* what) {
    return fail(ctx, SZB_ERR_CUDA, "CUDA error %s (%d) at %s", cudaGetErrorString(e), (int)e, what);
}
void* ctx_stage(szb_ctx* ctx, size_t bytes) {
    if (bytes > ctx->stage_bytes) {
        if (ctx->stage) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->stage); }
        ctx->stage = nullptr;
        ctx->stage_bytes = 0;
        size_t want = std::max(bytes, (size_t)1 << 20);
        if (cudaMalloc(&ctx->stage, want) != cudaSuccess) return nullptr;
        ctx->stage_bytes = want;
    }
    return ctx->stage;
}
}  // namespace szb

template <class T>
static int dev_alloc(szb_ctx* ctx, T** out, size_t count) {
    void* p = nullptr;
    SZB_CUDA(ctx, cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
    SZB_CUDA(ctx, cudaMemsetAsync(p, 0, std::max<size_t>(count, 1) * sizeof(T), ctx->stream));
    ctx->allocs.push_back(p);
    *out = (T*)p;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_tables(Tables* sm, const Tables* g) {
    const uint64_t* src = reinterpret_cast<const uint64_t*>(g);
    uint64_t* dst = reinterpret_cast<uint64_t*>(sm);
    for (int i = threadIdx.x; i < (int)(sizeof(Tables) / 8); i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}
__device__ __forceinline__ int state_slot(const Dev& d, int g, int node) { return node == 0 ? d.cur[g] : RING + node; }

// predecessor slots of the position in `slot`, whose direct predecessor sits in prev_slot (NO_PREV: a game's first position)
__device__ __forceinline__ void set_ancestors(const Dev& d, int g, int slot, uint32_t prev_slot) {
    uint4* row = reinterpret_cast<uint4*>(d.anc + ((size_t)g * d.pool_stride + slot) * 8);
    if (prev_slot == NO_PREV) { *row = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu); return; }
    const uint4 o = *reinterpret_cast<const uint4*>(d.anc + ((size_t)g * d.pool_stride + prev_slot) * 8);
    *row = make_uint4((o.x << 16) | (prev_slot & 0xFFFFu), (o.y << 16) | (o.x >> 16), (o.z << 16) | (o.y >> 16), (o.w << 16) | (o.z >> 16));
}

__device__ __forceinline__ void analyse(const Tables& T, Pos& p, uint16_t* mv, int& n) {
    n = gen_legal(T, p, mv);
    p.n_legal = (uint8_t)n;
    p.outcome = outcome_of(T, p, n);
}

// ------------------------------------------------------------------------------------------------
// games
// ------------------------------------------------------------------------------------------------
__global__ void k_games_init(Dev d, const Pos* start, int n) {
    __shared__ Tables T;
    load_tables(&T, d.tables);
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    Pos p = start[g];
    uint16_t mv[MAX_MOVES];
    int cnt;
    finish_setup(T, p);
    analyse(T, p, mv, cnt);
    const int slot = p.ply & (RING - 1);
    d.pool[(size_t)g * d.pool_stride + slot] = p;
    set_ancestors(d, g, slot, NO_PREV);
    d.cur[g] = slot;
}

__global__ void k_games_push(Dev d, int n, const int32_t* game, const uint16_t* index, int32_t* status) {
    __shared__ Tables T;
    load_tables(&T, d.tables);
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int g = game ? game[i] : i;
    if (g < 0 || g >= d.n_games) { status[i] = SZB_ERR_ARG; return; }
    Pos* gp = d.pool + (size_t)g * d.pool_stride;
    const Pos p = gp[d.cur[g]];
    uint16_t mv[MAX_MOVES];
    const uint16_t m = index[i] < N_ACTIONS ? index_to_move(p, index[i]) : MOVE_NONE;
    bool ok = false;
    if (m != MOVE_NONE) {
        int cnt = gen_legal(T, p, mv);
        for (int k = 0; k < cnt; k++) ok |= mv[k] == m;
    }
    if (!ok) { status[i] = SZB_ERR_ILLEGAL_MOVE; return; }
    Pos q;
    make_move(T, p, m, q);
    q.prev = (uint32_t)d.cur[g];
    set_repetition_flags(gp, q);
    int cnt;
    analyse(T, q, mv, cnt);
    const int slot = q.ply & (RING - 1);
    gp[slot] = q;
    set_ancestors(d, g, slot, q.prev);
    d.cur[g] = slot;
    status[i] = 0;
}

__global__ void k_games_get(Dev d, int n, const int32_t* game, szb_pos* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int g = game ? game[i] : i;
    szb_pos o;
    memset(&o, 0, sizeof o);
    if (g >= 0 && g < d.n_games) {
        const Pos& p = d.pool[(size_t)g * d.pool_stride + d.cur[g]];
        for (int t = 0; t < 6; t++) {
            o.pieces[t] = p.bb[BB_P + t] & p.bb[BB_WHITE];
            o.pieces[6 + t] = p.bb[BB_P + t] & p.bb[BB_BLACK];
        }
        o.turn = (p.flags & F_WHITE) ? 1 : 0;
        o.castling_w = p.rights_w; o.castling_b = p.rights_b;
        o.ep_square = p.ep; o.halfmove_clock = p.halfmove; o.ply = p.ply;
        o.chess960 = (p.flags & F_960) ? 1 : 0;
        o.outcome = p.outcome;
        o.rep_flags = (uint8_t)(((p.flags & F_REP2) ? 1 : 0) | ((p.flags & F_REP3) ? 2 : 0));
        o.n_legal = p.n_legal;
    }
    out[i] = o;
}

__global__ void k_unpack_planes_f32(int n, const uint64_t* planes, float* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;       // one output element
    size_t total = (size_t)n * N_PLANES * 64;
    if (i >= total) return;
    size_t row = i >> 6;
    out[i] = (float)((planes[row] >> (i & 63)) & 1ull);
}

// ------------------------------------------------------------------------------------------------
// search step kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_search_begin(Dev d, int num_searches) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) *d.edge_top = 0ull;
    if (g >= d.n_games) return;
    const size_t r = (size_t)g * d.nodes_per_game;
    d.node_count[g] = 0;
    d.sims_done[g] = 0;
    d.node_edge0[r] = -1;
    d.node_nchild[r] = 0;
    d.node_pedge[r] = -1;
    d.node_pnode[r] = 0;
    const Pos& p = d.pool[(size_t)g * d.pool_stride + d.cur[g]];
    const bool term = p.outcome != OUT_NONE;
    const float tval = p.outcome == OUT_CHECKMATE ? -1.0f : 0.0f;
    d.node_term[r] = term;
    d.node_tval[r] = tval;
    if (!term) {
        d.root_n[g] = 1;
        d.root_w[g] = 0.0;
    } else {
        // terminal root: every simulation of mcts.py:49 finds the childless root, reads its constant value and backs it up
        // (:104-109) -- done here in closed form (the sum of num_searches equal doubles 0 or -1 is exact); the game takes no slot
        d.root_n[g] = 1 + num_searches;
        d.root_w[g] = (double)tval * (double)num_searches;
        unsigned long long* gs = d.gstats + (size_t)g * 8;
        gs[0] += (unsigned long long)num_searches;
        gs[2] += (unsigned long long)num_searches;
    }
}

// slot -> game list of the games to search (root not terminal), ascending.  One block.
__global__ void __launch_bounds__(1024) k_active_list(Dev d) {
    __shared__ int warp_tot[32];
    __shared__ int base_sh;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) base_sh = 0;
    __syncthreads();
    for (int g0 = 0; g0 < d.n_games; g0 += 1024) {
        const int g = g0 + threadIdx.x;
        const bool live = g < d.n_games && !d.node_term[(size_t)g * d.nodes_per_game];
        const unsigned ballot = __ballot_sync(0xFFFFFFFFu, live);
        if (lane == 0) warp_tot[wid] = __popc(ballot);
        __syncthreads();
        int before = base_sh;
        for (int w = 0; w < wid; w++) before += warp_tot[w];
        if (live) d.order[before + __popc(ballot & ((1u << lane) - 1))] = g;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 32; w++) t += warp_tot[w]; base_sh += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *d.n_active = base_sh;
}

// PUCT arg-max over the n children at edge e0 by one warp (mctsnode.py:23-37): lane t scores the children t, t + 32, ..., a shuffle
// reduction picks the winner, the first index winning ties.  Returns its index; its visit count and e_link go to cn / lk.  All three
// are the same in every lane.
__device__ __forceinline__ int puct_pick(const Dev& d, int e0, int n, float sq, float c_puct, int lane, int& cn, unsigned long long& lk) {
    float best = -INFINITY;
    int besti = 0x7FFFFFFF, best_n = 0;
    unsigned long long best_link = 0;
    for (int i = lane; i < n; i += 32) {
        const int c = d.e_n[e0 + i];
        const unsigned long long l = d.e_link[e0 + i];
        const float s = puct_score(c, d.e_w[e0 + i], d.e_p[e0 + i], sq, c_puct);
        if (s > best || besti == 0x7FFFFFFF) { best = s; besti = i; best_n = c; best_link = l; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float ob = __shfl_down_sync(0xFFFFFFFFu, best, off);
        const int oi = __shfl_down_sync(0xFFFFFFFFu, besti, off);
        if (oi != 0x7FFFFFFF && (besti == 0x7FFFFFFF || ob > best || (ob == best && oi < besti))) { best = ob; besti = oi; }
    }
    besti = __shfl_sync(0xFFFFFFFFu, besti, 0);
    // child i was scored by lane i % 32, which still holds its visit count and link
    cn = __shfl_sync(0xFFFFFFFFu, best_n, besti & 31);
    lk = __shfl_sync(0xFFFFFFFFu, best_link, besti & 31);
    return besti;
}

// PUCT descent of one tree by one warp (mctsnode.py:23-37, mcts.py:54-55).  One dependent memory round trip per level: the four
// edge arrays of the node's children are read side by side, and the chosen child's header (child count, first edge) rides on its
// edge (e_link), like its visit count and node index: the winning lane already holds them.  The edges walked are recorded
// (d.path) so that the backup of this simulation is one parallel read-modify-write instead of a pointer chase.
__device__ __forceinline__ void select_tree(const Dev& d, int slot, int lane, float c_puct) {
    const int g = d.order[slot];
    const size_t r = (size_t)g * d.nodes_per_game;
    int32_t* path = d.path + (size_t)slot * PATH_CAP;
    int node = 0, depth = 0;
    int np = d.root_n[g];                                  // visit count of the node being expanded (root: mcts.py:46)
    int n = d.node_nchild[r], e0 = d.node_edge0[r];        // the root's header; deeper headers come with the chosen edge
    unsigned long long scanned = 0;
    for (;;) {
        if (n == 0) {
            if (lane == 0) { d.sel_node[slot] = node; d.sel_edge[slot] = -1; }
            break;
        }
        unsigned long long lk;
        const int e = e0 + puct_pick(d, e0, n, sqrt_parent(np), c_puct, lane, np, lk);
        if (lane == 0 && depth < PATH_CAP) path[depth] = e;
        depth++;
        scanned += (unsigned long long)n;
        const uint16_t c = link_child(lk);
        if (c == NO_CHILD) {
            if (lane == 0) { d.sel_node[slot] = node; d.sel_edge[slot] = e; }
            break;
        }
        node = c;
        n = link_nchild(lk);
        e0 = link_edge0(lk);
    }
    if (lane == 0) {
        d.path_len[slot] = depth;
        unsigned long long* gs = d.gstats + (size_t)g * 8;
        if ((unsigned long long)depth > gs[3]) gs[3] = (unsigned long long)depth;
        gs[4] += scanned;
        gs[5] += (unsigned long long)depth;
    }
}

// warp per tree
__global__ void __launch_bounds__(128) k_select(Dev d, float c_puct) {
    const int slot = d.g_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (slot >= d.g_end) return;
    select_tree(d, slot, threadIdx.x & 31, c_puct);
}

// Legal moves of p by a whole warp (same SET as gen_legal, chess.cuh: the order differs, and nothing downstream depends on it).
// Lane l owns the pieces on squares 2 l and 2 l + 1; besides, lanes 0..7 own the king's steps, lanes 8 / 9 the en-passant capturers,
// lanes 10..17 castling with the rook on file l - 10.  Check / pin masks are computed by every lane (uniform, no communication).
// The moves land in `out` (shared memory) through one warp scan of the per-lane counts; returns their number (uniform).
__device__ __forceinline__ int gen_legal_warp(const Tables& T, const Pos& p, uint16_t* out, int lane) {
    const bool white = p.flags & F_WHITE;
    const uint64_t own = p.bb[white ? BB_WHITE : BB_BLACK], opp = p.bb[white ? BB_BLACK : BB_WHITE];
    const uint64_t occ = own | opp;
    const uint64_t P = p.bb[BB_P], N = p.bb[BB_N], B = p.bb[BB_B], R = p.bb[BB_R], Q = p.bb[BB_Q], K = p.bb[BB_K];
    const uint64_t kbb = K & own;
    if (!kbb) return 0;
    const int ksq = lsb(kbb);
    const uint64_t checkers = attackers_to(T, p.bb, ksq, occ) & opp;
    const bool dbl = (checkers & (checkers - 1)) != 0;              // double check: king moves only
    const uint64_t last = white ? RANK_8 : RANK_1;
    // ---- special duty of this lane: at most one move --------------------------------------------------------------------
    uint16_t special = MOVE_NONE;
    if (lane < 8) {
        uint64_t kt = T.king[ksq] & ~own;
        for (int j = 0; j < lane; j++) kt &= kt - 1;                  // the lane-th step of the king
        if (kt) {
            const int t = lsb(kt);
            if (!(attackers_to(T, p.bb, t, occ ^ kbb) & opp)) special = mk_move(ksq, t, 0);
        }
    } else if (lane < 10) {
        if (!dbl && p.ep >= 0 && !(occ & bit(p.ep))) {
            const uint64_t eb = bit(p.ep);
            uint64_t caps = (white ? wpawn_sources(eb) : bpawn_sources(eb)) & P & own & (white ? 0x000000FF00000000ull : 0x00000000FF000000ull);
            if (lane == 9) caps &= caps - 1;
            if (caps) {
                const int s = lsb(caps);
                const uint64_t victim = white ? (eb >> 8) : (eb << 8);
                const uint64_t occ2 = (occ ^ bit(s) ^ victim) | eb;
                if (!(attackers_to(T, p.bb, ksq, occ2) & opp & ~victim)) special = mk_move(s, p.ep, 0);
            }
        }
    } else if (lane < 18) {
        const uint8_t rights = white ? p.rights_w : p.rights_b;
        const int br = white ? 0 : 56, rf = lane - 10;
        if (!dbl && (rights & (1u << rf)) && (kbb & (0xFFull << br))) {
            const int rook = br + rf;
            const uint64_t rb = bit(rook);
            if (R & own & rb) {
                const bool a_side = rook < ksq;
                const int kto = br + (a_side ? 2 : 6), rto = br + (a_side ? 3 : 5);
                const uint64_t kpath = between(T, ksq, kto);
                const uint64_t must_empty = kpath | between(T, rook, rto) | bit(kto) | bit(rto);
                if (!((occ ^ kbb ^ rb) & must_empty)) {
                    uint64_t chk = kpath | kbb;
                    bool bad = false;
                    while (chk && !bad) {
                        const int sq = lsb(chk);
                        chk &= chk - 1;
                        bad = (attackers_to(T, p.bb, sq, occ ^ kbb) & opp) != 0;
                    }
                    if (!bad && !(attackers_to(T, p.bb, kto, occ ^ kbb ^ rb ^ bit(rto)) & opp)) special = mk_move(ksq, rook, 0);
                }
            }
        }
    }
    // ---- the two squares of this lane ---------------------------------------------------------------------------------------
    uint64_t tgt[2] = {0, 0};
    bool pawn[2] = {false, false};
    if (!dbl) {
        uint64_t target_mask = ~own;
        if (checkers) target_mask &= between(T, ksq, lsb(checkers)) | checkers;
        uint64_t pinned = 0;
        uint64_t snipers = (((rank_mask(ksq) | file_mask(ksq)) & (R | Q)) | ((T.diag[ksq] | T.anti[ksq]) & (B | Q))) & opp;
        while (snipers) {
            const int sn = lsb(snipers);
            snipers &= snipers - 1;
            const uint64_t b = between(T, ksq, sn) & occ;
            if (b && !(b & (b - 1)) && (b & own)) pinned |= b;
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int s = 2 * lane + h;
            const uint64_t sb = bit(s);
            if (!(own & sb) || (K & sb)) continue;
            uint64_t a = 0;
            if (N & sb) {
                if (!(pinned & sb)) a = T.knight[s] & target_mask;
            } else if (P & sb) {
                if (white) {
                    const uint64_t one = (sb << 8) & ~occ;
                    a = one | (((one << 8) & ~occ) & 0x00000000FF000000ull);
                    a |= (((sb << 7) & ~FILE_H) | ((sb << 9) & ~FILE_A)) & opp;
                } else {
                    const uint64_t one = (sb >> 8) & ~occ;
                    a = one | (((one >> 8) & ~occ) & 0x000000FF00000000ull);
                    a |= (((sb >> 7) & ~FILE_A) | ((sb >> 9) & ~FILE_H)) & opp;
                }
                a &= target_mask;
                if (pinned & sb) a &= line_through(T, ksq, s);
                pawn[h] = true;
            } else {
                if ((B | Q) & sb) a |= bishop_att(T, s, occ);
                if ((R | Q) & sb) a |= rook_att(s, occ);
                a &= target_mask;
                if (pinned & sb) a &= line_through(T, ksq, s);
            }
            tgt[h] = a;
        }
    }
    int mine = special != MOVE_NONE;
#pragma unroll
    for (int h = 0; h < 2; h++) mine += pawn[h] ? popc(tgt[h] & ~last) + 4 * popc(tgt[h] & last) : popc(tgt[h]);
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xFFFFFFFFu, incl, off);
        if (lane >= off) incl += y;
    }
    int at = incl - mine;
    if (special != MOVE_NONE) out[at++] = special;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        uint64_t a = tgt[h];
        const int s = 2 * lane + h;
        while (a) {
            const int t = lsb(a);
            a &= a - 1;
            if (pawn[h] && (bit(t) & last)) {
                out[at++] = mk_move(s, t, PT_QUEEN);
                out[at++] = mk_move(s, t, PT_ROOK);
                out[at++] = mk_move(s, t, PT_BISHOP);
                out[at++] = mk_move(s, t, PT_KNIGHT);
            } else {
                out[at++] = mk_move(s, t, 0);
            }
        }
    }
    return __shfl_sync(0xFFFFFFFFu, incl, 31);
}

// The 119 planes of `now` (pool slot qslot of game g) by nine lanes: lane t < 8 packs history step t, whose position it loads
// through the recorded predecessor slots (d.anc) -- eight independent loads instead of a walk along Pos::prev -- and lane 8 the
// seven constant planes.  Same planes as pack_planes (chess.cuh), the host harness's form: a step exists when every link up to
// it holds (predecessor recorded and exactly one ply older: a recycled ring slot breaks the chain).
__device__ __forceinline__ void pack_planes_warp(const Dev& d, int g, const Pos* gp, int qslot, const Pos& now, uint64_t* out, int lane) {
    const bool white = now.flags & F_WHITE;
    const int own = white ? BB_WHITE : BB_BLACK, opp = white ? BB_BLACK : BB_WHITE;
    Pos P = now;
    bool link = lane == 0;
    if (lane >= 1 && lane < 8) {
        const uint16_t A = d.anc[((size_t)g * d.pool_stride + qslot) * 8 + lane - 1];
        if (A != 0xFFFFu) { P = gp[A]; link = true; }
    }
    const int ply = link ? (int)P.ply : -7;
    const int ply_next = __shfl_up_sync(0xFFFFFFFFu, ply, 1);                 // the step nearer to `now`
    if (lane >= 1) link = link && (uint16_t)(ply + 1) == (uint16_t)ply_next && ply_next >= 0;
    const unsigned ok = __ballot_sync(0xFFFFFFFFu, link);
    const int steps = __ffs(~ok) - 1;                                         // trailing ones: steps 0 .. steps-1 exist
    if (lane < 8) {
        uint64_t* o = out + 14 * lane;
        if (lane < steps) {
#pragma unroll
            for (int k = 0; k < 6; k++) {
                o[k] = view_bb(P.bb[BB_P + k] & P.bb[own], white);
                o[6 + k] = view_bb(P.bb[BB_P + k] & P.bb[opp], white);
            }
            o[12] = (P.flags & F_REP2) ? ~0ull : 0ull;
            o[13] = (P.flags & F_REP3) ? ~0ull : 0ull;
        } else {
#pragma unroll
            for (int k = 0; k < 14; k++) o[k] = 0;
        }
    } else if (lane == 8) {
        const int cf = now.ply ? castling_flags(now) : 15;       // hard-coded ones before the first move (chess_tensor.py:82)
        const int ownc = white ? (cf & 3) : (cf >> 2), oppc = white ? (cf >> 2) : (cf & 3);
        out[112] = white ? ~0ull : 0ull;
        out[113] = now.ply ? ~0ull : 0ull;
        out[114] = (ownc & 1) ? ~0ull : 0ull;
        out[115] = (ownc & 2) ? ~0ull : 0ull;
        out[116] = (oppc & 1) ? ~0ull : 0ull;
        out[117] = (oppc & 2) ? ~0ull : 0ull;
        out[118] = (now.ply && now.halfmove) ? ~0ull : 0ull;
    }
}

// the legal moves mv[0 .. cnt) of p -> their policy indices in the 4672-bit mask (shared memory, zeroed by the caller), by a warp
__device__ __forceinline__ void mask_moves(const Pos& p, const uint16_t* mv, int cnt, uint64_t* mask, int lane) {
    for (int k = lane; k < cnt; k += 32) {
        const int idx = move_to_index(p, mv[k]);
        atomicOr(reinterpret_cast<unsigned long long*>(&mask[idx >> 6]), 1ull << (idx & 63));
    }
}

// legal indices (ascending) and/or planes + mask of the current positions.  Warp per game, with the search step's own code for
// moves, mask and planes (gen_legal_warp, mask_moves, pack_planes_warp): every szb_legal_moves / szb_encode call -- and every
// test built on them -- checks what a search feeds its evaluator.  Perft and szb_games_push use the one-thread move generation
// (gen_legal, chess.cuh).
__global__ void __launch_bounds__(128) k_games_encode(Dev d, int n, const int32_t* game, uint16_t* index_out, uint16_t* count_out,
                                                      uint64_t* planes_out, uint64_t* mask_out) {
    __shared__ Tables T;
    __shared__ Pos p_sh[4];
    __shared__ uint16_t mv_sh[4][MAX_MOVES];
    __shared__ uint64_t m_sh[4][MASK_STRIDE];
    load_tables(&T, d.tables);
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (i >= n) return;
    const int g = game ? game[i] : i;
    if (g < 0 || g >= d.n_games) { if (count_out && lane == 0) count_out[i] = 0; return; }
    const Pos* gp = d.pool + (size_t)g * d.pool_stride;
    const int qslot = d.cur[g];
    if (lane == 0) p_sh[wib] = gp[qslot];
    for (int w = lane; w < MASK_STRIDE; w += 32) m_sh[wib][w] = 0;
    __syncwarp();
    const Pos& p = p_sh[wib];
    const int cnt = gen_legal_warp(T, p, mv_sh[wib], lane);
    __syncwarp();
    mask_moves(p, mv_sh[wib], cnt, m_sh[wib], lane);
    __syncwarp();
    if (mask_out) for (int w = lane; w < MASK_WORDS; w += 32) mask_out[(size_t)i * MASK_WORDS + w] = m_sh[wib][w];
    if (lane == 0) {
        if (index_out) {
            int k = 0;
            for (int w = 0; w < MASK_WORDS; w++) {
                uint64_t x = m_sh[wib][w];
                while (x) { index_out[(size_t)i * SZB_MAX_MOVES + k++] = (uint16_t)(w * 64 + lsb(x)); x &= x - 1; }
            }
        }
        if (count_out) count_out[i] = (uint16_t)cnt;
    }
    if (planes_out) pack_planes_warp(d, g, gp, qslot, p, planes_out + (size_t)i * N_PLANES, lane);
}

// Expansion of path slot ps by its warp (mcts.py:57-70, chess_tensor.py:88-172,190-218): make the selected move, repetition
// flags, legal moves, outcome, the 4672-bit legal mask and the 119 planes.  Lane 0 makes the move, the whole warp generates the
// legal moves into shared memory, then the lanes share the rest -- policy indices of the moves into the shared-memory legal mask,
// history planes from eight independent position loads, coalesced copies out.  Returns whether the leaf needs the evaluator.
// K1 = true: the caller (k_tree_step) runs the reference-exact mode only, so the step kernel carries none of the multi-leaf mode's
// code; K1 = false: K is read from d -- the tree is order[ps / K], and with K > 1 k_select_vl numbers the new nodes and may have
// dropped the path.
struct ExpandShared {
    Pos q;
    uint16_t mv[MAX_MOVES];
    uint64_t mask[MASK_STRIDE];
    uint64_t planes[PLANE_STRIDE];
};
template <bool K1>
__device__ __forceinline__ bool expand_warp(const Dev& d, const Tables& T, int ps, int lane, ExpandShared& S, unsigned long long* tr = nullptr) {
    if (!K1 && d.sel_edge[ps] == PATH_DROPPED) {
        if (lane == 0) d.need_eval[ps] = 0;
        return false;
    }
    const int g = d.order[K1 ? ps : ps / d.K];
    const size_t r = (size_t)g * d.nodes_per_game;
    Pos* gp = d.pool + (size_t)g * d.pool_stride;
    for (int w = lane; w < MASK_STRIDE; w += 32) S.mask[w] = 0;
    // lane 0: the position the leaf stands for (a new node: the parent's position + the selected move; else the node's own)
    int qslot = 0, term = -1, node = 0, e = 0, parent = 0;      // term: -1 = not known yet (a new node)
    if (lane == 0) {
        e = d.sel_edge[ps];
        node = d.sel_node[ps];
        if (e >= 0) {
            parent = node;
            node = K1 || d.K == 1 ? ++d.node_count[g] : d.sel_new[ps];
            const int pslot = state_slot(d, g, parent);
            const Pos pp = gp[pslot];
            const uint16_t m = index_to_move(pp, d.e_move[e]);
            Pos q;
            make_move(T, pp, m, q);
            q.prev = (uint32_t)pslot;
            set_repetition_flags(gp, q);
            S.q = q;
            qslot = RING + node;
            set_ancestors(d, g, qslot, (uint32_t)pslot);
        } else {
            qslot = state_slot(d, g, node);
            S.q = gp[qslot];
            term = d.node_term[r + node];
        }
    }
    __syncwarp();                                              // lane 0's shared / global writes -> the other lanes
    if (tr) tr[4] = global_ns();
    term = __shfl_sync(0xFFFFFFFFu, term, 0);
    qslot = __shfl_sync(0xFFFFFFFFu, qslot, 0);
    // all lanes: legal moves into shared memory (a terminal node that already exists needs none), then the outcome
    int cnt = 0;
    if (term != 1) cnt = gen_legal_warp(T, S.q, S.mv, lane);
    __syncwarp();
    if (lane == 0) {
        if (e >= 0) {
            S.q.n_legal = (uint8_t)cnt;
            S.q.outcome = outcome_of(T, S.q, cnt);
            term = S.q.outcome != OUT_NONE;
            gp[qslot] = S.q;
            d.node_pedge[r + node] = e;
            d.node_pnode[r + node] = (uint16_t)parent;
            d.node_nchild[r + node] = 0;
            d.node_edge0[r + node] = -1;
            d.node_term[r + node] = (uint8_t)term;
            d.node_tval[r + node] = S.q.outcome == OUT_CHECKMATE ? -1.0f : 0.0f;
            d.e_link[e] = link_pack(-1, 0, (uint32_t)node);
            d.sel_node[ps] = node;
        }
        if (term) {
            d.leaf_value[ps] = d.node_tval[r + node];
            d.need_eval[ps] = 0;
        } else {
            d.need_eval[ps] = 1;
        }
    }
    __syncwarp();
    if (tr) tr[5] = global_ns();
    term = __shfl_sync(0xFFFFFFFFu, term, 0);
    if (term) return false;
    mask_moves(S.q, S.mv, cnt, S.mask, lane);
    pack_planes_warp(d, g, gp, qslot, S.q, S.planes, lane);
    __syncwarp();
    uint64_t* mrow = d.mask + (size_t)ps * MASK_STRIDE;
    for (int w = lane; w < MASK_STRIDE; w += 32) mrow[w] = S.mask[w];
    uint64_t* prow = d.planes + (size_t)ps * PLANE_STRIDE;
    for (int i = lane; i < N_PLANES; i += 32) prow[i] = S.planes[i];
    return true;
}

// warp per path slot: the expansion phase of a search that runs the phase kernels (profiling, the multi-leaf mode).  A path slot
// is one in-flight simulation: slot * K + j (K = leaves per tree and step; 1 in the reference-exact mode).
__global__ void __launch_bounds__(128) k_expand(Dev d) {
    __shared__ Tables T;
    __shared__ ExpandShared ex_sh[4];
    load_tables(&T, d.tables);
    const int ps = d.g_begin * d.K + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (ps >= d.g_end * d.K) return;
    expand_warp<false>(d, T, ps, threadIdx.x & 31, ex_sh[threadIdx.x >> 5]);
}

// block per tree: policy[i] / value from the integer hash of the packed planes.  EC (evaluation cache, fused step): block i serves
// compacted row g_begin + i while i is below the step's device count, and the row's slot (d.row_slot) addresses everything.
template <bool EC>
__global__ void __launch_bounds__(128) k_hash_eval(Dev d) {
    int ps = d.g_begin * d.K + blockIdx.x;
    if (EC) {
        if ((int)blockIdx.x >= d.ec_cnt[d.ec_par]) return;
        ps = d.row_slot[ps];
    }
    if (!d.need_eval[ps]) return;
    __shared__ uint64_t h_sh;
    if (threadIdx.x == 0) {
        h_sh = he_fold(d.planes + (size_t)ps * PLANE_STRIDE);
        d.value[ps] = he_value(h_sh);
    }
    __syncthreads();
    const uint64_t h = h_sh;
    float* pol = d.policy + (size_t)ps * N_ACTIONS;
    for (int i = threadIdx.x; i < N_ACTIONS; i += blockDim.x) pol[i] = he_policy(h, i);
}

// warp-cooperative pieces of the expansion (mcts.py:77-96, mctsnode.py:39-54), shared by k_finish and k_finish_vl
__device__ __forceinline__ int count_legal(const uint64_t* mk, int lane) {
    int n = 0;
    for (int w = lane; w < MASK_WORDS; w += 32) n += popc(mk[w]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) n += __shfl_xor_sync(0xFFFFFFFFu, n, off);
    return n;
}
// Children of the node evaluated in path slot ps (legal-move bitset mk, evaluator output pol), written from edge e0 on in ascending
// move-index order; returns how many (zero-prior moves are dropped, mcts.py:87-89).
//   1. the legal moves are compacted into shared memory (idx_sh / p_sh: index and evaluator output, ascending): the 73 mask words
//      are dealt to the lanes in three rounds, a warp scan places each lane's set bits, and ALL prior loads are in flight at once;
//   2. torch.sum's cascade order over the masked policy (tree.cuh): lane t adds the entries with index = t (mod 32) in ascending
//      order, closing a 16-step block when the next entry belongs to a later one -- cascade_lane_sparse on the compact list;
//   3. every lane normalises entries lane, lane + 32, ... and a ballot places the survivors;
//   4. the root of a search with exploration on (PRIOR_ROOT_NOISE) mixes Dirichlet noise into the survivors' priors (root_noise).
// How the priors of the expanded node are set: the normalised policy (learning == 0, and every non-root node when exploration is
// on), the reference's constant rule (learning != 0, exploration off), or the normalised policy mixed with the root's noise.
enum { PRIOR_RAW = 0, PRIOR_CONST = 1, PRIOR_ROOT_NOISE = 2 };
__device__ __forceinline__ int prior_rule(const Dev& d, int learning, int node) {
    if (!learning) return PRIOR_RAW;
    if (!(d.dir_alpha > 0.0f)) return PRIOR_CONST;
    return node == 0 ? PRIOR_ROOT_NOISE : PRIOR_RAW;
}
// The noise key of game g's root: (seed, global game id, the root position's ply).
__device__ __forceinline__ uint64_t root_noise_key(const Dev& d, int g) {
    return dir_root_key(d.dir_seed, d.game_id_base + (uint64_t)g, d.pool[(size_t)g * d.pool_stride + d.cur[g]].ply);
}
// Priors of the root's `count` children at e0 (ascending policy index) -> fl32((1 - eps) p + eps fl32(eta)), eta ~ Dir(alpha) over
// them (tree.cuh).  Lane t owns the children t, t + 32, ...; their log-gamma draws wait in e_w (these new edges' value sums, zeroed
// again at the end) between the passes.  Max and sum are reduced in a fixed order, so its host build (tests/host_harness/exploration.cpp) recomputes eta.
__device__ __forceinline__ void root_noise(const Dev& d, unsigned long long e0, int count, uint64_t key, int lane) {
    __syncwarp();                                            // the ballot pass wrote the children from other lanes
    double mx = -INFINITY;
    for (int k = lane; k < count; k += 32) {
        const double l = dir_log_gamma(key, d.e_move[e0 + k], (double)d.dir_alpha);
        d.e_w[e0 + k] = l;
        mx = fmax(mx, l);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mx = fmax(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, off));
    double part = 0.0;
    for (int k = lane; k < count; k += 32) part = d_add(part, exp(d_add(d.e_w[e0 + k], -mx)));
    const double total = dir_combine([&](int t) -> double { return __shfl_sync(0xFFFFFFFFu, part, t); });
    for (int k = lane; k < count; k += 32) {
        const double eta = exp(d_add(d.e_w[e0 + k], -mx)) / total;
        d.e_p[e0 + k] = dir_mix(d.e_p[e0 + k], d2f(eta), d.dir_eps);
        d.e_w[e0 + k] = 0.0;
    }
}
// EC (evaluation cache, k_tree_step<true>): hit != null takes the compacted evaluator output from a cache entry instead of pol
// (k-th legal move, ascending); ins != null copies the compacted output into the entry reserved for this leaf.
template <bool EC = false>
__device__ __forceinline__ int create_children(const Dev& d, const uint64_t* mk, const float* pol, unsigned long long e0, int rule,
                                               uint64_t noise_key, int lane, uint16_t* idx_sh, float* p_sh,
                                               const float* hit = nullptr, float* ins = nullptr) {
    int n = 0;
#pragma unroll 1
    for (int w = lane; w < 96; w += 32) {
        uint64_t x = w < MASK_WORDS ? mk[w] : 0ull;
        const int mine = popc(x);
        int incl = mine;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int y = __shfl_up_sync(0xFFFFFFFFu, incl, off);
            if (lane >= off) incl += y;
        }
        int at = n + incl - mine;
        while (x) {
            const int e = w * 64 + lsb(x);
            x &= x - 1;
            idx_sh[at] = (uint16_t)e;
            p_sh[at] = (EC && hit) ? hit[at] : pol[e];
            at++;
        }
        n += __shfl_sync(0xFFFFFFFFu, incl, 31);
    }
    __syncwarp();
    if (EC && ins)
        for (int k = lane; k < n; k += 32) ins[k] = p_sh[k];
    float a0 = 0.0f, a1 = 0.0f;
    int cur = 0;                                             // 16-step block the pending a0 belongs to
    for (int k = 0; k < n; k++) {
        const int e = idx_sh[k];
        if ((e & 31) != lane) continue;
        const int blk = e >> 9;                              // step e / 32, block step / 16
        if (blk != cur) { a1 = f_add(a1, a0); a0 = 0.0f; cur = blk; }
        a0 = f_add(a0, p_sh[k]);
    }
    if (cur < CASCADE_STEPS / 16) { a1 = f_add(a1, a0); a0 = 0.0f; }   // pending block was a complete one; the tail block stays in a0
    const float part = f_add(a0, a1);
    const float total = cascade_combine([&](int t) -> float { return __shfl_sync(0xFFFFFFFFu, part, t); });
    int count = 0;
    for (int k0 = 0; k0 < n; k0 += 32) {
        const int k = k0 + lane;
        float pr = 0.0f;
        bool has = false;
        if (k < n) { pr = f_div(p_sh[k], total); has = pr != 0.0f; }     // zero-prior children are dropped
        const unsigned ballot = __ballot_sync(0xFFFFFFFFu, has);
        if (has) {
            const unsigned long long at = e0 + (unsigned long long)(count + __popc(ballot & ((1u << lane) - 1)));
            d.e_n[at] = 0;
            d.e_w[at] = 0.0;
            d.e_p[at] = rule == PRIOR_CONST ? noisy_prior(pr) : pr;
            d.e_move[at] = idx_sh[k];
            d.e_link[at] = link_pack(-1, 0, NO_CHILD);
        }
        count += __popc(ballot);
    }
    if (rule == PRIOR_ROOT_NOISE) root_noise(d, e0, count, noise_key, lane);
    return count;
}

// Trees per block of the finish / tree-step kernels.  Two, not four: a block of k_tree_step must fit NEXT TO a tower CTA of the other
// cohort (k_tower_tc2 leaves ~9 KB of an SM's shared memory and half its registers), otherwise the tree kernel of one cohort cannot run
// under the other cohort's tower and every step pays it in full (measured: tower busy share 1.01 -> 0.976 with four trees and a 4 KB
// look-up table per block, i.e. 17 KB of shared memory).
constexpr int FINISH_WARPS = 2;

// Second half of a simulation for the block's four trees (mcts.py:77-109): children of the evaluated node, then backup.  Called by
// ALL threads of the block (two block-wide barriers inside); mk: 80 words of shared memory of this warp.
// EC (evaluation cache): a leaf that hit takes its evaluator output (compacted priors, value) from its cache entry; a leaf that
// missed with an entry reserved writes the evaluator's output there.  Everything after that runs on the same bits either way.
template <bool EC = false>
__device__ __forceinline__ void finish_block(const Dev& d, int learning, int slot, bool active, int lane, int wib, int* want_sh,
                                             unsigned long long* base_sh, uint64_t* mk, uint16_t* idx_sh, float* p_sh) {
    const int g = active ? d.order[slot] : 0;
    const bool eval = active && d.need_eval[slot];
    int ec_ent = -1;
    bool ec_hit = false;
    if (EC && eval) { ec_ent = d.ec_ent[slot]; ec_hit = d.ec_hit[slot] != 0; }
    const size_t ec_e = (size_t)g * d.ec_slots + (size_t)(ec_ent < 0 ? 0 : ec_ent);
    // Everything the backup needs is requested NOW, so that these round trips run under the mask -> arena bump -> priors chain
    // below instead of after it: the path, the statistics of its edges (only this warp touches them; the children created below
    // are new edges), the leaf's value, the root's sums.
    const size_t r = (size_t)g * d.nodes_per_game;
    const int node = active ? d.sel_node[slot] : 0;
    const int L = active ? d.path_len[slot] : 0;
    const bool fast = L <= PATH_CAP;
    const int32_t* path = d.path + (size_t)slot * PATH_CAP;
    const int pe0 = (fast && lane < L) ? path[lane] : -1, pe1 = (fast && lane + 32 < L) ? path[lane + 32] : -1;
    double w0 = 0.0, w1 = 0.0;
    int n0 = 0, n1 = 0;
    if (pe0 >= 0) { w0 = d.e_w[pe0]; n0 = d.e_n[pe0]; }
    if (pe1 >= 0) { w1 = d.e_w[pe1]; n1 = d.e_n[pe1]; }
    const float v = !active ? 0.f : (eval ? ((EC && ec_hit) ? d.ec_meta[ec_e].value : d.value[slot]) : d.leaf_value[slot]);
    double root_w = 0.0;
    int root_n = 0, pedge = -1;
    if (active && lane == 0) { root_w = d.root_w[g]; root_n = d.root_n[g]; pedge = d.node_pedge[r + node]; }
    // children to allocate: one bump of the shared edge arena per BLOCK (four trees), not one same-address atomic per tree
    int n_legal = 0;
    if (eval) {
        const uint64_t* src = d.mask + (size_t)slot * MASK_STRIDE;
        for (int w = lane; w < MASK_WORDS; w += 32) mk[w] = src[w];
        __syncwarp();
        n_legal = count_legal(mk, lane);
    }
    if (lane == 0) want_sh[wib] = n_legal;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int k = 0; k < FINISH_WARPS; k++) tot += want_sh[k];
        *base_sh = tot ? atomicAdd(d.edge_top, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    if (!active) return;
    int count = 0;
    if (eval) {
        unsigned long long e0 = *base_sh;
        for (int k = 0; k < wib; k++) e0 += (unsigned long long)want_sh[k];
        if (e0 + (unsigned long long)n_legal > d.edge_cap) {
            if (lane == 0) atomicExch(d.error_flag, SZB_ERR_ARENA);
        } else {
            const int rule = prior_rule(d, learning, node);
            float* ec_p = EC && ec_ent >= 0 ? d.ec_pri + ec_e * EC_PRI_STRIDE : nullptr;
            count = create_children<EC>(d, mk, d.policy + (size_t)slot * N_ACTIONS, e0, rule, rule == PRIOR_ROOT_NOISE ? root_noise_key(d, g) : 0ull,
                                        lane, idx_sh, p_sh, ec_hit ? ec_p : nullptr, ec_hit ? nullptr : ec_p);
            if (EC && ec_p && !ec_hit && lane == 0) {
                EcMeta m;
                m.k0 = d.ec_key[2 * (size_t)slot];
                m.k1 = d.ec_key[2 * (size_t)slot + 1];
                m.epoch = d.ec_epoch;
                m.gen = d.ec_gen;
                m.n_legal = (uint32_t)n_legal;
                m.value = v;
                d.ec_meta[ec_e] = m;
                d.ec_gstats[(size_t)g * 4 + 2] += 1ull;
            }
        }
        if (lane == 0) {
            d.node_edge0[r + node] = (int32_t)e0;
            d.node_nchild[r + node] = (uint16_t)count;
            if (pedge >= 0) d.e_link[pedge] = link_pack((int32_t)e0, (uint32_t)count, (uint32_t)node);     // the header select reads
            if (node == 0) d.root_val[g] = v;
        }
    }
    // backup (mctsnode.py:56-63): value_sum accumulates python doubles; the edge k levels above the leaf gets (-1)^k * value
    const double val = (double)v;
    if (fast) {
        if (pe0 >= 0) { d.e_w[pe0] = w0 + (((L - 1 - lane) & 1) ? -val : val); d.e_n[pe0] = n0 + 1; }
        if (pe1 >= 0) { d.e_w[pe1] = w1 + (((L - 1 - lane - 32) & 1) ? -val : val); d.e_n[pe1] = n1 + 1; }
    } else if (lane == 0) {
        double x = val;
        for (int nd = node;;) {
            const int pe = d.node_pedge[r + nd];
            if (pe < 0) break;
            d.e_w[pe] += x;
            d.e_n[pe] += 1;
            x = -x;
            nd = d.node_pnode[r + nd];
        }
    }
    if (lane == 0) {
        unsigned long long* gs = d.gstats + (size_t)g * 8;
        gs[6] += (unsigned long long)L;
        if (eval) gs[7] += (unsigned long long)count;
        d.root_w[g] = root_w + ((L & 1) ? -val : val);
        d.root_n[g] = root_n + 1;
        gs[0] += 1ull;
        gs[eval ? 1 : 2] += 1ull;
    }
}

// warp per tree
__global__ void __launch_bounds__(32 * FINISH_WARPS) k_finish(Dev d, int learning) {
    __shared__ int want_sh[FINISH_WARPS];
    __shared__ unsigned long long base_sh;
    __shared__ uint64_t mk_sh[FINISH_WARPS * MASK_STRIDE];
    __shared__ uint16_t idx_sh[FINISH_WARPS][MAX_MOVES];
    __shared__ float p_sh[FINISH_WARPS][MAX_MOVES];
    const int slot = d.g_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5), wib = threadIdx.x >> 5;
    finish_block(d, learning, slot, slot < d.g_end, threadIdx.x & 31, wib, want_sh, &base_sh, mk_sh + wib * MASK_STRIDE, idx_sh[wib], p_sh[wib]);
}

// Evaluation cache lookup (szb_set_eval_cache) of the non-terminal leaf in S (planes and legal mask in shared memory) by its warp;
// returns whether it hit.
//   key: lane l mixes the words l, l + 32, ... of (119 planes, 73 mask words) together with their index into two 64-bit wrapping
//        sums of independent mixes; the warp reduction of a sum does not depend on the order it combines in; the evaluator id is
//        mixed into the result.  The mask belongs to the key because the fused heads emit a softmax over the legal moves only and
//        the planes do not encode every legality detail (en passant).  Two different inputs share a key with probability ~2^-128
//        per comparison: the one accepted risk, as in a transposition table.
//   probe: lane i reads entry (h + i) mod S of game g's table, 32 entries in one round trip.  An entry is live while its epoch is
//        current and this search or the previous one wrote or hit it.  A hit refreshes the entry's generation; a miss reserves the
//        window's first dead entry for finish_block to fill in the next step (none: the insert is dropped).
//   Only game g's warp touches g's table, one leaf per step: no races, and the hits do not depend on slot, cohort or shard.
__device__ __forceinline__ bool ec_lookup(const Dev& d, int slot, int lane, const ExpandShared& S) {
    uint64_t a = 0, b = 0;
    for (int i = lane; i < N_PLANES + MASK_WORDS; i += 32) {
        const uint64_t x = (i < N_PLANES ? S.planes[i] : S.mask[i - N_PLANES]) + (uint64_t)(i + 1) * 0x9E3779B97F4A7C15ull;
        a += mix64(x);
        b += mix64(x ^ 0xD1B54A32D192ED03ull);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        a += __shfl_xor_sync(0xFFFFFFFFu, a, off);
        b += __shfl_xor_sync(0xFFFFFFFFu, b, off);
    }
    const uint64_t k0 = mix64(a ^ ((uint64_t)d.ec_eval << 56)), k1 = mix64(b + (uint64_t)d.ec_eval + 1ull);
    const int g = d.order[slot];
    const uint32_t wrap = (uint32_t)d.ec_slots - 1u, h = (uint32_t)(k0 >> 32);
    EcMeta* tab = d.ec_meta + (size_t)g * d.ec_slots;
    const EcMeta m = tab[(h + (uint32_t)lane) & wrap];
    const bool live = m.epoch == d.ec_epoch && d.ec_gen - m.gen <= 1u;
    const unsigned hit = __ballot_sync(0xFFFFFFFFu, live && m.k0 == k0 && m.k1 == k1);
    const unsigned dead = __ballot_sync(0xFFFFFFFFu, !live);
    const int first = __ffs(hit ? hit : dead) - 1;
    const int ent = first < 0 ? -1 : (int)((h + (uint32_t)first) & wrap);
    if (lane == 0) {
        d.ec_key[2 * (size_t)slot] = k0;
        d.ec_key[2 * (size_t)slot + 1] = k1;
        d.ec_ent[slot] = ent;
        d.ec_hit[slot] = hit != 0;
        unsigned long long* gs = d.ec_gstats + (size_t)g * 4;
        gs[0] += 1ull;
        if (hit) {
            tab[ent].gen = d.ec_gen;
            gs[1] += 1ull;
            d.ec_ghits[g] += 1u;
        } else if (ent < 0) {
            gs[3] += 1ull;
        }
    }
    return hit != 0;
}

// One launch per simulation step and cohort in the reference-exact mode: the second half of step s-1 (children + backup of the
// evaluated leaves), the first half of step s (PUCT descent, then move / legality / planes / mask of the new leaf) -- the same
// warp owns its tree through all of it -- and the hand-over to the network: the leaf's input planes are written straight into the
// tower's bf16 NHWC input rows and the tower's per-item completion counters are cleared, so a step is this kernel + one tower
// launch (k_tower_tc2, whose last layer's epilogue emits the priors and the value k_finish reads: net.cu).
// EC: the evaluation cache is consulted (a template parameter, so that the step without it keeps its 6.4 KB of shared memory and its
// registers): a leaf that hits takes no input row; a miss takes the next compacted row of its cohort (d.row_slot records its slot).
constexpr int STEP_FINISH = 1, STEP_SELECT = 2;
template <bool EC>
__global__ void __launch_bounds__(32 * FINISH_WARPS) k_tree_step(Dev d, float c_puct, int learning, int phases) {
    __shared__ Tables T;
    __shared__ int want_sh[FINISH_WARPS];
    __shared__ unsigned long long base_sh;
    __shared__ ExpandShared ex_sh[FINISH_WARPS];               // (its mask also stages the finish phase's legal mask: 6.4 KB per block)
    const int slot = d.g_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const bool active = slot < d.g_end;
    unsigned long long* tr = (d.step_trace && slot == d.g_begin && lane == 0) ? d.step_trace : nullptr;
    auto stamp = [&](int k) { if (tr) tr[k] = global_ns(); };
    pdl_trigger();                                             // the tower launch behind me may begin its set-up and weight prefetch
    if (phases & STEP_SELECT) load_tables(&T, d.tables);       // (constant tables: before the wait)
    pdl_wait();                                                // the evaluator's priors / values; its completion counters are idle now
    // the next step's row counter: its last reader, the evaluator of the step before this one, has completed (never zeroed by the
    // step that increments it, and no host memset inside the chain of programmatic dependent launches)
    // Before zeroing, the count it holds (the rows the previous step's evaluator ran on; 0 at step 0) goes into the cohort's running
    // total of evaluated boards (szb_eval_cache_stats.boards_evaluated).
    if (EC && blockIdx.x == 0 && threadIdx.x == 0) {
        *d.ec_boards += (unsigned long long)d.ec_cnt[d.ec_par ^ 1];
        d.ec_cnt[d.ec_par ^ 1] = 0;
    }
    stamp(0);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.net_ready_n; i += gridDim.x * blockDim.x) d.net_ready[i] = 0;
    stamp(1);
    if (phases & STEP_FINISH)      // (the expansion's shared memory is idle during the finish phase: mask, move list and planes serve as its scratch)
        finish_block<EC>(d, learning, slot, active, lane, wib, want_sh, &base_sh, ex_sh[wib].mask, ex_sh[wib].mv, reinterpret_cast<float*>(ex_sh[wib].planes));
    if (!(phases & STEP_SELECT) || !active) return;
    __syncwarp();                                              // this warp's tree updates -> every lane of the descent
    stamp(2);
    select_tree(d, slot, lane, c_puct);
    __syncwarp();
    stamp(3);
    ExpandShared& S = ex_sh[wib];
    if (!expand_warp<true>(d, T, slot, lane, S, tr)) return;
    stamp(6);
    int row = slot;
    if (EC) {
        if (ec_lookup(d, slot, lane, S)) return;
        // Rows are handed out in whatever order the warps get here, so a leaf's row is not deterministic; its results are, because
        // a board's evaluation does not depend on its row, its batch or its neighbours (DESIGN.md 3).
        if (lane == 0) {
            row = d.g_begin + atomicAdd(d.ec_cnt + d.ec_par, 1);
            d.row_slot[row] = slot;
        }
        row = __shfl_sync(0xFFFFFFFFu, row, 0);
    }
    const uint64_t* pl = S.planes;
    if (d.net_in16) {
        // 64 squares x 128 channels of bf16 (0 / 1.0) into the interior of the slot's zero-haloed [10][10][128] input row.  A lane takes
        // an 8-plane x 8-square block (channel group cg, board row r): the planes' bytes of that row, an 8 x 8 bit transpose, and
        // every byte of the result is one square's 8 channels -> one 16-byte store through a 256-entry table (byte -> 8 bf16, 4 KB in
        // global memory: L1-resident, and not part of the block's shared-memory footprint).
        // Lanes 0..15 / 16..31 write two squares' 256 contiguous bytes per store.
        uint4* in = reinterpret_cast<uint4*>(d.net_in16 + (size_t)row * 100 * 128);
        const int cg = lane & 15;
#pragma unroll
        for (int it = 0; it < 4; it++) {
            const int r = it * 2 + (lane >> 4);
            uint64_t x = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int c = cg * 8 + j;
                if (c < N_PLANES) x |= ((pl[c] >> (8 * r)) & 0xFFull) << (8 * j);
            }
            uint64_t t = (x ^ (x >> 7)) & 0x00AA00AA00AA00AAull;
            x ^= t ^ (t << 7);
            t = (x ^ (x >> 14)) & 0x0000CCCC0000CCCCull;
            x ^= t ^ (t << 14);
            t = (x ^ (x >> 28)) & 0x00000000F0F0F0F0ull;
            x ^= t ^ (t << 28);
#pragma unroll
            for (int i = 0; i < 8; i++) in[(size_t)((r + 1) * 10 + i + 1) * 16 + cg] = __ldg(d.lut_bf16 + ((x >> (8 * i)) & 0xFFull));
        }
    }
    stamp(7);
}

// ------------------------------------------------------------------------------------------------
// multi-leaf mode (szb_config.leaves_per_tree = K > 1): K simulations of a tree in flight per step, kept apart by virtual loss.
// A DIFFERENT ALGORITHM from the reference's one-simulation-at-a-time search (different visit counts): opt-in, for the
// latency-bound regime of few games (interactive play, arena, the tail of a self-play iteration), never used by the parity tests
// or the benchmark.  Deterministic: one warp walks a tree's K paths one after the other, one thread backs them up in order.
// ------------------------------------------------------------------------------------------------
// warp per tree.  Every edge of an in-flight path carries a virtual visit that counts as a loss for the side choosing it
// (N + 1, W + 1: the child's value sum is from the child's mover's view), so later paths of the step look elsewhere.  A path that
// runs into a node still being created by an earlier path of the step is dropped (its virtual loss taken back).
__global__ void __launch_bounds__(128) k_select_vl(Dev d, float c_puct, int num_searches) {
    const int slot = d.g_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (slot >= d.g_end) return;
    const int g = d.order[slot];
    const size_t r = (size_t)g * d.nodes_per_game;
    const int budget = num_searches - d.sims_done[g];
    const int nc = d.node_count[g];
    int new_nodes = 0, inflight = 0, max_depth = 0;
    bool root_pending = false;
    unsigned long long scanned = 0, levels = 0;
    for (int j = 0; j < d.K; j++) {
        const int ps = slot * d.K + j;
        if (inflight >= budget) {
            if (lane == 0) d.sel_edge[ps] = PATH_DROPPED;
            continue;
        }
        int node = 0, depth = 0;
        int np = d.root_n[g] + inflight;
        bool dropped = false;
        for (;;) {
            const int n = d.node_nchild[r + node];
            const int e0 = d.node_edge0[r + node];
            if (n == 0) {
                // a node without children that already exists: a terminal node, or the root before its first expansion
                if (!d.node_term[r + node]) {
                    if (root_pending) { dropped = true; break; }
                    root_pending = true;
                }
                if (lane == 0) { d.sel_node[ps] = node; d.sel_edge[ps] = -1; }
                break;
            }
            // (only the pick: the headers come from node_nchild / node_edge0, because k_finish_vl does not keep e_link's up to date)
            unsigned long long lk;
            const int e = e0 + puct_pick(d, e0, n, sqrt_parent(np), c_puct, lane, np, lk);
            const uint16_t c = link_child(lk);
            depth++;
            scanned += (unsigned long long)n;
            if (c == CHILD_PENDING) { dropped = true; break; }
            if (lane == 0) {
                d.e_n[e] += 1;                                   // virtual visit ...
                d.e_w[e] += 1.0;                                 // ... lost by the side that chose this edge
                if (c == NO_CHILD) {
                    d.e_link[e] = link_pack(-1, 0, CHILD_PENDING);
                    d.sel_node[ps] = node;
                    d.sel_edge[ps] = e;
                    d.sel_new[ps] = nc + 1 + new_nodes;
                }
            }
            __syncwarp();
            if (c == NO_CHILD) { new_nodes++; break; }
            node = c;
        }
        if (dropped) {
            if (lane == 0) {
                d.sel_edge[ps] = PATH_DROPPED;
                for (int nd = node;;) {                          // take the virtual loss of this path back
                    const int pe = d.node_pedge[r + nd];
                    if (pe < 0) break;
                    d.e_n[pe] -= 1;
                    d.e_w[pe] -= 1.0;
                    nd = d.node_pnode[r + nd];
                }
            }
            __syncwarp();
            continue;
        }
        inflight++;
        levels += (unsigned long long)depth;
        max_depth = depth > max_depth ? depth : max_depth;
    }
    if (lane == 0) {
        d.node_count[g] = nc + new_nodes;
        unsigned long long* gs = d.gstats + (size_t)g * 8;
        if ((unsigned long long)max_depth > gs[3]) gs[3] = (unsigned long long)max_depth;
        gs[4] += scanned;
        gs[5] += levels;
    }
}

// block per tree, warp j = path j: expansions in parallel, then one thread backs the paths up in order (the virtual loss of an edge
// becomes the real result: N keeps its + 1, W gets value - 1)
__global__ void __launch_bounds__(32 * MAX_LEAVES) k_finish_vl(Dev d, int learning) {
    __shared__ int want_sh[MAX_LEAVES];
    __shared__ uint16_t idx_vl[MAX_LEAVES][MAX_MOVES];
    __shared__ float p_vl[MAX_LEAVES][MAX_MOVES];
    __shared__ unsigned long long base_sh;
    const int slot = d.g_begin + blockIdx.x;
    const int lane = threadIdx.x & 31, j = threadIdx.x >> 5;
    const int g = d.order[slot];
    const size_t r = (size_t)g * d.nodes_per_game;
    const int ps = slot * d.K + j;
    const bool live = j < d.K && d.sel_edge[ps] != PATH_DROPPED;
    const bool eval = live && d.need_eval[ps];
    const uint64_t* mk = d.mask + (size_t)ps * MASK_STRIDE;
    const int n_legal = eval ? count_legal(mk, lane) : 0;
    if (lane == 0) want_sh[j] = n_legal;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int k = 0; k < MAX_LEAVES; k++) tot += want_sh[k];
        base_sh = tot ? atomicAdd(d.edge_top, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    if (eval) {
        const int node = d.sel_node[ps];
        unsigned long long e0 = base_sh;
        for (int k = 0; k < j; k++) e0 += (unsigned long long)want_sh[k];
        int count = 0;
        if (e0 + (unsigned long long)n_legal > d.edge_cap) {
            if (lane == 0) atomicExch(d.error_flag, SZB_ERR_ARENA);
        } else {
            const int rule = prior_rule(d, learning, node);
            count = create_children(d, mk, d.policy + (size_t)ps * N_ACTIONS, e0, rule, rule == PRIOR_ROOT_NOISE ? root_noise_key(d, g) : 0ull,
                                    lane, idx_vl[j], p_vl[j]);
        }
        if (lane == 0) {
            d.node_edge0[r + node] = (int32_t)e0;
            d.node_nchild[r + node] = (uint16_t)count;
            if (node == 0) d.root_val[g] = d.value[ps];
        }
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    unsigned long long* gs = d.gstats + (size_t)g * 8;
    int done = 0;
    for (int k = 0; k < d.K; k++) {
        const int pk = slot * d.K + k;
        if (d.sel_edge[pk] == PATH_DROPPED) continue;
        const bool ev = d.need_eval[pk];
        const int node = d.sel_node[pk];
        double val = (double)(ev ? d.value[pk] : d.leaf_value[pk]);
        unsigned long long levels = 0;
        for (int nd = node;;) {
            const int pe = d.node_pedge[r + nd];
            if (pe < 0) break;
            d.e_w[pe] += val - 1.0;
            val = -val;
            nd = d.node_pnode[r + nd];
            levels++;
        }
        d.root_w[g] += val;
        gs[6] += levels;
        if (ev) gs[7] += (unsigned long long)d.node_nchild[r + node];
        gs[ev ? 1 : 2] += 1ull;
        done++;
    }
    d.root_n[g] += done;
    d.sims_done[g] += done;
    gs[0] += (unsigned long long)done;
}

// fewest simulations completed over the slots of this search.  One block.
__global__ void __launch_bounds__(256) k_min_done(Dev d, int n_slots, int32_t* out) {
    __shared__ int part[256];
    int m = 0x7FFFFFFF;
    for (int i = threadIdx.x; i < n_slots; i += 256) m = min(m, d.sims_done[d.order[i]]);
    part[threadIdx.x] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 256; i++) m = min(m, part[i]);
        *out = m;
    }
}

// per-game counter rows -> totals (sum, except max depth); rows are cleared.  One block.
__global__ void __launch_bounds__(256) k_fold_stats(Dev d, int n_games) {
    __shared__ unsigned long long part[256][8];
    unsigned long long acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int g = threadIdx.x; g < n_games; g += 256) {
        unsigned long long* gs = d.gstats + (size_t)g * 8;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const unsigned long long v = gs[k];
            acc[k] = k == 3 ? (v > acc[k] ? v : acc[k]) : acc[k] + v;
            gs[k] = 0;
        }
    }
#pragma unroll
    for (int k = 0; k < 8; k++) part[threadIdx.x][k] = acc[k];
    __syncthreads();
    if (threadIdx.x < 8) {
        const int k = threadIdx.x;
        unsigned long long t = 0;
        for (int i = 0; i < 256; i++) t = k == 3 ? (part[i][k] > t ? part[i][k] : t) : t + part[i][k];
        if (k == 3) { if (t > d.stats[3]) d.stats[3] = t; } else d.stats[k] += t;
    }
}

__global__ void k_collect(Dev d, uint32_t* visits, uint64_t* child_mask, float* root_value) {
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= d.n_games) return;
    const size_t r = (size_t)g * d.nodes_per_game;
    if (visits) for (int i = lane; i < N_ACTIONS; i += 32) visits[(size_t)g * N_ACTIONS + i] = 0;
    if (child_mask) for (int i = lane; i < MASK_WORDS; i += 32) child_mask[(size_t)g * MASK_WORDS + i] = 0;
    __syncwarp();
    const int n = d.node_nchild[r], e0 = d.node_edge0[r];
    for (int i = lane; i < n; i += 32) {
        const int idx = d.e_move[e0 + i];
        if (visits) visits[(size_t)g * N_ACTIONS + idx] = (uint32_t)d.e_n[e0 + i];
        if (child_mask) atomicOr((unsigned long long*)&child_mask[(size_t)g * MASK_WORDS + (idx >> 6)], 1ull << (idx & 63));
    }
    if (root_value && lane == 0) root_value[g] = d.node_term[r] ? d.node_tval[r] : d.root_val[g];
}

// compact root children: index / visits / count per game
__global__ void k_root_children(Dev d, uint16_t* index, uint32_t* visits, uint16_t* count) {
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= d.n_games) return;
    const size_t r = (size_t)g * d.nodes_per_game;
    const int n = d.node_nchild[r], e0 = d.node_edge0[r];
    for (int i = lane; i < SZB_MAX_MOVES; i += 32) {
        index[(size_t)g * SZB_MAX_MOVES + i] = i < n ? d.e_move[e0 + i] : 0;
        visits[(size_t)g * SZB_MAX_MOVES + i] = i < n ? (uint32_t)d.e_n[e0 + i] : 0u;
    }
    if (lane == 0) count[g] = (uint16_t)n;
}

// gather one game's tree into contiguous arrays (inspection path; one warp)
__global__ void k_tree_export(Dev d, int g, int max_nodes, int max_edges, int32_t* node_first, int32_t* node_count,
                              int32_t* node_parent, int32_t* node_pedge, uint8_t* node_term, float* node_tval,
                              int32_t* e_n, double* e_w, float* e_p, uint16_t* e_move, int32_t* e_child, int32_t* totals) {
    const int lane = threadIdx.x;
    const size_t r = (size_t)g * d.nodes_per_game;
    const int n_nodes = d.node_count[g] + 1;
    int off = 0;
    bool overflow = n_nodes > max_nodes;
    for (int i = 0; i < n_nodes && !overflow; i++) {
        const int n = d.node_nchild[r + i], e0 = d.node_edge0[r + i];
        if (off + n > max_edges) { overflow = true; break; }
        if (lane == 0) {
            node_first[i] = off; node_count[i] = n;
            node_parent[i] = i == 0 ? -1 : (int)d.node_pnode[r + i];
            node_pedge[i] = -1;                       // patched below once the parent's range is known
            node_term[i] = d.node_term[r + i]; node_tval[i] = d.node_tval[r + i];
        }
        for (int k = lane; k < n; k += 32) {
            e_n[off + k] = d.e_n[e0 + k]; e_w[off + k] = d.e_w[e0 + k]; e_p[off + k] = d.e_p[e0 + k];
            e_move[off + k] = d.e_move[e0 + k];
            const uint16_t c = link_child(d.e_link[e0 + k]);
            e_child[off + k] = c == NO_CHILD ? -1 : (int)c;
        }
        off += n;
    }
    __syncwarp();
    if (!overflow)
        for (int i = 1 + lane; i < n_nodes; i += 32) {
            const int pn = d.node_pnode[r + i];
            node_pedge[i] = node_first[pn] + (d.node_pedge[r + i] - d.node_edge0[r + pn]);
        }
    if (lane == 0) { totals[0] = overflow ? -1 : n_nodes; totals[1] = off; totals[2] = d.root_n[g]; }
}

// choose a move from the root visit counts (sim.py:68 sampling, or arg-max first-index as in eval.py:92-100); with sample_plies > 0
// sampling stops at that ply of the game (szb_exploration)
__global__ void k_pick(Dev d, uint64_t seed, int sample, int sample_plies, int32_t* moves) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= d.n_games) return;
    const size_t r = (size_t)g * d.nodes_per_game;
    const int n = d.node_nchild[r], e0 = d.node_edge0[r];
    const Pos& p = d.pool[(size_t)g * d.pool_stride + d.cur[g]];
    if (p.outcome != OUT_NONE || n == 0) { moves[g] = -1; return; }
    long long total = 0;
    for (int i = 0; i < n; i++) total += d.e_n[e0 + i];
    int pick = 0;
    if (sample && (sample_plies == 0 || p.ply < sample_plies) && total > 0) {
        const uint64_t rnd = mix64(mix64(seed ^ (0x9E3779B97F4A7C15ull * (d.game_id_base + (uint64_t)g + 1))) + (uint64_t)p.ply);
        const long long target = (long long)__umul64hi(rnd, (uint64_t)total);      // uniform in [0, total)
        long long acc = 0;
        for (int i = 0; i < n; i++) { acc += d.e_n[e0 + i]; if (acc > target) { pick = i; break; } }
    } else {
        int best = -1;
        for (int i = 0; i < n; i++) if (d.e_n[e0 + i] > best) { best = d.e_n[e0 + i]; pick = i; }
    }
    moves[g] = d.e_move[e0 + pick];
}

__global__ void k_push_picked(Dev d, const int32_t* moves, int32_t* n_active) {
    __shared__ Tables T;
    load_tables(&T, d.tables);
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= d.n_games) return;
    if (moves[g] < 0) return;
    Pos* gp = d.pool + (size_t)g * d.pool_stride;
    const Pos p = gp[d.cur[g]];
    const uint16_t m = index_to_move(p, moves[g]);
    Pos q;
    make_move(T, p, m, q);
    q.prev = (uint32_t)d.cur[g];
    set_repetition_flags(gp, q);
    uint16_t mv[MAX_MOVES];
    int cnt;
    analyse(T, q, mv, cnt);
    const int slot = q.ply & (RING - 1);
    gp[slot] = q;
    set_ancestors(d, g, slot, q.prev);
    d.cur[g] = slot;
    if (q.outcome == OUT_NONE) atomicAdd(n_active, 1);
}

// ------------------------------------------------------------------------------------------------
// perft: breadth-first expansion with bulk counting at the last ply
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_perft_count(const Tables* tables, const Pos* in, size_t n, unsigned long long* total) {
    __shared__ Tables T;
    load_tables(&T, tables);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int cnt = 0;
    if (i < n) {
        uint16_t mv[MAX_MOVES];
        cnt = gen_legal(T, in[i], mv);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, off);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(total, (unsigned long long)cnt);
}

__global__ void __launch_bounds__(128) k_perft_expand(const Tables* tables, const Pos* in, size_t n, Pos* out, unsigned long long* top) {
    __shared__ Tables T;
    load_tables(&T, tables);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    uint16_t mv[MAX_MOVES];
    int cnt = 0;
    Pos p;
    if (i < n) { p = in[i]; cnt = gen_legal(T, p, mv); }
    int incl = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int y = __shfl_up_sync(0xFFFFFFFFu, incl, off);
        if (lane >= off) incl += y;
    }
    unsigned long long base = 0;
    if (lane == 31) base = atomicAdd(top, (unsigned long long)incl);
    base = __shfl_sync(0xFFFFFFFFu, base, 31) + (unsigned long long)(incl - cnt);
    for (int k = 0; k < cnt; k++) {
        Pos q;
        make_move(T, p, mv[k], q);
        q.prev = NO_PREV;
        out[base + k] = q;
    }
}

static uint64_t perft_rec(szb_ctx* ctx, const Pos* front, size_t n, int depth, int level, cudaError_t* err,
                          float* ms_last, uint64_t* n_last) {
    if (*err != cudaSuccess || n == 0) return 0;
    cudaStream_t st = ctx->stream;
    unsigned long long total = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (depth == 1 && ms_last) { cudaEventCreate(&e0); cudaEventCreate(&e1); }
    cudaMemsetAsync(ctx->perft_counter, 0, sizeof(unsigned long long), st);
    if (e0) cudaEventRecord(e0, st);
    k_perft_count<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(ctx->d.tables, front, n, ctx->perft_counter);
    if (e0) cudaEventRecord(e1, st);
    ctx->launches++;
    cudaMemcpyAsync(&total, ctx->perft_counter, sizeof total, cudaMemcpyDeviceToHost, st);
    *err = cudaStreamSynchronize(st);
    if (*err != cudaSuccess) return 0;
    if (e0) {
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (n >= *n_last) { *ms_last = ms; *n_last = n; }
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    if (depth == 1) return total;
    if (total > ctx->perft_cap) {
        if (n == 1) { *err = cudaErrorMemoryAllocation; return 0; }
        size_t h = n / 2;
        return perft_rec(ctx, front, h, depth, level, err, ms_last, n_last) +
               perft_rec(ctx, front + h, n - h, depth, level, err, ms_last, n_last);
    }
    while ((int)ctx->perft_levels.size() <= level + 1) ctx->perft_levels.push_back(nullptr);
    if (!ctx->perft_levels[level + 1]) {
        *err = cudaMalloc((void**)&ctx->perft_levels[level + 1], ctx->perft_cap * sizeof(Pos));
        if (*err != cudaSuccess) return 0;
    }
    Pos* next = ctx->perft_levels[level + 1];
    cudaMemsetAsync(ctx->perft_counter, 0, sizeof(unsigned long long), st);
    k_perft_expand<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(ctx->d.tables, front, n, next, ctx->perft_counter);
    ctx->launches++;
    return perft_rec(ctx, next, (size_t)total, depth - 1, level + 1, err, ms_last, n_last);
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
static void pos_from_wire(const szb_pos& w, Pos& p) {
    memset(&p, 0, sizeof p);
    for (int t = 0; t < 6; t++) {
        p.bb[BB_P + t] = w.pieces[t] | w.pieces[6 + t];
        p.bb[BB_WHITE] |= w.pieces[t];
        p.bb[BB_BLACK] |= w.pieces[6 + t];
    }
    p.flags = (uint8_t)((w.turn ? F_WHITE : 0) | (w.chess960 ? F_960 : 0));
    p.rights_w = w.castling_w; p.rights_b = w.castling_b;
    p.ep = w.ep_square;
    p.halfmove = (uint8_t)std::min<int>(w.halfmove_clock, 250);
    p.ply = w.ply;
    p.prev = NO_PREV;
}

extern "C" {

const char* szb_version(void) { return "szb200 0.1 (sm_100a)"; }

const char* szb_last_error(const szb_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

void* szb_stream(szb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int szb_synchronize(szb_ctx* ctx) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

void szb_destroy(szb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    trainer_destroy(ctx);
    net_destroy(ctx);
    for (void* p : ctx->allocs) cudaFree(p);
    for (cudaEvent_t e : ctx->prof_events) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->conv_events) cudaEventDestroy(e);
    for (Pos* p : ctx->perft_levels) if (p) cudaFree(p);
    if (ctx->perft_counter) cudaFree(ctx->perft_counter);
    if (ctx->stage) cudaFree(ctx->stage);
    if (ctx->ec_mem) cudaFree(ctx->ec_mem);
    for (int c = 0; c < 2; c++) {
        if (ctx->cohort_stream[c]) cudaStreamDestroy(ctx->cohort_stream[c]);
        if (ctx->ev_join[c]) cudaEventDestroy(ctx->ev_join[c]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int szb_create(int device, const szb_config* cfg, szb_ctx** out) {
    if (!out || !cfg || cfg->max_games <= 0 || cfg->max_searches <= 0 || cfg->max_searches > 65000) return SZB_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return SZB_ERR_CUDA;
    szb_ctx* ctx = new szb_ctx();
    ctx->device = device;
    ctx->cfg = *cfg;
    if (ctx->cfg.edges_per_node <= 0) ctx->cfg.edges_per_node = 48;
    *out = ctx;        // returned even on failure so the caller can read the message, then destroy
    SZB_CUDA(ctx, cudaSetDevice(device));
    SZB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->work = ctx->stream;
    for (int c = 0; c < 2; c++) {
        SZB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->cohort_stream[c], cudaStreamNonBlocking));
        SZB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_join[c], cudaEventDisableTiming));
    }
    SZB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    ctx->cohorts = cfg->cohorts;
    if (cfg->leaves_per_tree < 0 || cfg->leaves_per_tree > MAX_LEAVES)
        return fail(ctx, SZB_ERR_ARG, "szb_config.leaves_per_tree must be 0 / 1 (the reference's algorithm) or 2..%d", MAX_LEAVES);
    if (ctx->cohorts < 0 || ctx->cohorts > 2) return fail(ctx, SZB_ERR_ARG, "szb_config.cohorts must be 0 (automatic), 1 or 2");
    if (const char* e = getenv("SZB_COHORTS")) { if (e[0] == '1' || e[0] == '2') ctx->cohorts = e[0] - '0'; }   // measurement aid
    Dev& d = ctx->d;
    const size_t G = (size_t)cfg->max_games;
    d.K = cfg->leaves_per_tree > 1 ? cfg->leaves_per_tree : 1;
    d.nodes_per_game = cfg->max_searches + 1;
    d.pool_stride = RING + d.nodes_per_game + 1;
    d.n_games = 0;
    const size_t NN = G * (size_t)d.nodes_per_game;
    d.edge_cap = (unsigned long long)NN * (unsigned long long)ctx->cfg.edges_per_node;
    // edges are addressed with 32-bit indices everywhere (node_edge0, node_pedge, path, e_link)
    if (d.edge_cap > 0x7FFFFFFFull)
        return fail(ctx, SZB_ERR_ARG, "tree arena of %llu edges (max_games x (max_searches + 1) x edges_per_node) exceeds the 2^31 - 1 edges "
                    "a context can index: lower max_games / edges_per_node or use one context per game block", d.edge_cap);
    build_tables(ctx->host_tables);
    Tables* dt = nullptr;
    int rc;
    if ((rc = dev_alloc(ctx, &dt, 1))) return rc;
    SZB_CUDA(ctx, cudaMemcpyAsync(dt, &ctx->host_tables, sizeof(Tables), cudaMemcpyHostToDevice, ctx->stream));
    d.tables = dt;
    {
        // byte -> eight bf16 (bit ? 1.0 : 0): the table k_tree_step expands the input planes with
        std::vector<uint32_t> lut(256 * 4);
        for (int b = 0; b < 256; b++)
            for (int k = 0; k < 4; k++) lut[b * 4 + k] = (((b >> (2 * k)) & 1) ? 0x3F80u : 0u) | (((b >> (2 * k + 1)) & 1) ? 0x3F800000u : 0u);
        uint4* dl = nullptr;
        if ((rc = dev_alloc(ctx, &dl, 256))) return rc;
        SZB_CUDA(ctx, cudaMemcpyAsync(dl, lut.data(), 256 * sizeof(uint4), cudaMemcpyHostToDevice, ctx->stream));
        SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        d.lut_bf16 = dl;
    }
#define A(field, count) if ((rc = dev_alloc(ctx, &d.field, (count)))) return rc
    A(pool, G * (size_t)d.pool_stride);
    A(cur, G); A(anc, G * (size_t)d.pool_stride * 8);
    A(node_edge0, NN); A(node_nchild, NN); A(node_pedge, NN); A(node_pnode, NN); A(node_term, NN); A(node_tval, NN);
    A(node_count, G); A(root_n, G); A(root_w, G);
    A(e_n, d.edge_cap); A(e_w, d.edge_cap); A(e_p, d.edge_cap); A(e_move, d.edge_cap); A(e_link, d.edge_cap);
    A(edge_top, 1); A(error_flag, 1);
    const size_t P = G * (size_t)d.K;                       // path slots
    A(sel_node, P); A(sel_edge, P); A(sel_new, P); A(need_eval, P); A(leaf_value, P);
    A(path, G * PATH_CAP); A(path_len, G);
    A(order, G); A(n_active, 1); A(sims_done, G);
    A(planes, P * PLANE_STRIDE); A(mask, P * MASK_STRIDE);
    A(policy, P * N_ACTIONS); A(value, P); A(root_val, G);
    A(stats, 8); A(gstats, G * 8);
    // evaluation cache bookkeeping (small; the tables themselves come with szb_set_eval_cache)
    A(ec_key, G * 2); A(ec_ent, G); A(ec_hit, G); A(row_slot, G); A(ec_cnt, 4); A(ec_boards, 2); A(ec_gstats, G * 4); A(ec_ghits, G);
#undef A
    if ((rc = dev_alloc(ctx, &ctx->d_moves, G + 1))) return rc;
    SZB_CUDA(ctx, cudaMalloc((void**)&ctx->perft_counter, sizeof(unsigned long long)));
    ctx->perft_cap = (size_t)4 << 20;      // positions per breadth-first level buffer (384 MiB)
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int games_upload(szb_ctx* ctx, int n, const std::vector<Pos>& start) {
    Dev& d = ctx->d;
    Pos* st = (Pos*)ctx_stage(ctx, sizeof(Pos) * (size_t)n);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    SZB_CUDA(ctx, cudaMemcpyAsync(st, start.data(), sizeof(Pos) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    d.n_games = n;
    k_games_init<<<(n + 31) / 32, 32, 0, ctx->stream>>>(d, st, n);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int szb_games_reset(szb_ctx* ctx, int32_t n, const int16_t* start_id) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || n <= 0 || n > ctx->cfg.max_games) return fail(ctx, SZB_ERR_ARG, "szb_games_reset: n_games out of range");
    std::vector<Pos> start((size_t)n);
    for (int g = 0; g < n; g++) {
        int id = start_id ? start_id[g] : -1;
        if (id > 959) return fail(ctx, SZB_ERR_ARG, "chess960 position index not 0 <= %d <= 959", id);
        memset(&start[g], 0, sizeof(Pos));
        start_position(ctx->host_tables, id, start[g]);
    }
    return games_upload(ctx, n, start);
}

int szb_games_set(szb_ctx* ctx, int32_t n, const szb_pos* positions) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !positions || n <= 0 || n > ctx->cfg.max_games) return fail(ctx, SZB_ERR_ARG, "szb_games_set: bad arguments");
    std::vector<Pos> start((size_t)n);
    for (int g = 0; g < n; g++) pos_from_wire(positions[g], start[g]);
    return games_upload(ctx, n, start);
}

int szb_games_push(szb_ctx* ctx, int32_t n, const int32_t* game, const uint16_t* move_index, int32_t* status) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || n <= 0 || !move_index) return fail(ctx, SZB_ERR_ARG, "szb_games_push: bad arguments");
    if (ctx->d.n_games == 0) return fail(ctx, SZB_ERR_STATE, "no games");
    const size_t bytes = (size_t)n * (4 + 2 + 4) + 64;
    char* st = (char*)ctx_stage(ctx, bytes);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    int32_t* d_status = (int32_t*)st;
    int32_t* d_game = (int32_t*)(st + 4 * (size_t)n);
    uint16_t* d_idx = (uint16_t*)(st + 8 * (size_t)n);
    if (game) SZB_CUDA(ctx, cudaMemcpyAsync(d_game, game, 4 * (size_t)n, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaMemcpyAsync(d_idx, move_index, 2 * (size_t)n, cudaMemcpyDefault, ctx->stream));
    k_games_push<<<(n + 31) / 32, 32, 0, ctx->stream>>>(ctx->d, n, game ? d_game : nullptr, d_idx, d_status);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    std::vector<int32_t> h((size_t)n);
    SZB_CUDA(ctx, cudaMemcpyAsync(h.data(), d_status, 4 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (status) SZB_CUDA(ctx, cudaMemcpy(status, h.data(), 4 * (size_t)n, cudaMemcpyDefault));
    for (int i = 0; i < n; i++)
        if (h[i] != 0) return fail(ctx, h[i], "Invalid move (entry %d)", i);
    return 0;
}

int szb_games_get(szb_ctx* ctx, int32_t n, const int32_t* game, szb_pos* out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || n <= 0 || !out) return fail(ctx, SZB_ERR_ARG, "szb_games_get: bad arguments");
    char* st = (char*)ctx_stage(ctx, (size_t)n * (sizeof(szb_pos) + 4));
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    szb_pos* d_out = (szb_pos*)st;
    int32_t* d_game = (int32_t*)(st + sizeof(szb_pos) * (size_t)n);
    if (game) SZB_CUDA(ctx, cudaMemcpyAsync(d_game, game, 4 * (size_t)n, cudaMemcpyDefault, ctx->stream));
    k_games_get<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d, n, game ? d_game : nullptr, d_out);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    SZB_CUDA(ctx, cudaMemcpyAsync(out, d_out, sizeof(szb_pos) * (size_t)n, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int encode_common(szb_ctx* ctx, int32_t n, const int32_t* game, uint16_t* index_out, uint16_t* count_out,
                         uint64_t* planes_out, uint64_t* mask_out) {
    if (!ctx || n <= 0) return fail(ctx, SZB_ERR_ARG, "bad arguments");
    if (ctx->d.n_games == 0) return fail(ctx, SZB_ERR_STATE, "no games");
    const size_t b_game = 4 * (size_t)n, b_idx = index_out ? 2 * (size_t)n * SZB_MAX_MOVES : 0, b_cnt = count_out ? 2 * (size_t)n : 0;
    const size_t b_pl = planes_out ? 8 * (size_t)n * N_PLANES : 0, b_mk = mask_out ? 8 * (size_t)n * MASK_WORDS : 0;
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    char* st = (char*)ctx_stage(ctx, up(b_game) + up(b_idx) + up(b_cnt) + up(b_pl) + up(b_mk) + 256);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    int32_t* d_game = (int32_t*)st; st += up(b_game);
    uint16_t* d_idx = (uint16_t*)st; st += up(b_idx);
    uint16_t* d_cnt = (uint16_t*)st; st += up(b_cnt);
    uint64_t* d_pl = (uint64_t*)st; st += up(b_pl);
    uint64_t* d_mk = (uint64_t*)st;
    if (game) SZB_CUDA(ctx, cudaMemcpyAsync(d_game, game, b_game, cudaMemcpyDefault, ctx->stream));
    k_games_encode<<<(n + 3) / 4, 128, 0, ctx->stream>>>(ctx->d, n, game ? d_game : nullptr, index_out ? d_idx : nullptr,
                                                        count_out ? d_cnt : nullptr, planes_out ? d_pl : nullptr,
                                                        mask_out ? d_mk : nullptr);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    if (index_out) SZB_CUDA(ctx, cudaMemcpyAsync(index_out, d_idx, b_idx, cudaMemcpyDefault, ctx->stream));
    if (count_out) SZB_CUDA(ctx, cudaMemcpyAsync(count_out, d_cnt, b_cnt, cudaMemcpyDefault, ctx->stream));
    if (planes_out) SZB_CUDA(ctx, cudaMemcpyAsync(planes_out, d_pl, b_pl, cudaMemcpyDefault, ctx->stream));
    if (mask_out) SZB_CUDA(ctx, cudaMemcpyAsync(mask_out, d_mk, b_mk, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int szb_legal_moves(szb_ctx* ctx, int32_t n, const int32_t* game, uint16_t* index_out, uint16_t* count_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    return encode_common(ctx, n, game, index_out, count_out, nullptr, nullptr);
}

int szb_encode(szb_ctx* ctx, int32_t n, const int32_t* game, uint64_t* planes_out, uint64_t* mask_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    return encode_common(ctx, n, game, nullptr, nullptr, planes_out, mask_out);
}

int szb_unpack_planes_f32(szb_ctx* ctx, int32_t n, const uint64_t* planes_dev, float* out_dev) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || n <= 0 || !planes_dev || !out_dev) return fail(ctx, SZB_ERR_ARG, "bad arguments");
    const size_t total = (size_t)n * N_PLANES * 64;
    k_unpack_planes_f32<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(n, planes_dev, out_dev);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    return 0;
}

int szb_perft_timed(szb_ctx* ctx, const szb_pos* pos, int32_t depth, uint64_t* nodes_out, float* ms_last_level,
                    uint64_t* positions_last_level) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !pos || !nodes_out || depth < 0) return fail(ctx, SZB_ERR_ARG, "szb_perft: bad arguments");
    if (depth == 0) { *nodes_out = 1; return 0; }
    Pos p;
    pos_from_wire(*pos, p);
    finish_setup(ctx->host_tables, p);
    while (ctx->perft_levels.size() < 1) ctx->perft_levels.push_back(nullptr);
    if (!ctx->perft_levels[0]) SZB_CUDA(ctx, cudaMalloc((void**)&ctx->perft_levels[0], ctx->perft_cap * sizeof(Pos)));
    SZB_CUDA(ctx, cudaMemcpyAsync(ctx->perft_levels[0], &p, sizeof p, cudaMemcpyHostToDevice, ctx->stream));
    cudaError_t err = cudaSuccess;
    float ms = 0;
    uint64_t nl = 0;
    uint64_t total = perft_rec(ctx, ctx->perft_levels[0], 1, depth, 0, &err, ms_last_level ? &ms : nullptr, &nl);
    if (err != cudaSuccess) return cuda_fail(ctx, err, "perft");
    *nodes_out = total;
    if (ms_last_level) *ms_last_level = ms;
    if (positions_last_level) *positions_last_level = nl;
    return 0;
}

int szb_perft(szb_ctx* ctx, const szb_pos* pos, int32_t depth, uint64_t* nodes_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    return szb_perft_timed(ctx, pos, depth, nodes_out, nullptr, nullptr);
}

// ---- search ------------------------------------------------------------------------------------
static int run_search(szb_ctx* ctx, int num_searches, float c_puct, int learning, int evaluator) {
    Dev& d = ctx->d;
    const int G = d.n_games;
    if (G == 0) return fail(ctx, SZB_ERR_STATE, "no games");
    if (num_searches < 1 || num_searches > ctx->cfg.max_searches)
        return fail(ctx, SZB_ERR_ARG, "num_searches %d outside [1, max_searches=%d]", num_searches, ctx->cfg.max_searches);
    cudaStream_t st = ctx->stream;
    int rc0 = 0;
    SZB_CUDA(ctx, cudaMemsetAsync(d.error_flag, 0, sizeof(int32_t), st));
    if (evaluator == SZB_EVAL_NET_BF16 && (rc0 = net_reset_error(ctx))) return rc0;
    d.net_in16 = nullptr; d.net_ready = nullptr; d.net_ready_n = 0; d.step_trace = nullptr;
    d.g_begin = 0;
    d.g_end = G;
    k_search_begin<<<(G + 127) / 128, 128, 0, st>>>(d, num_searches);
    k_active_list<<<1, 1024, 0, st>>>(d);
    ctx->launches += 2;
    // the games still running take the slots 0 .. n_slots-1 of this search; everything below is sized by that count
    int32_t n_slots = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(&n_slots, d.n_active, sizeof n_slots, cudaMemcpyDeviceToHost, st));
    SZB_CUDA(ctx, cudaStreamSynchronize(st));
    const bool prof = ctx->profiling;
    const char* trace_path = getenv("SZB_TRACE");            // debugging aid: per-cohort phase timestamps of this search as CSV
    const bool trace = prof && trace_path && trace_path[0];
    // steps of this search: one simulation per tree and step in the reference's algorithm; in multi-leaf mode up to K per step
    // (a few steps more than num_searches / K are planned because paths can be dropped; stragglers are caught up below)
    const int K = d.K;
    const int n_steps = K == 1 ? num_searches : (num_searches + K - 1) / K + 2;
    if (prof) {
        while ((int)ctx->prof_events.size() < 5 * n_steps * (trace ? 2 : 1)) {
            cudaEvent_t e;
            SZB_CUDA(ctx, cudaEventCreate(&e));
            ctx->prof_events.push_back(e);
        }
    }
    // Cohorts: the games can be split into two halves that step independently on two streams, so that one half's tree
    // kernels (select / expand / finish: latency-bound, a few hundred resident warps) run under the other half's
    // tensor-bound network kernel.  Games never interact, so results do not depend on the split.  Measured on one box,
    // alternating (scripts/ab_cohorts.py, 1024 games): 2.33 ms per simulation step with two cohorts vs 2.37-2.44 with one
    // (the tower is power-capped either way, so only the ~0.2 ms of small kernels can be hidden).  Profiling keeps one
    // cohort on the context's stream so that per-phase and per-kernel durations mean what they say.
    const int NS = n_slots;
    // automatic: two cohorts from 768 path slots on.  Measured, alternating on one box (scripts/ab_cohorts.py): 640 games 1.66-1.71 ms
    // per step with one cohort vs 1.77 with two (a 320-board tower launch is latency-bound and costs more than the overlap saves),
    // 800 games 2.03 vs 1.98, 1024 games 2.39 vs 2.33.  The count is the RUNNING games: a 1024-game batch with a few finished
    // games must still pipeline (it fell back to one cohort for a while in round 1: -5 %).
    int n_cohorts = ctx->cohorts ? ctx->cohorts : (NS * K >= 768 ? 2 : 1);
    if ((prof && !trace) || NS < 8) n_cohorts = 1;
    int bounds[3] = {0, NS, NS};
    if (n_cohorts == 2) bounds[1] = ((NS / 2 + 3) / 4) * 4;       // network tiles are 4 boards wide
    // one simulation step of the slots [dc.g_begin, dc.g_end) on stream cs; ev: five events around its four phases, or null
    auto launch_step = [&](const Dev& dc, cudaStream_t cs, cudaEvent_t* ev) -> int {
        const int n = dc.g_end - dc.g_begin, paths = n * K;
        const int warp_blocks = (n * 32 + 127) / 128;
        ctx->work = cs;
        if (ev) cudaEventRecord(ev[0], cs);
        if (K == 1) k_select<<<warp_blocks, 128, 0, cs>>>(dc, c_puct);
        else k_select_vl<<<warp_blocks, 128, 0, cs>>>(dc, c_puct, num_searches);
        if (ev) cudaEventRecord(ev[1], cs);
        k_expand<<<(paths + 3) / 4, 128, 0, cs>>>(dc);
        if (ev) cudaEventRecord(ev[2], cs);
        ctx->launches += 2;
        int rc_eval = 0;
        if (evaluator == SZB_EVAL_HASH) {
            k_hash_eval<false><<<paths, 128, 0, cs>>>(dc);
            ctx->launches++;
        } else {
            rc_eval = net_evaluate_batch(ctx, evaluator, dc.g_begin * K, paths, false);
        }
        if (ev) cudaEventRecord(ev[3], cs);
        if (K == 1) k_finish<<<(n + FINISH_WARPS - 1) / FINISH_WARPS, 32 * FINISH_WARPS, 0, cs>>>(dc, learning);
        else k_finish_vl<<<n, 32 * MAX_LEAVES, 0, cs>>>(dc, learning);
        if (ev) cudaEventRecord(ev[4], cs);
        ctx->launches++;
        return rc_eval;
    };
    // The reference-exact mode outside profiling runs a step as TWO launches: k_tree_step (children + backup of the previous step's
    // leaves, descent, expansion of the new leaf, the network's input rows) and the evaluator -- for the bf16 network ONE tower launch
    // whose last epilogue emits the priors of the legal moves and the value (net.cu).  Profiling keeps the phase kernels apart so
    // that per-phase times mean what they say; both give the same trees (test_fused_step_equals_phase_kernels).
    const bool fused = K == 1 && !prof && !getenv("SZB_NO_FUSE");
    // measurement aid: SZB_STEP_TRACE=<csv> -- device timestamps of the first tree's warp inside every k_tree_step of this search
    const char* step_trace_path = getenv("SZB_STEP_TRACE");
    unsigned long long* d_step_trace = nullptr;
    if (fused && step_trace_path && step_trace_path[0] && NS > 0) {
        SZB_CUDA(ctx, cudaMalloc((void**)&d_step_trace, (size_t)(n_steps + 1) * 8 * sizeof(unsigned long long)));
        SZB_CUDA(ctx, cudaMemsetAsync(d_step_trace, 0, (size_t)(n_steps + 1) * 8 * sizeof(unsigned long long), st));
    }
    const bool net_fused = fused && net_fused_step(ctx, evaluator);
    // evaluation cache: consulted by the fused reference-exact step with the bf16 network or the hash evaluator; every other path
    // (fp32 evaluator, profiling, SZB_NO_FUSE, phase kernels) runs without it and leaves it untouched
    const bool ec = d.ec_slots > 0 && fused && (evaluator == SZB_EVAL_HASH || net_fused);
    if (d.ec_slots > 0) SZB_CUDA(ctx, cudaMemsetAsync(d.ec_ghits, 0, sizeof(uint32_t) * (size_t)G, st));
    if (ec) {
        d.ec_gen++;
        d.ec_eval = (uint32_t)evaluator;
        SZB_CUDA(ctx, cudaMemsetAsync(d.ec_cnt, 0, 4 * sizeof(int32_t), st));
    }
    // the cohort streams fork from the context's stream only here, after everything enqueued on it for this search (the memsets
    // above included): the streams are non-blocking, so work recorded after the fork would not be ordered before the cohorts' kernels
    if (n_cohorts == 2) {
        SZB_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
        for (int c = 0; c < 2; c++) SZB_CUDA(ctx, cudaStreamWaitEvent(ctx->cohort_stream[c], ctx->ev_fork, 0));
    }
    // programmatic dependent launch chains the two kernels of a step when one cohort runs alone (the latency-bound regime); the
    // two-cohort pipeline already overlaps one cohort's tree kernel with the other's tower
    ctx->pdl = net_fused && n_cohorts == 1 && !getenv("SZB_NO_PDL");
    auto launch_fused = [&](const Dev& dc0, cudaStream_t cs, int phases) -> int {
        Dev dc = dc0;
        const int n = dc.g_end - dc.g_begin;
        ctx->work = cs;
        dc.net_in16 = nullptr; dc.net_ready = nullptr; dc.net_ready_n = 0;
        if (net_fused && (phases & STEP_SELECT)) net_handover(ctx, dc.g_begin, n, &dc.net_in16, &dc.net_ready, &dc.net_ready_n);
        const dim3 grid((n + FINISH_WARPS - 1) / FINISH_WARPS), block(32 * FINISH_WARPS);
        if (ec) launch_kernel(k_tree_step<true>, grid, block, 0, cs, ctx->pdl, dc, c_puct, learning, phases);
        else launch_kernel(k_tree_step<false>, grid, block, 0, cs, ctx->pdl, dc, c_puct, learning, phases);
        ctx->launches++;
        if (!(phases & STEP_SELECT)) return 0;
        if (evaluator == SZB_EVAL_HASH) {
            if (ec) k_hash_eval<true><<<n, 128, 0, cs>>>(dc);
            else k_hash_eval<false><<<n, 128, 0, cs>>>(dc);
            ctx->launches++;
            return 0;
        }
        return net_evaluate_batch(ctx, evaluator, dc.g_begin, n, net_fused, ec ? dc.ec_cnt + dc.ec_par : nullptr);
    };
    int rc = 0;
    for (int s = 0; s <= n_steps && !rc && NS > 0; s++) {
        if (s == n_steps && !fused) break;
        for (int c = 0; c < n_cohorts && !rc; c++) {
            Dev dc = d;
            dc.g_begin = bounds[c];
            dc.g_end = bounds[c + 1];
            cudaStream_t cs = n_cohorts == 2 ? ctx->cohort_stream[c] : st;
            if (fused) {
                dc.step_trace = (d_step_trace && c == 0) ? d_step_trace + (size_t)s * 8 : nullptr;
                dc.ec_cnt = d.ec_cnt + 2 * c;                    // per cohort, per step parity
                dc.ec_par = s & 1;
                dc.ec_boards = d.ec_boards + c;
                rc = launch_fused(dc, cs, (s > 0 ? STEP_FINISH : 0) | (s < n_steps ? STEP_SELECT : 0));
            } else {
                cudaEvent_t* ev = prof ? &ctx->prof_events[5 * ((size_t)s * (trace ? 2 : 1) + (trace ? c : 0))] : nullptr;
                rc = launch_step(dc, cs, ev);
            }
        }
    }
    ctx->work = st;
    ctx->pdl = false;
    if (n_cohorts == 2) {
        for (int c = 0; c < 2; c++) {
            SZB_CUDA(ctx, cudaEventRecord(ctx->ev_join[c], ctx->cohort_stream[c]));
            SZB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join[c], 0));
        }
    }
    if (d_step_trace) {
        std::vector<unsigned long long> h((size_t)(n_steps + 1) * 8);
        cudaStreamSynchronize(st);
        cudaMemcpy(h.data(), d_step_trace, h.size() * 8, cudaMemcpyDeviceToHost);
        cudaFree(d_step_trace);
        if (FILE* f = fopen(step_trace_path, "w")) {
            fprintf(f, "step,start_ns,tables_ns,finish_ns,select_ns,move_made_ns,movegen_ns,planes_mask_ns,input_rows_ns\n");
            for (int s = 0; s <= n_steps; s++) {
                fprintf(f, "%d", s);
                for (int k = 0; k < 8; k++) fprintf(f, ",%lld", h[(size_t)s * 8 + k] ? (long long)(h[(size_t)s * 8 + k] - h[0]) : -1ll);
                fprintf(f, "\n");
            }
            fclose(f);
        }
    }
    if (rc) { cudaStreamSynchronize(st); return rc; }
    SZB_CUDA(ctx, cudaGetLastError());
    if (K > 1 && NS > 0) {
        // multi-leaf mode: trees that dropped paths are still short of num_searches simulations -- step everything (finished trees
        // select nothing) until the slowest tree is done
        Dev dc = d;
        dc.g_begin = 0;
        dc.g_end = NS;
        for (int guard = 0; guard <= 2 * num_searches; guard++) {
            int32_t least = 0;
            k_min_done<<<1, 256, 0, st>>>(d, NS, d.n_active);
            ctx->launches++;
            SZB_CUDA(ctx, cudaMemcpyAsync(&least, d.n_active, sizeof least, cudaMemcpyDeviceToHost, st));
            SZB_CUDA(ctx, cudaStreamSynchronize(st));
            if (least >= num_searches) break;
            const int more = (num_searches - least + K - 1) / K;
            for (int k = 0; k < more && !rc; k++) rc = launch_step(dc, st, nullptr);
            if (rc) { cudaStreamSynchronize(st); return rc; }
        }
        ctx->work = st;
    }
    int32_t flag = 0;
    unsigned long long top = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(&flag, d.error_flag, sizeof flag, cudaMemcpyDeviceToHost, st));
    SZB_CUDA(ctx, cudaMemcpyAsync(&top, d.edge_top, sizeof top, cudaMemcpyDeviceToHost, st));
    SZB_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->edges_high_water = std::max<uint64_t>(ctx->edges_high_water, top);
    if (flag) return fail(ctx, flag, "tree arena exhausted (%llu edges): raise szb_config.edges_per_node", d.edge_cap);
    if (trace && NS > 0) {
        if (FILE* f = fopen(trace_path, "w")) {
            fprintf(f, "step,cohort,select_start_ms,expand_start_ms,eval_start_ms,finish_start_ms,finish_end_ms\n");
            for (int s = 0; s < n_steps; s++)
                for (int c = 0; c < n_cohorts; c++) {
                    cudaEvent_t* ev = &ctx->prof_events[5 * ((size_t)s * 2 + c)];
                    fprintf(f, "%d,%d", s, c);
                    for (int k = 0; k < 5; k++) {
                        float ms = 0;
                        cudaEventElapsedTime(&ms, ctx->prof_events[0], ev[k]);
                        fprintf(f, ",%.4f", ms);
                    }
                    fprintf(f, "\n");
                }
            fclose(f);
        }
        return 0;
    }
    if (prof && NS > 0) {
        for (int s = 0; s < n_steps; s++) {
            cudaEvent_t* ev = &ctx->prof_events[5 * (size_t)s];
            for (int k = 0; k < 4; k++) {
                float ms = 0;
                cudaEventElapsedTime(&ms, ev[k], ev[k + 1]);
                ctx->phase_ms[k] += ms;
            }
        }
        ctx->phase_steps += n_steps;
        net_collect_conv_times(ctx);
    }
    if (evaluator == SZB_EVAL_NET_BF16) return net_check_error(ctx);
    return 0;
}

int szb_search(szb_ctx* ctx, int32_t num_searches, float c_puct, int32_t learning, int32_t evaluator,
               uint32_t* visits_out, uint64_t* child_mask_out, float* root_value_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    int rc = run_search(ctx, num_searches, c_puct, learning, evaluator);
    if (rc) return rc;
    Dev& d = ctx->d;
    const size_t G = (size_t)d.n_games;
    const size_t b_v = visits_out ? G * N_ACTIONS * 4 : 0, b_m = child_mask_out ? G * MASK_WORDS * 8 : 0, b_r = root_value_out ? G * 4 : 0;
    if (b_v + b_m + b_r == 0) return 0;
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    char* st = (char*)ctx_stage(ctx, up(b_v) + up(b_m) + up(b_r) + 256);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    uint32_t* d_v = (uint32_t*)st; st += up(b_v);
    uint64_t* d_m = (uint64_t*)st; st += up(b_m);
    float* d_r = (float*)st;
    k_collect<<<(unsigned)((G * 32 + 127) / 128), 128, 0, ctx->stream>>>(d, visits_out ? d_v : nullptr, child_mask_out ? d_m : nullptr,
                                                                       root_value_out ? d_r : nullptr);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    if (visits_out) SZB_CUDA(ctx, cudaMemcpyAsync(visits_out, d_v, b_v, cudaMemcpyDefault, ctx->stream));
    if (child_mask_out) SZB_CUDA(ctx, cudaMemcpyAsync(child_mask_out, d_m, b_m, cudaMemcpyDefault, ctx->stream));
    if (root_value_out) SZB_CUDA(ctx, cudaMemcpyAsync(root_value_out, d_r, b_r, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int szb_root_children(szb_ctx* ctx, uint16_t* index_out, uint32_t* visits_out, uint16_t* count_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !index_out || !visits_out || !count_out) return fail(ctx, SZB_ERR_ARG, "szb_root_children: bad arguments");
    Dev& d = ctx->d;
    const size_t G = (size_t)d.n_games;
    if (G == 0) return fail(ctx, SZB_ERR_STATE, "no games");
    const size_t b_i = G * SZB_MAX_MOVES * 2, b_v = G * SZB_MAX_MOVES * 4, b_c = (G * 2 + 255) & ~(size_t)255;
    char* st = (char*)ctx_stage(ctx, b_i + b_v + b_c);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    uint32_t* d_v = (uint32_t*)st;
    uint16_t* d_i = (uint16_t*)(st + b_v);
    uint16_t* d_c = (uint16_t*)(st + b_v + b_i);
    k_root_children<<<(unsigned)((G * 32 + 127) / 128), 128, 0, ctx->stream>>>(d, d_i, d_v, d_c);
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    SZB_CUDA(ctx, cudaMemcpyAsync(index_out, d_i, b_i, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaMemcpyAsync(visits_out, d_v, b_v, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaMemcpyAsync(count_out, d_c, G * 2, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int szb_tree_export(szb_ctx* ctx, int32_t game, int32_t max_nodes, int32_t max_edges, int32_t* node_first, int32_t* node_count,
                    int32_t* node_parent, int32_t* node_parent_edge, uint8_t* node_terminal, float* node_terminal_value,
                    int32_t* edge_visits, double* edge_value_sum, float* edge_prior, uint16_t* edge_move, int32_t* edge_child,
                    int32_t* root_visits_out, double* root_value_sum_out, int32_t* n_nodes_out, int32_t* n_edges_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || game < 0 || game >= ctx->d.n_games || max_nodes <= 0 || max_edges <= 0) return fail(ctx, SZB_ERR_ARG, "szb_tree_export: bad arguments");
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t mn = (size_t)max_nodes, me = (size_t)max_edges;
    const size_t o_nf = 0, o_nc = o_nf + up(mn * 4), o_np = o_nc + up(mn * 4), o_ne = o_np + up(mn * 4), o_nt = o_ne + up(mn * 4),
                 o_nv = o_nt + up(mn), o_ew = o_nv + up(mn * 4), o_en = o_ew + up(me * 8), o_ep = o_en + up(me * 4),
                 o_ec = o_ep + up(me * 4), o_em = o_ec + up(me * 4), o_tot = o_em + up(me * 2), total = o_tot + 256;
    char* st = (char*)ctx_stage(ctx, total);
    if (!st) return fail(ctx, SZB_ERR_CUDA, "staging allocation failed");
    k_tree_export<<<1, 32, 0, ctx->stream>>>(ctx->d, game, max_nodes, max_edges, (int32_t*)(st + o_nf), (int32_t*)(st + o_nc),
                                            (int32_t*)(st + o_np), (int32_t*)(st + o_ne), (uint8_t*)(st + o_nt), (float*)(st + o_nv),
                                            (int32_t*)(st + o_en), (double*)(st + o_ew), (float*)(st + o_ep), (uint16_t*)(st + o_em),
                                            (int32_t*)(st + o_ec), (int32_t*)(st + o_tot));
    ctx->launches++;
    SZB_CUDA(ctx, cudaGetLastError());
    int32_t tot[3];
    double rw = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(tot, st + o_tot, sizeof tot, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaMemcpyAsync(&rw, ctx->d.root_w + game, 8, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (tot[0] < 0) return fail(ctx, SZB_ERR_ARG, "szb_tree_export: capacity too small");
    const size_t nn = (size_t)tot[0], ne = (size_t)tot[1];
    struct { void* dst; size_t off, bytes; } cp[] = {
        {node_first, o_nf, nn * 4}, {node_count, o_nc, nn * 4}, {node_parent, o_np, nn * 4}, {node_parent_edge, o_ne, nn * 4},
        {node_terminal, o_nt, nn}, {node_terminal_value, o_nv, nn * 4}, {edge_visits, o_en, ne * 4}, {edge_value_sum, o_ew, ne * 8},
        {edge_prior, o_ep, ne * 4}, {edge_move, o_em, ne * 2}, {edge_child, o_ec, ne * 4}};
    for (auto& c : cp)
        if (c.dst && c.bytes) SZB_CUDA(ctx, cudaMemcpyAsync(c.dst, st + c.off, c.bytes, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (root_visits_out) *root_visits_out = tot[2];
    if (root_value_sum_out) *root_value_sum_out = rw;
    if (n_nodes_out) *n_nodes_out = (int32_t)nn;
    if (n_edges_out) *n_edges_out = (int32_t)ne;
    return 0;
}

int szb_selfplay_ply(szb_ctx* ctx, int32_t num_searches, float c_puct, int32_t learning, int32_t evaluator,
                     uint64_t seed, int32_t sample, int32_t* moves_out, int32_t* n_active_out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    int rc = run_search(ctx, num_searches, c_puct, learning, evaluator);
    if (rc) return rc;
    Dev& d = ctx->d;
    const int G = d.n_games;
    int32_t* d_active = ctx->d_moves + ctx->cfg.max_games;
    SZB_CUDA(ctx, cudaMemsetAsync(d_active, 0, sizeof(int32_t), ctx->stream));
    k_pick<<<(G + 127) / 128, 128, 0, ctx->stream>>>(d, seed, sample, ctx->sample_plies, ctx->d_moves);
    k_push_picked<<<(G + 31) / 32, 32, 0, ctx->stream>>>(d, ctx->d_moves, d_active);
    ctx->launches += 2;
    SZB_CUDA(ctx, cudaGetLastError());
    if (moves_out) SZB_CUDA(ctx, cudaMemcpyAsync(moves_out, ctx->d_moves, 4 * (size_t)G, cudaMemcpyDefault, ctx->stream));
    int32_t act = 0;
    SZB_CUDA(ctx, cudaMemcpyAsync(&act, d_active, 4, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (n_active_out) *n_active_out = act;
    return 0;
}

int szb_set_game_id_base(szb_ctx* ctx, uint64_t base) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    ctx->d.game_id_base = base;
    return 0;
}

int szb_set_exploration(szb_ctx* ctx, const szb_exploration* x) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    const szb_exploration off{};
    const szb_exploration& e = x ? *x : off;
    if (!std::isfinite(e.dirichlet_alpha) || e.dirichlet_alpha < 0.0f)
        return fail(ctx, SZB_ERR_ARG, "szb_set_exploration: dirichlet_alpha %g is not a finite value >= 0", (double)e.dirichlet_alpha);
    if (!(e.dirichlet_epsilon >= 0.0f && e.dirichlet_epsilon <= 1.0f))
        return fail(ctx, SZB_ERR_ARG, "szb_set_exploration: dirichlet_epsilon %g outside [0, 1]", (double)e.dirichlet_epsilon);
    if (e.sample_plies < 0) return fail(ctx, SZB_ERR_ARG, "szb_set_exploration: sample_plies %d < 0", e.sample_plies);
    ctx->d.dir_alpha = e.dirichlet_alpha;
    ctx->d.dir_eps = e.dirichlet_epsilon;
    ctx->d.dir_seed = e.seed;
    ctx->sample_plies = e.sample_plies;
    return 0;
}

int szb_set_eval_cache(szb_ctx* ctx, int32_t slots_per_game) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    Dev& d = ctx->d;
    if (slots_per_game == 0) {
        if (ctx->ec_mem) {
            SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->ec_mem);
        }
        ctx->ec_mem = nullptr;
        ctx->ec_bytes = 0;
        d.ec_slots = 0; d.ec_meta = nullptr; d.ec_pri = nullptr;
        return 0;
    }
    if (slots_per_game < EC_MIN_SLOTS || slots_per_game > EC_MAX_SLOTS || (slots_per_game & (slots_per_game - 1)))
        return fail(ctx, SZB_ERR_ARG, "szb_set_eval_cache: %d slots per game is not 0 or a power of two in [%d, %d]", slots_per_game,
                    EC_MIN_SLOTS, EC_MAX_SLOTS);
    if (d.K > 1)
        return fail(ctx, SZB_ERR_UNSUPPORTED, "szb_set_eval_cache: the evaluation cache serves one leaf per tree and step (leaves_per_tree = %d)", d.K);
    if (slots_per_game == d.ec_slots) return 0;
    const size_t entries = (size_t)ctx->cfg.max_games * (size_t)slots_per_game;
    const size_t meta_bytes = entries * sizeof(EcMeta), bytes = meta_bytes + entries * EC_PRI_STRIDE * sizeof(float);
    void* mem = nullptr;
    const cudaError_t e = cudaMalloc(&mem, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, SZB_ERR_CUDA, "szb_set_eval_cache: cannot allocate %zu bytes (%d games x %d slots x %zu B): %s", bytes,
                    ctx->cfg.max_games, slots_per_game, sizeof(EcMeta) + EC_PRI_STRIDE * sizeof(float), cudaGetErrorString(e));
    }
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SZB_CUDA(ctx, cudaMemsetAsync(mem, 0, meta_bytes, ctx->stream));
    if (ctx->ec_mem) cudaFree(ctx->ec_mem);
    ctx->ec_mem = mem;
    ctx->ec_bytes = bytes;
    d.ec_slots = slots_per_game;
    d.ec_meta = (EcMeta*)mem;
    d.ec_pri = (float*)((char*)mem + meta_bytes);
    d.ec_epoch++;                              // a new table: nothing in it is live (the zeroed entries carry epoch 0)
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int szb_get_eval_cache_stats(szb_ctx* ctx, szb_eval_cache_stats* out, uint32_t* game_hits) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !out) return fail(ctx, SZB_ERR_ARG, "szb_get_eval_cache_stats: bad arguments");
    const size_t G = (size_t)ctx->cfg.max_games;
    std::vector<unsigned long long> h(G * 4);
    unsigned long long boards[2] = {0, 0};
    SZB_CUDA(ctx, cudaMemcpyAsync(h.data(), ctx->d.ec_gstats, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaMemcpyAsync(boards, ctx->d.ec_boards, sizeof boards, cudaMemcpyDeviceToHost, ctx->stream));
    if (game_hits && ctx->d.n_games > 0)
        SZB_CUDA(ctx, cudaMemcpyAsync(game_hits, ctx->d.ec_ghits, sizeof(uint32_t) * (size_t)ctx->d.n_games, cudaMemcpyDefault, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    unsigned long long t[4] = {0, 0, 0, 0};
    for (size_t g = 0; g < G; g++)
        for (int k = 0; k < 4; k++) t[k] += h[g * 4 + k];
    memset(out, 0, sizeof *out);
    out->lookups = t[0];
    out->hits = t[1];
    out->inserts = t[2];
    out->dropped_inserts = t[3];
    out->boards_evaluated = boards[0] + boards[1];     // the evaluator's own row counts, summed by the tree kernels
    out->bytes = ctx->ec_bytes;
    out->slots_per_game = ctx->d.ec_slots;
    return 0;
}

int szb_set_profiling(szb_ctx* ctx, int32_t on) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx) return SZB_ERR_ARG;
    ctx->profiling = on != 0;
    for (int k = 0; k < 4; k++) ctx->phase_ms[k] = 0;
    ctx->phase_steps = 0;
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->conv_events_used = 0;
    ctx->conv_ms = 0; ctx->conv_launches = 0;
    ctx->conv_recorded = 0; ctx->conv_boards = 0; ctx->conv_flop = 0;
    k_fold_stats<<<1, 256, 0, ctx->stream>>>(ctx->d, ctx->cfg.max_games);
    SZB_CUDA(ctx, cudaMemsetAsync(ctx->d.stats + 4, 0, 4 * sizeof(unsigned long long), ctx->stream));
    return 0;
}

int szb_get_phase_times(szb_ctx* ctx, szb_phase_times* out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !out) return SZB_ERR_ARG;
    unsigned long long h[8];
    k_fold_stats<<<1, 256, 0, ctx->stream>>>(ctx->d, ctx->cfg.max_games);
    SZB_CUDA(ctx, cudaMemcpyAsync(h, ctx->d.stats, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    out->select_ms = ctx->phase_ms[0]; out->expand_ms = ctx->phase_ms[1];
    out->eval_ms = ctx->phase_ms[2]; out->finish_ms = ctx->phase_ms[3];
    out->steps = ctx->phase_steps; out->reserved = 0;
    out->select_edges = h[4]; out->select_levels = h[5]; out->backup_levels = h[6]; out->edges_written = h[7];
    net_collect_conv_times(ctx);
    out->conv_ms = ctx->conv_ms; out->conv_launches = ctx->conv_launches; out->conv_kind = ctx->net_tower_mode;
    // per-launch averages (the launches of a chunked evaluation need not be equally large)
    const uint64_t rec = ctx->conv_recorded > 0 ? (uint64_t)ctx->conv_recorded : 1;
    out->conv_boards = (int32_t)(ctx->conv_boards / rec);
    out->conv_flop = ctx->conv_flop / rec;
    return 0;
}

int szb_get_stats(szb_ctx* ctx, szb_stats* out) {
    if (ctx) cudaSetDevice(ctx->device);       // whichever device the calling thread had current
    if (!ctx || !out) return SZB_ERR_ARG;
    unsigned long long h[8];
    k_fold_stats<<<1, 256, 0, ctx->stream>>>(ctx->d, ctx->cfg.max_games);
    SZB_CUDA(ctx, cudaMemcpyAsync(h, ctx->d.stats, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    SZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    out->simulations = h[0];
    out->evaluations = h[1];
    out->terminal_visits = h[2];
    out->max_depth = h[3];
    out->edges_allocated = ctx->edges_high_water;
    out->kernel_launches = ctx->launches;
    return 0;
}

}  // extern "C"
