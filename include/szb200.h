/*
 * szb200.h -- C ABI of libszb200.so: the B200-native replacement for the self-play hot path of
 * DidItWork/Sigma-Zero (batched AlphaZero MCTS over many concurrent chess / Chess960 games) and, at the
 * end of this header, for the fine-tuning step of the same loop (szb_train_*, train_RL.py:77-154).
 *
 * The reference has no FFI of its own: its boundary for this path is a Python call surface
 * (SURVEY.md 8b).  Each entry point below names the reference call it replaces (file:line into the
 * reference repository); the Python facade in sigma-zero_b200/ keeps the reference's names
 * (mcts.MCTS0, mctsnode.Node, chess_tensor.ChessTensor, network.policyNN, sim.play_game) and calls
 * these functions through ctypes.  INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - plain C types, opaque context, no torch / C++ types in any signature;
 *   - every function returns 0 on success and a negative code on failure; szb_last_error(ctx) gives
 *     the message;
 *   - one context per GPU, used from one host thread; work is issued on the context's stream;
 *   - I/O buffers belong to the caller and may be host (pageable or pinned) or device memory -- the
 *     library copies with cudaMemcpyDefault on its stream and synchronises before returning when the
 *     destination is host data;
 *   - there is no CPU fallback: without a CUDA device every call fails with SZB_ERR_CUDA.
 *
 * Move indices are the reference's policy indices: plane*64 + row*8 + col in the mover's view,
 * 0 <= index < 4672 (chess_tensor.py:221-306).  Planes are the reference's 119 input planes
 * (chess_tensor.py:8-26,38-142), bit-packed: one uint64 per plane, bit (row*8+col).
 */
#ifndef SZB200_H
#define SZB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SZB_N_PLANES 119
#define SZB_N_ACTIONS 4672
#define SZB_MASK_WORDS 73
#define SZB_MAX_MOVES 256          /* row stride of move-index outputs (>= 218) */

enum {
    SZB_OK = 0,
    SZB_ERR_ARG = -1,              /* bad argument */
    SZB_ERR_CUDA = -2,             /* CUDA runtime failure or no device */
    SZB_ERR_ILLEGAL_MOVE = -3,     /* szb_games_push: at least one move was not legal (chess_tensor.py:91-92) */
    SZB_ERR_ARENA = -4,            /* tree arena exhausted: raise szb_config.edges_per_node */
    SZB_ERR_STATE = -5,            /* call made in the wrong state (no games, no weights, ...) */
    SZB_ERR_UNSUPPORTED = -6,
    SZB_ERR_INTERNAL = -7          /* a kernel reported a failure (pipeline time-out, bad record row) */
};

/* evaluator used by szb_search / szb_selfplay */
enum {
    SZB_EVAL_NET_BF16 = 0,         /* tcgen05/TMEM implicit-GEMM tower, bf16 in / fp32 accumulate */
    SZB_EVAL_NET_FP32 = 1,         /* fp32 SIMT tower (parity mode, <= 1e-5 abs vs torch CPU fp32) */
    SZB_EVAL_HASH = 2              /* integer-hash evaluator (exact-parity tests, tree-only benchmarks) */
};

typedef struct szb_ctx szb_ctx;

typedef struct szb_config {
    int32_t max_games;             /* capacity: concurrent games (trees) */
    int32_t max_searches;          /* capacity: num_searches per move (train_RL.py:170) */
    int32_t edges_per_node;        /* tree arena = max_games * (max_searches+1) * edges_per_node edges; 0 -> 48 */
    int32_t cohorts;               /* search pipelining: 2 = the games step as two independent halves on two streams (one half's
                                      tree kernels run under the other half's network kernel), 1 = one batch, 0 = automatic (2 from 768 running games) */
    int32_t leaves_per_tree;       /* 0 / 1: the reference's algorithm, one simulation of a tree at a time (mcts.py:49) -- every parity
                                      statement of this library is about this mode.  2..8: that many simulations of a tree in flight per
                                      step, kept apart by virtual loss: a DIFFERENT search (other visit counts, still exactly
                                      num_searches simulations per move, deterministic) for the latency-bound regime of few games */
} szb_config;

/* A position crossing the ABI. */
typedef struct szb_pos {
    uint64_t pieces[12];           /* white P N B R Q K, black P N B R Q K; bit s = square s, a1 = 0, h8 = 63 */
    uint8_t turn;                  /* 1 = white to move */
    uint8_t castling_w;            /* files (bit f) of white rooks that may castle */
    uint8_t castling_b;
    int8_t ep_square;              /* -1 = none */
    uint16_t halfmove_clock;
    uint16_t ply;                  /* moves already played in this game object (len(board.move_stack)) */
    uint8_t chess960;              /* castling written king-takes-rook (Board.from_chess960_pos) */
    uint8_t outcome;               /* out: 0 running, 1 checkmate, 2 insufficient material, 3 stalemate,
                                      4 seventy-five moves, 5 fivefold repetition (Board.outcome()) */
    uint8_t rep_flags;             /* out: bit0 is_repetition(2), bit1 is_repetition(3) */
    uint8_t n_legal;               /* out */
    uint8_t pad[4];
} szb_pos;

/* ---- lifecycle --------------------------------------------------------------------------------- */
const char *szb_version(void);
int szb_create(int device_ordinal, const szb_config *cfg, szb_ctx **out);
void szb_destroy(szb_ctx *ctx);
const char *szb_last_error(const szb_ctx *ctx);
/* the CUDA stream (cudaStream_t) all work of this context is ordered on */
void *szb_stream(szb_ctx *ctx);
int szb_synchronize(szb_ctx *ctx);

/* ---- games: replaces ChessTensor.__init__/start_board/move_piece (chess_tensor.py:30-35,65-129) -- */
/* start n_games games; start_id[g] = -1 -> chess.Board(), 0..959 -> Board.from_chess960_pos(id) */
int szb_games_reset(szb_ctx *ctx, int32_t n_games, const int16_t *start_id);
/* start n_games games from arbitrary positions (empty history) */
int szb_games_set(szb_ctx *ctx, int32_t n_games, const szb_pos *positions);
/* play move_index[i] in game game[i] (i < n; each game at most once per call).  status[i] (optional) is 0
 * or SZB_ERR_ILLEGAL_MOVE; illegal moves leave their game untouched ("Invalid move", chess_tensor.py:91). */
int szb_games_push(szb_ctx *ctx, int32_t n, const int32_t *game, const uint16_t *move_index, int32_t *status);
/* current position of each listed game (game == NULL: games 0..n-1) */
int szb_games_get(szb_ctx *ctx, int32_t n, const int32_t *game, szb_pos *out);
/* replaces list(board.legal_moves) + actionsToTensor (chess_tensor.py:146,190-218): ascending policy
 * indices of the legal moves, row stride SZB_MAX_MOVES, and their count */
int szb_legal_moves(szb_ctx *ctx, int32_t n, const int32_t *game, uint16_t *index_out, uint16_t *count_out);
/* replaces get_representation (chess_tensor.py:131-142) and actionsToTensor's mask: planes_out is
 * uint64[n][119], mask_out (optional) uint64[n][73] with bit index = policy index */
int szb_encode(szb_ctx *ctx, int32_t n, const int32_t *game, uint64_t *planes_out, uint64_t *mask_out);
/* bit-packed planes -> float32 [n][119][8][8] (what mcts.py:73 feeds the network).  Both device pointers. */
int szb_unpack_planes_f32(szb_ctx *ctx, int32_t n, const uint64_t *planes_dev, float *out_dev);

/* ---- perft: bulk legal move generation + make-move (correctness config c1, movegen roofline) ---- */
int szb_perft(szb_ctx *ctx, const szb_pos *pos, int32_t depth, uint64_t *nodes_out);
/* timing hook for benchmarks: one breadth-first ply over the context's current frontier; see bench.py */
int szb_perft_timed(szb_ctx *ctx, const szb_pos *pos, int32_t depth, uint64_t *nodes_out,
                    float *ms_last_level, uint64_t *positions_last_level);

/* ---- network: replaces policyNN.load_state_dict / forward (network.py:100-192, play.py:25-28) ---- */
/* tensors of the fp32 state_dict by name (252 entries; *.num_batches_tracked may be omitted).
 * data[i] are HOST pointers to contiguous fp32; the library stages them on the device, folds BatchNorm (eval mode) into the
 * convolutions there and builds the fp32 and bf16 device packs.  The whole state_dict is validated before anything loaded
 * earlier is touched. */
int szb_net_load(szb_ctx *ctx, int32_t n_tensors, const char *const *names, const float *const *data,
                 const int64_t *numel);
/* The same with DEVICE pointers (e.g. slices of the flat fp32 buffer torch.distributed just broadcast over NCCL: the weight
 * path of train_RL.py:211-227 with no host round trip).  BatchNorm folding and all packing run on the GPU, asynchronously on the
 * context's stream; the tensors may be released once the stream has passed this call.  A context that already holds a network
 * refills its buffers in place (no allocation, no synchronisation). */
int szb_net_load_device(szb_ctx *ctx, int32_t n_tensors, const char *const *names, const float *const *data_dev,
                        const int64_t *numel);
/* 64-bit digest of the packed device weights (what the kernels actually read): equal on every rank after a broadcast */
int szb_net_checksum(szb_ctx *ctx, uint64_t *digest_out);
/* policyNN.forward(x, inference=True): planes uint64[n][119] -> softmax policy float[n][4672], value float[n] */
int szb_net_forward(szb_ctx *ctx, int32_t n, const uint64_t *planes, int32_t evaluator,
                    float *policy_out, float *value_out);
/* raw logits variant (inference=False) */
int szb_net_forward_logits(szb_ctx *ctx, int32_t n, const uint64_t *planes, int32_t evaluator,
                           float *logits_out, float *value_out);

/* ---- search: replaces MCTS0.search (mcts.py:39-122) for every current game at once ---------------- */
/* num_searches, c_puct = args['num_searches'], args['C']; learning as in mcts.py:91-96.
 * visits_out (optional): uint32[n_games][4672], visit count of every root child at its policy index
 *   (the reference returns count / sum(count), mcts.py:113-122);
 * child_mask_out (optional): uint64[n_games][73], bit set for every root child (children with zero visits
 *   are part of the reference's result dict);
 * root_value_out (optional): float[n_games] network value of the root. */
int szb_search(szb_ctx *ctx, int32_t num_searches, float c_puct, int32_t learning, int32_t evaluator,
               uint32_t *visits_out, uint64_t *child_mask_out, float *root_value_out);

/* compact form of the last search's result: for every game the root children in ascending policy-index order
 * (row stride SZB_MAX_MOVES), their visit counts and their number -- the (move, visit_count) pairs of
 * mcts.py:113-116.  Valid until the next search. */
int szb_root_children(szb_ctx *ctx, uint16_t *index_out, uint32_t *visits_out, uint16_t *count_out);

/* read-only export of one game's search tree (backs the mctsnode.Node view, mctsnode.py:8-18).
 * Nodes are the visited nodes in creation order (node 0 = root); node_* arrays have max_nodes entries,
 * edge_* arrays max_edges entries; each node's children are edges [node_first[i], node_first[i]+node_count[i]).
 * edge_child is the visited-node index behind an edge or -1.  n_nodes_out / n_edges_out receive the totals
 * (SZB_ERR_ARG if a capacity is too small). */
int szb_tree_export(szb_ctx *ctx, int32_t game, int32_t max_nodes, int32_t max_edges,
                    int32_t *node_first, int32_t *node_count, int32_t *node_parent, int32_t *node_parent_edge,
                    uint8_t *node_terminal, float *node_terminal_value,
                    int32_t *edge_visits, double *edge_value_sum, float *edge_prior, uint16_t *edge_move,
                    int32_t *edge_child, int32_t *root_visits_out, double *root_value_sum_out,
                    int32_t *n_nodes_out, int32_t *n_edges_out);

/* ---- self-play: replaces sim.play_game's ply loop (sim.py:46-76) ---------------------------------- */
/* One ply for every unfinished game: search, pick a move (sample proportional to visits, sim.py:68, with a
 * counter-based RNG keyed (seed, global game id, ply); or argmax with lowest index on ties when sample == 0), record
 * (planes, visits, colour) and push the move.  moves_out (optional): int32[n_games] chosen policy index or -1
 * for games already over.  n_active_out (optional): games still running afterwards. */
int szb_selfplay_ply(szb_ctx *ctx, int32_t num_searches, float c_puct, int32_t learning, int32_t evaluator,
                     uint64_t seed, int32_t sample, int32_t *moves_out, int32_t *n_active_out);

/* Global id of this context's game 0 (default 0).  The move-sampling RNG is keyed (seed, global game id, ply), so a game's
 * moves do not depend on which rank / shard plays it (train_RL.py:219-239 fans games out to workers). */
int szb_set_game_id_base(szb_ctx *ctx, uint64_t base);

/* Opt-in AlphaZero exploration for self-play (NOT the reference's rule: every parity statement of this library is about the
 * default, which is off).  Applies to the szb_search / szb_selfplay_ply calls made after it, until it is changed.
 *   - Root noise, when dirichlet_alpha > 0 and the search runs with learning != 0: when a search expands its root, the normalised
 *     priors of the children that survive the zero-prior drop (ascending policy index) become
 *     fl32((1 - (double)eps) * (double)p + (double)eps * (double)fl32(eta)), eta ~ Dir(alpha) over those children, mixed in double
 *     without FMA contraction and rounded once (at eps = 1 a root prior is exactly fl32(eta)).  Every other node of such a search
 *     gets the raw normalised priors: the reference's constant rule (mcts.py:91-96, a one-category Dirichlet) is not applied.
 *     eta of a child is a function of (seed, global game id = game id base + game, the root position's ply, the child's policy
 *     index) only: not of the slot, the cohort split, the shard, leaves_per_tree or the other children.
 *     With learning == 0 or dirichlet_alpha == 0 nothing changes (the constant rule still applies under learning != 0).
 *   - Sampling horizon, for szb_selfplay_ply(..., sample = 1, ...): moves are sampled proportional to visits (with the same RNG
 *     key, so the same moves as without the horizon) while the root position's ply < sample_plies, and from then on the arg-max
 *     (first maximum, lowest index on ties) is played.  0 = sample every ply (sim.py:68).
 * x == NULL switches everything off.  SZB_ERR_ARG (setting unchanged) for an alpha that is not finite or is negative, an epsilon
 * outside [0, 1] or sample_plies < 0. */
typedef struct szb_exploration {
    float dirichlet_alpha;         /* 0 = off (the reference's rule); AlphaZero chess: 0.3 */
    float dirichlet_epsilon;       /* in [0, 1]; 0.25 */
    uint64_t seed;                 /* keys the root noise */
    int32_t sample_plies;          /* 0 = sample every ply (sim.py:68); k = arg-max from ply k on */
    int32_t reserved;
} szb_exploration;
int szb_set_exploration(szb_ctx *ctx, const szb_exploration *x);

/* Opt-in evaluation cache (off by default).  Per game an open-addressed table of slots_per_game entries keyed on the EXACT evaluator
 * input: a 128-bit hash of the leaf's 119 packed planes, its legal-move mask and the evaluator id.  A leaf whose key is live in its
 * game's table (written or hit by this search or the previous one, under the current weights) takes the stored priors and value
 * instead of an evaluation, and the evaluator runs only on the leaves that missed.  A board's evaluation does not depend on its batch,
 * so every visit count, prior, value, move and record is bit-identical with the cache on and off; szb_stats counts a hit as an
 * evaluation either way.  The one accepted risk is a 128-bit key collision (~2^-128 per comparison), as in a transposition table.
 * Consulted by szb_search / szb_selfplay_ply with leaves_per_tree = 1 and the bf16 network (fused step) or the hash evaluator; the
 * fp32 evaluator, profiling and SZB_NO_FUSE run without it.  Loading weights (szb_net_load, szb_net_load_device) or resizing
 * invalidates every entry.  Memory: max_games x slots_per_game x 928 bytes (1024 games x 2048 slots: 1.9 GB).
 * slots_per_game: 0 = off (frees the table), otherwise a power of two in [64, 65536] (SZB_ERR_ARG otherwise); the current size keeps
 * the table.  SZB_ERR_UNSUPPORTED for leaves_per_tree > 1, SZB_ERR_CUDA if the table cannot be allocated; the setting is unchanged
 * on any failure. */
int szb_set_eval_cache(szb_ctx *ctx, int32_t slots_per_game);

typedef struct szb_eval_cache_stats {
    uint64_t lookups;              /* non-terminal leaves that consulted the cache (cumulative) */
    uint64_t hits;
    uint64_t inserts;              /* entries written */
    uint64_t dropped_inserts;      /* misses whose probe window had no free entry */
    uint64_t boards_evaluated;     /* boards the evaluator ran on in those searches: the sum of its per-step input-row counts, kept
                                      on the device (every lookup that misses takes one row, so it equals lookups - hits) */
    uint64_t bytes;                /* device memory of the table */
    int32_t slots_per_game;        /* 0 = off */
    int32_t reserved;
} szb_eval_cache_stats;
/* game_hits (optional, [n_games]): hits of each game in the last search. */
int szb_get_eval_cache_stats(szb_ctx *ctx, szb_eval_cache_stats *out, uint32_t *game_hits);

/* ---- counters (SURVEY.md 5: metrics) -------------------------------------------------------------- */
typedef struct szb_stats {
    uint64_t simulations;          /* iterations of mcts.py:49 executed */
    uint64_t evaluations;          /* network / evaluator calls (non-terminal leaves) */
    uint64_t terminal_visits;
    uint64_t edges_allocated;      /* high-water mark of the edge arena in the last search */
    uint64_t kernel_launches;      /* kernels of this library launched since creation */
    uint64_t max_depth;
} szb_stats;
int szb_get_stats(szb_ctx *ctx, szb_stats *out);

/* ---- measurement hooks (bench.py; CUDA events recorded on the context's stream) ------------------ */
/* per-phase device time of the simulation steps of searches run while profiling is on */
typedef struct szb_phase_times {
    float select_ms, expand_ms, eval_ms, finish_ms;   /* totals over `steps` simulation steps */
    int32_t steps;
    int32_t reserved;
    uint64_t select_edges;     /* children scanned by PUCT selection (16 B each: N 4 + W 8 + P 4) */
    uint64_t select_levels;    /* tree levels descended (16 B node header each) */
    uint64_t backup_levels;    /* edges updated by backup (24 B read-modify-write each) */
    uint64_t edges_written;    /* children created by expansion (20 B each) */
    float conv_ms;             /* total device time of the timed network launches, CUDA events on the context's stream */
    int32_t conv_launches;     /* how many launches conv_ms covers (a bf16 forward of more than 512 boards is several launches) */
    int32_t conv_boards;       /* boards per timed launch, averaged (the GEMM's M / 64) */
    int32_t conv_kind;         /* what is timed: 2 = k_tower_tc2, the whole tower (stem + 38 convolutions + policy 1x1) in one
                                  launch; 1 = k_tower_tc2 on one 3x3 256->256 layer; 0 = k_conv_tc<256,0> on one such layer */
    uint64_t conv_flop;        /* algorithmic FLOP (2 x MAC, no padding credit) per timed launch, averaged */
} szb_phase_times;
int szb_set_profiling(szb_ctx *ctx, int32_t on);
int szb_get_phase_times(szb_ctx *ctx, szb_phase_times *out);
/* device-side timing of the network's whole-tower launches (k_tower_tc2 stamps %globaltimer when its first CTA starts and when
 * its last CTA ends): unlike event pairs this also works while the two cohorts of a search overlap on two streams.
 * on = 1: clear and start recording; on = 0: stop and report what was recorded (at most 8192 launches). */
typedef struct szb_tower_spans {
    int32_t launches;          /* launches recorded */
    int32_t reserved;
    uint64_t boards;           /* boards of those launches (sum) */
    uint64_t busy_ns;          /* sum of (end - start) over the launches */
    uint64_t wall_ns;          /* last end - first start */
    uint64_t flop;             /* algorithmic FLOP of those launches (sum) */
    uint64_t sm_cycles;        /* SM clock cycles CTA 0 of every launch lived (clock64), summed ... */
    uint64_t sm_ns;            /* ... and the nanoseconds it lived (%globaltimer): sm_cycles / sm_ns = the SM clock INSIDE the launches in GHz */
} szb_tower_spans;
int szb_tower_spans_record(szb_ctx *ctx, int32_t on, szb_tower_spans *out);
/* average duration (ms) of one launch of a kernel run `iters` times back to back on n boards:
 * which = 0: one 3x3 256->256 tower convolution (single-CTA tcgen05 kernel, with residual) ; 1: whole bf16 forward ;
 * 2: whole fp32 forward ; 3: one 3x3 256->256 fp32 SIMT convolution ; 4: one 3x3 256->256 tower convolution
 * (CTA-pair kernel) ; 5: the whole tower in one CTA-pair launch ; 6: the whole forward (tower + heads) in the cluster-resident
 * kernel that serves batches of at most 18 boards */
/* NOTE: the tower kernels run on whatever the activation buffers hold.  On a fresh context that is all-zero input planes --
 * constant activations, little switching, far less power -- so many back-to-back launches then sustain a higher clock than real
 * positions allow (1.5 vs 1.3 PFLOP/s, profiles/r01o_*).  Run a search first when a sustained figure is wanted. */
int szb_time_kernel(szb_ctx *ctx, int32_t which, int32_t n, int32_t iters, float *ms_avg_out);

/* ---- trainer: the fine-tuning half of the self-play loop (train_RL.py:77-154) ---------------------------------------------
 * Replaces chessDataset / collatefn / train() of the reference for packed self-play records: per batch
 *     loss = mse_loss(v, z) + cross_entropy(logits, pi)      (train_RL.py:103-113, pi = soft visit-fraction target)
 *     Adam(lr, weight_decay) with torch's update rule (train_RL.py:187), StepLR(lr_step, lr_gamma) stepped per batch (:199, :123)
 * on network.py:100-192 in training mode (BatchNorm with batch statistics; running buffers updated with `bn_momentum`).
 * Mixed precision: fp32 master weights / moments / BatchNorm arithmetic, bf16 tensor-core operands with fp32 accumulation.
 * One trainer per context; tensors are named as in the reference's state_dict and laid out as torch lays them out. */
typedef struct szb_train_config {
    int32_t batch;            /* largest batch (boards) a step may carry */
    float lr, beta1, beta2, eps, weight_decay;     /* torch.optim.Adam: 1e-4, 0.9, 0.999, 1e-8, 1e-4 in the reference */
    int32_t lr_step;          /* StepLR step_size (500) */
    float lr_gamma;           /* StepLR gamma (0.95) */
    float bn_momentum, bn_eps;                     /* torch.nn.BatchNorm2d defaults 0.1, 1e-5 */
    int64_t step0;            /* optimiser steps already taken (resume): Adam's bias correction and StepLR continue from here */
    int32_t probe_lbo, probe_sbo;                  /* 0 (measurement aid: override the wgrad operand descriptor strides) */
} szb_train_config;
enum { SZB_TRAIN_FORWARD_ONLY = 1,   /* losses only */
       SZB_TRAIN_NO_UPDATE = 2 };    /* forward + backward, gradients kept, no optimiser step */
enum { SZB_TRAIN_PARAMS = 0,         /* parameters and BatchNorm running buffers */
       SZB_TRAIN_GRADS = 1,          /* gradients of the last step */
       SZB_TRAIN_EXP_AVG = 2, SZB_TRAIN_EXP_AVG_SQ = 3,    /* Adam moments */
       SZB_TRAIN_ACTIVATIONS = 4,    /* read-only: "logits" [n][4672], "value" [n] of the last step */
       SZB_TRAIN_MOMENTUM_BUFFER = 5 };  /* SGD with momentum only: torch's per-parameter "momentum_buffer"; setting it marks the
                                          * buffers as existing (a resumed state), so the next step blends into them */
enum { SZB_TRAIN_ADAM = 0, SZB_TRAIN_SGD = 1 };
int szb_train_create(szb_ctx *ctx, const szb_train_config *cfg);
/* the optimiser of the trainer: Adam (the default, train_RL.py:187) or torch.optim.SGD(lr, momentum, dampening, weight_decay,
 * nesterov) with StepLR(lr_step, lr_gamma) stepped per batch, the supervised recipe of train_supervised.py:84-92.  SGD reads lr,
 * weight_decay, lr_step, lr_gamma and step0 from the config and ignores beta1, beta2 and eps; weight decay applies to every
 * parameter, BatchNorm's included.  Call after szb_train_create and before the first szb_train_step (SZB_ERR_STATE after it);
 * SZB_ERR_ARG for an unknown kind, negative momentum or dampening, or nesterov without momentum or with dampening.  Under SGD
 * the Adam moment kinds of szb_train_get / szb_train_set return SZB_ERR_STATE, and SZB_TRAIN_MOMENTUM_BUFFER is valid when
 * momentum is not 0. */
int szb_train_set_optimizer(szb_ctx *ctx, int32_t kind, float momentum, float dampening, int32_t nesterov);
int szb_train_destroy(szb_ctx *ctx);
/* copy named tensors (host or device pointers, fp32, torch layout) into / out of the trainer; `kind` as above.  Setting
 * SZB_TRAIN_PARAMS needs every parameter and running buffer of the state_dict once before the first step. */
int szb_train_set(szb_ctx *ctx, int32_t kind, int32_t n_tensors, const char *const *names, const float *const *data,
                  const int64_t *numel);
int szb_train_get(szb_ctx *ctx, int32_t kind, int32_t n_tensors, const char *const *names, float *const *data,
                  const int64_t *numel);
/* the packed self-play records the steps draw from (copied to the device once): states [n][119] as szb_encode emits them,
 * CSR policy targets (pi_off [n+1] starting at 0, policy indices, visit fractions), outcomes z [n] from the mover's side */
int szb_train_records(szb_ctx *ctx, int64_t n, const uint64_t *states, const int64_t *pi_off, const uint16_t *pi_index,
                      const float *pi_prob, const int8_t *z);
/* one optimiser step on the batch of record rows `rows` [n] (2 <= n <= cfg.batch); losses_out (may be null: no synchronisation)
 * receives {mse, cross entropy} of the batch BEFORE the update, as the reference prints them */
int szb_train_step(szb_ctx *ctx, int32_t n, const int32_t *rows, int32_t flags, float *losses_out);
/* {mse, cross entropy} of steps [first, first + count) since szb_train_create (every szb_train_step counts), from a device ring of
 * the last 65,536 steps: a loop can queue steps with losses_out = null and read the history in bulk.  Synchronises; reports a
 * kernel-side failure of any step run since the last check. */
int szb_train_loss_history(szb_ctx *ctx, int64_t first, int32_t count, float *out);
/* optimiser step counter: read (set = 0) or overwrite (set = 1) */
int szb_train_state(szb_ctx *ctx, int64_t *step_inout, int32_t set);

#ifdef __cplusplus
}
#endif
#endif /* SZB200_H */
