"""ctypes binding of include/szb200.h.  Fails loudly when the CUDA library is missing: there is no fallback."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SZB_LIB") or os.path.join(HERE, "libszb200.so")     # SZB_LIB: A/B-test another build of the library

N_PLANES, N_ACTIONS, MASK_WORDS, MAX_MOVES = 119, 4672, 73, 256
EVAL_NET_BF16, EVAL_NET_FP32, EVAL_HASH = 0, 1, 2
ERR_ILLEGAL_MOVE = -3


class SzbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("szb200 error %d: %s" % (code, msg))
        self.code = code


class Config(ctypes.Structure):
    _fields_ = [("max_games", ctypes.c_int32), ("max_searches", ctypes.c_int32),
                ("edges_per_node", ctypes.c_int32), ("cohorts", ctypes.c_int32), ("leaves_per_tree", ctypes.c_int32)]


class Pos(ctypes.Structure):
    _fields_ = [("pieces", ctypes.c_uint64 * 12), ("turn", ctypes.c_uint8), ("castling_w", ctypes.c_uint8),
                ("castling_b", ctypes.c_uint8), ("ep_square", ctypes.c_int8), ("halfmove_clock", ctypes.c_uint16),
                ("ply", ctypes.c_uint16), ("chess960", ctypes.c_uint8), ("outcome", ctypes.c_uint8),
                ("rep_flags", ctypes.c_uint8), ("n_legal", ctypes.c_uint8), ("pad", ctypes.c_uint8 * 4)]


class Stats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint64) for n in
                ("simulations", "evaluations", "terminal_visits", "edges_allocated", "kernel_launches", "max_depth")]


class PhaseTimes(ctypes.Structure):
    _fields_ = [("select_ms", ctypes.c_float), ("expand_ms", ctypes.c_float), ("eval_ms", ctypes.c_float),
                ("finish_ms", ctypes.c_float), ("steps", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("select_edges", ctypes.c_uint64), ("select_levels", ctypes.c_uint64),
                ("backup_levels", ctypes.c_uint64), ("edges_written", ctypes.c_uint64),
                ("conv_ms", ctypes.c_float), ("conv_launches", ctypes.c_int32), ("conv_boards", ctypes.c_int32),
                ("conv_kind", ctypes.c_int32), ("conv_flop", ctypes.c_uint64)]


class TowerSpans(ctypes.Structure):
    _fields_ = [("launches", ctypes.c_int32), ("reserved", ctypes.c_int32), ("boards", ctypes.c_uint64),
                ("busy_ns", ctypes.c_uint64), ("wall_ns", ctypes.c_uint64), ("flop", ctypes.c_uint64),
                ("sm_cycles", ctypes.c_uint64), ("sm_ns", ctypes.c_uint64)]


class TrainConfig(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("lr", ctypes.c_float), ("beta1", ctypes.c_float), ("beta2", ctypes.c_float),
                ("eps", ctypes.c_float), ("weight_decay", ctypes.c_float), ("lr_step", ctypes.c_int32), ("lr_gamma", ctypes.c_float),
                ("bn_momentum", ctypes.c_float), ("bn_eps", ctypes.c_float), ("step0", ctypes.c_int64),
                ("probe_lbo", ctypes.c_int32), ("probe_sbo", ctypes.c_int32)]


class Exploration(ctypes.Structure):
    _fields_ = [("dirichlet_alpha", ctypes.c_float), ("dirichlet_epsilon", ctypes.c_float), ("seed", ctypes.c_uint64),
                ("sample_plies", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class EvalCacheStats(ctypes.Structure):
    _fields_ = [("lookups", ctypes.c_uint64), ("hits", ctypes.c_uint64), ("inserts", ctypes.c_uint64),
                ("dropped_inserts", ctypes.c_uint64), ("boards_evaluated", ctypes.c_uint64), ("bytes", ctypes.c_uint64),
                ("slots_per_game", ctypes.c_int32), ("reserved", ctypes.c_int32)]


TRAIN_FORWARD_ONLY, TRAIN_NO_UPDATE = 1, 2
TRAIN_PARAMS, TRAIN_GRADS, TRAIN_EXP_AVG, TRAIN_EXP_AVG_SQ, TRAIN_ACTIVATIONS, TRAIN_MOMENTUM_BUFFER = 0, 1, 2, 3, 4, 5
TRAIN_ADAM, TRAIN_SGD = 0, 1

_vp, _i32, _u64, _f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_uint64, ctypes.c_float
SIGNATURES = {
    "szb_version": (ctypes.c_char_p, []),
    "szb_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(Config), ctypes.POINTER(_vp)]),
    "szb_destroy": (None, [_vp]),
    "szb_last_error": (ctypes.c_char_p, [_vp]),
    "szb_stream": (_vp, [_vp]),
    "szb_synchronize": (ctypes.c_int, [_vp]),
    "szb_games_reset": (ctypes.c_int, [_vp, _i32, _vp]),
    "szb_games_set": (ctypes.c_int, [_vp, _i32, _vp]),
    "szb_games_push": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "szb_games_get": (ctypes.c_int, [_vp, _i32, _vp, _vp]),
    "szb_legal_moves": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "szb_encode": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "szb_unpack_planes_f32": (ctypes.c_int, [_vp, _i32, _vp, _vp]),
    "szb_perft": (ctypes.c_int, [_vp, ctypes.POINTER(Pos), _i32, ctypes.POINTER(_u64)]),
    "szb_perft_timed": (ctypes.c_int, [_vp, ctypes.POINTER(Pos), _i32, ctypes.POINTER(_u64),
                                       ctypes.POINTER(_f32), ctypes.POINTER(_u64)]),
    "szb_net_load": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "szb_net_load_device": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "szb_net_checksum": (ctypes.c_int, [_vp, ctypes.POINTER(_u64)]),
    "szb_net_forward": (ctypes.c_int, [_vp, _i32, _vp, _i32, _vp, _vp]),
    "szb_net_forward_logits": (ctypes.c_int, [_vp, _i32, _vp, _i32, _vp, _vp]),
    "szb_search": (ctypes.c_int, [_vp, _i32, _f32, _i32, _i32, _vp, _vp, _vp]),
    "szb_root_children": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "szb_tree_export": (ctypes.c_int, [_vp, _i32, _i32, _i32] + [_vp] * 11 + [ctypes.POINTER(_i32), ctypes.POINTER(ctypes.c_double),
                                                                          ctypes.POINTER(_i32), ctypes.POINTER(_i32)]),
    "szb_selfplay_ply": (ctypes.c_int, [_vp, _i32, _f32, _i32, _i32, _u64, _i32, _vp, _vp]),
    "szb_set_game_id_base": (ctypes.c_int, [_vp, _u64]),
    "szb_set_exploration": (ctypes.c_int, [_vp, ctypes.POINTER(Exploration)]),
    "szb_set_eval_cache": (ctypes.c_int, [_vp, _i32]),
    "szb_get_eval_cache_stats": (ctypes.c_int, [_vp, ctypes.POINTER(EvalCacheStats), _vp]),
    "szb_get_stats": (ctypes.c_int, [_vp, ctypes.POINTER(Stats)]),
    "szb_set_profiling": (ctypes.c_int, [_vp, _i32]),
    "szb_get_phase_times": (ctypes.c_int, [_vp, ctypes.POINTER(PhaseTimes)]),
    "szb_time_kernel": (ctypes.c_int, [_vp, _i32, _i32, _i32, ctypes.POINTER(_f32)]),
    "szb_tower_spans_record": (ctypes.c_int, [_vp, _i32, ctypes.POINTER(TowerSpans)]),
    "szb_train_create": (ctypes.c_int, [_vp, ctypes.POINTER(TrainConfig)]),
    "szb_train_set_optimizer": (ctypes.c_int, [_vp, _i32, _f32, _f32, _i32]),
    "szb_train_destroy": (ctypes.c_int, [_vp]),
    "szb_train_set": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "szb_train_get": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "szb_train_records": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "szb_train_step": (ctypes.c_int, [_vp, _i32, _vp, _i32, _vp]),
    "szb_train_loss_history": (ctypes.c_int, [_vp, ctypes.c_int64, _i32, _vp]),
    "szb_train_state": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_int64), _i32]),
}

_lib = None


def load():
    """Returns the loaded library; raises if libszb200.so has not been built (python sigma-zero_b200/build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SzbError(-2, "libszb200.so is not built (%s); run `python __graft_entry__.py` or "
                               "`python sigma-zero_b200/build.py`. There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here == header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
