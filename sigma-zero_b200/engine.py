"""Engine: one libszb200 context (one GPU) with numpy-friendly methods.  Host logic only -- all compute is in
the CUDA library."""
import ctypes

import numpy as np

from . import _lib
from ._lib import EVAL_HASH, EVAL_NET_BF16, EVAL_NET_FP32, MASK_WORDS, MAX_MOVES, N_ACTIONS, N_PLANES, SzbError

__all__ = ["Engine", "EVAL_HASH", "EVAL_NET_BF16", "EVAL_NET_FP32", "SzbError"]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class Engine:
    def __init__(self, max_games=1024, max_searches=800, device=0, edges_per_node=0, cohorts=0, leaves_per_tree=1):
        """leaves_per_tree: 1 = the reference's search (one simulation of a tree at a time; what every parity test runs);
        2..8 = that many simulations of a tree in flight per step with virtual loss -- a different, opt-in search"""
        self.lib = _lib.load()
        self.max_games, self.max_searches = int(max_games), int(max_searches)
        self.leaves_per_tree = int(leaves_per_tree)
        cfg = _lib.Config(self.max_games, self.max_searches, int(edges_per_node), int(cohorts), self.leaves_per_tree)
        h = ctypes.c_void_p()
        rc = self.lib.szb_create(int(device), ctypes.byref(cfg), ctypes.byref(h))
        self._h = h
        if rc != 0:
            msg = self.lib.szb_last_error(h).decode() if h else "szb_create failed (no CUDA device?)"
            if h:
                self.lib.szb_destroy(h)
            self._h = None
            raise SzbError(rc, msg)
        self.device = int(device)
        self.n_games = 0
        self.weights_loaded = False

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.szb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise SzbError(rc, self.lib.szb_last_error(self._h).decode())

    @property
    def stream(self):
        return self.lib.szb_stream(self._h)

    def synchronize(self):
        self._check(self.lib.szb_synchronize(self._h))

    # ---- games -------------------------------------------------------------------------------
    def reset(self, start_ids):
        ids = np.ascontiguousarray(start_ids, dtype=np.int16)
        self._check(self.lib.szb_games_reset(self._h, len(ids), _ptr(ids)))
        self.n_games = len(ids)

    def set_positions(self, positions):
        arr = (_lib.Pos * len(positions))(*positions)
        self._check(self.lib.szb_games_set(self._h, len(positions), ctypes.cast(arr, ctypes.c_void_p)))
        self.n_games = len(positions)

    def set_positions_buffer(self, buf, n):
        """buf: contiguous host array holding n szb_pos structs (112 bytes each), e.g. a view of pinned memory"""
        assert buf.nbytes >= n * ctypes.sizeof(_lib.Pos)
        self._check(self.lib.szb_games_set(self._h, int(n), _ptr(buf)))
        self.n_games = int(n)

    def push(self, games, move_indices, raise_on_illegal=True):
        games = None if games is None else np.ascontiguousarray(games, dtype=np.int32)
        idx = np.ascontiguousarray(move_indices, dtype=np.uint16)
        status = np.zeros(len(idx), dtype=np.int32)
        rc = self.lib.szb_games_push(self._h, len(idx), _ptr(games), _ptr(idx), _ptr(status))
        if rc == _lib.ERR_ILLEGAL_MOVE and not raise_on_illegal:
            return status
        if rc == _lib.ERR_ILLEGAL_MOVE:
            raise ValueError("Invalid move")
        self._check(rc)
        return status

    def positions(self, games=None, n=None):
        games = None if games is None else np.ascontiguousarray(games, dtype=np.int32)
        n = len(games) if games is not None else (self.n_games if n is None else n)
        out = (_lib.Pos * n)()
        self._check(self.lib.szb_games_get(self._h, n, _ptr(games), ctypes.cast(out, ctypes.c_void_p)))
        return out

    def outcomes(self):
        return np.array([p.outcome for p in self.positions()], dtype=np.uint8)

    def legal_moves(self, games=None):
        games = None if games is None else np.ascontiguousarray(games, dtype=np.int32)
        n = len(games) if games is not None else self.n_games
        idx = np.zeros((n, MAX_MOVES), dtype=np.uint16)
        cnt = np.zeros(n, dtype=np.uint16)
        self._check(self.lib.szb_legal_moves(self._h, n, _ptr(games), _ptr(idx), _ptr(cnt)))
        return idx, cnt

    def encode(self, games=None, want_mask=True):
        games = None if games is None else np.ascontiguousarray(games, dtype=np.int32)
        n = len(games) if games is not None else self.n_games
        planes = np.zeros((n, N_PLANES), dtype=np.uint64)
        mask = np.zeros((n, MASK_WORDS), dtype=np.uint64) if want_mask else None
        self._check(self.lib.szb_encode(self._h, n, _ptr(games), _ptr(planes), _ptr(mask)))
        return planes, mask

    # ---- perft -------------------------------------------------------------------------------
    def perft(self, pos, depth, timed=False):
        nodes = ctypes.c_uint64()
        if not timed:
            self._check(self.lib.szb_perft(self._h, ctypes.byref(pos), int(depth), ctypes.byref(nodes)))
            return nodes.value
        ms, npos = ctypes.c_float(), ctypes.c_uint64()
        self._check(self.lib.szb_perft_timed(self._h, ctypes.byref(pos), int(depth), ctypes.byref(nodes),
                                             ctypes.byref(ms), ctypes.byref(npos)))
        return nodes.value, ms.value, npos.value

    # ---- network -----------------------------------------------------------------------------
    def load_state_dict(self, state_dict):
        """state_dict: mapping name -> torch tensor / ndarray with network.py's 252 keys."""
        names, arrays = [], []
        for k, v in state_dict.items():
            if k.endswith("num_batches_tracked"):
                continue
            a = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
            names.append(k.encode())
            arrays.append(np.ascontiguousarray(a, dtype=np.float32))
        n = len(names)
        c_names = (ctypes.c_char_p * n)(*names)
        c_data = (ctypes.c_void_p * n)(*[a.ctypes.data for a in arrays])
        c_numel = (ctypes.c_int64 * n)(*[a.size for a in arrays])
        self._check(self.lib.szb_net_load(self._h, n, ctypes.cast(c_names, ctypes.c_void_p),
                                          ctypes.cast(c_data, ctypes.c_void_p), ctypes.cast(c_numel, ctypes.c_void_p)))
        self.weights_loaded = True

    def load_flat_device(self, keys, numels, flat):
        """Weights from ONE flat fp32 CUDA tensor (torch) laid out as the concatenation of the state_dict tensors `keys` with
        `numels` elements each -- e.g. the buffer torch.distributed just broadcast.  Folding and packing run on the GPU
        (szb_net_load_device); nothing crosses the host."""
        import torch
        assert flat.is_cuda and flat.dtype == torch.float32 and flat.is_contiguous() and flat.device.index == self.device
        base, n = flat.data_ptr(), len(keys)
        offs = np.concatenate([[0], np.cumsum(numels)])
        assert int(offs[-1]) == flat.numel()
        c_names = (ctypes.c_char_p * n)(*[k.encode() for k in keys])
        c_data = (ctypes.c_void_p * n)(*[base + 4 * int(o) for o in offs[:-1]])
        c_numel = (ctypes.c_int64 * n)(*[int(x) for x in numels])
        # the fold kernels run on the library's stream: order them after the producer of `flat` on torch's current stream
        torch.cuda.current_stream(flat.device).synchronize()
        self._check(self.lib.szb_net_load_device(self._h, n, ctypes.cast(c_names, ctypes.c_void_p),
                                                 ctypes.cast(c_data, ctypes.c_void_p), ctypes.cast(c_numel, ctypes.c_void_p)))
        self.synchronize()                                   # `flat` may be freed or overwritten by the caller from here on
        self.weights_loaded = True

    def net_checksum(self):
        h = ctypes.c_uint64()
        self._check(self.lib.szb_net_checksum(self._h, ctypes.byref(h)))
        return h.value

    def net_forward(self, planes, evaluator=EVAL_NET_BF16, logits=False):
        planes = np.ascontiguousarray(planes, dtype=np.uint64).reshape(-1, N_PLANES)
        n = planes.shape[0]
        pol = np.zeros((n, N_ACTIONS), dtype=np.float32)
        val = np.zeros(n, dtype=np.float32)
        fn = self.lib.szb_net_forward_logits if logits else self.lib.szb_net_forward
        self._check(fn(self._h, n, _ptr(planes), int(evaluator), _ptr(pol), _ptr(val)))
        return pol, val

    # ---- search ------------------------------------------------------------------------------
    def search(self, num_searches, c_puct=2.0, learning=False, evaluator=EVAL_NET_BF16,
               want_visits=True, want_children=True, want_value=False, out=None):
        """out: optional (visits uint32[G,4672], child_mask uint64[G,73], root_value float32[G]) host arrays to fill
        (e.g. views of pinned memory); entries may be None."""
        G = self.n_games
        if out is not None:
            visits, child, val = out
        else:
            visits = np.zeros((G, N_ACTIONS), dtype=np.uint32) if want_visits else None
            child = np.zeros((G, MASK_WORDS), dtype=np.uint64) if want_children else None
            val = np.zeros(G, dtype=np.float32) if want_value else None
        self._check(self.lib.szb_search(self._h, int(num_searches), float(c_puct), int(bool(learning)), int(evaluator),
                                        _ptr(visits), _ptr(child), _ptr(val)))
        return visits, child, val

    def root_children(self):
        """(index uint16[G,256], visits uint32[G,256], count uint16[G]) of the last search"""
        G = self.n_games
        idx = np.zeros((G, MAX_MOVES), dtype=np.uint16)
        vis = np.zeros((G, MAX_MOVES), dtype=np.uint32)
        cnt = np.zeros(G, dtype=np.uint16)
        self._check(self.lib.szb_root_children(self._h, _ptr(idx), _ptr(vis), _ptr(cnt)))
        return idx, vis, cnt

    def tree_export(self, game=0):
        """dict of numpy arrays describing one game's search tree (see szb_tree_export)"""
        mn = self.max_searches + 1
        me = mn * 218
        a = dict(node_first=np.zeros(mn, np.int32), node_count=np.zeros(mn, np.int32), node_parent=np.zeros(mn, np.int32),
                 node_parent_edge=np.zeros(mn, np.int32), node_terminal=np.zeros(mn, np.uint8),
                 node_terminal_value=np.zeros(mn, np.float32), edge_visits=np.zeros(me, np.int32),
                 edge_value_sum=np.zeros(me, np.float64), edge_prior=np.zeros(me, np.float32),
                 edge_move=np.zeros(me, np.uint16), edge_child=np.zeros(me, np.int32))
        rn, rw, nn, ne = ctypes.c_int32(), ctypes.c_double(), ctypes.c_int32(), ctypes.c_int32()
        self._check(self.lib.szb_tree_export(self._h, int(game), mn, me, *[_ptr(v) for v in a.values()],
                                             ctypes.byref(rn), ctypes.byref(rw), ctypes.byref(nn), ctypes.byref(ne)))
        out = {k: (v[:nn.value] if k.startswith("node_") else v[:ne.value]) for k, v in a.items()}
        out["root_visits"], out["root_value_sum"] = rn.value, rw.value
        return out

    def selfplay_ply(self, num_searches, c_puct=2.0, learning=True, evaluator=EVAL_NET_BF16, seed=0, sample=True):
        moves = np.zeros(self.n_games, dtype=np.int32)
        active = ctypes.c_int32()
        self._check(self.lib.szb_selfplay_ply(self._h, int(num_searches), float(c_puct), int(bool(learning)),
                                              int(evaluator), int(seed), int(bool(sample)), _ptr(moves),
                                              ctypes.cast(ctypes.byref(active), ctypes.c_void_p)))
        return moves, active.value

    def set_game_id_base(self, base):
        """global id of game 0 (keys the move-sampling RNG so that shards of one job play the same games)"""
        self._check(self.lib.szb_set_game_id_base(self._h, int(base)))

    def set_exploration(self, alpha=0.0, epsilon=0.25, seed=0, sample_plies=0):
        """Opt-in AlphaZero exploration for the searches and self-play plies that follow (szb_set_exploration): with alpha > 0,
        searches with learning=True mix Dirichlet(alpha) noise into the root's priors with weight epsilon (keyed by seed, global
        game id and ply) and give every other node its raw priors; sample_plies > 0 makes selfplay_ply(sample=True) play the
        arg-max from that ply of the game on.  alpha=0, sample_plies=0: the reference's behaviour."""
        x = _lib.Exploration(float(alpha), float(epsilon), int(seed) & (2 ** 64 - 1), int(sample_plies), 0)
        self._check(self.lib.szb_set_exploration(self._h, ctypes.byref(x)))

    def set_eval_cache(self, slots_per_game=0):
        """Opt-in exact evaluation cache for the searches that follow (szb_set_eval_cache): per game a table of slots_per_game
        entries (0 = off, else a power of two in [64, 65536]) keyed on the exact evaluator input, so that positions an earlier
        search of the same game evaluated skip the network.  Results are bit-identical with the cache on and off."""
        self._check(self.lib.szb_set_eval_cache(self._h, int(slots_per_game)))

    def eval_cache_stats(self, game_hits=False):
        """Cumulative counters of the evaluation cache (lookups, hits, inserts, dropped_inserts, boards_evaluated, bytes,
        slots_per_game); with game_hits=True also each game's hits in the last search (uint32[n_games])."""
        s = _lib.EvalCacheStats()
        hits = np.zeros(max(self.n_games, 1), dtype=np.uint32) if game_hits else None
        self._check(self.lib.szb_get_eval_cache_stats(self._h, ctypes.byref(s), _ptr(hits) if game_hits else None))
        out = {n: getattr(s, n) for n, _ in _lib.EvalCacheStats._fields_ if n != "reserved"}
        if game_hits:
            out["game_hits"] = hits[:self.n_games]
        return out

    def set_profiling(self, on=True):
        self._check(self.lib.szb_set_profiling(self._h, int(bool(on))))

    def phase_times(self):
        t = _lib.PhaseTimes()
        self._check(self.lib.szb_get_phase_times(self._h, ctypes.byref(t)))
        return {n: getattr(t, n) for n, _ in _lib.PhaseTimes._fields_ if n != "reserved"}

    def time_kernel(self, which, n, iters=20):
        ms = ctypes.c_float()
        self._check(self.lib.szb_time_kernel(self._h, int(which), int(n), int(iters), ctypes.byref(ms)))
        return ms.value

    def tower_spans(self, on):
        """on=True: start recording the device start / end time of every whole-tower launch; on=False: stop and return the totals"""
        if on:
            self._check(self.lib.szb_tower_spans_record(self._h, 1, None))
            return None
        t = _lib.TowerSpans()
        self._check(self.lib.szb_tower_spans_record(self._h, 0, ctypes.byref(t)))
        return {n: getattr(t, n) for n, _ in _lib.TowerSpans._fields_ if n != "reserved"}

    def stats(self):
        s = _lib.Stats()
        self._check(self.lib.szb_get_stats(self._h, ctypes.byref(s)))
        return {n: getattr(s, n) for n, _ in _lib.Stats._fields_}


def child_indices(child_mask_row):
    """uint64[73] bitset -> ascending policy indices."""
    bits = np.unpackbits(np.ascontiguousarray(child_mask_row, dtype="<u8").view(np.uint8), bitorder="little")
    return np.nonzero(bits[:N_ACTIONS])[0]
