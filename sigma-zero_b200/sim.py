"""Drop-in for the reference's sim.py.  `play_game` keeps the reference signature (one game);
`generate_training_data` plays all `num_games` games concurrently on the GPU -- that batch is the product's
hot path (szb_selfplay_ply: search for every game, sample a move proportional to visits, push it)."""
import os

import numpy as np
import torch

from . import chess_compat as chess
from . import runtime
from .chess_tensor import index_move


def _empty_history():
    return {'states': [], 'actions': [], 'rewards': [], 'colours': []}


def selfplay_batch(model, args, num_games, c960=False, seed=None, start_ids=None, max_plies=None, learning=True,
                   sample=True, record=True, game_id_base=0):
    """Plays num_games games in lock step.  Returns one history dict per game (sim.py:38-43 schema) plus counters.

    With a `seed`, everything random about a game -- its Chess960 start position (the reference draws random.randint(0,
    959), chess_tensor.py:69), the moves sampled from the visit counts (sim.py:68) and the root noise of the opt-in exploration
    -- is a function of (seed, global game id = game_id_base + index) only, so a job sharded over ranks plays exactly the games
    a single process would.  args may carry 'dirichlet_alpha', 'dirichlet_epsilon' and 'sample_plies' (runtime.exploration_of);
    without them the engine's exploration is switched off.  'eval_cache_slots' (runtime.eval_cache_of) switches the exact
    evaluation cache on: the same games, fewer network evaluations."""
    n_search = int(args['num_searches'])
    explore = runtime.exploration_of(args)
    cache_slots = runtime.eval_cache_of(args)
    eng = runtime.get_engine(min_games=num_games, min_searches=n_search, leaves_per_tree=runtime.leaves_of(args))
    runtime.sync_weights(eng, model)
    eng.owner = None
    if seed is None:
        seed = int(np.random.default_rng().integers(0, 2 ** 62))
    if start_ids is None:
        start_ids = ([int(np.random.default_rng([int(seed), int(game_id_base) + g]).integers(0, 960)) for g in range(num_games)]
                     if c960 else np.full(num_games, -1))
    eng.reset(start_ids)
    eng.set_game_id_base(game_id_base)
    eng.set_exploration(seed=int(seed), **explore)
    eng.set_eval_cache(cache_slots)
    seed64 = int(seed)
    games = [_empty_history() for _ in range(num_games)]
    evaluator = runtime.evaluator_of(model)
    plies = 0
    active = num_games
    while active > 0 and (max_plies is None or plies < max_plies):
        if record:
            planes, _ = eng.encode(want_mask=False)
            pos = eng.positions()
        moves, active = eng.selfplay_ply(n_search, float(args['C']), learning, evaluator, seed=seed64, sample=sample)
        if record:
            idx, vis, cnt = eng.root_children()
            states = runtime.unpack_planes(planes)
            for g in range(num_games):
                if moves[g] < 0:
                    continue
                white = bool(pos[g].turn)
                k = int(cnt[g])
                total = int(vis[g, :k].sum())
                pawns = pos[g].pieces[0 if white else 6]
                probs = {}
                for i, c in zip(idx[g, :k], vis[g, :k]):
                    m = index_move(int(i), white)
                    if m.promotion is None and (pawns >> m.from_square) & 1 and m.to_square // 8 in (0, 7):
                        m = chess.make_move(m.from_square, m.to_square, chess.QUEEN)
                    probs[m] = int(c) / total
                h = games[g]
                h['states'].append(torch.from_numpy(states[g]))
                h['actions'].append(probs)
                h['colours'].append(white)
        plies += 1
    final = eng.positions()
    for g, h in enumerate(games):
        o = final[g].outcome
        result = "*" if o == 0 else ("1/2-1/2" if o != 1 else ("0-1" if final[g].turn else "1-0"))
        reward = 1 if result == "1-0" else (-1 if result == "0-1" else 0)
        h['rewards'] = [reward if i % 2 == 0 else -reward for i in range(len(h['actions']))]
        h['result'] = result
    return games, {"plies": plies, "simulations": plies * n_search * num_games}


def selfplay_records(model, args, num_games, c960=False, seed=None, start_ids=None, max_plies=None, learning=True,
                     sample=True, game_id_base=0):
    """The same games as selfplay_batch, recorded straight into the packed training format of records.py (no per-move
    Python objects): returns (records, counters).  records["game"] numbers the games of this call from 0; rows are ordered
    by game, then ply -- exactly records.pack_records(selfplay_batch(...)[0]).  records["result"] holds one outcome code
    per game: 1 white won, -1 black won, 0 draw, 2 unfinished (max_plies)."""
    n_search = int(args['num_searches'])
    explore = runtime.exploration_of(args)
    cache_slots = runtime.eval_cache_of(args)
    eng = runtime.get_engine(min_games=num_games, min_searches=n_search, leaves_per_tree=runtime.leaves_of(args))
    runtime.sync_weights(eng, model)
    eng.owner = None
    if seed is None:
        seed = int(np.random.default_rng().integers(0, 2 ** 62))
    if start_ids is None:
        start_ids = ([int(np.random.default_rng([int(seed), int(game_id_base) + g]).integers(0, 960)) for g in range(num_games)]
                     if c960 else np.full(num_games, -1))
    eng.reset(start_ids)
    eng.set_game_id_base(game_id_base)
    eng.set_exploration(seed=int(seed), **explore)
    eng.set_eval_cache(cache_slots)
    evaluator = runtime.evaluator_of(model)
    col = np.arange(256)[None, :]
    st, gm, pl, ix, pr, ln = [], [], [], [], [], []
    plies, active, sims = 0, num_games, 0
    while active > 0 and (max_plies is None or plies < max_plies):
        planes, _ = eng.encode(want_mask=False)
        moves, active = eng.selfplay_ply(n_search, float(args['C']), learning, evaluator, seed=int(seed), sample=sample)
        idx, vis, cnt = eng.root_children()
        live = np.nonzero(moves >= 0)[0]
        if len(live):
            k = cnt[live].astype(np.int64)
            sel = col < k[:, None]
            v = vis[live].astype(np.int64)
            tot = (v * sel).sum(axis=1)
            st.append(planes[live])
            gm.append(live.astype(np.int32))
            pl.append(np.full(len(live), plies, dtype=np.int32))
            ix.append(idx[live][sel])
            pr.append((v / tot[:, None])[sel].astype(np.float32))      # count / sum(count) in double, like mcts.py:113-122
            ln.append(k)
            sims += len(live) * n_search
        plies += 1
    final = eng.positions()
    result = np.array([2 if p.outcome == 0 else (0 if p.outcome != 1 else (-1 if p.turn else 1)) for p in final], dtype=np.int8)
    if not st:
        rec = {"states": np.zeros((0, 119), np.uint64), "pi_index": np.zeros(0, np.uint16), "pi_prob": np.zeros(0, np.float32),
               "pi_off": np.zeros(1, np.int64), "z": np.zeros(0, np.int8), "colour": np.zeros(0, bool), "game": np.zeros(0, np.int32),
               "result": result}
        return rec, {"plies": plies, "simulations": sims}
    states, game, ply, length = np.concatenate(st), np.concatenate(gm), np.concatenate(pl), np.concatenate(ln)
    start = np.concatenate([[0], np.cumsum(length)])[:-1]              # CSR start of every recorded position, in recording order
    order = np.lexsort((ply, game))                                     # by game, then ply
    flat_i, flat_p = np.concatenate(ix), np.concatenate(pr)
    game, ply, length = game[order], ply[order], length[order]
    new_off = np.concatenate([[0], np.cumsum(length)])
    rows = np.repeat(start[order] - new_off[:-1], length) + np.arange(new_off[-1])      # gather of the CSR payload
    reward = np.where(result == 2, 0, result).astype(np.int8)[game]
    z = np.where(ply % 2 == 0, reward, -reward).astype(np.int8)          # sim.py:86-97: +r for even positions, -r for odd
    rec = {"states": states[order], "pi_index": flat_i[rows].astype(np.uint16), "pi_prob": flat_p[rows],
           "pi_off": new_off.astype(np.int64), "z": z,
           "colour": states[order][:, 112] != 0, "game": game, "result": result}
    return rec, {"plies": plies, "simulations": sims}


def play_game(model, args, c960=False):
    """One self-play game (reference signature, sim.py:31-99)."""
    games, _ = selfplay_batch(model, args, 1, c960=c960)
    h = games[0]
    print("Result", h.pop('result'))
    return h


def generate_training_data(model, num_games=1, args=None, return_dict=None, c960=False):
    """num_games self-play games, concatenated like sim.py:102-123 -- but played concurrently on the GPU."""
    games, _ = selfplay_batch(model, args, num_games, c960=c960)
    out = _empty_history()
    for h in games:
        for key in out:
            out[key] += h[key]
    if return_dict is not None:
        return_dict[os.getpid()] = out
    return out
