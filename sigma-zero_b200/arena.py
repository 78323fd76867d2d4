"""Arena play between two networks -- the promotion check of the reference's test_update.py (:26-83) -- with every
game of the match running concurrently on the GPU (SURVEY.md 8f rank 2; a "next" row: same engine, learning=False,
arg-max move with the lowest index on ties, as eval.py:92-100 / test_update.py:19-23 pick it).

Each network gets its own libszb200 context (its own weights, tree arenas and a full copy of the games); the two
contexts are kept in step by pushing every chosen move to both.  In game g the first network plays White when g is
even and Black when g is odd (the reference plays one game per colour per match).  Every ply both contexts search all
games (szb_search works on a context's whole batch) and each game takes the move of the context whose network is to
move in it.  Host logic only -- all chess and all search runs in the CUDA library."""
import numpy as np

from . import runtime
from .engine import Engine, EVAL_NET_BF16, EVAL_NET_FP32


def _evaluator(model):
    return EVAL_NET_FP32 if getattr(model, "precision", "bf16") == "fp32" else EVAL_NET_BF16


def play_match(model_a, model_b, num_games, args, c960=False, seed=0, max_plies=None, device=0, leaves_per_tree=None,
               eval_cache_slots=None):
    """Plays num_games games between model_a and model_b (arg-max of the visit counts, learning=False).  eval_cache_slots (default:
    args' 'eval_cache_slots', absent = off) gives each side's engine the exact evaluation cache: the same games, fewer evaluations.

    Returns {"score_a": points of model_a (win 1, draw 0.5), "results": per-game "1-0" / "0-1" / "1/2-1/2" / "*",
             "a_is_white": per-game bool, "plies": plies played, "moves": per-game list of the policy indices played}."""
    n_search = int(args["num_searches"])
    c_puct = float(args["C"])
    a_white = np.arange(num_games) % 2 == 0
    start_ids = ([int(np.random.default_rng([int(seed), g // 2]).integers(0, 960)) for g in range(num_games)]
                 if c960 else [-1] * num_games)                       # both colours of a pair start from the same position
    cache_slots = runtime.eval_cache_of(args if eval_cache_slots is None else {"eval_cache_slots": eval_cache_slots})
    engines = []
    for model in (model_a, model_b):
        e = Engine(max_games=num_games, max_searches=n_search, device=device, cohorts=1,
                   leaves_per_tree=int(args.get("leaves_per_tree", 1)) if leaves_per_tree is None else int(leaves_per_tree))
        e.load_state_dict(model.state_dict())
        e.reset(start_ids)
        e.set_eval_cache(cache_slots)
        engines.append(e)
    ev = (_evaluator(model_a), _evaluator(model_b))
    moves = [[] for _ in range(num_games)]
    plies = 0
    try:
        while max_plies is None or plies < max_plies:
            outcomes = engines[0].outcomes()
            live = outcomes == 0
            if not live.any():
                break
            white_to_move = plies % 2 == 0
            chosen = np.full(num_games, -1, dtype=np.int64)
            for k, e in enumerate(engines):
                mine = live & ((a_white == white_to_move) if k == 0 else (a_white != white_to_move))
                if not mine.any():
                    continue
                e.search(n_search, c_puct, False, ev[k], want_visits=False, want_children=False)
                idx, vis, cnt = e.root_children()
                for g in np.nonzero(mine)[0]:
                    n = int(cnt[g])
                    chosen[g] = int(idx[g, int(np.argmax(vis[g, :n]))])          # first maximum = lowest move index on ties
            who = np.nonzero(chosen >= 0)[0]
            for g in who:
                moves[g].append(int(chosen[g]))
            for e in engines:
                e.push(who, chosen[who])
            plies += 1
        final = engines[0].positions()
    finally:
        for e in engines:
            e.close()
    results, score_a = [], 0.0
    for g in range(num_games):
        o = final[g].outcome
        if o == 0:
            res = "*"
        elif o == 1:                                              # checkmate: the side to move lost
            res = "0-1" if final[g].turn else "1-0"
        else:
            res = "1/2-1/2"
        results.append(res)
        if res == "1/2-1/2":
            score_a += 0.5
        elif res != "*" and ((res == "1-0") == bool(a_white[g])):
            score_a += 1.0
    return {"score_a": score_a, "results": results, "a_is_white": a_white.tolist(), "plies": plies, "moves": moves}


def update_model(current_model, new_model, matches=1, args=None, threshold=0.55, c960=False, seed=0, max_plies=None):
    """test_update.update_model (:26-83) with its evident intent: True when the new network scores >= threshold of the
    points over `matches` pairs of games (one per colour).  (The reference compares a bound method with a colour at
    :72-77, so every game scores 0.5 there -- SURVEY.md Appendix H, not preserved.)"""
    args = args or {"C": 2, "num_searches": 800}
    out = play_match(new_model, current_model, 2 * matches, args, c960=c960, seed=seed, max_plies=max_plies)
    finished = sum(r != "*" for r in out["results"])
    return finished > 0 and out["score_a"] / finished >= threshold
