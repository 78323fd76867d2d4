"""What the opt-in exact evaluation cache (szb_set_eval_cache) saves in self-play, in one call with the arms alternating:

  * off: every non-terminal leaf goes through the network;
  * on:  2048 entries per game; leaves whose exact input an earlier search of the same game evaluated skip the network.

Config c2's size: 1024 vanilla games x 800 simulations per move, bf16 network, `--plies` self-play plies per repetition (search +
pick + push, each call ends in a device synchronisation).  Per ply it reports the median time over the repetitions of each arm,
and for the cache arm the hit rate, the boards the network evaluated, and the played child's mean share of the previous
search's root visits -- the share of the previous tree the next search can find in the cache.  Both arms must play the same moves
(asserted).

Two networks: policyNN as initialised with torch seed 0 ("random": flat visit distributions), and the same network with its policy
output layer scaled by --policy-scale ("synthetic_peaked": visits concentrate roughly as a trained network's do; NOT a trained
network).  Also one game's 800-simulation search (PlayTensor-style: arg-max move, learning=False), off vs on.

Writes eval_cache_cost.json into --out with the card's name and power limit read in the same run.  One network at c2's size takes
about five minutes, so the two can run as separate calls: the second with --merge <the first's file> carries the first's sections
(and its card reading, under "card_by_network") into its own file.

    python scripts/eval_cache_cost.py [--plies 24] [--reps 5] [--policy-scale 8] [--networks random,synthetic_peaked]
                                      [--merge FILE] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sigma_zero_b200.engine import EVAL_NET_BF16, Engine
from sigma_zero_b200.network import policyNN

SLOTS = 2048


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def weights(scale):
    torch.manual_seed(0)
    sd = policyNN({}).eval().state_dict()
    return {k: (v * scale if k.startswith("conv_p2.") and scale != 1.0 else v) for k, v in sd.items()}


def run_arm(eng, games, sims, plies, slots, seed):
    """times of `plies` self-play plies; per ply the moves, cache counters and the played child's share of the root visits"""
    eng.set_eval_cache(0)                                # a fresh table per repetition
    eng.set_eval_cache(slots)
    eng.reset(np.full(games, -1))
    rows = []
    prev = eng.eval_cache_stats()
    for _ in range(plies):
        t0 = time.perf_counter()
        mv, _ = eng.selfplay_ply(sims, 2.0, True, EVAL_NET_BF16, seed=seed, sample=True)
        ms = (time.perf_counter() - t0) * 1e3
        idx, vis, cnt = eng.root_children()
        shares = []
        for g in np.nonzero(mv >= 0)[0]:
            k = int(cnt[g])
            tot = float(vis[g, :k].sum())
            shares.append(float(vis[g, :k][idx[g, :k] == mv[g]].sum()) / tot if tot else 0.0)
        cur = eng.eval_cache_stats()
        rows.append({"ms": ms, "moves": mv, "lookups": cur["lookups"] - prev["lookups"], "hits": cur["hits"] - prev["hits"],
                     "boards_evaluated": cur["boards_evaluated"] - prev["boards_evaluated"],
                     "dropped_inserts": cur["dropped_inserts"] - prev["dropped_inserts"],
                     "played_share": float(np.mean(shares)) if shares else 0.0})
        prev = cur
    return rows


def selfplay_study(eng, a):
    arms = {"off": 0, "on": SLOTS}
    for slots in arms.values():                           # warm-up: modules, staging buffers, the network's first launches
        run_arm(eng, a.games, a.sims, 1, slots, seed=1)
    runs = {k: [] for k in arms}
    for _ in range(a.reps):                               # alternate the arms: drift of the shared host hits both alike
        for k, slots in arms.items():
            runs[k].append(run_arm(eng, a.games, a.sims, a.plies, slots, seed=1))
    for r in runs["off"] + runs["on"]:
        assert all(np.array_equal(x["moves"], y["moves"]) for x, y in zip(r, runs["off"][0])), "cache on must play the same moves"
    per_ply = []
    for p in range(a.plies):
        off = [r[p]["ms"] for r in runs["off"]]
        on = [r[p]["ms"] for r in runs["on"]]
        c = runs["on"][0][p]
        per_ply.append({"ply": p, "ms_off_median": float(np.median(off)), "ms_on_median": float(np.median(on)),
                        "ms_off_each_rep": off, "ms_on_each_rep": on,
                        "lookups": c["lookups"], "hits": c["hits"], "hit_rate": c["hits"] / max(c["lookups"], 1),
                        "boards_evaluated": c["boards_evaluated"], "dropped_inserts": c["dropped_inserts"],
                        "played_child_share_of_previous_search": runs["off"][0][p - 1]["played_share"] if p else None})
    tot_off = [sum(x["ms"] for x in r) for r in runs["off"]]
    tot_on = [sum(x["ms"] for x in r) for r in runs["on"]]
    c = runs["on"][0]
    return {"per_ply": per_ply,
            "total_ms_off_median": float(np.median(tot_off)), "total_ms_on_median": float(np.median(tot_on)),
            "total_ms_off_each_rep": tot_off, "total_ms_on_each_rep": tot_on,
            "on_over_off": float(np.median(tot_on) / np.median(tot_off)),
            "hit_rate_all_plies": sum(x["hits"] for x in c) / max(sum(x["lookups"] for x in c), 1),
            "mean_played_child_share": float(np.mean([x["played_share"] for x in runs["off"][0][:-1]]))}


def single_game_study(sd, a):
    """one game, arg-max move, learning=False: per-move time of a `--sims` search, off vs on, over `--single-moves` moves"""
    out = {}
    moves_of = {}
    for k, slots in (("off", 0), ("on", SLOTS)):
        eng = Engine(max_games=1, max_searches=a.sims, device=0)
        eng.load_state_dict(sd)
        ms_all = []
        for rep in range(a.reps + 1):                     # repetition 0 warms up
            eng.set_eval_cache(0)
            eng.set_eval_cache(slots)
            eng.reset([-1])
            ms, mv = [], []
            for _ in range(a.single_moves):
                t0 = time.perf_counter()
                eng.search(a.sims, 2.0, False, EVAL_NET_BF16, want_visits=False, want_children=False)
                ms.append((time.perf_counter() - t0) * 1e3)
                idx, vis, cnt = eng.root_children()
                best = int(idx[0, int(np.argmax(vis[0, :cnt[0]]))])
                mv.append(best)
                eng.push([0], [best])
                if eng.outcomes()[0] != 0:
                    break
            if rep:
                ms_all.append(float(np.mean(ms[1:])) if len(ms) > 1 else float(ms[0]))
            moves_of[k] = mv
        st = eng.eval_cache_stats()
        out[k] = {"ms_per_move_median": float(np.median(ms_all)), "ms_per_move_each_rep": ms_all,
                  "hit_rate": st["hits"] / max(st["lookups"], 1) if slots else None}
        eng.close()
    assert moves_of["off"] == moves_of["on"], "cache on must play the same moves"
    out["on_over_off"] = out["on"]["ms_per_move_median"] / out["off"]["ms_per_move_median"]
    out["note"] = "mean over moves 2.. of a game (move 1 starts from an empty table), median over repetitions"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--plies", type=int, default=24)
    ap.add_argument("--single-moves", type=int, default=8)
    ap.add_argument("--policy-scale", type=float, default=8.0)
    ap.add_argument("--networks", default="random,synthetic_peaked", help="comma-separated subset of random, synthetic_peaked")
    ap.add_argument("--merge", default=None, help="eval_cache_cost.json of an earlier run whose network sections to carry over")
    ap.add_argument("--out", default=".")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    before = card()
    result = {"card": before, "torch": torch.__version__,
              "config": {"games": a.games, "simulations_per_move": a.sims, "plies": a.plies, "reps": a.reps, "slots_per_game": SLOTS,
                         "start": "vanilla", "c_puct": 2.0, "learning": True, "sampled_moves": True, "policy_scale": a.policy_scale}}
    nets = [(n, s) for n, s in (("random", 1.0), ("synthetic_peaked", a.policy_scale)) if n in a.networks.split(",")]
    eng = Engine(max_games=a.games, max_searches=a.sims, device=0)
    for name, scale in nets:
        eng.load_state_dict(weights(scale))
        result[name] = selfplay_study(eng, a)
        result[name]["network"] = ("policyNN({}) with torch seed 0" if scale == 1.0 else
                                   "SYNTHETIC: policyNN({}) with torch seed 0, conv_p2 weight and bias x %g (not a trained network)" % scale)
        r = result[name]
        print("%s: %.0f ms off, %.0f ms on for %d plies (x%.3f); hit rate %.3f; played child's share %.3f"
              % (name, r["total_ms_off_median"], r["total_ms_on_median"], a.plies, r["on_over_off"], r["hit_rate_all_plies"],
                 r["mean_played_child_share"]))
    eng.close()
    result["single_game"] = {name: single_game_study(weights(scale), a) for name, scale in nets}
    for name, r in result["single_game"].items():
        print("single game, %s: %.2f ms off, %.2f ms on per move (x%.3f)" % (name, r["off"]["ms_per_move_median"],
                                                                             r["on"]["ms_per_move_median"], r["on_over_off"]))
    result["card_after"] = card()["nvidia_smi"]
    result["card_by_network"] = {name: {"card": before, "card_after": result["card_after"], "config": result["config"]} for name, _ in nets}
    if a.merge:
        with open(a.merge) as f:
            prev = json.load(f)
        for name in ("random", "synthetic_peaked"):
            if name in prev and name not in result:
                result[name] = prev[name]
                result["single_game"][name] = prev["single_game"][name]
                result["card_by_network"][name] = prev["card_by_network"][name]
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, "eval_cache_cost.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]), "->", path)


if __name__ == "__main__":
    main()
