"""Cost of the opt-in root exploration in self-play (szb_set_exploration), in one call with the arms alternating:

  * off: the reference's rule (learning=True, constant noise at every expansion, every move sampled);
  * on:  AlphaZero's settings -- Dirichlet(0.3) noise on the root's priors with epsilon 0.25, moves sampled for 30 plies.

Config c2's size: 1024 vanilla games x 800 simulations per move, bf16 network (policyNN as initialised with torch seed 0).  A
repetition resets the games and times `--plies` calls of selfplay_ply (search + pick + push; each call ends in a device
synchronisation); the reported figure is the median over the repetitions of the mean ms per ply.

Writes exploration_cost.json into the --out directory with the card's name and power limit read in the same run.

    python scripts/exploration_cost.py [--reps 5] [--plies 2] [--out DIR]
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

ARMS = {"off": dict(alpha=0.0, epsilon=0.25, sample_plies=0), "on": dict(alpha=0.3, epsilon=0.25, sample_plies=30)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def run_arm(eng, games, sims, plies, setting, seed):
    eng.reset(np.full(games, -1))
    eng.set_exploration(seed=seed, **setting)
    ms, moves = [], []
    for _ in range(plies):
        t0 = time.perf_counter()
        mv, _ = eng.selfplay_ply(sims, 2.0, True, EVAL_NET_BF16, seed=seed, sample=True)
        ms.append((time.perf_counter() - t0) * 1e3)
        moves.append(mv)
    return float(np.mean(ms)), moves


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--plies", type=int, default=2)
    ap.add_argument("--out", default=".")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.manual_seed(0)
    eng = Engine(max_games=a.games, max_searches=a.sims, device=0)
    eng.load_state_dict(policyNN({}).eval().state_dict())
    before = card()
    for setting in ARMS.values():                        # warm-up: modules, staging buffers, the network's first launches
        run_arm(eng, a.games, a.sims, 1, setting, seed=1)
    times = {k: [] for k in ARMS}
    first_moves = {}
    for rep in range(a.reps):                            # alternate the arms: drift of the shared host hits both alike
        for k, setting in ARMS.items():
            t, moves = run_arm(eng, a.games, a.sims, a.plies, setting, seed=1)
            times[k].append(t)
            if rep == 0:
                first_moves[k] = moves
            else:
                assert all(np.array_equal(x, y) for x, y in zip(moves, first_moves[k])), "repetitions must play the same moves"
    result = {"card": before, "torch": torch.__version__,
              "config": {"games": a.games, "simulations_per_move": a.sims, "network": "bf16, policyNN({}) with torch seed 0",
                         "start": "vanilla", "plies_per_rep": a.plies, "reps": a.reps, "c_puct": 2.0, "learning": True},
              "arms": {k: dict(ARMS[k]) for k in ARMS}}
    for k, t in times.items():
        result[k] = {"ms_per_ply_median": float(np.median(t)), "ms_per_ply_min": float(np.min(t)), "ms_per_ply_max": float(np.max(t)),
                     "ms_per_ply_each_rep": t}
    result["on_over_off_median"] = result["on"]["ms_per_ply_median"] / result["off"]["ms_per_ply_median"]
    result["moves_differ_on_first_ply"] = int((first_moves["on"][0] != first_moves["off"][0]).sum())
    result["card_after"] = card()["nvidia_smi"]
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, "exploration_cost.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    for k in ARMS:
        r = result[k]
        print("exploration %s: %.1f ms per ply (median of %d; min %.1f, max %.1f)"
              % (k, r["ms_per_ply_median"], a.reps, r["ms_per_ply_min"], r["ms_per_ply_max"]))
    print(json.dumps(result["card"]), "->", path)


if __name__ == "__main__":
    main()
