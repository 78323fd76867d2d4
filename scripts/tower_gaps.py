"""Where the tensor pipe of the 512-board k_tower_tc2 launch sits idle: device timestamps of every work item of the last 64
large-batch launches of a c2-sized search (1024 vanilla games, two cohorts of 512, 800 simulations after an 800-simulation warm-up
search, policyNN initialised with torch seed 0).

The library records them with SZB_TOWER_TRACE (TowerArgs::trace, five %globaltimer stamps per item of the leader CTA: 0 dependency
resolved, 1 first activation chunk in shared memory, 2 accumulator complete, 3 stored and released, 4 last MMA of the item issued)
and SZB_TOWER_SPAN (first CTA start, last CTA end), and writes them when the engine closes.  Per launch it reports, as means over
items and launches:

  * the MMA warp's wait per item: the previous item of the same CTA pair's last MMA issued -> this item's first chunk in shared
    memory, split into the part before the producer had acquired the item's dependency and the TMA latency after it;
  * the same wait for the items whose dependency (layer - 1, same tile) was dealt in the round right before (one round = one item
    per pair) and for the others;
  * the MMA issue span of an item (first chunk -> last MMA issued), the drain (last MMA issued -> accumulator complete) and the
    epilogue (accumulator complete -> stored and released);
  * the launch's head (first CTA start -> last release of layer 0) and tail (last release of layer 38 -> last CTA end).

    python scripts/tower_gaps.py [--label NAME] [--out DIR]       (SZB_LIB=<build> selects the library, as bench.py)
Writes tower_gaps_<label>.txt and the raw trace tower_gaps_<label>.csv into --out (default: <temp dir>/tower_gaps), with the card's
name and power limit.
"""
import argparse
import collections
import csv
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--label", default="current")
ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "tower_gaps"))
ap.add_argument("--sims", type=int, default=800)
ap.add_argument("--analyse", metavar="CSV", help="only summarise an earlier run's raw trace")
args = ap.parse_args()
os.makedirs(args.out, exist_ok=True)
trace_csv = args.analyse or os.path.join(args.out, "tower_gaps_%s.csv" % args.label)
card = ["not read (--analyse)"]
if not args.analyse:
    if os.path.exists(trace_csv):
        os.remove(trace_csv)
    os.environ["SZB_TOWER_TRACE"] = trace_csv
    os.environ["SZB_TOWER_SPAN"] = os.path.join(args.out, "tower_gaps_%s_span.csv" % args.label)
    import torch
    from oracle import ref_path
    from sigma_zero_b200.engine import EVAL_NET_BF16, Engine

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[:1]
    torch.manual_seed(0)
    model = ref_path.build_policy_nn().eval()
    eng = Engine(max_games=1024, max_searches=args.sims, cohorts=2)
    eng.load_state_dict(model.state_dict())
    eng.reset([-1] * 1024)
    for _ in range(2):                               # warm-up search, then the traced one (the ring keeps its last 64 launches)
        eng.search(args.sims, 2.0, True, EVAL_NET_BF16, want_visits=False, want_children=False)
    eng.close()

launches = collections.defaultdict(list)
for r in csv.DictReader(open(trace_csv)):
    if r["launch"] == "launch":
        continue
    launches[int(r["launch"])].append({k: int(v) for k, v in r.items()})

acc = collections.defaultdict(list)
for key in sorted(launches):
    R = sorted(launches[key], key=lambda r: r["item"])
    P = R[0]["pairs"]
    tiles = max(r["tile"] for r in R) + 1
    n_layers = len(R) // tiles
    if any(r["operands_ns"] < 0 or r["last_mma_ns"] < 0 or r["acc_ns"] < 0 for r in R):
        continue
    acc["launch_us"].append((R[0]["end_ns"] - R[0]["start_ns"]) / 1e3)
    busy = 0
    for i, r in enumerate(R):
        busy += r["last_mma_ns"] - r["operands_ns"]
        acc["issue_us"].append((r["last_mma_ns"] - r["operands_ns"]) / 1e3)
        acc["drain_us"].append((r["acc_ns"] - r["last_mma_ns"]) / 1e3)
        if r["layer"] < n_layers - 1:
            acc["epilogue_us"].append((r["released_ns"] - r["acc_ns"]) / 1e3)
        if i < P:
            acc["first_item_wait_us"].append((r["operands_ns"] - r["start_ns"]) / 1e3)
            continue
        prev = R[i - P]["last_mma_ns"]
        wait = r["operands_ns"] - prev
        dep_part = max(0, min(r["dep_ns"], r["operands_ns"]) - prev) if r["layer"] > 0 else 0
        acc["wait_us"].append(wait / 1e3)
        acc["wait_dependency_us"].append(dep_part / 1e3)
        acc["wait_after_dependency_us"].append((wait - dep_part) / 1e3)
        if i >= 2 * P and R[i - 2 * P]["layer"] < n_layers - 1 and R[i - 2 * P]["released_ns"] > prev:
            acc["accumulator_not_free_us"].append((R[i - 2 * P]["released_ns"] - prev) / 1e3)
        if r["layer"] > 0:
            tight = i // P - (i - tiles) // P == 1
            acc["wait_tight_us" if tight else "wait_slack_us"].append(wait / 1e3)
            acc["wait_tight_dependency_us" if tight else "wait_slack_dependency_us"].append(dep_part / 1e3)
    last = R[-1]["end_ns"]
    l0 = max(r["released_ns"] for r in R if r["layer"] == 0)
    l38 = max(r["released_ns"] for r in R if r["layer"] == n_layers - 3)
    acc["head_us"].append(l0 / 1e3)
    acc["tail_us"].append((last - l38) / 1e3)
    acc["tail_last2_issue_us"].append(sum(r["last_mma_ns"] - r["operands_ns"] for r in R if r["layer"] >= n_layers - 2) / P / 1e3)
    acc["mma_issue_share"].append(busy / P / (last - R[0]["start_ns"]))

LAUNCH_KEYS = ("launch_us", "mma_issue_share", "head_us", "tail_us", "tail_last2_issue_us")
lines = ["k_tower_tc2, 512-board launches inside a c2-sized search (1024 vanilla games, 2 cohorts, %d simulations after warm-up)" % args.sims,
         "library: %s   card: %s" % (os.environ.get("SZB_LIB", "in-tree build"), card),
         "launches analysed: %d (pairs %d, tiles %d)" % (len(acc["launch_us"]), P, tiles), ""]
for k in ["launch_us", "mma_issue_share", "first_item_wait_us", "wait_us", "wait_dependency_us", "wait_after_dependency_us",
          "wait_tight_us", "wait_tight_dependency_us", "wait_slack_us", "wait_slack_dependency_us", "accumulator_not_free_us",
          "issue_us", "drain_us", "epilogue_us", "head_us", "tail_us", "tail_last2_issue_us"]:
    v = [x for x in acc[k] if x is not None]
    if not v:
        lines.append("%-28s -" % k)
        continue
    v.sort()
    per = len(acc["launch_us"]) * (1 if k in LAUNCH_KEYS else P)
    lines.append("%-28s n %6d  mean %8.3f  median %8.3f  p10 %8.3f  p90 %8.3f  sum per %s launch %9.1f" % (
        k, len(v), statistics.fmean(v), v[len(v) // 2], v[len(v) // 10], v[9 * len(v) // 10], "" if k in LAUNCH_KEYS else "pair per", sum(v) / per))
lines += ["",
          "wait: previous item's last MMA issued -> first chunk in shared memory (same pair); dependency: the part before the producer had",
          "acquired (layer - 1, tile); tight: that dependency was dealt in the round right before; accumulator_not_free: items whose",
          "accumulator (item - 2 rounds) was released after the previous item's last MMA; mma_issue_share: sum of issue spans / pairs / launch",
          "time (an upper bound of the tensor pipe's busy share); tail_last2_issue: MMA issue time per pair of layers 39-40."]
text = "\n".join(lines)
print(text)
open(os.path.join(args.out, "tower_gaps_%s.txt" % args.label), "w").write(text + "\n")
