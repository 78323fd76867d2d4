"""Throughput of supervised training on one GPU, in one call with the arms alternating:

  * ms per optimiser step (forward + backward + update) at batch 128 and 512 on synthetic records resident on the GPU: the library's
    trainer with SGD (the supervised recipe), the library's trainer with Adam (the self-play recipe), and torch eager SGD on the same GPU
    (fp32 parameters, torch's default TF32 setting: cuDNN convolutions in TF32, matmuls in fp32 -- the torch arm of bench.py's
    f1_trainer);
  * positions/s of supervised.pgn_to_records (PGN text -> records: lock-step replay on the GPU, SAN resolved on the host), on the
    three finished games of tests/util.PGN_SAMPLE repeated to `--games` games (short games: 4-33 plies, so the lock-step batches are
    as full as the longest game allows).

Writes one JSON file (default: supervised_throughput.json in the current directory) with the card's name and power limit read in the
same run.

    python scripts/supervised_throughput.py [--steps 20] [--reps 5] [--games 1020] [--out FILE]
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
from sigma_zero_b200 import records as records_mod, supervised
from sigma_zero_b200.engine import Engine
from sigma_zero_b200.network import policyNN
from sigma_zero_b200.trainer import Trainer
from tests import util


def synthetic_records(n, seed=0):
    rng = np.random.default_rng(seed)
    bits = rng.random((n, 119, 64)) < 0.12
    idx, prob, off = [], [], [0]
    for _ in range(n):
        k = int(rng.integers(5, 45))
        idx.extend(np.sort(rng.choice(4672, size=k, replace=False)).tolist())
        p = rng.random(k).astype(np.float32)
        prob.extend((p / p.sum()).tolist())
        off.append(len(idx))
    return {"states": np.packbits(bits, axis=-1, bitorder="little").view("<u8").reshape(n, 119).astype(np.uint64),
            "pi_index": np.array(idx, np.uint16), "pi_prob": np.array(prob, np.float32), "pi_off": np.array(off, np.int64),
            "z": rng.integers(-1, 2, n).astype(np.int8)}


class LibArm:
    """one library trainer on its own context (one trainer per context)"""

    def __init__(self, model, rec, batch, optimizer):
        self.eng = Engine(max_games=2, max_searches=8, device=0)
        self.tr = Trainer(self.eng, model, batch_size=batch, optimizer=optimizer)
        self.tr.set_records(rec)
        self.ext = torch.cuda.ExternalStream(self.eng.stream, device=torch.device("cuda", 0))

    def run(self, batches, steps, warmup):
        for i in range(warmup):
            self.tr.step(batches[i % len(batches)], want_losses=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.ext)
        for i in range(steps):
            self.tr.step(batches[i % len(batches)], want_losses=False)
        e1.record(self.ext)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def close(self):
        self.tr.close()
        self.eng.close()


class TorchSgdArm:
    def __init__(self, model, rec, batch):
        dev = torch.device("cuda", 0)
        self.model = policyNN({}).to(dev).train()
        self.model.load_state_dict(model.state_dict())
        self.opt = torch.optim.SGD(self.model.parameters(), lr=0.1, weight_decay=1e-4)
        rows = np.arange(batch)
        self.x = torch.from_numpy(records_mod.unpack_states(rec, rows)).to(device=dev, dtype=torch.float32)
        self.pi = torch.from_numpy(records_mod.dense_policy(rec, rows)).to(dev)
        self.z = torch.from_numpy(rec["z"][rows].astype(np.float32)).to(dev)

    def step(self):
        self.opt.zero_grad(set_to_none=True)
        p, v = self.model.forward_torch(self.x)
        (torch.nn.functional.mse_loss(v.squeeze(-1), self.z) + torch.nn.functional.cross_entropy(p, self.pi)).backward()
        self.opt.step()

    def run(self, batches, steps, warmup):
        for _ in range(warmup):
            self.step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def close(self):
        pass


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def step_times(batch, steps, reps, warmup):
    torch.manual_seed(0)
    model = policyNN({})
    rec = synthetic_records(8 * batch, seed=batch)
    rng = np.random.default_rng(batch)
    batches = [rng.permutation(8 * batch)[:batch].astype(np.int32) for _ in range(8)]
    arms = {"library_sgd": LibArm(model, rec, batch, "sgd"), "library_adam": LibArm(model, rec, batch, "adam"),
            "torch_eager_sgd": TorchSgdArm(model, rec, batch)}
    times = {k: [] for k in arms}
    try:
        for rep in range(reps):                          # alternate the arms: drift of the shared host hits each of them alike
            for k, arm in arms.items():
                times[k].append(arm.run(batches, steps, warmup if rep == 0 else 1))
    finally:
        for arm in arms.values():
            arm.close()
    out = {"batch": batch, "steps_per_rep": steps, "reps": reps}
    for k, t in times.items():
        out[k] = {"ms_per_step_median": float(np.median(t)), "ms_per_step_min": float(np.min(t)), "ms_per_step_max": float(np.max(t)),
                  "positions_per_sec_median": batch / (float(np.median(t)) * 1e-3), "ms_per_step_each_rep": [float(x) for x in t]}
    out["sgd_over_adam"] = out["library_sgd"]["ms_per_step_median"] / out["library_adam"]["ms_per_step_median"]
    out["torch_sgd_over_library_sgd"] = out["torch_eager_sgd"]["ms_per_step_median"] / out["library_sgd"]["ms_per_step_median"]
    return out


def pgn_rate(n_games, reps):
    games = [g for g in supervised.read_pgn(util.PGN_SAMPLE) if g[0].get("Result") in supervised.RESULTS]
    text = "\n\n".join([util.PGN_SAMPLE] * (n_games // len(games) + 1))
    t0 = time.perf_counter()
    parsed = [g for g in supervised.read_pgn(text) if g[0].get("Result") in supervised.RESULTS][:n_games]
    parse_s = time.perf_counter() - t0
    supervised.pgn_to_records(parsed[:8])               # warm-up: the engine and its kernels
    secs, n_pos = [], 0
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rec = supervised.pgn_to_records(parsed)
        secs.append(time.perf_counter() - t0)
        n_pos = len(rec["z"])
    return {"games": len(parsed), "positions": n_pos, "plies_of_longest_game": max(len(m) for _, m in parsed),
            "read_pgn_seconds": parse_s, "pgn_to_records_seconds_each_rep": secs,
            "positions_per_sec_median": n_pos / float(np.median(secs)),
            "note": "tests/util.PGN_SAMPLE's three finished games repeated; host SAN resolution included, text parsing (read_pgn) not"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--games", type=int, default=1020)
    ap.add_argument("--out", default="supervised_throughput.json")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.backends.cudnn.allow_tf32 = True              # torch's defaults, stated: TF32 convolutions, fp32 matmuls
    torch.backends.cuda.matmul.allow_tf32 = False
    result = {"card": card(), "torch": torch.__version__, "tf32": {"cudnn": True, "matmul": False},
              "step_times": [step_times(b, a.steps, a.reps, a.warmup) for b in (128, 512)],
              "pgn_to_records": pgn_rate(a.games, 3)}
    result["card_after"] = card()["nvidia_smi"]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    for s in result["step_times"]:
        print("batch %d: library SGD %.3f ms, library Adam %.3f ms, torch eager SGD %.3f ms per step (medians of %d)"
              % (s["batch"], s["library_sgd"]["ms_per_step_median"], s["library_adam"]["ms_per_step_median"],
                 s["torch_eager_sgd"]["ms_per_step_median"], s["reps"]))
    p = result["pgn_to_records"]
    print("pgn_to_records: %d positions of %d games, %.0f positions/s" % (p["positions"], p["games"], p["positions_per_sec_median"]))
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
