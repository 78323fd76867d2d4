"""Self-play fan-out of the reference's train_RL.py (args + launcher, train_RL.py:156-244) and, as a "next" row
(SURVEY.md 8f rank 1), its fine-tuning step on the self-play records (train_RL.py:77-154): on the GPU library's own trainer
(trainer.py -> szb_train_*, csrc/train.cu) whenever the training device is a GPU, in torch otherwise.

The reference spawns `num_process` CPU workers that each play `num_games // num_process` games one after another
and merges their pickled dicts.  Here every rank (one process per GPU, torch.distributed over NCCL) plays its
shard of the games concurrently on its GPU; the only collective is the broadcast of the flat fp32 weight buffer
from the trainer rank at the start of an iteration.  `num_selfPlay_iterations` -- which the reference's args
carry but never read -- is defined as the number of self-play games per outer iteration.
Training (train_on_records / rl_iteration below) follows the reference's recipe -- loss = MSE(v, z) + CE(logits, pi) (:103-113),
Adam lr 1e-4 wd 1e-4 (:187), StepLR(500, 0.95) (:199) -- on the packed record format of records.py.  The CUDA trainer is deterministic,
so the ranks of a job, which all train on the same gathered records, keep identical weights; the trained flat weight buffer is folded
into the inference network on the device (Engine.load_flat_device), torch objects (module, optimiser, scheduler) carry the state
between iterations and into checkpoints."""
import os

import torch

from ._lib import EVAL_NET_BF16

DEFAULT_ARGS = {
    'C': 2,
    'num_searches': 100,
    'num_iterations': 3,
    'num_selfPlay_iterations': 500,
    'num_epochs': 4,
    'batch_size': 64,
    'chess960': True,
}


def shard_of(n_games, rank, world):
    """contiguous block of game indices owned by `rank` (sizes differ by at most one)"""
    base, extra = divmod(n_games, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def flatten_state_dict(sd):
    keys = [k for k in sd if not k.endswith("num_batches_tracked")]
    return keys, torch.cat([sd[k].detach().reshape(-1).float() for k in keys])


def unflatten_into(model, keys, flat):
    sd = model.state_dict()
    off = 0
    for k in keys:
        n = sd[k].numel()
        sd[k].copy_(flat[off:off + n].reshape(sd[k].shape))
        off += n


def broadcast_weights(model, src=0, device=None, engine=None):
    """One flat-buffer broadcast (NCCL over NVLink on GPUs, gloo in CPU tests); returns the buffer's bytes.
    With `engine` (and a CUDA device) the broadcast buffer never leaves the GPU: the library folds and packs it straight from
    there (szb_net_load_device) and the torch module is updated by a device-side copy when its parameters live on the GPU."""
    import torch.distributed as dist
    keys, flat = flatten_state_dict(model.state_dict())
    if device is not None:
        flat = flat.to(device)
    dist.broadcast(flat, src=src)
    param_dev = next(model.parameters()).device
    unflatten_into(model, keys, flat if flat.device == param_dev else flat.to(param_dev))
    if engine is not None and flat.is_cuda:
        from . import runtime
        sd = model.state_dict()
        engine.load_flat_device(keys, [int(sd[k].numel()) for k in keys], flat)
        runtime.mark_synced(engine, model)
    return flat.numel() * 4


def _iteration_shard(model, args):
    """broadcast rank 0's weights (the only collective of the path) and return this rank's block of the iteration's games"""
    import torch.distributed as dist
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    lo, hi = shard_of(int(args['num_selfPlay_iterations']), rank, world)
    if dist.is_initialized() and world > 1:
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))) if torch.cuda.is_available() else None
        engine = None
        if dev is not None:
            from . import runtime
            engine = runtime.get_engine(min_games=max(1, hi - lo), min_searches=int(args['num_searches']),
                                        leaves_per_tree=runtime.leaves_of(args))
        broadcast_weights(model, 0, dev, engine)
    return lo, hi


def selfplay_iteration(model, args, seed=0, max_plies=None):
    """One outer iteration's self-play: this rank's shard of args['num_selfPlay_iterations'] games, as the reference's
    per-game history dicts (sim.py:38-43)."""
    from .sim import selfplay_batch
    lo, hi = _iteration_shard(model, args)
    games, counters = selfplay_batch(model, args, hi - lo, c960=bool(args.get('chess960', False)),
                                     seed=seed, max_plies=max_plies, game_id_base=lo)
    return games, counters


def selfplay_iteration_records(model, args, seed=0, max_plies=None):
    """The same games recorded straight into the packed training format (sim.selfplay_records); `game` holds global game
    numbers so that the shards of all ranks concatenate into one record set."""
    from .sim import selfplay_records
    lo, hi = _iteration_shard(model, args)
    rec, counters = selfplay_records(model, args, hi - lo, c960=bool(args.get('chess960', False)),
                                     seed=seed, max_plies=max_plies, game_id_base=lo)
    rec["game"] = rec["game"] + lo
    return rec, counters


def concat_records(parts):
    """record sets of consecutive game blocks -> one record set (CSR offsets re-based)"""
    import numpy as np
    out = {k: np.concatenate([p[k] for p in parts]) for k in ("states", "pi_index", "pi_prob", "z", "colour", "game")}
    off, base = [np.zeros(1, dtype=np.int64)], 0
    for p in parts:
        off.append(p["pi_off"][1:] + base)
        base += int(p["pi_off"][-1])
    out["pi_off"] = np.concatenate(off)
    if all("result" in p for p in parts):
        out["result"] = np.concatenate([p["result"] for p in parts])
    return out


def make_optimiser(model, lr=1e-4, weight_decay=1e-4):
    """the reference's optimiser and schedule (train_RL.py:187,199)"""
    opt = torch.optim.Adam(model.parameters(), lr=lr, weight_decay=weight_decay)
    return opt, torch.optim.lr_scheduler.StepLR(opt, step_size=500, gamma=0.95)


def _batches(n, batch_size, epochs, seed):
    """the row numbers of every batch: a fresh permutation per epoch, short last batch dropped (DataLoader(drop_last=True),
    train_RL.py:241-246) unless the whole record set is smaller than one batch; BatchNorm needs more than one sample"""
    import numpy as np
    rng = np.random.default_rng(seed)
    for epoch in range(epochs):
        order = rng.permutation(n)
        for lo in range(0, n, batch_size):
            rows = order[lo:lo + batch_size]
            if (len(rows) < batch_size and n >= batch_size) or len(rows) < 2:
                continue
            yield rows


def trainer_hparams(optimiser, lr_scheduler):
    """(optimiser kind, Trainer hyper-parameters, step0) of a torch optimiser and StepLR scheduler (either may be None).
    torch.optim.Adam and torch.optim.SGD with one param group are what the library's trainer implements; anything else raises
    TypeError -- train it with backend="torch"."""
    kind, hp, step0 = "adam", {}, 0
    if optimiser is not None:
        if type(optimiser) not in (torch.optim.Adam, torch.optim.SGD):
            raise TypeError("the CUDA trainer implements torch.optim.Adam and torch.optim.SGD, not %s: use backend=\"torch\""
                            % type(optimiser).__name__)
        if len(optimiser.param_groups) != 1:
            raise TypeError("the CUDA trainer takes one param group, not %d: use backend=\"torch\"" % len(optimiser.param_groups))
        g = optimiser.param_groups[0]
        if g.get("maximize", False):
            raise TypeError("the CUDA trainer minimises; maximize=True needs backend=\"torch\"")
        if type(optimiser) is torch.optim.SGD:
            kind = "sgd"
            hp = dict(lr=float(g["initial_lr"] if lr_scheduler is not None and "initial_lr" in g else g["lr"]), weight_decay=float(g["weight_decay"]),
                      momentum=float(g["momentum"]), dampening=float(g["dampening"]), nesterov=bool(g["nesterov"]))
        else:
            hp = dict(lr=float(g.get("initial_lr", g["lr"])), beta1=float(g["betas"][0]), beta2=float(g["betas"][1]), eps=float(g["eps"]),
                      weight_decay=float(g["weight_decay"]))
    if lr_scheduler is not None:
        hp.update(lr_step=int(lr_scheduler.step_size), lr_gamma=float(lr_scheduler.gamma))
        step0 = int(lr_scheduler.last_epoch)
    else:
        hp.update(lr_step=1 << 30, lr_gamma=1.0)
    return kind, hp, step0


def train_on_records_cuda(model, rec, epochs=1, batch_size=64, optimiser=None, lr_scheduler=None, seed=0, log=None, engine=None):
    """train_on_records on the GPU library's trainer (szb_train_*, csrc/train.cu): same batches, same recipe, no torch op in the step.
    `optimiser` / `lr_scheduler` (torch objects, optional: torch.optim.Adam or torch.optim.SGD, StepLR) carry the state between calls
    and into checkpoints: their moments or momentum buffers, step counter and hyper-parameters are loaded into the trainer first and
    written back after the last batch."""
    from . import runtime
    from .trainer import Trainer
    kind, hp, step0 = trainer_hparams(optimiser, lr_scheduler)
    eng = engine if engine is not None else runtime.get_engine()
    tr = Trainer(eng, model, batch_size=batch_size, step0=step0, optimizer=kind, **hp)
    try:
        if optimiser is not None and optimiser.state_dict()["state"]:
            tr.load_optimiser_state(optimiser.state_dict())
            if lr_scheduler is not None:
                tr.step_count = step0                        # StepLR's counter is the one the learning rate follows
        tr.set_records(rec)
        history = []
        if log is not None:
            for rows in _batches(len(rec["z"]), batch_size, epochs, seed):
                history.append(tr.step(rows))
                log({"MSE Loss": history[-1][0], "CE Loss": history[-1][1]}, len(history))
        else:
            # nobody watches the losses step by step: queue the steps (the host runs ahead of the GPU) and read the history in bulk
            first = tr.steps_run
            for rows in _batches(len(rec["z"]), batch_size, epochs, seed):
                tr.step(rows, want_losses=False)
                if tr.steps_run - first == 32768:
                    history += tr.loss_history(first)
                    first = tr.steps_run
            history += tr.loss_history(first)
        flat = tr.write_back(model, steps_taken=len(history))
        if optimiser is not None:
            optimiser.load_state_dict(tr.optimiser_state(model))
        if lr_scheduler is not None:
            lr_scheduler.last_epoch += len(history)
            lr_scheduler._last_lr = [g["lr"] for g in optimiser.param_groups] if optimiser is not None else lr_scheduler._last_lr
        # the inference network of the same context gets the new weights straight from the trainer's device buffer
        eng.load_flat_device(tr.keys, tr.numels, flat)
        runtime.mark_synced(eng, model)
    finally:
        tr.close()
    model.eval()
    return history


def evaluate_records(model, rec, evaluator=EVAL_NET_BF16):
    """Held-out losses (mse, ce) of `model` on packed records, in eval mode: the library's inference network (`evaluator` EVAL_NET_BF16
    or EVAL_NET_FP32; BatchNorm with the running statistics; it already holds the weights train_on_records_cuda trained, else the
    model's are sent to it) gives the logits and values in chunks of the engine's capacity, and the host computes, in float64, the
    mean of (v - z)^2 and of the cross entropy -sum(pi * log_softmax(logits)) against the CSR policy targets.  Changes no weights,
    running statistics or trainer state."""
    import numpy as np
    from . import runtime
    n = len(rec["z"])
    if n == 0:
        raise ValueError("evaluate_records: no records")
    eng = runtime.get_engine(min_games=min(n, 1024))                  # grown (and the model's weights re-sent) only when it is smaller
    runtime.sync_weights(eng, model)
    chunk = eng.max_games * eng.leaves_per_tree
    off = np.asarray(rec["pi_off"], dtype=np.int64)
    se = ce = 0.0
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        logits, value = eng.net_forward(rec["states"][lo:hi], evaluator, logits=True)
        lg = logits.astype(np.float64)
        mx = lg.max(axis=1)
        lse = mx + np.log(np.exp(lg - mx[:, None]).sum(axis=1))
        a, b = int(off[lo]), int(off[hi])
        row = np.repeat(np.arange(hi - lo), np.diff(off[lo:hi + 1]))
        logp = lg[row, np.asarray(rec["pi_index"][a:b], dtype=np.int64)] - lse[row]
        ce -= float(np.dot(np.asarray(rec["pi_prob"][a:b], dtype=np.float64), logp))
        se += float(((value.astype(np.float64) - np.asarray(rec["z"][lo:hi], dtype=np.float64)) ** 2).sum())
    return se / n, ce / n


def train_on_records(model, rec, epochs=1, batch_size=64, optimiser=None, lr_scheduler=None, device=None, seed=0, log=None, backend=None):
    """Fine-tunes `model` on packed self-play records (records.pack_records): per batch
    loss = mse_loss(v, z) + cross_entropy(logits, pi) with pi the soft visit-fraction target (train_RL.py:103-113).
    Returns the per-batch (mse, ce) losses.  The model is left in eval() mode, ready for the next self-play iteration.

    backend "cuda" (the default whenever the training device is a GPU): the library's own trainer, train_on_records_cuda.
    backend "torch": torch autograd, the reference's own code path -- what the CUDA trainer is tested against, and what runs when
    device="cpu" is asked for explicitly."""
    import numpy as np
    from . import records
    if optimiser is None:
        optimiser, lr_scheduler = make_optimiser(model)
    device = torch.device(device) if device is not None else next(model.parameters()).device
    if backend is None:
        backend = "cuda" if device.type == "cuda" else "torch"
    if backend == "cuda":
        model.to(device)                                     # the module ends up where the caller asked for it, as with the torch path
        return train_on_records_cuda(model, rec, epochs=epochs, batch_size=batch_size, optimiser=optimiser, lr_scheduler=lr_scheduler, seed=seed, log=log)
    model.to(device).train()
    history = []
    for rows in _batches(len(rec["z"]), batch_size, epochs, seed):
        x = torch.from_numpy(records.unpack_states(rec, rows)).to(device=device, dtype=torch.float32)
        pi = torch.from_numpy(records.dense_policy(rec, rows)).to(device)
        z = torch.from_numpy(rec["z"][rows].astype(np.float32)).to(device)
        p, v = model(x)
        mse = torch.nn.functional.mse_loss(v.squeeze(-1), z)
        ce = torch.nn.functional.cross_entropy(p, pi)
        optimiser.zero_grad()
        (mse + ce).backward()
        optimiser.step()
        if lr_scheduler is not None:
            lr_scheduler.step()
        history.append((float(mse.detach()), float(ce.detach())))
        if log is not None:
            log({"MSE Loss": history[-1][0], "CE Loss": history[-1][1]}, len(history))
    model.eval()
    return history


def rl_iteration(model, args, seed=0, max_plies=None, epochs=None, optimiser=None, lr_scheduler=None, train_device=None):
    """One outer iteration of train_RL.main (:205-264): sharded self-play with the current weights (rank 0's are broadcast),
    records gathered on every rank, the same fine-tuning step everywhere (identical data + identical seed => identical
    weights, so the next iteration's broadcast is a formality).  Returns (records, loss history)."""
    import torch.distributed as dist
    rec, _ = selfplay_iteration_records(model, args, seed=seed, max_plies=max_plies)
    if dist.is_initialized() and dist.get_world_size() > 1:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, rec)
        rec = concat_records(parts)
    hist = train_on_records(model, rec, epochs=int(args.get('num_epochs', 1)) if epochs is None else epochs,
                            batch_size=int(args.get('batch_size', 64)), optimiser=optimiser, lr_scheduler=lr_scheduler,
                            device=train_device, seed=seed)
    return rec, hist


def main(args=None, model=None, weights=None, num_games=None, out_dir=".", seed=0, max_plies=None, passes_per_epoch=7,
         train_device=None, log=print):
    """The reference's outer loop (train_RL.py:156-264): for epoch in [start_epoch, num_epochs): self-play with the current
    weights, save the games, fine-tune on them, save weights and optimiser.

    Differences kept deliberately (SURVEY Appendix H, "do not preserve"): no hard-coded absolute paths -- `weights` is the
    checkpoint to start from (the reference loads supervised weights, :161-163) and everything is written under `out_dir`; the games
    are saved in the packed record format (games/RL_960_{epoch}.npz) instead of a pickled list of bool tensors; resuming reads
    the files this loop writes (saves/RL_960_{epoch}.pt, saves/RL_960_opt_{epoch}.pt -- the reference's resume reads names its
    training never writes, :191-194 vs :153).  `num_games` games per epoch (the reference's local num_games = 40, :165; default:
    args['num_selfPlay_iterations']) are split over the ranks of a torchrun job instead of num_process CPU workers; training runs
    `passes_per_epoch` passes over the epoch's records (the reference's train(total_steps=6) loops range(0, 7), :94,256)."""
    import time

    import torch.distributed as dist
    from . import records
    from .network import policyNN
    args = dict(DEFAULT_ARGS, **(args or {}))
    rank = dist.get_rank() if dist.is_initialized() else 0
    if model is None:
        model = policyNN({})
    if weights:
        model.load_state_dict(torch.load(weights, map_location="cpu"))
    if train_device is not None:
        model.to(train_device)           # before the optimiser exists: a resumed optimiser state must live where the parameters train
    model.eval()
    optimiser, scheduler = make_optimiser(model)
    start_epoch, num_epochs = int(args.get("start_epoch", 1)), int(args["num_epochs"])
    os.makedirs(os.path.join(out_dir, "saves"), exist_ok=True)
    os.makedirs(os.path.join(out_dir, "games"), exist_ok=True)
    if start_epoch > 1:
        try:
            model.load_state_dict(torch.load(os.path.join(out_dir, "saves", "RL_960_%d.pt" % (start_epoch - 1)), map_location="cpu"))
            optimiser.load_state_dict(torch.load(os.path.join(out_dir, "saves", "RL_960_opt_%d.pt" % (start_epoch - 1)), map_location="cpu"))
            sched_path = os.path.join(out_dir, "saves", "RL_960_sched_%d.pt" % (start_epoch - 1))
            if os.path.exists(sched_path):                   # the StepLR step counter continues instead of restarting
                scheduler.load_state_dict(torch.load(sched_path, map_location="cpu"))
        except OSError:
            log("No saved weights from epoch %d found!" % (start_epoch - 1))
            start_epoch = 1
    run_args = dict(args, num_selfPlay_iterations=int(num_games if num_games is not None else args["num_selfPlay_iterations"]))
    history = []
    for epoch in range(start_epoch, num_epochs):
        log("Epoch %d" % epoch)
        t1 = time.perf_counter()
        rec, hist = rl_iteration(model, run_args, seed=seed + epoch, max_plies=max_plies, epochs=passes_per_epoch,
                                 optimiser=optimiser, lr_scheduler=scheduler, train_device=train_device)
        if rank == 0:
            records.save(os.path.join(out_dir, "games", "RL_960_%d.npz" % epoch), rec)
            torch.save(model.state_dict(), os.path.join(out_dir, "saves", "RL_960_%d.pt" % epoch))
            torch.save(optimiser.state_dict(), os.path.join(out_dir, "saves", "RL_960_opt_%d.pt" % epoch))
            torch.save(scheduler.state_dict(), os.path.join(out_dir, "saves", "RL_960_sched_%d.pt" % epoch))
        history.append({"epoch": epoch, "positions": int(len(rec["z"])), "losses": hist, "seconds": time.perf_counter() - t1})
        log("Time taken: %0.4f seconds" % history[-1]["seconds"])
    return model, history


def build_parser():
    """the command line of `python -m sigma_zero_b200.train_RL`: DEFAULT_ARGS as flags plus the run's settings and the opt-in
    extensions of the args dict (--leaves_per_tree, --dirichlet_alpha / --dirichlet_epsilon / --sample_plies for AlphaZero's
    root noise and sampling horizon in self-play, and --eval_cache_slots for the exact evaluation cache; the defaults are the
    reference's behaviour)"""
    import argparse
    ap = argparse.ArgumentParser(description="self-play + fine-tuning loop of the reference's train_RL.py on the B200 engine "
                                             "(under torchrun the games of an epoch are split over the ranks)")
    for key, val in DEFAULT_ARGS.items():
        ap.add_argument("--" + key, type=type(val) if not isinstance(val, bool) else int, default=val)
    ap.add_argument("--start_epoch", type=int, default=1)
    ap.add_argument("--num_games", type=int, default=None)
    ap.add_argument("--weights", default=None, help="state_dict to start from, e.g. supervised_model_best.pt")
    ap.add_argument("--out_dir", default=".")
    ap.add_argument("--leaves_per_tree", type=int, default=1)
    ap.add_argument("--dirichlet_alpha", type=float, default=0.0,
                    help="Dirichlet noise on the root's priors in self-play (AlphaZero chess: 0.3); 0 = off, the reference's rule")
    ap.add_argument("--dirichlet_epsilon", type=float, default=0.25, help="weight of the root noise")
    ap.add_argument("--sample_plies", type=int, default=0,
                    help="sample moves from the visit counts for this many plies of a game, then play the arg-max; 0 = sample every ply")
    ap.add_argument("--eval_cache_slots", type=int, default=0,
                    help="exact evaluation cache for self-play: entries per game, a power of two in [64, 65536] (e.g. 2048; "
                         "max_games x slots x 928 bytes of GPU memory); 0 = off.  The games are bit-identical either way")
    return ap


CLI_ARGS = list(DEFAULT_ARGS) + ["start_epoch", "leaves_per_tree", "dirichlet_alpha", "dirichlet_epsilon", "sample_plies",
                                 "eval_cache_slots"]


if __name__ == "__main__":
    ns = vars(build_parser().parse_args())
    if "RANK" in os.environ:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    cli = {k: ns[k] for k in CLI_ARGS}
    cli["chess960"] = bool(cli["chess960"])
    main(cli, weights=ns["weights"], num_games=ns["num_games"], out_dir=ns["out_dir"], train_device="cuda")
