"""Supervised path of the reference (SURVEY.md 8f rank 3): PGN games -> packed training positions with the played move as
a one-hot policy target (generate_training_supervised.py:11-115), the SGD recipe of train_supervised.py:84-92, and main(), the
training loop from a PGN file to supervised_model_best.pt on the library's trainer.

The reference replays each PGN game through python-chess and ChessTensor one move at a time on the host and stores a
bit-compressed uint8[119,8] tensor per position.  Here all selected games are replayed IN LOCK STEP on the GPU engine: one
szb_encode (the 119 input planes of every game, bit-packed), one szb_legal_moves and one szb_games_push per ply for the whole
batch.  The host only reads PGN text and resolves each SAN token against its game's legal-move list -- no chess rule is
evaluated in Python: legality, castling, en passant and promotions come from the engine's move generator.  The packed state of
records.py (one uint64 per plane, bit row*8+col) viewed as bytes IS the reference's compressed layout (byte r of plane k = row
r with bit c = column c, generate_training_supervised.py:91): see compressed_states()."""
import bz2
import io
import re

import numpy as np

from . import chess_compat as chess
from .chess_tensor import index_move

RESULTS = ("1-0", "0-1", "1/2-1/2")
_TAG = re.compile(r'^\[(\w+)\s+"(.*)"\]\s*$')
_SAN = re.compile(r"^([NBRQK])?([a-h])?([1-8])?(x)?([a-h][1-8])(?:=?([NBRQnbrq]))?[+#]*[!?]*$")
_CASTLE = re.compile(r"^(O-O-O|O-O|0-0-0|0-0)[+#]*[!?]*$")
_PIECE = {"N": chess.KNIGHT, "B": chess.BISHOP, "R": chess.ROOK, "Q": chess.QUEEN, "K": chess.KING}


# ---------------------------------------------------------------------------------------------------
# PGN text
# ---------------------------------------------------------------------------------------------------
def _movetext_tokens(text):
    """SAN tokens of the main line: comments, variations, NAGs, move numbers and the result marker removed"""
    out, depth, i, n = [], 0, 0, len(text)
    buf = []
    while i < n:
        c = text[i]
        if c == "{":
            j = text.find("}", i)
            i = n if j < 0 else j + 1
            continue
        if c == ";":
            j = text.find("\n", i)
            i = n if j < 0 else j + 1
            continue
        if c == "(":
            depth += 1
        elif c == ")":
            depth = max(0, depth - 1)
        elif depth == 0:
            buf.append(c)
        i += 1
    for tok in "".join(buf).split():
        tok = re.sub(r"^\d+\.(\.\.)?\.*", "", tok)              # "12.e4", "12...e5", "12."
        if not tok or tok.startswith("$") or tok in RESULTS or tok == "*":
            continue
        out.append(tok)
    return out


def read_pgn(source):
    """source: PGN text, bytes, a path (optionally .bz2, like the reference's FICS dump) or a file object.
    Yields (headers: dict, san_moves: list[str]) per game."""
    if isinstance(source, bytes):
        source = source.decode("utf-8", errors="replace")
    if isinstance(source, str) and "\n" not in source and not source.lstrip().startswith("["):
        opener = bz2.open if source.endswith(".bz2") else open
        with opener(source, "rt", encoding="utf-8", errors="replace") as f:
            yield from read_pgn(f.read())
        return
    if hasattr(source, "read"):
        source = source.read()
        if isinstance(source, bytes):
            source = source.decode("utf-8", errors="replace")
    headers, body = {}, []
    for line in io.StringIO(source):
        text = line.strip()
        if not text or text.startswith("%"):
            continue
        m = _TAG.match(text)
        if m:
            if body:                                             # a tag pair after movetext: the next game begins
                yield headers, _movetext_tokens("".join(body))
                headers, body = {}, []
            headers[m.group(1)] = m.group(2)
        else:
            body.append(line)
    if headers or body:
        yield headers, _movetext_tokens("".join(body))


def select_balanced(games, num_games=0):
    """The reference's selection rule (generate_training_supervised.py:33-49,70-105): scan results until draws + 2 * min(white
    wins, black wins) reaches num_games (0 = the whole file); then take, in file order, that many white wins, as many black
    wins and every counted draw."""
    games = list(games)
    count = {r: 0 for r in RESULTS}
    for h, _ in games:
        r = h.get("Result")
        if r in count:
            count[r] += 1
        if num_games and count["1/2-1/2"] + 2 * min(count["1-0"], count["0-1"]) >= num_games:
            break
    left = {"1-0": min(count["1-0"], count["0-1"]), "0-1": min(count["1-0"], count["0-1"]), "1/2-1/2": count["1/2-1/2"]}
    out = []
    for h, mv in games:
        r = h.get("Result")
        if r not in left or left[r] == 0:
            continue
        out.append((h, mv))
        left[r] -= 1
        if sum(left.values()) == 0:
            break
    return out


# ---------------------------------------------------------------------------------------------------
# SAN -> one of the engine's legal moves
# ---------------------------------------------------------------------------------------------------
def resolve_san(san, legal, piece_at):
    """legal: iterable of (from_square, to_square, promotion|None) as the engine lists them (queen promotions may come as
    promotion None on a pawn reaching the last rank; castling as the king's two-square move or, in Chess960 games, king takes
    own rook); piece_at(square) -> (piece_type, is_white) or None.  Returns the position of the matching move in `legal`.
    Raises ValueError for unknown or ambiguous SAN."""
    legal = list(legal)
    m = _CASTLE.match(san)
    if m:
        long_side = m.group(1).count("-") == 2
        hits = []
        for k, (f, t, _) in enumerate(legal):
            p, q = piece_at(f), piece_at(t)
            if not p or p[0] != chess.KING or (f >> 3) != (t >> 3):
                continue
            own_rook = bool(q) and q[0] == chess.ROOK and q[1] == p[1]
            if own_rook or abs((t & 7) - (f & 7)) == 2:
                if ((t & 7) < (f & 7)) == long_side:
                    hits.append(k)
        if len(hits) != 1:
            raise ValueError("cannot resolve castling %r" % san)
        return hits[0]
    m = _SAN.match(san)
    if not m:
        raise ValueError("not a SAN move: %r" % san)
    piece = _PIECE.get(m.group(1), chess.PAWN)
    ffile = "abcdefgh".index(m.group(2)) if m.group(2) else None
    frank = int(m.group(3)) - 1 if m.group(3) else None
    to = chess.SQUARE_NAMES.index(m.group(5))
    promo = _PIECE[m.group(6).upper()] if m.group(6) else None
    hits = []
    for k, (f, t, pr) in enumerate(legal):
        p = piece_at(f)
        if t != to or not p or p[0] != piece:
            continue
        if ffile is not None and (f & 7) != ffile or frank is not None and (f >> 3) != frank:
            continue
        if piece == chess.PAWN and (t >> 3) in (0, 7):
            if (pr or chess.QUEEN) != (promo or chess.QUEEN):
                continue
        elif promo is not None:
            continue
        q = piece_at(t)
        if piece == chess.KING and q and q[1] == p[1]:
            continue                                             # king-takes-own-rook is castling, never written as a king move
        hits.append(k)
    if len(hits) != 1:
        raise ValueError("%s SAN move %r" % ("ambiguous" if hits else "illegal", san))
    return hits[0]


def _piece_lookup(pos):
    table = {}
    for t in range(12):
        bb = int(pos.pieces[t])
        while bb:
            low = bb & -bb
            table[low.bit_length() - 1] = (t % 6 + 1, t < 6)
            bb ^= low
    return table.get


# ---------------------------------------------------------------------------------------------------
# replay on the GPU engine -> packed records
# ---------------------------------------------------------------------------------------------------
def pgn_to_records(games, engine=None, batch=1024, strict=False):
    """games: iterable of (headers, san_moves) (read_pgn / select_balanced).  Returns packed records in the format of records.py
    with one policy entry of probability 1 per position (the move played, train_RL.collatefn's one-hot target), z = the game
    result from the mover's side (generate_training_supervised.py:76-81) and `game` = index into `games`.  A game whose SAN cannot
    be resolved is cut at that move (strict=True: ValueError)."""
    from . import runtime
    games = [(h, mv) for h, mv in games if h.get("Result") in RESULTS]
    parts = {k: [] for k in ("states", "pi_index", "z", "colour", "game", "ply")}
    for base in range(0, len(games), batch):
        block = games[base:base + batch]
        eng = engine or runtime.get_engine(min_games=len(block), min_searches=1)
        eng.owner = None
        eng.reset(np.full(len(block), -1))
        alive = np.ones(len(block), dtype=bool)
        reward = np.array([1 if h["Result"] == "1-0" else (-1 if h["Result"] == "0-1" else 0) for h, _ in block])
        longest = max((len(mv) for _, mv in block), default=0)
        for ply in range(longest):
            who = [g for g in range(len(block)) if alive[g] and ply < len(block[g][1])]
            if not who:
                break
            who_arr = np.array(who, dtype=np.int32)
            planes, _ = eng.encode(who_arr, want_mask=False)
            idx, cnt = eng.legal_moves(who_arr)
            pos = eng.positions(who_arr)
            keep, chosen = [], []
            for k, g in enumerate(who):
                white = bool(pos[k].turn)
                legal = []
                for i in idx[k, :cnt[k]]:
                    mv = index_move(int(i), white)
                    legal.append((mv.from_square, mv.to_square, mv.promotion))
                try:
                    j = resolve_san(block[g][1][ply], legal, _piece_lookup(pos[k]))
                except ValueError:
                    if strict:
                        raise ValueError("game %d ply %d: cannot play %r" % (base + g, ply, block[g][1][ply]))
                    alive[g] = False
                    continue
                keep.append(k)
                chosen.append(int(idx[k, j]))
            if not keep:
                continue
            keep = np.array(keep)
            gs = who_arr[keep]
            eng.push(gs, chosen)
            parts["states"].append(planes[keep])
            parts["pi_index"].append(np.array(chosen, dtype=np.uint16))
            parts["colour"].append(planes[keep][:, 112] != 0)
            parts["z"].append(np.where(ply % 2 == 0, reward[gs], -reward[gs]).astype(np.int8))
            parts["game"].append((base + gs).astype(np.int32))
            parts["ply"].append(np.full(len(gs), ply, dtype=np.int32))
    if not parts["z"]:
        return {"states": np.zeros((0, 119), np.uint64), "pi_index": np.zeros(0, np.uint16), "pi_prob": np.zeros(0, np.float32),
                "pi_off": np.zeros(1, np.int64), "z": np.zeros(0, np.int8), "colour": np.zeros(0, bool), "game": np.zeros(0, np.int32)}
    cat = {k: np.concatenate(v) for k, v in parts.items()}
    order = np.lexsort((cat["ply"], cat["game"]))                 # by game, then ply -- the reference's order
    n = len(order)
    return {"states": cat["states"][order], "pi_index": cat["pi_index"][order], "pi_prob": np.ones(n, np.float32),
            "pi_off": np.arange(n + 1, dtype=np.int64), "z": cat["z"][order], "colour": cat["colour"][order], "game": cat["game"][order]}


def compressed_states(records, rows=None):
    """uint8[n,119,8]: the reference's stored state (`(representation.byte() << arange(8)).sum(-1)`,
    generate_training_supervised.py:91) -- a byte view of the packed planes, no computation"""
    s = records["states"] if rows is None else records["states"][rows]
    return np.ascontiguousarray(s, dtype="<u8").view(np.uint8).reshape(len(s), 119, 8)


def make_supervised_optimiser(model, lr=0.1, weight_decay=1e-4, lr_step_size=4000):
    """SGD + StepLR(4000, 0.5) of train_supervised.py:84-92, the scheduler stepped per batch.  Train with
    train_RL.train_on_records(model, records, optimiser=opt, lr_scheduler=sched): on a CUDA device the library's trainer runs the
    SGD update (szb_train_set_optimizer), elsewhere torch does; main() below is the whole loop from PGN to checkpoint."""
    import torch
    opt = torch.optim.SGD(model.parameters(), lr=lr, weight_decay=weight_decay)
    return opt, torch.optim.lr_scheduler.StepLR(opt, step_size=lr_step_size, gamma=0.5)


# ---------------------------------------------------------------------------------------------------
# training from PGN: python -m sigma_zero_b200.supervised --pgn games.pgn.bz2
# ---------------------------------------------------------------------------------------------------
def split_holdout(games, fraction=0.02, seed=0):
    """(train, held_out): a seeded random `fraction` of the GAMES is held out, so that no position of a held-out game is trained on.
    At least one game is held out when fraction > 0 and at least one is kept for training; both lists keep file order."""
    games = list(games)
    n_hold = int(round(fraction * len(games)))
    if fraction > 0 and len(games) >= 2:
        n_hold = min(max(n_hold, 1), len(games) - 1)
    hold = set(np.random.default_rng(seed).permutation(len(games))[:n_hold].tolist())
    return [g for i, g in enumerate(games) if i not in hold], [g for i, g in enumerate(games) if i in hold]


def main(pgn, num_games=0, holdout=0.02, epochs=10, batch_size=128, weights=None, out_dir=".", start_epoch=1, seed=0, model=None, log=print):
    """Supervised pre-training, the loop of train_supervised.py on the GPU library: the balanced selection of `pgn`'s games
    (select_balanced), a seeded held-out fraction of them (split_holdout), both replayed into records (pgn_to_records); then for each
    epoch in [start_epoch, epochs]: one pass of SGD + StepLR (make_supervised_optimiser) over the training records on the library's
    trainer, the held-out losses in eval mode (train_RL.evaluate_records), and out_dir/saves/supervised_{epoch}.pt,
    supervised_opt_{epoch}.pt and supervised_sched_{epoch}.pt.  The epoch with the lowest held-out loss (mse + ce; the training loss
    when nothing is held out) is also written as out_dir/supervised_model_best.pt -- the file train_RL.main(weights=...) and
    PlayTensor(model_path=...) start from -- with its losses in supervised_model_best.json.  start_epoch N resumes weights,
    optimiser and scheduler from epoch N - 1, as train_RL.main does.  Returns (model, per-epoch history)."""
    import json
    import os
    import time

    import torch

    from .network import policyNN
    from .train_RL import evaluate_records, train_on_records
    games = select_balanced(read_pgn(pgn), num_games)
    train_games, held_games = split_holdout(games, holdout, seed)
    rec = pgn_to_records(train_games)
    held = pgn_to_records(held_games) if held_games else None
    if len(rec["z"]) < 2:
        raise ValueError("%d training positions: too few to train on" % len(rec["z"]))
    log("%d games (%d positions) to train on, %d held out (%d positions)"
        % (len(train_games), len(rec["z"]), len(held_games), 0 if held is None else len(held["z"])))
    if model is None:
        model = policyNN({})
    if weights:
        model.load_state_dict(torch.load(weights, map_location="cpu"))
    model.to("cuda")                     # before the optimiser exists: a resumed optimiser state must live where the parameters train
    optimiser, scheduler = make_supervised_optimiser(model)
    saves = os.path.join(out_dir, "saves")
    os.makedirs(saves, exist_ok=True)
    path = lambda kind, epoch: os.path.join(saves, "supervised_%s%d.pt" % (kind, epoch))
    best_pt, best_json = os.path.join(out_dir, "supervised_model_best.pt"), os.path.join(out_dir, "supervised_model_best.json")
    best = None
    if start_epoch > 1:
        try:
            model.load_state_dict(torch.load(path("", start_epoch - 1), map_location="cpu"))
            optimiser.load_state_dict(torch.load(path("opt_", start_epoch - 1), map_location="cpu"))
            scheduler.load_state_dict(torch.load(path("sched_", start_epoch - 1), map_location="cpu"))
            if os.path.exists(best_json):
                with open(best_json) as f:
                    best = json.load(f)
        except OSError:
            log("No saved weights from epoch %d found!" % (start_epoch - 1))
            start_epoch = 1
    history = []
    for epoch in range(start_epoch, epochs + 1):
        t0 = time.perf_counter()
        hist = train_on_records(model, rec, epochs=1, batch_size=batch_size, optimiser=optimiser, lr_scheduler=scheduler, device="cuda",
                                seed=seed + epoch)
        seconds = time.perf_counter() - t0
        mse, ce = (float(x) for x in np.mean(hist, axis=0))
        h_mse, h_ce = evaluate_records(model, held) if held is not None else (float("nan"), float("nan"))
        torch.save(model.state_dict(), path("", epoch))
        torch.save(optimiser.state_dict(), path("opt_", epoch))
        torch.save(scheduler.state_dict(), path("sched_", epoch))
        loss = h_mse + h_ce if held is not None else mse + ce
        if best is None or loss < best["loss"]:
            best = {"epoch": epoch, "loss": loss, "heldout_mse": h_mse, "heldout_ce": h_ce, "train_mse": mse, "train_ce": ce}
            torch.save(model.state_dict(), best_pt)
            with open(best_json, "w") as f:
                json.dump(best, f)
        positions = len(hist) * min(batch_size, len(rec["z"]))
        history.append({"epoch": epoch, "steps": len(hist), "train_mse": mse, "train_ce": ce, "heldout_mse": h_mse, "heldout_ce": h_ce,
                        "seconds": seconds, "positions_per_sec": positions / seconds, "lr": scheduler.get_last_lr()[0]})
        log("epoch %d: train mse %.4f ce %.4f | held-out mse %.4f ce %.4f | %.2f s, %.0f positions/s%s"
            % (epoch, mse, ce, h_mse, h_ce, seconds, positions / seconds, " (best)" if best["epoch"] == epoch else ""))
    return model, history


def parse_args(argv=None):
    """command line -> keyword arguments of main()"""
    import argparse
    ap = argparse.ArgumentParser(description="supervised pre-training on PGN games (SGD + StepLR, train_supervised.py) on the B200 "
                                             "library's trainer; writes supervised_model_best.pt for train_RL --weights")
    ap.add_argument("--pgn", required=True, help="PGN file, plain text or .bz2")
    ap.add_argument("--num_games", type=int, default=0, help="balanced selection of this many games (0: every game with a result)")
    ap.add_argument("--holdout", type=float, default=0.02, help="fraction of the games held out for the eval-mode loss")
    ap.add_argument("--epochs", type=int, default=10, help="last epoch to train")
    ap.add_argument("--batch_size", type=int, default=128)
    ap.add_argument("--weights", default=None, help="state_dict to start from")
    ap.add_argument("--out_dir", default=".")
    ap.add_argument("--start_epoch", type=int, default=1, help="resume from the files of epoch start_epoch - 1")
    ap.add_argument("--seed", type=int, default=0, help="held-out split and batch order")
    return vars(ap.parse_args(argv))


if __name__ == "__main__":
    main(**parse_args())
