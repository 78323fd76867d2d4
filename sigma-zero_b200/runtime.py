"""Process-wide engine management for the drop-in facade: one libszb200 context per GPU, grown on demand,
with the model's weights pushed to it whenever they change.  Host logic only."""
import math
import os

import numpy as np

from .engine import EVAL_NET_BF16, EVAL_NET_FP32, Engine

_engine = None
_weights_key = None

DEFAULT_PRECISION = os.environ.get("SZB_PRECISION", "bf16")     # "bf16" (tcgen05) or "fp32" (parity mode)


def device_ordinal():
    return int(os.environ.get("LOCAL_RANK", os.environ.get("SZB_DEVICE", "0")))


def get_engine(min_games=1, min_searches=800, leaves_per_tree=None):
    """An Engine with at least the requested capacity (re-created, and weights re-sent, when it must grow or when the
    search mode changes).  leaves_per_tree: None = keep the current engine's mode (1 for a new one)."""
    global _engine, _weights_key
    want_k = (_engine.leaves_per_tree if _engine else 1) if leaves_per_tree is None else int(leaves_per_tree)
    if _engine is None or _engine.max_games < min_games or _engine.max_searches < min_searches or _engine.leaves_per_tree != want_k:
        games = max(min_games, _engine.max_games if _engine else 1)
        searches = max(min_searches, _engine.max_searches if _engine else 1)
        if _engine is not None:
            _engine.close()
        _engine = Engine(max_games=games, max_searches=searches, device=device_ordinal(), leaves_per_tree=want_k)
        _engine.owner = None
        _weights_key = None
    return _engine


def leaves_of(args):
    """args['leaves_per_tree'] (an extension of the reference's args dict; default 1 = the reference's search)"""
    return int((args or {}).get('leaves_per_tree', 1))


def exploration_of(args):
    """Engine.set_exploration keywords (alpha, epsilon, sample_plies) from the args-dict extensions 'dirichlet_alpha' (absent = off),
    'dirichlet_epsilon' (default 0.25) and 'sample_plies' (default 0 = sample every ply).  Raises ValueError on a negative or
    non-finite alpha, an epsilon outside [0, 1] or a negative sample_plies."""
    args = args or {}
    alpha = float(args.get('dirichlet_alpha', 0.0))
    epsilon = float(args.get('dirichlet_epsilon', 0.25))
    sample_plies = args.get('sample_plies', 0)
    if not math.isfinite(alpha) or alpha < 0.0:
        raise ValueError("dirichlet_alpha must be a finite value >= 0, not %r" % (args.get('dirichlet_alpha'),))
    if not 0.0 <= epsilon <= 1.0:
        raise ValueError("dirichlet_epsilon must lie in [0, 1], not %r" % (args.get('dirichlet_epsilon'),))
    if int(sample_plies) != sample_plies or int(sample_plies) < 0:
        raise ValueError("sample_plies must be an integer >= 0, not %r" % (sample_plies,))
    return {"alpha": alpha, "epsilon": epsilon, "sample_plies": int(sample_plies)}


def eval_cache_of(args):
    """Engine.set_eval_cache's slots_per_game from the args-dict extension 'eval_cache_slots' (absent = 0 = off).  Raises
    ValueError unless it is 0 or a power of two in [64, 65536]."""
    slots = (args or {}).get('eval_cache_slots', 0)
    if slots is None:
        slots = 0
    if int(slots) != slots or not (int(slots) == 0 or (64 <= int(slots) <= 65536 and int(slots) & (int(slots) - 1) == 0)):
        raise ValueError("eval_cache_slots must be 0 or a power of two in [64, 65536], not %r" % (slots,))
    return int(slots)


def evaluator_of(model):
    prec = getattr(model, "precision", DEFAULT_PRECISION)
    return EVAL_NET_FP32 if prec == "fp32" else EVAL_NET_BF16


def _key_of(engine, model):
    sd = model.state_dict()
    return (id(model), id(engine), tuple(int(getattr(v, "_version", 0)) for v in sd.values()), tuple(v.data_ptr() for v in sd.values()))


def flat_weights(model, device):
    """(keys, element counts, ONE flat fp32 tensor on `device`) of the model's state_dict, num_batches_tracked left out"""
    import torch
    sd = model.state_dict()
    keys = [k for k in sd if not k.endswith("num_batches_tracked")]
    flat = torch.cat([sd[k].detach().reshape(-1).float() for k in keys]).to(device)
    return keys, [int(sd[k].numel()) for k in keys], flat


def sync_weights(engine, model):
    """Send the model's weights to the GPU library if they changed since the last call: one flat fp32 buffer on the device
    (wherever the parameters live), BatchNorm folding and packing by the library's own kernels (szb_net_load_device)."""
    global _weights_key
    key = _key_of(engine, model)
    if key != _weights_key:
        import torch
        keys, numels, flat = flat_weights(model, torch.device("cuda", engine.device))
        engine.load_flat_device(keys, numels, flat)
        _weights_key = key


def mark_synced(engine, model):
    """the engine was just loaded with exactly this model's weights by other means (train_RL.broadcast_weights)"""
    global _weights_key
    _weights_key = _key_of(engine, model)


def unpack_planes(words):
    """uint64[..., 119] -> bool[..., 119, 8, 8] (host-side view change of the GPU encoder's output)"""
    w = np.ascontiguousarray(words, dtype="<u8")
    bits = np.unpackbits(w.view(np.uint8).reshape(w.shape + (8,)), axis=-1, bitorder="little")
    return bits.reshape(w.shape + (8, 8)).astype(bool)


def pack_planes(planes):
    """bool/float[..., 119, 8, 8] -> uint64[..., 119]"""
    p = np.asarray(planes) != 0
    flat = p.reshape(p.shape[:-2] + (64,))
    return np.packbits(flat, axis=-1, bitorder="little").view("<u8").reshape(p.shape[:-2])
