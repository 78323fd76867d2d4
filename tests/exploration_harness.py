"""Host build of the root exploration sampler (tests/host_harness/exploration.cpp, compiled from tree.cuh) for the exploration
tests.  The library is built into a temporary directory, so a read-only checkout works."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from tests import util

_lib = None


def load():
    global _lib
    if _lib is None:
        src = os.path.join(util.ROOT, "tests", "host_harness", "exploration.cpp")
        out = os.path.join(tempfile.mkdtemp(prefix="szb_exploration_"), "exploration.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-Wno-unknown-pragmas",
                               "-o", out, src])
        lib = ctypes.CDLL(out)
        sig = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p]
        for f in (lib.hx_dirichlet, lib.hx_dirichlet_log):
            f.argtypes, f.restype = sig, None
        _lib = lib
    return _lib


def _call(fn, seed, game_id, ply, moves, alpha):
    moves = np.ascontiguousarray(moves, dtype=np.uint16)
    out = np.zeros(len(moves), dtype=np.float64)
    fn(seed, game_id, ply, len(moves), moves.ctypes.data, alpha, out.ctypes.data)
    return out


def eta(seed, game_id, ply, moves, alpha):
    """Dir(alpha) sample over the children `moves` for the key (seed, global game id, root ply), float64"""
    return _call(load().hx_dirichlet, seed, game_id, ply, moves, alpha)


def log_gamma(seed, game_id, ply, moves, alpha):
    """the children's log-gamma draws"""
    return _call(load().hx_dirichlet_log, seed, game_id, ply, moves, alpha)
