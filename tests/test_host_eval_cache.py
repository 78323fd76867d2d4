"""Opt-in evaluation cache without a GPU: the args-key validation of runtime.eval_cache_of, the train_RL command line, the
ABI struct and the header / ctypes signatures of the two new entry points."""
import ctypes
import os
import re

import pytest


def test_eval_cache_of_validates():
    from sigma_zero_b200 import runtime
    assert runtime.eval_cache_of(None) == 0
    assert runtime.eval_cache_of({"num_searches": 10}) == 0
    assert runtime.eval_cache_of({"eval_cache_slots": 0}) == 0
    for ok in (64, 128, 2048, 65536):
        assert runtime.eval_cache_of({"eval_cache_slots": ok}) == ok
    for bad in (-64, 1, 32, 63, 100, 96, 131072, 2048.5, "x"):
        with pytest.raises((ValueError, TypeError)):
            runtime.eval_cache_of({"eval_cache_slots": bad})


def test_train_rl_command_line_defaults_to_off():
    from sigma_zero_b200 import runtime, train_RL
    ns = vars(train_RL.build_parser().parse_args([]))
    assert ns["eval_cache_slots"] == 0
    assert runtime.eval_cache_of({k: ns[k] for k in train_RL.CLI_ARGS}) == 0
    ns = vars(train_RL.build_parser().parse_args(["--eval_cache_slots", "2048"]))
    assert runtime.eval_cache_of({k: ns[k] for k in train_RL.CLI_ARGS}) == 2048
    assert "eval_cache_slots" not in train_RL.DEFAULT_ARGS


def test_eval_cache_stats_struct_layout():
    from sigma_zero_b200 import _lib
    assert ctypes.sizeof(_lib.EvalCacheStats) == 56
    assert [(n, getattr(_lib.EvalCacheStats, n).offset) for n, _ in _lib.EvalCacheStats._fields_] == \
        [("lookups", 0), ("hits", 8), ("inserts", 16), ("dropped_inserts", 24), ("boards_evaluated", 32), ("bytes", 40),
         ("slots_per_game", 48), ("reserved", 52)]
    assert ctypes.sizeof(_lib.Stats) == 48                 # szb_stats did not grow


def test_header_matches_signatures():
    from sigma_zero_b200 import _lib
    from tests import util
    header = open(os.path.join(util.ROOT, "include", "szb200.h")).read()
    assert re.search(r"int szb_set_eval_cache\(szb_ctx \*ctx, int32_t slots_per_game\);", header)
    assert re.search(r"int szb_get_eval_cache_stats\(szb_ctx \*ctx, szb_eval_cache_stats \*out, uint32_t \*game_hits\);", header)
    fields = re.search(r"typedef struct szb_eval_cache_stats \{(.*?)\} szb_eval_cache_stats;", header, re.S).group(1)
    names = re.findall(r"(u?int\d+_t) (\w+);", fields)
    assert [n for _, n in names] == [n for n, _ in _lib.EvalCacheStats._fields_]
    assert _lib.SIGNATURES["szb_set_eval_cache"] == (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32])
    res, args = _lib.SIGNATURES["szb_get_eval_cache_stats"]
    assert res is ctypes.c_int and len(args) == 3 and args[1]._type_ is _lib.EvalCacheStats
