"""GPU: the leaf expansion where no other test reaches it -- a profiled search of more path slots than the other GPU tests use,
against the normal (fused) search, and szb_encode / szb_legal_moves on positions whose ring slots have wrapped."""
import numpy as np
import pytest

from oracle import hash_eval, ref_path
from tests import util

pytestmark = pytest.mark.gpu


def test_profiled_search_above_8192_paths_equals_fused():
    """~8,200 running games (vanilla and Chess960, short seeded random prefixes): the profiled search (phase kernels, one expansion
    per path slot in k_expand) and the normal search (k_tree_step) build the same trees -- visit counts, child masks, root values and
    the exported trees of a sample of games"""
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, S = 8200, 12
    rng = np.random.default_rng(17)
    eng = Engine(max_games=G, max_searches=S)
    eng.reset([-1 if g % 2 == 0 else int(rng.integers(960)) for g in range(G)])
    plies = rng.integers(0, 9, G)
    for ply in range(int(plies.max())):
        idx, cnt = eng.legal_moves()
        who = [g for g in range(G) if ply < plies[g] and cnt[g] > 0]
        eng.push(who, [int(idx[g, rng.integers(cnt[g])]) for g in who])
    running = eng.outcomes() == 0
    assert int(running.sum()) > 8192
    sample = range(0, G, 97)
    res = {}
    for prof in (False, True):
        eng.set_profiling(prof)
        v, c, val = eng.search(S, 2.0, True, EVAL_HASH, want_value=True)
        res[prof] = (v, c, val, [eng.tree_export(g) for g in sample])
    eng.set_profiling(False)
    eng.close()
    for a, b in zip(res[False][:3], res[True][:3]):
        assert np.array_equal(a, b)
    for ta, tb in zip(res[False][3], res[True][3]):
        for k in ta:
            assert np.array_equal(np.asarray(ta[k]), np.asarray(tb[k])), k
    assert (res[False][0][running].sum(axis=1) == S - 1).all() and res[False][0][~running].sum() == 0


def test_encode_past_the_position_ring():
    """games played in lock step with seeded random moves past the 256-position ring (seven of the eight reach 360 plies); from ply 200
    on, planes, legal masks and legal index lists are compared with the oracle at every ply.  From ply 256 on a position's ring slot
    is ply mod 256, so its history planes run back across slot 0 to slot 255."""
    from sigma_zero_b200.engine import Engine, child_indices
    G, PLIES = 8, 360
    rng = np.random.default_rng(5)
    eng = Engine(max_games=G, max_searches=4)
    games = util.setup_games(eng, [(g % 2 == 1, int(rng.integers(960)) if g % 2 else 518, []) for g in range(G)])
    checked = 0
    for ply in range(PLIES + 1):
        if ply >= 200:
            idx, cnt = eng.legal_moves()
            planes, mask = eng.encode()
            for g, og in enumerate(games):
                exp = util.legal_indices(og)
                assert idx[g, :cnt[g]].tolist() == exp, (g, ply)
                assert list(child_indices(mask[g])) == exp, (g, ply)
                assert np.array_equal(planes[g], hash_eval.pack_planes(og.get_representation())), (g, ply)
                checked += len(og.board.move_stack) >= 256
        who, mv = [], []
        for g, og in enumerate(games):
            if ply < PLIES and og.board.outcome() is None:
                legal = list(og.board.legal_moves)
                m = legal[rng.integers(len(legal))]
                who.append(g)
                mv.append(ref_path.move_to_index(m, og.board.turn))
                og.move_piece(m)
        if who:
            eng.push(who, mv)
    eng.close()
    assert sum(len(og.board.move_stack) >= PLIES for og in games) == 7
    assert checked > 500
