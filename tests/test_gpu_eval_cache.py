"""Opt-in exact evaluation cache on the GPU (szb_set_eval_cache): with the cache on, every move, visit count, root value, tree and
counter is bit-identical to the cache off -- with the bf16 network (pair tower, two cohorts, the one-game cluster tower) and the
hash evaluator -- while positions an earlier search of the same game evaluated skip the evaluator.  Also: exact hit accounting,
eviction, invalidation on new weights, refused settings and the product paths."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SLOTS = 2048


def make_engine(G, S, cohorts=0, leaves_per_tree=1, weights=None):
    from sigma_zero_b200.engine import Engine
    eng = Engine(max_games=G, max_searches=S, cohorts=cohorts, leaves_per_tree=leaves_per_tree)
    if weights is not None:
        eng.load_state_dict(weights)
    return eng


def random_weights(seed=0, policy_scale=1.0):
    from sigma_zero_b200.network import policyNN
    torch.manual_seed(seed)
    sd = policyNN({}).eval().state_dict()
    if policy_scale != 1.0:
        sd = {k: (v * policy_scale if k.startswith("conv_p2.") else v) for k, v in sd.items()}
    return sd


def start_ids(G):
    return [(g * 37) % 960 if g % 2 else -1 for g in range(G)]


def trajectory(eng, G, S, plies, ev, learning, seed=3, tree_games=(), explore=None):
    """self-play plies: per ply the moves, the root children, the root values and the exported trees of a few games"""
    eng.reset(start_ids(G))
    if explore:
        eng.set_exploration(**explore)
    out = []
    for _ in range(plies):
        moves, _ = eng.selfplay_ply(S, 2.0, learning, ev, seed=seed, sample=True)
        idx, vis, cnt = eng.root_children()
        trees = [eng.tree_export(g) for g in tree_games]
        out.append((moves, idx, vis, cnt, trees))
    st = eng.stats()
    return out, st


def assert_same(a, b):
    (ta, sa), (tb, sb) = a, b
    assert len(ta) == len(tb)
    for pa, pb in zip(ta, tb):
        for x, y in zip(pa[:4], pb[:4]):
            assert np.array_equal(x, y)
        for xa, xb in zip(pa[4], pb[4]):
            assert xa.keys() == xb.keys()
            for k in xa:
                assert np.array_equal(np.asarray(xa[k]), np.asarray(xb[k])), k
    assert sa == sb


def run_pair(G, S, plies, ev, learning, cohorts=0, weights=None, slots=SLOTS, explore=None, tree_games=(0,)):
    off = make_engine(G, S, cohorts, weights=weights)
    ref = trajectory(off, G, S, plies, ev, learning, tree_games=tree_games, explore=explore)
    off.close()
    on = make_engine(G, S, cohorts, weights=weights)
    on.set_eval_cache(slots)
    got = trajectory(on, G, S, plies, ev, learning, tree_games=tree_games, explore=explore)
    cs = on.eval_cache_stats()
    on.close()
    return ref, got, cs


@pytest.mark.parametrize("cohorts", [1, 2])
@pytest.mark.parametrize("learning", [True, False])
@pytest.mark.parametrize("explore", [None, {"alpha": 0.3, "epsilon": 0.25, "seed": 5, "sample_plies": 6}])
def test_hash_selfplay_is_bit_identical(cohorts, learning, explore):
    from sigma_zero_b200.engine import EVAL_HASH
    ref, got, cs = run_pair(64, 200, 16, EVAL_HASH, learning, cohorts=cohorts, explore=explore, tree_games=(0, 31, 63))
    assert_same(ref, got)
    assert cs["hits"] > 0 and cs["lookups"] == ref[1]["evaluations"]
    assert cs["boards_evaluated"] + cs["hits"] == cs["lookups"]


def test_bf16_selfplay_is_bit_identical_64_games():
    from sigma_zero_b200.engine import EVAL_NET_BF16
    ref, got, cs = run_pair(64, 200, 16, EVAL_NET_BF16, True, weights=random_weights(), tree_games=(0, 17, 63))
    assert_same(ref, got)
    assert cs["hits"] > 0 and cs["lookups"] == ref[1]["evaluations"]


def test_bf16_selfplay_is_bit_identical_1024_games_two_cohorts():
    from sigma_zero_b200.engine import EVAL_NET_BF16
    ref, got, cs = run_pair(1024, 800, 3, EVAL_NET_BF16, True, weights=random_weights(), tree_games=(0, 700))
    assert_same(ref, got)
    assert cs["hits"] > 0 and cs["boards_evaluated"] + cs["hits"] == ref[1]["evaluations"]


def test_bf16_chunked_tower_one_cohort_is_bit_identical():
    """one cohort of 1024 boards: the tower runs as chunks of 512, each clamped to the device count of compacted rows"""
    from sigma_zero_b200.engine import EVAL_NET_BF16
    ref, got, cs = run_pair(1024, 800, 2, EVAL_NET_BF16, True, cohorts=1, weights=random_weights(), tree_games=(0, 1023))
    assert_same(ref, got)
    assert cs["hits"] > 0 and cs["boards_evaluated"] + cs["hits"] == ref[1]["evaluations"]


def test_bf16_one_game_cluster_tower_is_bit_identical():
    from sigma_zero_b200.engine import EVAL_NET_BF16
    ref, got, cs = run_pair(1, 200, 8, EVAL_NET_BF16, False, weights=random_weights(), tree_games=(0,))
    assert_same(ref, got)
    assert cs["hits"] > 0


def test_second_search_of_the_same_positions_is_all_hits():
    from sigma_zero_b200.engine import EVAL_HASH, EVAL_NET_BF16
    for ev, w in ((EVAL_HASH, None), (EVAL_NET_BF16, random_weights())):
        G, S = 64, 200
        eng = make_engine(G, S, weights=w)
        eng.reset(start_ids(G))
        eng.set_eval_cache(SLOTS)
        v1, _, r1 = eng.search(S, 2.0, False, ev, want_value=True)
        c1 = eng.eval_cache_stats()
        assert c1["dropped_inserts"] == 0 and c1["inserts"] + c1["hits"] == c1["lookups"] > 0   # nothing dropped: all stored
        v2, _, r2 = eng.search(S, 2.0, False, ev, want_value=True)
        c2 = eng.eval_cache_stats(game_hits=True)
        assert np.array_equal(v1, v2) and np.array_equal(r1, r2)
        assert c2["lookups"] - c1["lookups"] == c2["hits"] - c1["hits"] > 0
        assert c2["boards_evaluated"] == c1["boards_evaluated"]
        assert int(c2["game_hits"].sum()) == c2["hits"] - c1["hits"]
        # after the arg-max move every game's new root (a visited child of the last root) is a hit
        idx, vis, cnt = eng.root_children()
        best = [int(idx[g, int(np.argmax(vis[g, :cnt[g]]))]) for g in range(G)]
        eng.push(list(range(G)), best)
        live = eng.outcomes() == 0
        eng.search(S, 2.0, False, ev, want_visits=False, want_children=False)
        c3 = eng.eval_cache_stats(game_hits=True)
        assert np.all(c3["game_hits"][live] >= 1)
        eng.close()


def test_game_hits_do_not_depend_on_reruns_or_cohorts():
    from sigma_zero_b200.engine import EVAL_HASH
    G, S = 96, 100
    per = []
    for cohorts in (1, 2, 1):
        eng = make_engine(G, S, cohorts)
        eng.set_eval_cache(SLOTS)
        eng.reset(start_ids(G))
        hits = []
        for _ in range(6):
            eng.selfplay_ply(S, 2.0, True, EVAL_HASH, seed=9, sample=True)
            hits.append(eng.eval_cache_stats(game_hits=True)["game_hits"].copy())
        per.append(np.stack(hits))
        eng.close()
    assert np.array_equal(per[0], per[1]) and np.array_equal(per[0], per[2])
    assert per[0].sum() > 0


def test_small_table_drops_inserts_and_stays_bit_identical():
    from sigma_zero_b200.engine import EVAL_HASH, EVAL_NET_BF16
    ref, got, cs = run_pair(16, 800, 4, EVAL_HASH, True, slots=64)
    assert_same(ref, got)
    assert cs["dropped_inserts"] > 0 and cs["hits"] > 0
    ref, got, cs = run_pair(16, 800, 2, EVAL_NET_BF16, True, slots=64, weights=random_weights())
    assert_same(ref, got)
    assert cs["dropped_inserts"] > 0


def test_new_weights_or_evaluator_invalidate():
    from sigma_zero_b200.engine import EVAL_HASH, EVAL_NET_BF16
    G, S = 32, 200
    w0, w1 = random_weights(0), random_weights(1)

    def fresh(w, ev):
        e = make_engine(G, S, weights=w)
        e.reset(start_ids(G))
        v, _, r = e.search(S, 2.0, False, ev, want_value=True)
        e.close()
        return v, r

    eng = make_engine(G, S, weights=w0)
    eng.set_eval_cache(SLOTS)
    eng.reset(start_ids(G))
    eng.search(S, 2.0, False, EVAL_NET_BF16)
    eng.load_state_dict(w1)                              # different weights: nothing of the previous search may be reused
    before = eng.eval_cache_stats()
    v, _, r = eng.search(S, 2.0, False, EVAL_NET_BF16, want_value=True)
    fv, fr = fresh(w1, EVAL_NET_BF16)
    assert np.array_equal(v, fv) and np.array_equal(r, fr)
    after = eng.eval_cache_stats()
    assert after["hits"] - before["hits"] < after["lookups"] - before["lookups"]
    # switch to the hash evaluator and back: keys carry the evaluator
    v, _, r = eng.search(S, 2.0, False, EVAL_HASH, want_value=True)
    hv, hr = fresh(None, EVAL_HASH)
    assert np.array_equal(v, hv) and np.array_equal(r, hr)
    v, _, r = eng.search(S, 2.0, False, EVAL_NET_BF16, want_value=True)
    assert np.array_equal(v, fv) and np.array_equal(r, fr)
    eng.close()


def test_refused_settings_leave_the_setting():
    from sigma_zero_b200.engine import SzbError
    eng = make_engine(8, 16)
    eng.set_eval_cache(256)
    s0 = eng.eval_cache_stats()
    assert s0["slots_per_game"] == 256 and s0["bytes"] == 8 * 256 * 928
    for bad in (32, 100, 96, 131072, -64, 1):
        with pytest.raises(SzbError) as ei:
            eng.set_eval_cache(bad)
        assert ei.value.code == -1
        assert eng.eval_cache_stats()["slots_per_game"] == 256
    eng.set_eval_cache(256)                              # the current size keeps the table
    assert eng.eval_cache_stats()["slots_per_game"] == 256
    eng.set_eval_cache(0)
    assert eng.eval_cache_stats()["slots_per_game"] == 0 and eng.eval_cache_stats()["bytes"] == 0
    eng.close()
    ml = make_engine(8, 16, leaves_per_tree=4)
    with pytest.raises(SzbError) as ei:
        ml.set_eval_cache(256)
    assert ei.value.code == -6
    assert ml.eval_cache_stats()["slots_per_game"] == 0
    ml.set_eval_cache(0)
    ml.close()


def test_product_paths_accept_the_key(tmp_path):
    from sigma_zero_b200.arena import play_match
    from sigma_zero_b200.chess_tensor import ChessTensor
    from sigma_zero_b200.mcts import MCTS0
    from sigma_zero_b200.network import policyNN
    from sigma_zero_b200.sim import selfplay_records
    from sigma_zero_b200.train_RL import main
    torch.manual_seed(0)
    model = policyNN({}).eval()
    # MCTS0.search: the same visit fractions with the key
    probs = []
    for key in ({}, {"eval_cache_slots": 1024}):
        game = ChessTensor()
        mcts = MCTS0(game, dict({"C": 2, "num_searches": 60}, **key), model)
        probs.append(mcts.search(game.board, verbose=False))
    assert probs[0] == probs[1]
    # selfplay_records: byte-equal records
    base = {"C": 2, "num_searches": 24}
    off, _ = selfplay_records(model, base, 10, c960=True, seed=7, max_plies=8)
    on, _ = selfplay_records(model, dict(base, eval_cache_slots=SLOTS), 10, c960=True, seed=7, max_plies=8)
    for k in ("states", "pi_index", "pi_prob", "pi_off", "z", "game", "result"):
        assert np.asarray(off[k]).tobytes() == np.asarray(on[k]).tobytes(), k
    # play_match: the same games
    other = policyNN({}).eval()
    a = play_match(model, other, 4, {"C": 2, "num_searches": 16}, seed=1, max_plies=6)
    b = play_match(model, other, 4, {"C": 2, "num_searches": 16}, seed=1, max_plies=6, eval_cache_slots=512)
    assert a["moves"] == b["moves"] and a["results"] == b["results"]
    # train_RL.main with the key: one tiny epoch end to end
    args = {"C": 2, "num_searches": 8, "num_epochs": 2, "batch_size": 4, "chess960": True, "eval_cache_slots": 256}
    _, hist = main(args, model=policyNN({}), num_games=4, out_dir=str(tmp_path), max_plies=6, passes_per_epoch=1,
                   train_device="cuda", log=lambda *x: None)
    assert [h["epoch"] for h in hist] == [1] and 0 < hist[0]["positions"] <= 24
