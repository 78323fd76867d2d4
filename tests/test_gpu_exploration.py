"""Opt-in root exploration on the GPU (szb_set_exploration): off is bit-identical to a context that never set it, the root
priors are the host harness's Dirichlet sample mixed by the documented formula, interior nodes get raw priors, the noise is
keyed by (seed, global game id, ply, move) only, the sampling horizon plays the first maximum, and the product path carries
the args keys through."""
import numpy as np
import pytest
import torch

from tests import exploration_harness

pytestmark = pytest.mark.gpu

EPS = np.float32(0.25)


def random_games(n, seed, max_plies=24):
    """start ids (vanilla and Chess960) and random legal move sequences of different lengths (0 .. max_plies) for n games"""
    from sigma_zero_b200.engine import Engine
    rng = np.random.default_rng(seed)
    starts = [int(rng.integers(0, 960)) if g % 2 else -1 for g in range(n)]
    target = [(g * 7) % (max_plies + 1) for g in range(n)]
    eng = Engine(max_games=n, max_searches=1)
    eng.reset(starts)
    hist = [[] for _ in range(n)]
    for p in range(max_plies):
        idx, cnt = eng.legal_moves()
        who = [g for g in range(n) if target[g] > p and cnt[g] > 0]
        mv = [int(idx[g, rng.integers(0, cnt[g])]) for g in who]
        if who:
            eng.push(who, mv)
        for g, m in zip(who, mv):
            hist[g].append(m)
    eng.close()
    return starts, hist


def replay(eng, starts, hist):
    eng.reset(starts)
    for r in range(max([len(h) for h in hist] + [0])):
        who = [g for g, h in enumerate(hist) if len(h) > r]
        eng.push(who, [hist[g][r] for g in who])


def root_priors(eng, g):
    t = eng.tree_export(g)
    f, k = int(t["node_first"][0]), int(t["node_count"][0])
    return t["edge_move"][f:f + k].copy(), t["edge_prior"][f:f + k].copy()


def test_off_is_today():
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, S = 64, 200
    starts, hist = random_games(G, seed=1)

    def run(eng, learning):
        replay(eng, starts, hist)
        vis, _, _ = eng.search(S, 2.0, learning, EVAL_HASH)
        priors = [eng.tree_export(g)["edge_prior"].copy() for g in range(0, G, 8)]
        moves = [eng.selfplay_ply(S, 2.0, learning, EVAL_HASH, seed=3, sample=True)[0] for _ in range(8)]
        return vis, priors, moves

    def same(a, b):
        assert np.array_equal(a[0], b[0])
        assert all(np.array_equal(x, y) for x, y in zip(a[1], b[1]))
        assert all(np.array_equal(x, y) for x, y in zip(a[2], b[2]))

    ref = Engine(G, S)
    today = {learning: run(ref, learning) for learning in (True, False)}
    eng = Engine(G, S)
    eng.set_exploration(alpha=0.3, epsilon=0.25, seed=5, sample_plies=3)
    assert eng.lib.szb_set_exploration(eng._h, None) == 0                  # NULL: off
    same(run(eng, True), today[True])
    eng.set_exploration(alpha=0.3, epsilon=0.25, seed=5)                   # noise on, but a learning=False search
    same(run(eng, False), today[False])
    eng.set_exploration(sample_plies=0)
    same(run(eng, True), today[True])


def test_bad_settings_are_refused_and_leave_the_setting():
    from sigma_zero_b200.engine import EVAL_HASH, Engine, SzbError
    eng = Engine(4, 8)
    eng.reset([-1, 0, 518, 959])
    eng.set_exploration(alpha=0.3, epsilon=1.0, seed=2)
    eng.search(1, 2.0, True, EVAL_HASH)
    want = [root_priors(eng, g)[1] for g in range(4)]
    for bad in (dict(alpha=-1.0), dict(alpha=float("nan")), dict(alpha=float("inf")), dict(epsilon=1.5), dict(epsilon=-0.5),
                dict(sample_plies=-2)):
        with pytest.raises(SzbError) as e:
            eng.set_exploration(**dict(dict(alpha=0.3, epsilon=0.25, seed=9), **bad))
        assert e.value.code == -1
    eng.search(1, 2.0, True, EVAL_HASH)
    assert all(np.array_equal(root_priors(eng, g)[1], want[g]) for g in range(4))


def test_root_priors_are_the_host_dirichlet_mixed_in_double():
    """at eps = 1 the root priors are fl32(eta) of the host harness's sampler for the same key; at eps = 0.25 they are
    fl32((1 - eps) p + eps eta) recomputed in float64, bit for bit, with p the learning=False priors"""
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, seed = 256, 77
    starts, hist = random_games(G, seed=2)
    eng = Engine(G, 4)
    replay(eng, starts, hist)
    ply = [p.ply for p in eng.positions()]
    assert min(ply) == 0 and max(ply) >= 20
    checked = 0
    for alpha in (0.3, 2.5):
        runs = {}
        for name, eps, learning in (("eta", 1.0, True), ("mixed", float(EPS), True), ("raw", 1.0, False)):
            eng.set_exploration(alpha=alpha, epsilon=eps, seed=seed)
            eng.search(1, 2.0, learning, EVAL_HASH, want_visits=False, want_children=False)
            runs[name] = [root_priors(eng, g) for g in range(G)]
        for g in range(G):
            moves, eta = runs["eta"][g]
            if len(moves) == 0:
                continue
            assert np.array_equal(moves, runs["raw"][g][0]) and np.array_equal(moves, runs["mixed"][g][0])
            host = exploration_harness.eta(seed, g, ply[g], moves, float(np.float32(alpha)))     # the ABI carries alpha as fp32
            np.testing.assert_allclose(eta, host.astype(np.float32), rtol=1e-6, atol=1e-38)
            assert abs(float(eta.astype(np.float64).sum()) - 1.0) < 1e-5
            p = runs["raw"][g][1].astype(np.float64)
            e = np.float64(EPS)
            want = ((1.0 - e) * p + e * eta.astype(np.float64)).astype(np.float32)
            assert np.array_equal(runs["mixed"][g][1], want), g
            checked += 1
    assert checked >= 2 * (G - 8)


def test_interior_nodes_get_raw_priors():
    """every expanded non-root node of a noised search holds the priors a learning=False search gives at the root of the same
    position (history and repetition planes included: the second context replays the game and the node's path)"""
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, S = 8, 64
    starts, hist = random_games(G, seed=3, max_plies=12)
    eng = Engine(G, S)
    replay(eng, starts, hist)
    eng.set_exploration(alpha=0.3, epsilon=0.25, seed=5)
    eng.search(S, 2.0, True, EVAL_HASH)
    cases = []
    for g in range(G):
        t = eng.tree_export(g)
        for i in range(1, len(t["node_count"])):
            f, k = int(t["node_first"][i]), int(t["node_count"][i])
            if k == 0:
                continue
            path, j = [], i
            while j != 0:
                path.append(int(t["edge_move"][t["node_parent_edge"][j]]))
                j = int(t["node_parent"][j])
            cases.append((g, path[::-1], t["edge_move"][f:f + k].copy(), t["edge_prior"][f:f + k].copy()))
    assert len(cases) >= G * S // 2
    chk = Engine(len(cases), 1)
    replay(chk, [starts[g] for g, *_ in cases], [hist[g] + path for g, path, *_ in cases])
    chk.search(1, 2.0, False, EVAL_HASH, want_visits=False, want_children=False)
    for c, (g, path, moves, priors) in enumerate(cases):
        m, p = root_priors(chk, c)
        assert np.array_equal(m, moves) and np.array_equal(p, priors), (g, path)


def test_noise_is_keyed_by_seed():
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, S = 64, 100
    starts, hist = random_games(G, seed=4)
    eng = Engine(G, S)
    replay(eng, starts, hist)
    out = []
    for seed in (1, 1, 2):
        eng.set_exploration(alpha=0.3, epsilon=0.25, seed=seed)
        vis, _, _ = eng.search(S, 2.0, True, EVAL_HASH)
        out.append((vis, [root_priors(eng, g)[1] for g in range(G)]))
    assert np.array_equal(out[0][0], out[1][0]) and all(np.array_equal(a, b) for a, b in zip(out[0][1], out[1][1]))
    differ = sum(not np.array_equal(a, b) for a, b in zip(out[0][1], out[2][1]) if len(a) > 1)
    assert differ >= G - 8


@pytest.mark.parametrize("network", [False, True])
def test_noise_does_not_depend_on_cohorts_or_context(network):
    """games 512..1023 of a 1024-game context (two cohorts) = the same games alone in a 512-game context with game id base 512"""
    from sigma_zero_b200.engine import EVAL_HASH, EVAL_NET_BF16, Engine
    from sigma_zero_b200.network import policyNN
    S = 100
    starts, hist = random_games(1024, seed=5, max_plies=10)
    big, small = Engine(1024, S), Engine(512, S)
    ev = EVAL_HASH
    if network:
        torch.manual_seed(0)
        sd = policyNN({}).eval().state_dict()
        big.load_state_dict(sd)
        small.load_state_dict(sd)
        ev = EVAL_NET_BF16
    replay(big, starts, hist)
    replay(small, starts[512:], hist[512:])
    small.set_game_id_base(512)
    for e in (big, small):
        e.set_exploration(alpha=0.3, epsilon=0.25, seed=6)
    vb, _, _ = big.search(S, 2.0, True, ev)
    vs, _, _ = small.search(S, 2.0, True, ev)
    assert np.array_equal(vb[512:], vs)
    for g in (512, 600, 777, 1023):
        mb, pb = root_priors(big, g)
        ms, ps = root_priors(small, g - 512)
        assert np.array_equal(mb, ms) and np.array_equal(pb, ps)


def test_noise_does_not_depend_on_leaves_per_tree():
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, S = 64, 100
    starts, hist = random_games(G, seed=6)
    pri = []
    for k in (1, 4):
        eng = Engine(G, S, leaves_per_tree=k)
        replay(eng, starts, hist)
        eng.set_exploration(alpha=0.3, epsilon=0.25, seed=8)
        eng.search(S, 2.0, True, EVAL_HASH)
        pri.append([root_priors(eng, g) for g in range(G)])
        eng.close()
    for (m1, p1), (m4, p4) in zip(*pri):
        assert np.array_equal(m1, m4) and np.array_equal(p1, p4)


def test_sampling_horizon():
    """sample_plies = 4: plies 0-3 are the moves sampling plays (same RNG key), from ply 4 on the first maximum of the visits"""
    from sigma_zero_b200.engine import EVAL_HASH, Engine
    G, S = 256, 32
    eng = Engine(G, S)
    runs = {}
    for sp in (4, 0):
        eng.reset([(g * 37) % 960 if g % 2 else -1 for g in range(G)])
        eng.set_exploration(alpha=0.3, epsilon=0.25, seed=11, sample_plies=sp)
        plies = []
        for _ in range(12):
            moves, _ = eng.selfplay_ply(S, 2.0, True, EVAL_HASH, seed=11, sample=True)
            plies.append((moves, *eng.root_children()))
        runs[sp] = plies
    for ply in range(4):
        assert np.array_equal(runs[4][ply][0], runs[0][ply][0])
    not_argmax = {4: 0, 0: 0}
    for sp in (4, 0):
        for ply in range(4, 12):
            moves, idx, vis, cnt = runs[sp][ply]
            for g in np.nonzero(moves >= 0)[0]:
                k = int(cnt[g])
                not_argmax[sp] += int(moves[g] != idx[g, int(np.argmax(vis[g, :k]))])
    assert not_argmax[4] == 0
    assert not_argmax[0] > 0                                        # without the horizon the later plies are still sampled


def test_product_path_carries_the_keys(tmp_path):
    from sigma_zero_b200.chess_tensor import ChessTensor
    from sigma_zero_b200.mcts import MCTS0
    from sigma_zero_b200.network import policyNN
    from sigma_zero_b200.sim import selfplay_records
    from sigma_zero_b200.train_RL import concat_records, main, shard_of
    torch.manual_seed(0)
    model = policyNN({}).eval()
    # MCTS0.search: noise at the root with learning=True
    game = ChessTensor()
    mcts = MCTS0(game, {"C": 2, "num_searches": 40, "dirichlet_alpha": 0.3, "seed": 3}, model)
    priors = {}
    for learning in (True, False):
        mcts.search(game.board, verbose=False, learning=learning)
        priors[learning] = np.array([c.prior for c in mcts.tree().children])
    assert len(priors[True]) == 20 and not np.array_equal(priors[True], priors[False])
    assert abs(priors[True].sum() - 1.0) < 1e-5
    # selfplay_records: deterministic for a seed, equal to its shards; without the keys the shared engine is off again
    keys = {"dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.25, "sample_plies": 3}
    base = {"C": 2, "num_searches": 12}
    off1, _ = selfplay_records(model, base, 10, c960=True, seed=7, max_plies=6)
    on1, _ = selfplay_records(model, dict(base, **keys), 10, c960=True, seed=7, max_plies=6)
    on2, _ = selfplay_records(model, dict(base, **keys), 10, c960=True, seed=7, max_plies=6)
    off2, _ = selfplay_records(model, base, 10, c960=True, seed=7, max_plies=6)
    parts = []
    for rank in range(2):
        lo, hi = shard_of(10, rank, 2)
        rec, _ = selfplay_records(model, dict(base, **keys), hi - lo, c960=True, seed=7, max_plies=6, game_id_base=lo)
        rec["game"] = rec["game"] + lo
        parts.append(rec)
    sharded = concat_records(parts)
    fields = ("states", "pi_index", "pi_prob", "pi_off", "z", "game", "result")
    assert all(np.array_equal(on1[k], on2[k]) and np.array_equal(on1[k], sharded[k]) for k in fields)
    assert all(np.array_equal(off1[k], off2[k]) for k in fields)
    assert not all(np.array_equal(on1[k], off1[k]) for k in fields)
    # train_RL.main with the keys: one tiny epoch end to end
    args = dict({"C": 2, "num_searches": 8, "num_epochs": 2, "batch_size": 4, "chess960": True}, **keys)
    _, hist = main(args, model=policyNN({}), num_games=4, out_dir=str(tmp_path), max_plies=6, passes_per_epoch=1,
                   train_device="cuda", log=lambda *a: None)
    assert [h["epoch"] for h in hist] == [1] and 0 < hist[0]["positions"] <= 24
    assert np.isfinite(np.array(hist[0]["losses"])).all()
