"""Opt-in root exploration without a GPU: the Dirichlet sampler of tree.cuh through its host build, the argument checks of
runtime.exploration_of, the train_RL command line and the ABI struct."""
import ctypes
import math

import numpy as np
import pytest
import scipy.stats

from tests.exploration_harness import eta, log_gamma


@pytest.mark.parametrize("alpha", [0.01, 0.3, 1.0, 2.5])
@pytest.mark.parametrize("n", [1, 2, 20, 218])
def test_dirichlet_is_a_distribution(alpha, n):
    moves = np.sort(np.random.default_rng(n).choice(4672, n, replace=False))
    for key in range(50):
        e = eta(1234 + key, key, key % 200, moves, alpha)
        assert np.all(np.isfinite(e)) and np.all(e >= 0.0)
        assert abs(e.sum() - 1.0) <= 1e-6
        if n == 1:
            assert e[0] == 1.0


@pytest.mark.parametrize("alpha", [0.3, 2.5])
def test_dirichlet_marginals(alpha):
    n, keys = 20, 20000
    moves = np.arange(100, 100 + 3 * n, 3)
    e = np.stack([eta(7, g, g % 97, moves, alpha) for g in range(keys)])
    a0 = n * alpha
    var = (alpha * (a0 - alpha)) / (a0 * a0 * (a0 + 1))             # Beta(alpha, (n - 1) alpha)
    se = math.sqrt(var / keys)
    for i in range(n):
        assert abs(e[:, i].mean() - 1.0 / n) <= 5 * se, (i, e[:, i].mean())
        assert abs(e[:, i].var() / var - 1.0) <= 0.10, (i, e[:, i].var(), var)
    p = scipy.stats.kstest(e[:, 0], scipy.stats.beta(alpha, (n - 1) * alpha).cdf).pvalue
    assert p > 1e-3, p


def test_draw_depends_on_the_child_alone():
    moves = np.array([3, 77, 400, 401, 1500, 2222, 4000, 4671])
    for alpha in (0.3, 2.5):
        full = log_gamma(99, 5, 12, moves, alpha)
        sub = log_gamma(99, 5, 12, moves[[6, 1, 3]], alpha)
        assert np.array_equal(sub, full[[6, 1, 3]])
        perm = np.random.default_rng(0).permutation(len(moves))
        assert np.array_equal(log_gamma(99, 5, 12, moves[perm], alpha), full[perm])
        # ... and the key: another seed, game or ply draws differently
        for other in ((100, 5, 12), (99, 6, 12), (99, 5, 13)):
            assert not np.array_equal(log_gamma(*other, moves, alpha), full)


def test_exploration_of_validates():
    from sigma_zero_b200 import runtime
    assert runtime.exploration_of(None) == {"alpha": 0.0, "epsilon": 0.25, "sample_plies": 0}
    assert runtime.exploration_of({"num_searches": 10}) == {"alpha": 0.0, "epsilon": 0.25, "sample_plies": 0}
    assert runtime.exploration_of({"dirichlet_alpha": 0.3, "dirichlet_epsilon": 1.0, "sample_plies": 30}) == \
        {"alpha": 0.3, "epsilon": 1.0, "sample_plies": 30}
    assert runtime.exploration_of({"dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.0})["epsilon"] == 0.0
    for bad in ({"dirichlet_alpha": -0.1}, {"dirichlet_alpha": float("nan")}, {"dirichlet_alpha": float("inf")},
                {"dirichlet_epsilon": -0.01}, {"dirichlet_epsilon": 1.5}, {"dirichlet_epsilon": float("nan")},
                {"sample_plies": -1}, {"sample_plies": 2.5}):
        with pytest.raises(ValueError):
            runtime.exploration_of(bad)


def test_train_rl_command_line_defaults_to_off():
    from sigma_zero_b200 import runtime, train_RL
    ns = vars(train_RL.build_parser().parse_args([]))
    assert ns["dirichlet_alpha"] == 0.0 and ns["dirichlet_epsilon"] == 0.25 and ns["sample_plies"] == 0
    assert ns["leaves_per_tree"] == 1 and ns["num_searches"] == train_RL.DEFAULT_ARGS["num_searches"]
    assert runtime.exploration_of({k: ns[k] for k in train_RL.CLI_ARGS})["alpha"] == 0.0
    ns = vars(train_RL.build_parser().parse_args(["--dirichlet_alpha", "0.3", "--sample_plies", "30"]))
    assert runtime.exploration_of({k: ns[k] for k in train_RL.CLI_ARGS}) == {"alpha": 0.3, "epsilon": 0.25, "sample_plies": 30}
    assert "dirichlet_alpha" not in train_RL.DEFAULT_ARGS


def test_exploration_struct_layout():
    from sigma_zero_b200 import _lib
    assert ctypes.sizeof(_lib.Exploration) == 24
    assert [(n, getattr(_lib.Exploration, n).offset) for n, _ in _lib.Exploration._fields_] == \
        [("dirichlet_alpha", 0), ("dirichlet_epsilon", 4), ("seed", 8), ("sample_plies", 16), ("reserved", 20)]
