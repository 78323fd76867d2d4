"""Host logic of supervised training (no GPU): the torch optimiser -> trainer hyper-parameter mapping, its refusals, the held-out split
by game and the command line of `python -m sigma_zero_b200.supervised`."""
import pytest
import torch


def _params():
    return [torch.nn.Parameter(torch.zeros(3)), torch.nn.Parameter(torch.zeros(2))]


def test_adam_hparams_are_unchanged():
    """the values train_on_records_cuda derived before SGD existed: initial_lr when present, StepLR's counter as step0"""
    from sigma_zero_b200.train_RL import make_optimiser, trainer_hparams
    model = torch.nn.Linear(3, 2)
    opt, sched = make_optimiser(model)
    for _ in range(7):
        opt.step()
        sched.step()
    kind, hp, step0 = trainer_hparams(opt, sched)
    assert kind == "adam" and step0 == 7
    assert hp == dict(lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-4, lr_step=500, lr_gamma=0.95)
    opt = torch.optim.Adam(_params(), lr=3e-4, betas=(0.8, 0.99), eps=1e-6, weight_decay=0.0)
    kind, hp, step0 = trainer_hparams(opt, None)
    assert kind == "adam" and step0 == 0
    assert hp == dict(lr=3e-4, beta1=0.8, beta2=0.99, eps=1e-6, weight_decay=0.0, lr_step=1 << 30, lr_gamma=1.0)
    assert trainer_hparams(None, None) == ("adam", dict(lr_step=1 << 30, lr_gamma=1.0), 0)


def test_sgd_hparams_with_and_without_scheduler():
    from sigma_zero_b200.supervised import make_supervised_optimiser
    from sigma_zero_b200.train_RL import trainer_hparams
    model = torch.nn.Linear(3, 2)
    opt, sched = make_supervised_optimiser(model)
    for _ in range(4001):
        opt.step()
        sched.step()                                                      # the scheduler's lr is now halved; initial_lr is not
    assert opt.param_groups[0]["lr"] == pytest.approx(0.05)
    kind, hp, step0 = trainer_hparams(opt, sched)
    assert kind == "sgd" and step0 == 4001
    assert hp == dict(lr=0.1, weight_decay=1e-4, momentum=0.0, dampening=0.0, nesterov=False, lr_step=4000, lr_gamma=0.5)
    # no scheduler: the group's current lr, a constant schedule and step 0 -- even when a scheduler once set initial_lr
    kind, hp, step0 = trainer_hparams(opt, None)
    assert kind == "sgd" and step0 == 0
    assert hp == dict(lr=pytest.approx(0.05), weight_decay=1e-4, momentum=0.0, dampening=0.0, nesterov=False, lr_step=1 << 30, lr_gamma=1.0)
    opt = torch.optim.SGD(_params(), lr=0.02, momentum=0.9, dampening=0.0, weight_decay=0.0, nesterov=True)
    assert trainer_hparams(opt, None) == ("sgd", dict(lr=0.02, weight_decay=0.0, momentum=0.9, dampening=0.0, nesterov=True,
                                                      lr_step=1 << 30, lr_gamma=1.0), 0)


@pytest.mark.parametrize("make", [
    lambda: torch.optim.RMSprop(_params(), lr=0.01),
    lambda: torch.optim.AdamW(_params(), lr=0.01),
    lambda: torch.optim.SGD([{"params": _params()[:1]}, {"params": _params()[1:], "lr": 0.5}], lr=0.1),
    lambda: torch.optim.SGD(_params(), lr=0.1, maximize=True),
    lambda: torch.optim.Adam(_params(), lr=0.1, maximize=True),
], ids=["rmsprop", "adamw", "two_param_groups", "sgd_maximize", "adam_maximize"])
def test_unsupported_optimisers_name_the_torch_backend(make):
    """what the CUDA trainer does not implement is refused up front, before any GPU work, and the message says what to use instead"""
    from sigma_zero_b200.train_RL import train_on_records_cuda, trainer_hparams
    opt = make()
    with pytest.raises(TypeError, match='backend="torch"'):
        trainer_hparams(opt, None)
    with pytest.raises(TypeError, match='backend="torch"'):
        train_on_records_cuda(torch.nn.Linear(3, 2), {"z": []}, optimiser=opt)


def test_holdout_split_is_by_game_seeded_and_disjoint():
    from sigma_zero_b200.supervised import split_holdout
    games = [({"Result": "1-0", "Game": str(i)}, ["e4"] * (i % 7 + 1)) for i in range(200)]
    train, held = split_holdout(games, 0.1, seed=3)
    assert len(held) == 20 and len(train) == 180
    ids = lambda gs: [h["Game"] for h, _ in gs]
    assert not set(ids(train)) & set(ids(held)) and sorted(ids(train) + ids(held), key=int) == ids(games)
    assert ids(train) == sorted(ids(train), key=int) and ids(held) == sorted(ids(held), key=int)         # file order kept
    again = split_holdout(games, 0.1, seed=3)
    assert ids(again[0]) == ids(train) and ids(again[1]) == ids(held)
    assert ids(split_holdout(games, 0.1, seed=4)[1]) != ids(held)
    # a tiny file still holds out one game and trains on the rest; fraction 0 holds out none
    assert [len(x) for x in split_holdout(games[:3], 0.02)] == [2, 1]
    assert [len(x) for x in split_holdout(games[:1], 0.5)] == [1, 0]
    assert [len(x) for x in split_holdout(games, 0.0)] == [200, 0]


def test_command_line():
    from sigma_zero_b200.supervised import main, parse_args
    import inspect
    kw = parse_args(["--pgn", "games.pgn.bz2", "--num_games", "5000", "--holdout", "0.05", "--epochs", "3", "--batch_size", "256",
                     "--weights", "w.pt", "--out_dir", "run", "--start_epoch", "2", "--seed", "9"])
    assert kw == dict(pgn="games.pgn.bz2", num_games=5000, holdout=0.05, epochs=3, batch_size=256, weights="w.pt", out_dir="run",
                      start_epoch=2, seed=9)
    assert set(kw) <= set(inspect.signature(main).parameters)
    kw = parse_args(["--pgn", "g.pgn"])
    assert kw == dict(pgn="g.pgn", num_games=0, holdout=0.02, epochs=10, batch_size=128, weights=None, out_dir=".", start_epoch=1, seed=0)
    with pytest.raises(SystemExit):
        parse_args([])                                                    # --pgn is required
