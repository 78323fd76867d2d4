"""GPU tests of supervised training: the trainer's SGD update (szb_train_set_optimizer, csrc/train.cu) against torch.optim.SGD, StepLR,
resume through torch's SGD state_dict, the product path with make_supervised_optimiser, the eval-mode held-out loss and supervised.main
from PGN text to supervised_model_best.pt.

Tolerances follow test_gpu_trainer.py: the optimiser arithmetic is fp32 on both sides (torch may contract a + alpha * b into an FMA, so
1e-6 x max(1, max|w|) per tensor rather than exact bits); the loss trajectory is held to 0.05 nat, or to 1.25x the gap of torch's own
bf16-autocast run + 0.02 when that is larger; eval-mode losses to bf16 tolerance (MSE 2e-2 abs, CE 2 % rel)."""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _records(n, seed=0, moves=4672):
    """synthetic records; `moves` < 4672 draws the policy targets from the first `moves` indices only, a pattern the network can learn"""
    rng = np.random.default_rng(seed)
    bits = rng.random((n, 119, 64)) < 0.12
    states = np.packbits(bits, axis=-1, bitorder="little").view("<u8").reshape(n, 119).astype(np.uint64)
    idx, prob, off = [], [], [0]
    for _ in range(n):
        k = int(rng.integers(1, 30))
        ind = np.sort(rng.choice(moves, size=min(k, moves), replace=False))
        k = len(ind)
        p = rng.random(k).astype(np.float32) ** 3
        p /= p.sum()
        idx.extend(ind.tolist())
        prob.extend(p.tolist())
        off.append(len(idx))
    return {"states": states, "pi_index": np.array(idx, np.uint16), "pi_prob": np.array(prob, np.float32), "pi_off": np.array(off, np.int64),
            "z": rng.integers(-1, 2, n).astype(np.int8), "colour": np.ones(n, bool), "game": np.zeros(n, np.int32)}


def _model(seed=0):
    from sigma_zero_b200.network import policyNN
    torch.manual_seed(seed)
    model = policyNN({})
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for mod in model.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.weight.copy_(0.5 + torch.rand(mod.weight.shape, generator=g))
                mod.bias.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_mean.copy_(0.1 * torch.randn(mod.running_mean.shape, generator=g))
                mod.running_var.copy_(0.5 + torch.rand(mod.running_var.shape, generator=g))
    return model


def _torch_batch(rec, rows, dev):
    from sigma_zero_b200 import records
    x = torch.from_numpy(records.unpack_states(rec, rows)).to(device=dev, dtype=torch.float32)
    pi = torch.from_numpy(records.dense_policy(rec, rows)).to(dev)
    z = torch.from_numpy(rec["z"][rows].astype(np.float32)).to(dev)
    return x, pi, z


def _torch_losses(model, x, pi, z, autocast=False):
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        p, v = model.forward_torch(x)
    p, v = p.float(), v.float()
    return torch.nn.functional.mse_loss(v.squeeze(-1), z), torch.nn.functional.cross_entropy(p, pi)


@pytest.fixture(scope="module")
def setup():
    from sigma_zero_b200.engine import Engine
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    eng = Engine(max_games=2, max_searches=8, device=0)
    yield eng, torch.device("cuda", 0)
    eng.close()


SGD_CASES = {"recipe": dict(momentum=0.0), "momentum": dict(momentum=0.9), "nesterov": dict(momentum=0.9, nesterov=True),
             "dampening": dict(momentum=0.9, dampening=0.5)}


@pytest.mark.parametrize("case", list(SGD_CASES))
def test_sgd_update_is_torch_sgd(setup, case):
    """two steps (the second blends into the momentum buffers the first created): torch.optim.SGD fed the trainer's own gradients
    reproduces the trainer's weights and momentum buffers"""
    from sigma_zero_b200 import _lib
    from sigma_zero_b200.trainer import Trainer
    eng, dev = setup
    kw = SGD_CASES[case]
    rec = _records(48, seed=21)
    rows = [np.arange(16, dtype=np.int32), np.arange(16, 32, dtype=np.int32)]
    model = _model(11).to(dev)
    tr = Trainer(eng, model, batch_size=16, optimizer="sgd", lr=0.1, weight_decay=1e-4, **kw)
    tr.set_records(rec)
    grads = []
    for r in rows:
        tr.step(r)
        grads.append(tr.get_tensors(_lib.TRAIN_GRADS))
    got = tr.get_tensors(_lib.TRAIN_PARAMS, tr.param_keys)
    buf = tr.get_tensors(_lib.TRAIN_MOMENTUM_BUFFER) if kw["momentum"] else None
    state = tr.optimiser_state(model)
    assert tr.step_count == 2
    tr.close()
    opt = torch.optim.SGD(model.parameters(), lr=0.1, weight_decay=1e-4, **kw)
    params = dict(model.named_parameters())
    for g in grads:
        for k, p in params.items():
            p.grad = g[k].view(p.shape).to(dev)
        opt.step()
    worst = 0.0
    for k, p in params.items():
        want = p.detach().flatten().cpu()
        err = (got[k] - want).abs().max().item() / max(1.0, want.abs().max().item())
        worst = max(worst, err)
        assert err <= 1e-6, (k, err)
        if buf is not None:
            tb = opt.state[p]["momentum_buffer"].flatten().cpu()
            err = (buf[k] - tb).abs().max().item() / max(1.0, tb.abs().max().item())
            worst = max(worst, err)
            assert err <= 1e-6, (k, "momentum_buffer", err)
    print("SGD %s: worst error %.3g (relative to max(1, max|w|) per tensor)" % (case, worst))
    # the written-back state is what torch keeps: momentum buffers only with momentum, and torch accepts it
    assert (len(state["state"]) == 129) == bool(kw["momentum"]) and (state["state"] == {}) == (not kw["momentum"])
    torch.optim.SGD(model.parameters(), lr=0.1, weight_decay=1e-4, **kw).load_state_dict(state)


def test_step_lr_halves_at_step_4000(setup):
    """step0 = 3999 (StepLR(4000, 0.5) after 3999 batches): the next update still takes lr 0.1, the one after it 0.05 -- measured as the
    size of the update against the step's own gradient (momentum 0, no weight decay: w1 = w0 - lr * g)"""
    from sigma_zero_b200 import _lib
    from sigma_zero_b200.trainer import Trainer
    eng, dev = setup
    rec = _records(32, seed=22)
    model = _model(12)
    tr = Trainer(eng, model, batch_size=16, step0=3999, optimizer="sgd", weight_decay=0.0)
    tr.set_records(rec)
    lrs, state_lrs = [], []
    w = torch.cat(list(tr.get_tensors(_lib.TRAIN_PARAMS, tr.param_keys).values()))
    for r in (np.arange(16, dtype=np.int32), np.arange(16, 32, dtype=np.int32)):
        tr.step(r)
        g = torch.cat(list(tr.get_tensors(_lib.TRAIN_GRADS).values())).double()
        w1 = torch.cat(list(tr.get_tensors(_lib.TRAIN_PARAMS, tr.param_keys).values()))
        lrs.append(float(((w - w1).double() @ g) / (g @ g)))
        state_lrs.append(tr.optimiser_state(model)["param_groups"][0]["lr"])
        w = w1
    assert tr.step_count == 4001
    tr.close()
    print("learning rates measured from the updates:", lrs)
    assert abs(lrs[0] - 0.1) <= 1e-4 and abs(lrs[1] - 0.05) <= 5e-5, lrs
    assert state_lrs == [pytest.approx(0.05), pytest.approx(0.05)]


def test_loss_trajectory_tracks_torch_sgd(setup):
    """25 steps of the recipe (SGD lr 0.1, wd 1e-4) from the same start: the losses follow torch's fp32 run and the cross entropy falls.
    At lr 0.1 two runs that differ only in rounding drift apart, and the size of that drift jumps from step to step (torch's own
    bf16-autocast run against fp32: 0.001 to 0.45 nat of CE, up to 0.27 of MSE on these records), so the gap at one step says little.
    The yardstick is the largest gap the autocast run reaches over the 25 steps: every step within 0.05, or within 1.25x that gap
    + 0.02 when that is larger."""
    from sigma_zero_b200.trainer import Trainer
    eng, dev = setup
    rec = _records(128, seed=23)
    rng = np.random.default_rng(24)
    batches = [rng.permutation(128)[:32].astype(np.int32) for _ in range(25)]
    ref_sd = {k: v.detach().clone() for k, v in _model(13).state_dict().items()}

    def torch_run(autocast):
        model = _model(13).to(dev).train()
        opt = torch.optim.SGD(model.parameters(), lr=0.1, weight_decay=1e-4)
        out = []
        for rows in batches:
            mse, ce = _torch_losses(model, *_torch_batch(rec, rows, dev), autocast=autocast)
            opt.zero_grad(set_to_none=True)
            (mse + ce).backward()
            opt.step()
            out.append((float(mse.detach()), float(ce.detach())))
        return out

    traj_t, traj_a = torch_run(False), torch_run(True)
    model = _model(13)
    model.load_state_dict(ref_sd)
    tr = Trainer(eng, model, batch_size=32, optimizer="sgd")
    tr.set_records(rec)
    traj_o = [tr.step(rows) for rows in batches]
    tr.close()
    gap_a = [max(abs(a[j] - t[j]) for a, t in zip(traj_a, traj_t)) for j in (0, 1)]
    worst = 0.0
    for i, ((mt, ct), (mo, co)) in enumerate(zip(traj_t, traj_o)):
        for j, (o, t) in enumerate(((mo, mt), (co, ct))):
            bound = max(0.05, 1.25 * gap_a[j] + 0.02)
            worst = max(worst, abs(o - t) / bound)
            assert abs(o - t) <= bound, (i, j, o, t, gap_a, traj_t, traj_a, traj_o)
    print("SGD trajectory: autocast's largest gap mse %.3f ce %.3f; tightest bound used to %.2f; ce %.3f -> %.3f (torch %.3f -> %.3f)"
          % (gap_a[0], gap_a[1], worst, traj_o[0][1], traj_o[-1][1], traj_t[0][1], traj_t[-1][1]))
    assert traj_o[-1][1] < traj_o[0][1]


def test_sgd_deterministic_resumable_and_graph_free_path_identical(setup):
    """(a) two runs are bit-identical; (b) 10 steps, the state saved through torch's SGD state_dict (momentum 0.9) and resumed in a NEW
    trainer, 10 more == 20 uninterrupted steps, bit for bit; (c) captured graph and plain launches (SZB_TRAIN_NO_GRAPH=1) agree"""
    from sigma_zero_b200 import _lib
    from sigma_zero_b200.trainer import Trainer
    eng, dev = setup
    rec = _records(96, seed=25)
    rng = np.random.default_rng(26)
    batches = [rng.permutation(96)[:24].astype(np.int32) for _ in range(20)]
    kw = dict(optimizer="sgd", momentum=0.9, lr=0.02)

    def run(split=None, no_graph=False):
        m = _model(14)
        if no_graph:
            os.environ["SZB_TRAIN_NO_GRAPH"] = "1"
        try:
            tr = Trainer(eng, m, batch_size=24, **kw)
        finally:
            os.environ.pop("SZB_TRAIN_NO_GRAPH", None)
        tr.set_records(rec)
        for i, rows in enumerate(batches):
            if split is not None and i == split:
                tr.write_back(m, steps_taken=i)
                opt = torch.optim.SGD(m.parameters(), lr=0.02, momentum=0.9, weight_decay=1e-4)
                opt.load_state_dict(tr.optimiser_state(m))
                saved = opt.state_dict()
                assert len(saved["state"]) == 129
                tr.close()
                tr = Trainer(eng, m, batch_size=24, step0=i, **kw)
                tr.load_optimiser_state(saved)
                tr.set_records(rec)
            tr.step(rows, want_losses=(i % 3 == 0))
        out = tr.get_tensors(_lib.TRAIN_PARAMS)
        out.update({"buf." + k: v for k, v in tr.get_tensors(_lib.TRAIN_MOMENTUM_BUFFER).items()})
        tr.close()
        return out

    a, b, c, d = run(), run(), run(split=10), run(no_graph=True)
    for k in a:
        assert torch.equal(a[k], b[k]), "not deterministic: " + k
        assert torch.equal(a[k], c[k]), "resume differs: " + k
        assert torch.equal(a[k], d[k]), "graph and plain launches differ: " + k
    assert not torch.equal(a["conv1.weight"], _model(14).state_dict()["conv1.weight"].flatten())


def test_train_on_records_with_the_supervised_optimiser(setup):
    """train_on_records(..., make_supervised_optimiser) on a CUDA device runs the library's SGD: the written-back state loads into
    torch.optim.SGD, the scheduler counter advanced by the number of batches, and the inference network holds the trained weights"""
    from sigma_zero_b200 import runtime
    from sigma_zero_b200.engine import Engine
    from sigma_zero_b200.supervised import make_supervised_optimiser
    from sigma_zero_b200.train_RL import train_on_records
    rec = _records(64, seed=27)
    model = _model(15)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    opt, sched = make_supervised_optimiser(model)
    hist = train_on_records(model, rec, epochs=2, batch_size=16, optimiser=opt, lr_scheduler=sched, device="cuda", seed=1)
    assert len(hist) == 8 and all(np.isfinite(h).all() for h in hist)
    assert sched.last_epoch == 8 and opt.param_groups[0]["lr"] == pytest.approx(0.1) and opt.state_dict()["state"] == {}
    torch.optim.SGD(model.parameters(), lr=0.1, weight_decay=1e-4).load_state_dict(opt.state_dict())
    sd = model.state_dict()
    assert not torch.equal(sd["conv1.weight"].cpu(), before["conv1.weight"])
    assert int(sd["norm_layer.num_batches_tracked"]) == int(before["norm_layer.num_batches_tracked"]) + 8
    digest = runtime.get_engine().net_checksum()
    fresh = Engine(max_games=2, max_searches=8, device=0)
    try:
        fresh.load_state_dict(model.state_dict())
        assert fresh.net_checksum() == digest
    finally:
        fresh.close()
    # a second call continues the schedule
    train_on_records(model, rec, epochs=1, batch_size=16, optimiser=opt, lr_scheduler=sched, device="cuda", seed=2)
    assert sched.last_epoch == 12


def test_optimiser_refusals(setup):
    from sigma_zero_b200 import _lib
    from sigma_zero_b200._lib import SzbError
    from sigma_zero_b200.trainer import Trainer
    eng, dev = setup
    rec = _records(16, seed=28)
    lib, h = eng.lib, eng._h

    def code(fn):
        with pytest.raises(SzbError) as e:
            fn()
        return e.value.code

    tr = Trainer(eng, _model(16), batch_size=8)                                 # Adam
    try:
        assert code(lambda: tr.get_tensors(_lib.TRAIN_MOMENTUM_BUFFER)) == -5
        assert lib.szb_train_set_optimizer(h, 7, 0.0, 0.0, 0) == -1                  # unknown kind
        assert lib.szb_train_set_optimizer(h, _lib.TRAIN_SGD, -0.1, 0.0, 0) == -1    # negative momentum
        assert lib.szb_train_set_optimizer(h, _lib.TRAIN_SGD, 0.9, -0.5, 0) == -1    # negative dampening
        assert lib.szb_train_set_optimizer(h, _lib.TRAIN_SGD, 0.0, 0.0, 1) == -1     # nesterov without momentum
        assert lib.szb_train_set_optimizer(h, _lib.TRAIN_SGD, 0.9, 0.1, 1) == -1     # nesterov with dampening
        tr.set_records(rec)
        tr.step(np.arange(8, dtype=np.int32))
        assert lib.szb_train_set_optimizer(h, _lib.TRAIN_SGD, 0.0, 0.0, 0) == -5     # a step has run
        assert len(tr.get_tensors(_lib.TRAIN_EXP_AVG)) == 129                        # still Adam
    finally:
        tr.close()
    tr = Trainer(eng, _model(16), batch_size=8, optimizer="sgd", momentum=0.9)
    try:
        assert code(lambda: tr.get_tensors(_lib.TRAIN_EXP_AVG)) == -5
        assert code(lambda: tr.get_tensors(_lib.TRAIN_EXP_AVG_SQ)) == -5
        assert len(tr.get_tensors(_lib.TRAIN_MOMENTUM_BUFFER)) == 129
    finally:
        tr.close()
    tr = Trainer(eng, _model(16), batch_size=8, optimizer="sgd")                # momentum 0: no buffers at all
    try:
        assert code(lambda: tr.get_tensors(_lib.TRAIN_MOMENTUM_BUFFER)) == -5
    finally:
        tr.close()
    with pytest.raises(ValueError):
        Trainer(eng, _model(16), batch_size=8, optimizer="rmsprop")
    assert ctypes.sizeof(_lib.TrainConfig) == 56


def test_evaluate_records_matches_torch_eval(setup):
    """held-out losses through the inference network after training equal torch's model.eval() fp32 losses within bf16 tolerance, and
    the call changes no weight, running statistic or step counter"""
    from sigma_zero_b200 import runtime
    from sigma_zero_b200.supervised import make_supervised_optimiser
    from sigma_zero_b200.train_RL import evaluate_records, train_on_records
    eng, dev = setup
    train, held = _records(64, seed=29), _records(300, seed=30)
    model = _model(17)
    opt, sched = make_supervised_optimiser(model)
    train_on_records(model, train, epochs=1, batch_size=16, optimiser=opt, lr_scheduler=sched, device="cuda", seed=3)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    opt_sd, last_epoch = opt.state_dict(), sched.last_epoch
    mse, ce = evaluate_records(model, held)
    assert sched.last_epoch == last_epoch and opt.state_dict() == opt_sd
    for k, v in model.state_dict().items():
        assert torch.equal(v, sd[k]), k
    digest = runtime.get_engine().net_checksum()
    assert evaluate_records(model, held) == (pytest.approx(mse, rel=1e-6), pytest.approx(ce, rel=1e-6))
    assert runtime.get_engine().net_checksum() == digest
    model.eval()
    rows = np.arange(300)
    with torch.no_grad():
        x, pi, z = _torch_batch(held, rows, next(model.parameters()).device)
        mse_t, ce_t = (float(t) for t in _torch_losses(model, x, pi, z))
    print("evaluate_records: mse %.5f (torch eval fp32 %.5f, diff %.2g), ce %.5f (torch %.5f, rel diff %.2g)"
          % (mse, mse_t, abs(mse - mse_t), ce, ce_t, abs(ce - ce_t) / ce_t))
    assert abs(mse - mse_t) <= 2e-2 and abs(ce - ce_t) <= 2e-2 * ce_t
    assert not model.training


def test_supervised_main_end_to_end(tmp_path):
    """PGN text -> records -> epochs of SGD -> checkpoints; the best file is the epoch with the lowest held-out loss and loads into
    policyNN; --start_epoch resumes the scheduler; train_RL.main starts from the best file"""
    from sigma_zero_b200 import supervised, train_RL
    from sigma_zero_b200.network import policyNN
    from tests import util
    lines = []
    out = str(tmp_path / "sup")
    _, hist = supervised.main(util.PGN_SAMPLE, holdout=0.02, epochs=4, batch_size=8, out_dir=out, seed=0, log=lines.append)
    assert [h["epoch"] for h in hist] == [1, 2, 3, 4] and len(lines) == 5
    for e in range(1, 5):
        for kind in ("", "opt_", "sched_"):
            assert os.path.exists(os.path.join(out, "saves", "supervised_%s%d.pt" % (kind, e)))
    assert hist[-1]["train_ce"] < hist[0]["train_ce"], hist
    assert all(np.isfinite([h["heldout_mse"], h["heldout_ce"]]).all() for h in hist)
    best_epoch = min(hist, key=lambda h: h["heldout_mse"] + h["heldout_ce"])["epoch"]
    best = torch.load(os.path.join(out, "supervised_model_best.pt"), map_location="cpu")
    ref = torch.load(os.path.join(out, "saves", "supervised_%d.pt" % best_epoch), map_location="cpu")
    assert set(best) == set(ref) and all(torch.equal(best[k], ref[k]) for k in best)
    policyNN({}).load_state_dict(best)
    # resume epoch 5 from epoch 4's files: the StepLR counter continues
    sched4 = torch.load(os.path.join(out, "saves", "supervised_sched_4.pt"))
    _, hist5 = supervised.main(util.PGN_SAMPLE, holdout=0.02, epochs=5, batch_size=8, out_dir=out, seed=0, start_epoch=5, log=lines.append)
    sched5 = torch.load(os.path.join(out, "saves", "supervised_sched_5.pt"))
    assert [h["epoch"] for h in hist5] == [5] and sched4["last_epoch"] == 4 * hist[0]["steps"]
    assert sched5["last_epoch"] == sched4["last_epoch"] + hist5[0]["steps"]
    # the self-play loop starts from the pre-trained weights
    args = dict(num_epochs=2, num_selfPlay_iterations=2, num_searches=8, batch_size=4, chess960=False)
    _, rl = train_RL.main(args, weights=os.path.join(out, "supervised_model_best.pt"), out_dir=str(tmp_path / "rl"), max_plies=4,
                          passes_per_epoch=1, train_device="cuda", log=lambda *a: None)
    assert len(rl) == 1 and rl[0]["positions"] > 0 and all(np.isfinite(l).all() for l in rl[0]["losses"])
