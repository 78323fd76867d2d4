"""The fine-tuning half of the self-play loop on the GPU library (train_RL.py:77-154): host-side mirror of szb_train_*.

    loss = mse_loss(v, z) + cross_entropy(logits, pi)    (train_RL.py:103-113)
    Adam(lr 1e-4, weight_decay 1e-4) (:187), StepLR(500, 0.95) stepped per batch (:199, :123-124)
    or, optimizer="sgd", the supervised recipe: SGD(lr 0.1, weight_decay 1e-4), StepLR(4000, 0.5) (train_supervised.py:84-92)

`Trainer` owns the library's training state for one model: fp32 master weights, Adam moments or SGD momentum buffers, BatchNorm
buffers.  Records (records.pack_records) are copied to the GPU once; a step sends only the row numbers of its batch.  After training,
`write_back(model)` puts the weights (and running statistics) back into the torch module and `optimiser_state(...)` produces a
torch.optim.Adam or torch.optim.SGD state_dict, so checkpoints stay interchangeable with the torch trainer's.  There is no CPU path:
without libszb200.so or a GPU the constructor raises."""
import ctypes

import numpy as np

from . import _lib

ADAM_DEFAULTS = dict(lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-4, lr_step=500, lr_gamma=0.95)
SGD_DEFAULTS = dict(lr=0.1, weight_decay=1e-4, lr_step=4000, lr_gamma=0.5)          # supervised.make_supervised_optimiser


def _names(keys):
    return (ctypes.c_char_p * len(keys))(*[k.encode() for k in keys])


class Trainer:
    def __init__(self, engine, model, batch_size=128, step0=0, bn_momentum=0.1, bn_eps=1e-5, _probe=(0, 0), optimizer="adam", momentum=0.0,
                 dampening=0.0, nesterov=False, **hp):
        """optimizer "adam" (hp: lr, beta1, beta2, eps, weight_decay, lr_step, lr_gamma; ADAM_DEFAULTS) or "sgd" (hp: lr, weight_decay,
        lr_step, lr_gamma; SGD_DEFAULTS) with torch.optim.SGD's momentum, dampening and nesterov"""
        import torch
        if optimizer not in ("adam", "sgd"):
            raise ValueError("optimizer must be 'adam' or 'sgd', not %r" % (optimizer,))
        self.engine, self.lib, self.batch_size = engine, engine.lib, int(batch_size)
        self.optimizer = optimizer
        full = dict(ADAM_DEFAULTS)
        if optimizer == "sgd":
            unknown = set(hp) - set(SGD_DEFAULTS)
            if unknown:
                raise TypeError("SGD has no hyper-parameter %s" % ", ".join(sorted(unknown)))
            full.update(SGD_DEFAULTS)
        full.update(hp)
        hp = full
        self.hp = hp
        self.momentum, self.dampening, self.nesterov = float(momentum), float(dampening), bool(nesterov)
        self._have_buffers = False                   # SGD with momentum: torch's "momentum_buffer" state exists (after a step or a load)
        cfg = _lib.TrainConfig(self.batch_size, hp["lr"], hp["beta1"], hp["beta2"], hp["eps"], hp["weight_decay"], hp["lr_step"], hp["lr_gamma"],
                               bn_momentum, bn_eps, int(step0), int(_probe[0]), int(_probe[1]))
        engine._check(self.lib.szb_train_create(engine._h, ctypes.byref(cfg)))
        if optimizer == "sgd":
            engine._check(self.lib.szb_train_set_optimizer(engine._h, _lib.TRAIN_SGD, self.momentum, self.dampening, int(self.nesterov)))
        sd = model.state_dict()
        self.keys = [k for k in sd if not k.endswith("num_batches_tracked")]
        self.param_keys = [k for k, _ in model.named_parameters()]
        self.numels = [int(sd[k].numel()) for k in self.keys]
        self.device = torch.device("cuda", engine.device)
        self.n_records = 0
        self.steps_run = 0
        self.set_tensors(_lib.TRAIN_PARAMS, {k: sd[k] for k in self.keys})

    def close(self):
        if self.engine is not None and self.engine._h:
            self.lib.szb_train_destroy(self.engine._h)
        self.engine = None

    # ---- named tensors -----------------------------------------------------------------------
    def _call(self, fn, kind, keys, tensors):
        n = len(keys)
        data = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors])
        numel = (ctypes.c_int64 * n)(*[int(t.numel()) for t in tensors])
        self.engine._check(fn(self.engine._h, kind, n, ctypes.cast(_names(keys), ctypes.c_void_p), ctypes.cast(data, ctypes.c_void_p),
                              ctypes.cast(numel, ctypes.c_void_p)))

    def set_tensors(self, kind, tensors):
        import torch
        keys = list(tensors)
        vals = [tensors[k].detach().to(dtype=torch.float32).contiguous() for k in keys]
        if any(v.is_cuda for v in vals):
            torch.cuda.synchronize()
        self._call(self.lib.szb_train_set, kind, keys, vals)

    def get_tensors(self, kind, keys=None, shapes=None, device="cpu"):
        """{name: fp32 tensor} of the parameters (+ running buffers), gradients or Adam moments, in torch layout"""
        import torch
        if keys is None:
            keys = self.keys if kind == _lib.TRAIN_PARAMS else self.param_keys
        numel = dict(zip(self.keys, self.numels))
        out = [torch.empty(int(np.prod(shapes[k])) if shapes and k in shapes else numel[k], dtype=torch.float32, device=device) for k in keys]
        self._call(self.lib.szb_train_get, kind, keys, out)
        return dict(zip(keys, out))

    def activations(self, n):
        """(logits [n, 4672], value [n]) of the last step"""
        import torch
        lg, v = torch.empty(n * 4672, dtype=torch.float32), torch.empty(n, dtype=torch.float32)
        self._call(self.lib.szb_train_get, _lib.TRAIN_ACTIVATIONS, ["logits", "value"], [lg, v])
        return lg.view(n, 4672), v

    @property
    def step_count(self):
        s = ctypes.c_int64(0)
        self.engine._check(self.lib.szb_train_state(self.engine._h, ctypes.byref(s), 0))
        return s.value

    @step_count.setter
    def step_count(self, value):
        s = ctypes.c_int64(int(value))
        self.engine._check(self.lib.szb_train_state(self.engine._h, ctypes.byref(s), 1))

    # ---- data + steps ------------------------------------------------------------------------
    def set_records(self, rec):
        states = np.ascontiguousarray(rec["states"], dtype=np.uint64).reshape(-1, 119)
        off = np.ascontiguousarray(rec["pi_off"], dtype=np.int64)
        idx = np.ascontiguousarray(rec["pi_index"], dtype=np.uint16)
        prob = np.ascontiguousarray(rec["pi_prob"], dtype=np.float32)
        z = np.ascontiguousarray(rec["z"], dtype=np.int8)
        assert len(off) == len(states) + 1 == len(z) + 1 and off[0] == 0 and off[-1] == len(idx) == len(prob)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        self.engine._check(self.lib.szb_train_records(self.engine._h, len(states), p(states), p(off), p(idx), p(prob), p(z)))
        self.n_records = len(states)

    def step(self, rows, flags=0, want_losses=True):
        """one optimiser step on the records `rows`; returns (mse, ce) of the batch before the update"""
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        losses = (ctypes.c_float * 2)()
        self.engine._check(self.lib.szb_train_step(self.engine._h, len(rows), rows.ctypes.data_as(ctypes.c_void_p), int(flags),
                                                   ctypes.cast(losses, ctypes.c_void_p) if want_losses else None))
        self.steps_run += 1
        self._have_buffers = self._have_buffers or not (flags & (_lib.TRAIN_NO_UPDATE | _lib.TRAIN_FORWARD_ONLY))
        return (float(losses[0]), float(losses[1])) if want_losses else None

    def loss_history(self, first=0, count=None):
        """[(mse, ce)] of steps [first, first + count) since the trainer was created (the library keeps the last 65,536): lets a loop
        queue its steps with want_losses=False -- no host round trip per step -- and collect the losses in bulk"""
        count = self.steps_run - first if count is None else count
        out = np.empty((count, 2), dtype=np.float32)
        self.engine._check(self.lib.szb_train_loss_history(self.engine._h, int(first), int(count), out.ctypes.data_as(ctypes.c_void_p)))
        return [(float(a), float(b)) for a, b in out]

    # ---- back to torch -----------------------------------------------------------------------
    def flat_weights(self):
        """(keys, numels, ONE flat fp32 CUDA tensor) in the model's state_dict order: the buffer train_RL.broadcast_weights sends
        over NCCL and Engine.load_flat_device folds into the inference network, with no host round trip"""
        import torch
        flat = torch.empty(int(sum(self.numels)), dtype=torch.float32, device=self.device)
        offs = np.concatenate([[0], np.cumsum(self.numels)])
        views = [flat[int(offs[i]):int(offs[i + 1])] for i in range(len(self.keys))]
        torch.cuda.synchronize(self.device)
        self._call(self.lib.szb_train_get, _lib.TRAIN_PARAMS, self.keys, views)
        return self.keys, self.numels, flat

    def write_back(self, model, steps_taken=0):
        """trained weights and BatchNorm running statistics -> the torch module (state_dict layout, dtype and device kept)"""
        import torch
        keys, numels, flat = self.flat_weights()
        sd = model.state_dict()
        off = 0
        with torch.no_grad():
            for k, n in zip(keys, numels):
                sd[k].copy_(flat[off:off + n].view(sd[k].shape).to(sd[k].device))
                off += n
            for k, v in sd.items():
                if k.endswith("num_batches_tracked"):
                    v += int(steps_taken)
        return flat

    def optimiser_state(self, model):
        """a torch.optim.Adam state_dict (per-parameter step / exp_avg / exp_avg_sq, one param group) of the trainer's state, or under
        SGD a torch.optim.SGD one (per-parameter momentum_buffer when momentum is not 0 and the buffers exist, else an empty state)"""
        import torch
        shapes = {k: tuple(p.shape) for k, p in model.named_parameters()}
        if self.optimizer == "sgd":
            return self._sgd_state(shapes)
        m = self.get_tensors(_lib.TRAIN_EXP_AVG)
        v = self.get_tensors(_lib.TRAIN_EXP_AVG_SQ)
        step, hp = self.step_count, self.hp
        state = {i: {"step": torch.tensor(float(step)), "exp_avg": m[k].view(shapes[k]), "exp_avg_sq": v[k].view(shapes[k])}
                 for i, k in enumerate(self.param_keys)}
        lr = hp["lr"] * hp["lr_gamma"] ** (step // hp["lr_step"])
        group = {"lr": lr, "betas": (hp["beta1"], hp["beta2"]), "eps": hp["eps"], "weight_decay": hp["weight_decay"], "amsgrad": False,
                 "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None, "initial_lr": hp["lr"],
                 "params": list(range(len(self.param_keys)))}
        return {"state": state, "param_groups": [group]}

    def _sgd_state(self, shapes):
        hp, state = self.hp, {}
        if self.momentum != 0 and self._have_buffers:
            buf = self.get_tensors(_lib.TRAIN_MOMENTUM_BUFFER)
            state = {i: {"momentum_buffer": buf[k].view(shapes[k])} for i, k in enumerate(self.param_keys)}
        lr = hp["lr"] * hp["lr_gamma"] ** (self.step_count // hp["lr_step"])
        group = {"lr": lr, "momentum": self.momentum, "dampening": self.dampening, "weight_decay": hp["weight_decay"], "nesterov": self.nesterov,
                 "maximize": False, "foreach": None, "differentiable": False, "fused": None, "initial_lr": hp["lr"],
                 "params": list(range(len(self.param_keys)))}
        return {"state": state, "param_groups": [group]}

    def load_optimiser_state(self, opt_state):
        """continue from a torch.optim.Adam state_dict (moments and step counter) or, under SGD, a torch.optim.SGD one (momentum
        buffers; SGD keeps no step counter, the learning rate follows step0 / step_count)"""
        st = opt_state.get("state", {})
        if not st:
            return
        if self.optimizer == "sgd":
            buf = {k: st[i]["momentum_buffer"] for i, k in enumerate(self.param_keys) if st.get(i, {}).get("momentum_buffer") is not None}
            if buf and self.momentum != 0:
                if len(buf) != len(self.param_keys):
                    raise ValueError("the SGD state has momentum buffers for %d of %d parameters" % (len(buf), len(self.param_keys)))
                self.set_tensors(_lib.TRAIN_MOMENTUM_BUFFER, buf)
                self._have_buffers = True
            return
        m = {k: st[i]["exp_avg"] for i, k in enumerate(self.param_keys) if i in st}
        v = {k: st[i]["exp_avg_sq"] for i, k in enumerate(self.param_keys) if i in st}
        self.set_tensors(_lib.TRAIN_EXP_AVG, m)
        self.set_tensors(_lib.TRAIN_EXP_AVG_SQ, v)
        self.step_count = int(float(next(iter(st.values()))["step"]))
