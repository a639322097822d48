"""Training the learned human-motion models (world_model.AttentionWorld / MlpWorld) on the device.

The fork's model-based loop trains a world model on transitions of the ORCA simulator and then lets `ModelCrowdSim` move
the humans with it.  Here both halves run on the GPU:

- `collect_world_transitions` runs a BatchedCrowdSim with ORCA humans and records, per step and env, every human's state
  before the step and the velocity ORCA gave it (cn_env_copy_world_pairs), with no host read per step.
- `WorldTrainer` takes optimisation steps -- MSELoss, backward, torch.optim.Adam -- as two CUDA kernels on one flat fp32
  parameter block (cn_world_trainer_*, csrc/world_trainer.cu).  The container's parameters become views of that block, so
  `state_dict()`, `torch.save` and loading into a fresh container keep working, and after every call the model's
  `cn_world` handle is refreshed from the block on the device: `predict_into`, `ModelCrowdSim` and `Explorer` use the
  trained weights with no copy through the host.
"""
import ctypes as C

import torch

from . import _capi
from ._capi import check


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class EarlyStopping(object):
    """The rule of the public `pytorchtools.EarlyStopping`: a validation loss `val <= best - delta` is an improvement
    (the caller keeps the weights and the counter restarts); otherwise the counter grows and training stops when it reaches
    `patience`.  The first loss is always an improvement."""

    def __init__(self, patience, delta=0.0):
        self.patience, self.delta = int(patience), float(delta)
        self.best, self.counter = None, 0

    def update(self, val):
        """-> (improved, stop)"""
        if self.best is None or val <= self.best - self.delta:
            self.best, self.counter = val, 0
            return True, False
        self.counter += 1
        return False, self.counter >= self.patience


class WorldTrainer(object):
    """Adam on an AttentionWorld or MlpWorld container.  MlpWorld trains with its Dropout layers on (p = world.drop_rate;
    the masks are Philox draws keyed by `seed` and the step count); AttentionWorld has none.  `max_humans` bounds the humans
    per sample of an AttentionWorld's data (MlpWorld is built for world.num_human)."""

    def __init__(self, world, device, lr, betas=(0.9, 0.999), eps=1e-8, max_batch=4096, seed=0, max_humans=16):
        self.lib = _capi.load()
        self.device = torch.device(device)
        self.index = self.device.index or 0
        self.world = world
        self.lr, self.betas, self.eps, self.seed = float(lr), (float(betas[0]), float(betas[1])), float(eps), int(seed)
        params = list(world.parameters())
        if [k for k, _ in world.named_parameters()] != list(world.state_dict().keys()):
            raise ValueError("the world trainer needs a model whose parameters are its whole state dict, in order")
        n = sum(p.numel() for p in params)
        self.flat = torch.empty(n, dtype=torch.float32, device=self.device)
        off = 0
        for p in params:                       # re-home every parameter inside the flat block (same values, same names)
            k = p.numel()
            self.flat[off:off + k].copy_(p.detach().reshape(-1))
            p.data = self.flat[off:off + k].view(p.shape)
            off += k
        self.mlp = world.kind == _capi.WORLD_MLP
        humans = world.num_human if self.mlp else max_humans
        drop = float(getattr(world, "drop_rate", 0.0)) if self.mlp else 0.0
        self.handle = C.c_void_p()
        check(self.lib.cn_world_trainer_create(world.kind, humans, self.index, int(max_batch), drop, C.byref(self.handle)))
        if int(self.lib.cn_world_trainer_param_count(self.handle)) != n:
            raise ValueError("world-model layout does not match the trainer's (%d parameters vs %d)" % (
                n, int(self.lib.cn_world_trainer_param_count(self.handle))))
        self.max_batch = int(max_batch)
        self.grad = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._synced = None
        self.sync(reset_optimizer=True)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.cn_world_trainer_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _stamp(self):
        return tuple((p.data_ptr(), p._version) for p in self.world.parameters())

    def sync(self, reset_optimizer=False):
        """The parameters were written by someone else (load_state_dict, a broadcast); reset_optimizer also zeroes Adam's
        moments and step count."""
        check(self.lib.cn_world_trainer_sync_weights(self.handle, _ptr(self.flat), int(bool(reset_optimizer)), self._stream()))
        self._synced = self._stamp()

    def _publish(self):
        """Point the model's cn_world handle at the trained block (device to device).  The kernels update the block in
        place, which bumps no parameter version, so the handle's own upload stamp is set here."""
        h = self.world.handle(self.index)
        check(self.lib.cn_world_load_weights_device(h, _ptr(self.flat), self.flat.numel(), self._stream()))
        self.world._uploaded = (self.index, self._stamp())

    def _data(self, x, y):
        x = x.to(self.device, torch.float32).contiguous()
        y = y.to(self.device, torch.float32).contiguous()
        B = x.shape[0]
        x, y = x.reshape(B, -1, 4), y.reshape(B, -1, 2)
        if x.shape[1] != y.shape[1]:
            raise ValueError("states (%s) and velocities (%s) disagree on the human count" % (tuple(x.shape), tuple(y.shape)))
        return x, y

    def _step(self, x, y, index, batch, loss_sum, grad=None, mask=None):
        if self._synced != self._stamp():
            self.sync()
        check(self.lib.cn_world_trainer_step(self.handle, _ptr(self.flat), _ptr(x), _ptr(y), _ptr(index), int(batch),
                                             int(x.shape[1]), self.lr, self.betas[0], self.betas[1], self.eps, self.seed,
                                             _ptr(grad), _ptr(loss_sum), _ptr(mask), self._stream()))

    def step(self, x, y, index=None):
        """One Adam step on x (B, H, 4) -> y (B, H, 2) (or the samples index (int64 device vector) of x / y); returns the
        batch MSE as a 0-d device tensor."""
        x, y = self._data(x, y)
        batch = x.shape[0] if index is None else int(index.shape[0])
        loss = torch.zeros((), dtype=torch.float32, device=self.device)
        self._step(x, y, index, batch, loss)
        self._publish()
        return loss

    def gradient(self, x, y, index=None, mask=None):
        """The gradient of the batch MSE alone (into self.grad, no update): the data-parallel form, followed by an
        all-reduce and apply().  mask (optional, MlpWorld): uint8 device tensor (B, 192) <- the dropout masks drawn."""
        x, y = self._data(x, y)
        batch = x.shape[0] if index is None else int(index.shape[0])
        loss = torch.zeros((), dtype=torch.float32, device=self.device)
        self._step(x, y, index, batch, loss, grad=self.grad, mask=mask)
        return loss

    def apply(self, grad=None, scale=1.0):
        """Adam with a gradient computed elsewhere (default self.grad) times `scale`."""
        if self._synced != self._stamp():
            self.sync()
        g = self.grad if grad is None else grad
        check(self.lib.cn_world_trainer_apply(self.handle, _ptr(self.flat), _ptr(g), float(scale), self.lr, self.betas[0],
                                              self.betas[1], self.eps, self._stream()))
        self._publish()

    def _validate(self, X, Y):
        """MSE of the model (dropout off) over all of X / Y, as a 0-d device tensor."""
        out = torch.zeros((), dtype=torch.float32, device=self.device)
        check(self.lib.cn_world_trainer_eval(self.handle, _ptr(X), _ptr(Y), None, int(X.shape[0]), int(X.shape[1]),
                                             _ptr(out), self._stream()))
        return out

    def evaluate(self, X, Y):
        if self._synced != self._stamp():
            self.sync()
        X, Y = self._data(X, Y)
        return self._validate(X, Y)

    def optimize_epoch(self, X, Y, batch_size, num_epochs, val=None, patience=None, delta=0.0, generator=None):
        """Epochs of shuffled mini-batches (one torch.randperm per epoch, the last partial batch kept, as a DataLoader with
        shuffle=True): every batch is one indexed step, gathered inside the kernel.  Returns one dict per epoch run:
        {"train": mean of the batch MSEs, "val": validation MSE (dropout off) or None}, read back once per epoch.  With
        `patience` (needs `val`), early stopping by the EarlyStopping rule; the weights of the best validation loss are
        restored at the end."""
        if batch_size < 1 or batch_size > self.max_batch:
            raise ValueError("batch_size %d outside 1..max_batch (%d)" % (batch_size, self.max_batch))
        if patience is not None and val is None:
            raise ValueError("early stopping needs validation data")
        X, Y = self._data(X, Y)
        if val is not None:
            Xv, Yv = self._data(*val)
        N = X.shape[0]
        stopper = EarlyStopping(patience, delta) if patience is not None else None
        best = None
        history = []
        for _ in range(int(num_epochs)):
            perm = torch.randperm(N, generator=generator).to(self.device)
            train = torch.zeros((), dtype=torch.float32, device=self.device)
            nb = (N + batch_size - 1) // batch_size
            for b in range(nb):
                idx = perm[b * batch_size:(b + 1) * batch_size]
                self._step(X, Y, idx, idx.shape[0], train)
            v = self._validate(Xv, Yv) if val is not None else torch.zeros((), device=self.device)
            got = torch.stack([train, v]).cpu()
            history.append({"train": float(got[0]) / nb, "val": float(got[1]) if val is not None else None})
            if stopper is not None:
                improved, stop = stopper.update(history[-1]["val"])
                if improved:
                    best = self.flat.clone()
                if stop:
                    break
        if best is not None:
            self.flat.copy_(best)
            self.sync()
        self._publish()
        return history


def collect_world_transitions(batch, max_steps=None, robot="orca", safety_space=0.0, query_env=False, epsilon=0.0):
    """Roll the envs of `batch` (a BatchedCrowdSim with ORCA humans) forward and record the world-model training pairs of
    every step: X (N, H, 4) fp32 human states (px, py, vx, vy) before the step, Y (N, H, 2) fp32 the velocities ORCA gave
    them in that step, env (N,) int64 the env of each pair -- compacted device tensors over the envs still running (with
    auto_reset off, each env runs one episode and then freezes).  Per step: ORCA -> copy pairs -> robot action ->
    step(update), enqueued with no host read.  robot: a BatchedSARL (its lookahead, query_env / epsilon as in
    cn_policy_lookahead), "orca" (the robot's own ORCA with safety_space) or "keep" (the pending action).  max_steps
    defaults to the episode time limit in steps."""
    lib = batch.lib
    E, H = batch.E, batch.H
    if max_steps is None:
        max_steps = int(round(batch.cfg.time_limit / batch.cfg.time_step)) + 1
    if not (robot in ("orca", "keep") or hasattr(robot, "lookahead")):
        raise ValueError("robot must be a BatchedSARL, 'orca' or 'keep'")
    dev = torch.device("cuda", batch.device)
    X = torch.empty((max_steps, E, H, 4), dtype=torch.float32, device=dev)
    Y = torch.empty((max_steps, E, H, 2), dtype=torch.float32, device=dev)
    V = torch.zeros((max_steps, E), dtype=torch.uint8, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    for t in range(max_steps):
        check(lib.cn_env_orca(batch.handle, stream))
        check(lib.cn_env_copy_world_pairs(batch.handle, _ptr(X[t]), _ptr(Y[t]), _ptr(V[t]), stream))
        if robot == "orca":
            check(lib.cn_env_robot_orca(batch.handle, float(safety_space), stream))
        elif robot != "keep":
            check(robot.lib.cn_policy_lookahead(robot.handle, batch.handle, int(bool(query_env)), float(epsilon), stream))
        check(lib.cn_env_step(batch.handle, None, 1, stream))
    keep = V.bool()
    env = keep.nonzero()[:, 1]
    return X[keep], Y[keep], env
