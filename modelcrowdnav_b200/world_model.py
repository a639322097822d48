"""Learned human-motion models of the fork (crowd_nav/policy/world_model.py:20-106) on the device.

`MlpWorld` / `AttentionWorld` here are PARAMETER CONTAINERS -- torch modules whose state-dict keys and shapes are the
reference's (mlp.0 / mlp.3 / mlp.6 / mlp.8; mlp1.* mlp2.* attention.* mlp3.*), so its checkpoints load unchanged and
`env.sim_world = model` keeps working -- while the prediction itself is `cn_world_predict` (csrc/world_model.cu): it reads the
humans' states from the env batch on the device and leaves every human's next velocity where the env step expects the ORCA
result.  `ModelCrowdSim` (envs.py) calls it instead of solving ORCA; no state or velocity crosses PCIe.

There is no CPU / eager forward: `forward(x)` runs the same CUDA kernel on a throw-away env batch holding `x`.
SGANWorld (world_model.py:108-268) wraps the third-party Social-GAN generator and its trajectory datasets; it is outside
the hot path and not provided.
"""
import ctypes as C

import numpy as np
import torch
from torch import nn

from . import _capi
from ._capi import check


def _linear_stack(dims, slots):
    """nn.Sequential whose Linear layers sit at the given indices (what fixes the state-dict keys `<i>.weight`); the slots
    in between hold Identity placeholders for the reference's activation / dropout modules, which carry no state."""
    mods = [nn.Identity() for _ in range(max(slots) + 1)]
    for (i, o), k in zip(zip(dims[:-1], dims[1:]), slots):
        mods[k] = nn.Linear(i, o)
    return nn.Sequential(*mods)


class _DeviceWorld(nn.Module):
    kind = None

    def _init_device_state(self):
        self._handle = None
        self._uploaded = None          # (device ordinal, parameter version stamp) of the weights the handle holds
        self.mse = 0
        self.device = None

    def flat_weights(self):
        return np.concatenate([v.detach().cpu().numpy().astype(np.float32).ravel() for v in self.state_dict().values()])

    def handle(self, device_index=0):
        """cn_world handle holding the CURRENT parameters (re-uploaded when a parameter was modified in place or replaced)."""
        lib = _capi.load()
        stamp = (device_index, tuple((p.data_ptr(), p._version) for p in self.parameters()))
        if self._handle is None or self._uploaded is None or self._uploaded[0] != device_index:
            if self._handle is not None:
                lib.cn_world_destroy(self._handle)
            self._handle = C.c_void_p()
            check(lib.cn_world_create(self.kind, int(getattr(self, "num_human", 0)), device_index, C.byref(self._handle)))
            self._uploaded = None
        if self._uploaded != stamp:
            w = np.ascontiguousarray(self.flat_weights())
            check(lib.cn_world_load_weights(self._handle, w.ctypes.data_as(C.c_void_p), w.size, None))
            self._uploaded = stamp
        return self._handle

    def predict_into(self, batch):
        """Next human velocities for every env of a BatchedCrowdSim, left on the device in place of the ORCA result."""
        check(_capi.load().cn_world_predict(self.handle(batch.device), batch.handle, None))

    def forward(self, x):
        """(B, H * 4) or (B, H, 4) human states (px, py, vx, vy) -> (B, H * 2) velocities, through the CUDA kernel."""
        from .batch import BatchedCrowdSim
        if not x.is_cuda:
            raise RuntimeError("world models run on the GPU only (cn_world_predict); there is no CPU fallback")
        B = x.shape[0]
        xs = x.detach().reshape(B, -1, 4).double().cpu().numpy()
        H = xs.shape[1]
        agents = np.zeros((B, H + 1, _capi.AGENT_STRIDE))
        agents[:, 1:, :4] = xs
        agents[:, :, 6] = 0.3; agents[:, :, 7] = 1.0
        env = BatchedCrowdSim(B, H, device=x.device.index or 0)
        try:
            env.set_state(agents)
            self.predict_into(env)
            v = env.human_actions()
        finally:
            env.close()
        return torch.from_numpy(v.reshape(B, H * 2)).to(device=x.device, dtype=torch.float32)

    def __del__(self):
        try:
            if self._handle is not None:
                _capi.load().cn_world_destroy(self._handle)
        except Exception:
            pass


class MlpWorld(_DeviceWorld):
    """world_model.py:20-50: (B, num_human * 4) -> (B, num_human * 2), tanh-bounded velocities (dropout = identity in eval)."""
    kind = _capi.WORLD_MLP

    def __init__(self, num_human, drop_rate=0.5, multihuman=True):
        super().__init__()
        self.num_human = num_human if multihuman else 1
        self.drop_rate = drop_rate          # the Dropout layers' p in training mode (world_trainer.WorldTrainer)
        self.mlp = _linear_stack([self.num_human * 4, 128, 64, 12, self.num_human * 2], [0, 3, 6, 8])
        self._init_device_state()


class AttentionWorld(_DeviceWorld):
    """world_model.py:53-106: the SARL block structure on (px, py, vx, vy) rows, one (vx, vy) per human."""
    kind = _capi.WORLD_ATTENTION

    def __init__(self, input_dim=4, with_global_state=True):
        super().__init__()
        if input_dim != 4 or not with_global_state:
            raise NotImplementedError("the device AttentionWorld is the default configuration (input_dim 4, global state)")
        self.input_dim = input_dim
        self.with_global_state = with_global_state
        self.mlp1 = _linear_stack([4, 150, 100], [0, 2])
        self.mlp2 = _linear_stack([100, 100, 50], [0, 2])
        self.attention = _linear_stack([200, 100, 100, 1], [0, 2, 4])
        self.mlp3 = _linear_stack([54, 150, 100, 100, 2], [0, 2, 4, 6])
        self._init_device_state()


class SGANWorld(object):
    def __init__(self, *a, **kw):
        raise NotImplementedError("SGANWorld wraps the third-party Social-GAN generator (outside the B200 hot path)")
