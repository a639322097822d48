"""Device-side optimisation step of a value network (csrc/trainer.cu and csrc/trainer_nets.cu behind cn_trainer_*): the
`fused` mode of `Trainer` (trainer.py), for SARL and OM-SARL (with or without the global state), CADRL, and LSTM-RL
(ValueNetwork1 and 2, with or without occupancy maps).  The torch model stays the owner of the parameters -- checkpoints, `state_dict()`, the upload to the
CUDA lookahead keep working -- but its parameters become VIEWS of one flat fp32 block in state-dict order, which the two
kernels of a step (forward + backward, reduce + SGD momentum) update in place.  Reference: crowd_nav/utils/trainer.py:61-82.
"""
import ctypes as C

import torch

from . import _capi
from ._capi import check


class FusedTrainer(object):
    """The network is read off the torch model: CADRL has `value_network`, LSTM-RL has `lstm` (and `mlp1` for
    ValueNetwork2), SARL has `mlp1` / `mlp2` / `attention` / `mlp3`; occupancy maps follow from the first layer's input
    width.  CADRL trains on single-human states: its batches are (B, 13), one human per sample."""

    def __init__(self, model, device, momentum=0.9, max_batch=128, max_humans=16):
        self.lib = _capi.load()
        self.device = torch.device(device)
        self.momentum = float(momentum)
        self.lr = None
        params = list(model.parameters())
        names = [k for k, _ in model.named_parameters()]
        if names != list(model.state_dict().keys()):
            raise ValueError("the fused trainer needs a model whose parameters are its whole state dict, in order")
        n = sum(p.numel() for p in params)
        self.flat = torch.empty(n, dtype=torch.float32, device=self.device)
        off = 0
        for p in params:                       # re-home every parameter inside the flat block (same values, same names)
            k = p.numel()
            self.flat[off:off + k].copy_(p.detach().reshape(-1))
            p.data = self.flat[off:off + k].view(p.shape)
            off += k
        self.model = model
        dims = _layer_dims(model)
        self.cfg = _capi.default_sarl_cfg(**dims)
        self.single_human = dims.get("network") == _capi.NET_CADRL
        if self.single_human:
            max_humans = 1
        self.handle = C.c_void_p()
        check(self.lib.cn_trainer_create(C.byref(self.cfg), self.device.index or 0, max_batch, max_humans, C.byref(self.handle)))
        if int(self.lib.cn_trainer_param_count(self.handle)) != n:
            raise ValueError("value-network layout does not match the fused trainer's (%d parameters vs %d)" % (
                n, int(self.lib.cn_trainer_param_count(self.handle))))
        self.grad = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.loss = torch.zeros((), dtype=torch.float32, device=self.device)
        self._synced = False
        self.max_batch, self.max_humans = max_batch, max_humans

    def close(self):
        if getattr(self, "handle", None):
            self.lib.cn_trainer_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def sync_from_model(self, zero_momentum=False):
        """The parameters were written by someone else (load_state_dict, broadcast, another optimiser)."""
        check(self.lib.cn_trainer_sync_weights(self.handle, C.c_void_p(self.flat.data_ptr()), int(zero_momentum), self._stream()))
        self._synced = True

    def flush_to_model(self):
        """Nothing to copy -- the parameters ARE the flat block; the next optimize_* call re-syncs the transposed copy in
        case the model is modified in between."""
        self._synced = False

    def step(self, inputs, values, dist_group=None):
        """One SGD-momentum step on (inputs (B, H, D), or (B, D) for CADRL, values (B, 1)); returns the batch MSE as a 0-d
        device tensor."""
        if self.lr is None:
            raise ValueError("Learning rate is not set!")
        if not self._synced:
            self.sync_from_model()
        inputs = inputs.contiguous().float()
        values = values.contiguous().float().reshape(-1)
        B, H = inputs.shape[0], self._humans(inputs)
        loss = torch.empty((), dtype=torch.float32, device=self.device)
        if dist_group is None:
            check(self.lib.cn_trainer_step(self.handle, C.c_void_p(self.flat.data_ptr()), C.c_void_p(inputs.data_ptr()),
                                           C.c_void_p(values.data_ptr()), B, H, self.lr, self.momentum, None,
                                           C.c_void_p(loss.data_ptr()), self._stream()))
            return loss
        import torch.distributed as dist
        check(self.lib.cn_trainer_step(self.handle, C.c_void_p(self.flat.data_ptr()), C.c_void_p(inputs.data_ptr()),
                                       C.c_void_p(values.data_ptr()), B, H, self.lr, self.momentum,
                                       C.c_void_p(self.grad.data_ptr()), C.c_void_p(loss.data_ptr()), self._stream()))
        dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=dist_group)        # one 386 kB bucket over NVLink
        check(self.lib.cn_trainer_apply(self.handle, C.c_void_p(self.flat.data_ptr()), C.c_void_p(self.grad.data_ptr()),
                                        1.0 / dist.get_world_size(dist_group), self.lr, self.momentum, self._stream()))
        return loss


    def step_indexed(self, states, values, idx, loss_sum, dist_group=None):
        """One SGD-momentum step on the batch memory[idx], gathered inside the kernel: states (capacity, H, D) fp32 and
        values (capacity, 1) fp32 are the replay tensors themselves (CADRL: states (capacity, D)), idx an int64 device vector; the batch MSE is ADDED to
        the 0-d device tensor loss_sum.  One C call, two kernels (+ the all-reduce and the apply kernel under dist_group)."""
        if self.lr is None:
            raise ValueError("Learning rate is not set!")
        if not self._synced:
            self.sync_from_model()
        B, H = int(idx.shape[0]), self._humans(states)
        grad = None if dist_group is None else C.c_void_p(self.grad.data_ptr())
        check(self.lib.cn_trainer_step_indexed(self.handle, C.c_void_p(self.flat.data_ptr()), C.c_void_p(states.data_ptr()),
                                               C.c_void_p(values.data_ptr()), C.c_void_p(idx.data_ptr()), B, H, self.lr,
                                               self.momentum, grad, C.c_void_p(loss_sum.data_ptr()), self._stream()))
        if dist_group is not None:
            import torch.distributed as dist
            dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=dist_group)
            check(self.lib.cn_trainer_apply(self.handle, C.c_void_p(self.flat.data_ptr()), C.c_void_p(self.grad.data_ptr()),
                                            1.0 / dist.get_world_size(dist_group), self.lr, self.momentum, self._stream()))


    def _humans(self, states):
        """Humans per sample of a batch or replay tensor: its second axis, or 1 for CADRL's (N, D) rows."""
        if self.single_human:
            if states.dim() != 2:
                raise ValueError("CADRL trains on single-human states: expected (N, %d), got %s" % (
                    self.cfg.input_dim, tuple(states.shape)))
            return 1
        return int(states.shape[1])


class FusedSarlTrainer(FusedTrainer):
    """The SARL trainer under its original name (FusedTrainer covers every value network)."""


def _widths(seq):
    return [m.out_features for m in seq if isinstance(m, torch.nn.Linear)]


def _om_kwargs(input_dim):
    """cn_sarl_cfg occupancy-map fields for a first layer reading `input_dim` columns: 13 + cell_num^2 * om_channel_size
    (multi_human_rl.py:106-107) with maps; {} for 13 columns, or any width that is no map layout."""
    om = input_dim - 13
    for ch in (3, 2, 1):
        cells = int(round((om / ch) ** 0.5)) if om > 0 and om % ch == 0 else 0
        if 1 <= cells <= 8 and cells * cells * ch == om:
            return dict(with_om=1, cell_num=cells, om_channel_size=ch)
    return {}


def _layer_dims(model):
    """cn_sarl_cfg of the torch value network: CADRL (policy.make_cadrl_network), LSTM-RL (make_lstm_network) or SARL
    (make_value_network), with the layer widths of its Linear layers."""
    if hasattr(model, "value_network"):
        first = [m for m in model.value_network if isinstance(m, torch.nn.Linear)][0]
        return dict(network=_capi.NET_CADRL, input_dim=first.in_features, mlp3_dims=_widths(model.value_network))
    if hasattr(model, "lstm"):
        mlp1 = getattr(model, "mlp1", None)
        first = [m for m in mlp1 if isinstance(m, torch.nn.Linear)][0] if mlp1 is not None else None
        input_dim = first.in_features if first is not None else model.lstm.input_size
        return dict(network=_capi.NET_LSTM_RL, input_dim=input_dim, self_state_dim=model.self_state_dim,
                    mlp3_dims=_widths(model.mlp), lstm_hidden=model.lstm.hidden_size,
                    lstm_mlp1_dims=_widths(mlp1) if mlp1 is not None else [0, 0, 0, 0], **_om_kwargs(input_dim))
    first = [m for m in model.mlp1 if isinstance(m, torch.nn.Linear)][0]
    return dict(input_dim=first.in_features, self_state_dim=model.self_state_dim, mlp1_dims=_widths(model.mlp1),
                mlp2_dims=_widths(model.mlp2), attn_dims=_widths(model.attention), mlp3_dims=_widths(model.mlp3),
                without_global_state=int(not model.with_global_state), **_om_kwargs(first.in_features))
