"""Fused trainer (cn_trainer_*, csrc/trainer.cu + csrc/trainer_nets.cu) for the value networks other than plain SARL:
OM-SARL, CADRL, and LSTM-RL ValueNetwork1 / 2 with and without occupancy maps.

Ground truth is torch autograd on the torch modules of policy.py (the reference's networks).  The LSTM references run with
cuDNN's TF32 off (fixture `no_tf32`), so they are FP32 like the kernels."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

M1, M2, M3, ATT, LM1 = [150, 100], [100, 50], [150, 100, 100, 1], [100, 100, 1], [150, 100, 100, 50]


def _make(name):
    from modelcrowdnav_b200.policy import make_cadrl_network, make_lstm_network, make_value_network
    if name == "om_sarl":
        return make_value_network(61, 6, M1, M2, M3, ATT)
    if name == "cadrl":
        return make_cadrl_network(13, M3)
    om = name.startswith("om_")
    return make_lstm_network(61 if om else 13, 6, LM1 if name.endswith("vn2") else None, M3, 50)


# network -> parameter count at the default shapes (None: not part of the published table)
NETS = {"om_sarl": 103702, "cadrl": 27401, "lstm_rl": 46851, "om_lstm_rl": 56451, "lstm_rl_vn2": 86601, "om_lstm_rl_vn2": None}


@pytest.fixture(scope="module")
def dev():
    import torch
    import modelcrowdnav_b200 as mcn
    assert mcn._capi.load().cn_device_count() > 0, "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture
def no_tf32():
    import torch
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


def _model(name, dev, seed=0):
    import torch
    torch.manual_seed(seed)
    return _make(name).to(dev)


def _in_dim(name):
    return 61 if name.startswith("om_") else 13


def _states(name, n, H, seed):
    """Random joint states: (n, H, D), or CADRL's single-human rows (n, D)."""
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    shape = (n, _in_dim(name)) if name == "cadrl" else (n, H, _in_dim(name))
    x = torch.rand(shape, generator=g) * 4 - 2
    x[..., 2] = 0.0                                          # theta, zero for holonomic robots
    if _in_dim(name) > 13:
        x[..., 13::3] = (x[..., 13::3] > 0).float()            # occupancy flags of the map cells
    y = torch.rand((n, 1), generator=g) - 0.25
    return x, y


def _flat(model):
    import torch
    return torch.cat([v.detach().reshape(-1) for v in model.state_dict().values()]).cpu().numpy()


def _step_grad(ft, x, y, H):
    import torch
    from modelcrowdnav_b200._capi import check
    loss = torch.zeros((), device=x.device)
    check(ft.lib.cn_trainer_step(ft.handle, C.c_void_p(ft.flat.data_ptr()), C.c_void_p(x.data_ptr()),
                                 C.c_void_p(y.reshape(-1).contiguous().data_ptr()), x.shape[0], H, 0.01, 0.9,
                                 C.c_void_p(ft.grad.data_ptr()), C.c_void_p(loss.data_ptr()), ft._stream()))
    torch.cuda.synchronize()
    return float(loss)


@pytest.mark.parametrize("B,H", [(100, 5), (37, 10), (1, 1), (64, 16)])
@pytest.mark.parametrize("name", list(NETS))
def test_gradient_matches_autograd(dev, no_tf32, name, B, H):
    """One cn_trainer_step with grad_out against torch autograd on the same batch: loss within 1e-6 relative, every gradient
    entry within 2e-5 of the largest.  CADRL runs every case with one human per sample."""
    import torch
    from modelcrowdnav_b200.fused_trainer import FusedTrainer
    if name == "cadrl":
        H = 1
    model = _model(name, dev)
    x, y = _states(name, B, H, seed=B * 100 + H)
    x, y = x.to(dev).contiguous(), y.to(dev)
    out = model(x)
    loss = torch.nn.functional.mse_loss(out, y)
    loss.backward()
    ref_loss = float(((out.detach().double() - y.double()) ** 2).mean())       # the same outputs, reduced in float64
    ref = torch.cat([p.grad.reshape(-1) for p in model.parameters()]).cpu().numpy()
    ft = FusedTrainer(model, dev)
    ft.sync_from_model()
    got_loss = _step_grad(ft, x, y, H)
    got = ft.grad.cpu().numpy()
    assert got.size == ref.size
    assert abs(got_loss - ref_loss) <= 1e-6 * abs(ref_loss) + 1e-12, (got_loss, ref_loss)
    scale = np.abs(ref).max()
    assert scale > 0
    assert np.max(np.abs(got - ref)) <= 2e-5 * scale, (np.max(np.abs(got - ref)), scale)
    ft.close()


def _memory(name, dev, n=600, H=5):
    import modelcrowdnav_b200 as mcn
    x, y = _states(name, n, H, seed=7)
    memory = mcn.ReplayMemory(100000, device=dev)
    memory.push_batch(x.to(dev), y.to(dev))
    return memory


@pytest.mark.parametrize("name", list(NETS))
def test_100_steps_match_eager(dev, no_tf32, name):
    """Trainer(mode="fused") against Trainer(mode="eager") (torch SGD with momentum): 100 steps on the same index batches from
    the same weights; weights within 1e-5, and the steps moved them."""
    import torch
    from modelcrowdnav_b200.trainer import Trainer
    memory = _memory(name, dev)
    idx = torch.randint(len(memory), (100, 100), generator=torch.Generator().manual_seed(2)).to(dev)
    w0 = _flat(_model(name, dev))
    out = {}
    for mode in ("eager", "fused"):
        model = _model(name, dev)
        tr = Trainer(model, memory, dev, 100, mode=mode)
        tr.set_learning_rate(0.01)
        if mode == "fused":
            assert tr._fused_indexed_ok()
        for i in range(idx.shape[0]):
            tr._step(idx[i])
        tr._after()
        out[mode] = _flat(model)
    assert np.max(np.abs(out["fused"] - out["eager"])) <= 1e-5, np.max(np.abs(out["fused"] - out["eager"]))
    assert np.max(np.abs(out["eager"] - w0)) > 1e-3


@pytest.mark.parametrize("name", list(NETS))
def test_step_forms_agree(dev, name):
    """step_indexed (batch gathered inside the kernel) equals step on the gathered batch, and grad_out + cn_trainer_apply with
    scale 1 equals the in-place step, bit for bit over three steps."""
    import torch
    from modelcrowdnav_b200._capi import check
    from modelcrowdnav_b200.fused_trainer import FusedTrainer
    memory = _memory(name, dev, n=300)
    S, V = memory.states[:len(memory)].contiguous(), memory.values[:len(memory)].contiguous()
    H = 1 if name == "cadrl" else S.shape[1]
    fts = []
    for _ in range(3):
        ft = FusedTrainer(_model(name, dev), dev)
        ft.lr = 0.01
        fts.append(ft)
    fts[2].sync_from_model()
    loss_sum = torch.zeros((), device=dev)
    g = torch.Generator().manual_seed(3)
    for _ in range(3):
        idx = torch.randperm(S.shape[0], generator=g)[:64].to(dev)
        fts[0].step_indexed(S, V, idx, loss_sum)
        fts[1].step(S[idx], V[idx])
        x, y = S[idx].contiguous(), V[idx].reshape(-1).contiguous()
        f = fts[2]
        check(f.lib.cn_trainer_step(f.handle, C.c_void_p(f.flat.data_ptr()), C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()),
                                    64, H, f.lr, f.momentum, C.c_void_p(f.grad.data_ptr()), None, f._stream()))
        check(f.lib.cn_trainer_apply(f.handle, C.c_void_p(f.flat.data_ptr()), C.c_void_p(f.grad.data_ptr()), 1.0, f.lr,
                                     f.momentum, f._stream()))
    torch.cuda.synchronize()
    assert torch.equal(fts[0].flat, fts[1].flat)
    assert torch.equal(fts[2].flat, fts[1].flat)
    assert np.isfinite(float(loss_sum)) and float(loss_sum) > 0
    for f in fts:
        f.close()


@pytest.mark.parametrize("name", list(NETS))
def test_parameters_are_shared(dev, name):
    """cn_trainer_param_count = the torch model's count = cn_policy_param_count of the same config; a step moves
    model.state_dict() itself, because the parameters are views of the trainer's block."""
    from modelcrowdnav_b200.fused_trainer import FusedTrainer
    model = _model(name, dev)
    n = sum(p.numel() for p in model.parameters())
    if NETS[name] is not None:
        assert n == NETS[name]
    ft = FusedTrainer(model, dev)
    assert int(ft.lib.cn_trainer_param_count(ft.handle)) == n
    assert int(ft.lib.cn_policy_param_count(C.byref(ft.cfg))) == n
    before = _flat(model)
    x, y = _states(name, 32, 5, seed=5)
    ft.lr = 0.01
    ft.step(x.to(dev), y.to(dev))
    after = _flat(model)
    assert np.max(np.abs(after - before)) > 0
    for v in model.state_dict().values():
        assert ft.flat.data_ptr() <= v.data_ptr() < ft.flat.data_ptr() + 4 * ft.flat.numel()
    ft.close()


def test_refusals(dev):
    """Configurations the fused trainer cannot run fail at creation (or at the step) with the right code and a message."""
    import torch
    from modelcrowdnav_b200 import _capi
    lib = _capi.load()

    def create(max_humans=5, **kw):
        h = C.c_void_p()
        rc = lib.cn_trainer_create(C.byref(_capi.default_sarl_cfg(**kw)), 0, 128, max_humans, C.byref(h))
        if rc == _capi.CN_OK:
            lib.cn_trainer_destroy(h)
        else:
            assert lib.cn_last_error().decode()
        return rc

    cadrl = dict(network=_capi.NET_CADRL)
    lstm = dict(network=_capi.NET_LSTM_RL)
    om = dict(with_om=1, cell_num=4, om_channel_size=3)
    assert create(1, **cadrl) == _capi.CN_OK
    assert create(2, **cadrl) == _capi.CN_EINVAL                                  # CADRL trains on one human per sample
    assert create(16, **lstm) == _capi.CN_OK
    assert create(17, **lstm) == _capi.CN_EUNSUPPORTED                            # over the 16-human cap
    assert create(16, lstm_mlp1_dims=LM1, **lstm) == _capi.CN_OK
    assert create(17, lstm_mlp1_dims=LM1, **lstm) == _capi.CN_EUNSUPPORTED
    assert create(5, lstm_hidden=256, **lstm) == _capi.CN_EUNSUPPORTED            # W_hh does not fit the shared-memory plan
    assert create(5, self_state_dim=14, **lstm) == _capi.CN_EINVAL                # the self state is part of row 0
    assert create(5, input_dim=61, **om) == _capi.CN_OK                           # OM-SARL
    assert create(5, input_dim=61, **om, **lstm) == _capi.CN_OK                   # OM-LSTM-RL
    assert create(5, input_dim=13, **om) == _capi.CN_EINVAL                       # with_om and input_dim disagree
    assert create(5, input_dim=60, **om, **lstm) == _capi.CN_EINVAL
    assert create(1, input_dim=61, **om, **cadrl) == _capi.CN_EINVAL               # CADRL has no maps
    # a CADRL step with more than one human per sample
    h = C.c_void_p()
    _capi.check(lib.cn_trainer_create(C.byref(_capi.default_sarl_cfg(**cadrl)), 0, 128, 1, C.byref(h)))
    w = torch.zeros(int(lib.cn_trainer_param_count(h)), device=dev)
    x, y = torch.zeros((8, 2, 13), device=dev), torch.zeros(8, device=dev)
    rc = lib.cn_trainer_step(h, C.c_void_p(w.data_ptr()), C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), 8, 2, 0.01, 0.9,
                             None, None, None)
    assert rc == _capi.CN_EINVAL and "human_num" in lib.cn_last_error().decode()
    lib.cn_trainer_destroy(h)
    # the Python trainer: CADRL batches are (B, 13)
    from modelcrowdnav_b200.fused_trainer import FusedTrainer
    ft = FusedTrainer(_model("cadrl", dev), dev)
    ft.lr = 0.01
    with pytest.raises(ValueError):
        ft.step(x, y.reshape(-1, 1))
    ft.close()


@pytest.mark.parametrize("policy_name,with_om", [("cadrl", False), ("lstm_rl", False), ("sarl", True)])
def test_training_loop_fused(dev, no_tf32, tmp_path, policy_name, with_om):
    """TrainingLoop(trainer_mode="fused") end to end: a small imitation-learning phase, two RL iterations; finite losses, and
    the lookahead's FP32 network afterwards computes the trained torch model's values (1e-5)."""
    import torch
    from modelcrowdnav_b200.train_loop import TrainingLoop
    cfg = None
    if with_om:
        cfg = tmp_path / "policy.config"
        cfg.write_text("[sarl]\nwith_om = true\n")
        cfg = str(cfg)
    loop = TrainingLoop(dev, policy_name=policy_name, trainer_mode="fused", sample_episodes=8, policy_config=cfg)
    il_loss = loop.imitation_learning(il_episodes=16, il_epochs=2)
    assert loop.trainer._fused is not None and loop.trainer._fused_indexed_ok()
    loop.start_rl()
    losses = [loop.rl_iteration(0.5, train_batches=10) for _ in range(2)]
    assert np.isfinite(il_loss) and all(np.isfinite(losses)), (il_loss, losses)
    x = loop.memory.states[:min(len(loop.memory), 256)].contiguous()
    got = loop.policy.handle(1.0, precision="f32").forward(x).cpu().numpy()
    with torch.no_grad():
        ref = loop.model(x).reshape(-1).cpu().numpy()
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)
    assert err.max() <= 1e-5, err.max()
