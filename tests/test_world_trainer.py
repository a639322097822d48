"""Training the world models on the device (cn_world_trainer_*, csrc/world_trainer.cu; cn_env_copy_world_pairs;
modelcrowdnav_b200/world_trainer.py).

Ground truth is torch autograd on a torch restatement of AttentionWorld / MlpWorld written here, which is first pinned to
the reference's own predictions (tests/golden/model_world_*.npz) on the CPU.  The GPU references run with TF32 off."""
import ctypes as C

import numpy as np
import pytest

from conftest import MODEL_WORLD_NAMES, load_model_world


# ---- the torch restatement of both forwards ----------------------------------------------------------------------------
def _lin(p, name, x):
    import torch
    return torch.nn.functional.linear(x, p[name + ".weight"], p[name + ".bias"])


def attention_forward(p, x):
    """AttentionWorld.forward (world_model.py:71-106): x (B, H, 4) -> (B, H, 2)"""
    import torch
    relu = torch.relu
    e = relu(_lin(p, "mlp1.2", relu(_lin(p, "mlp1.0", x))))
    f = _lin(p, "mlp2.2", relu(_lin(p, "mlp2.0", e)))
    u = torch.cat([e, e.mean(dim=1, keepdim=True).expand_as(e)], dim=-1)
    s = _lin(p, "attention.4", relu(_lin(p, "attention.2", relu(_lin(p, "attention.0", u)))))[..., 0]
    ex = torch.exp(s) * (s != 0).to(s.dtype)
    w = ex / ex.sum(dim=1, keepdim=True)
    feat = (w.unsqueeze(-1) * f).sum(dim=1)
    j = torch.cat([x, feat.unsqueeze(1).expand(-1, x.shape[1], -1)], dim=-1)
    g = relu(_lin(p, "mlp3.4", relu(_lin(p, "mlp3.2", relu(_lin(p, "mlp3.0", j))))))
    return _lin(p, "mlp3.6", g)


def mlp_forward(p, x, masks=None, drop=0.0):
    """MlpWorld.forward (world_model.py:20-50) on x (B, H, 4) -> (B, H, 2); masks = the (B, 128) and (B, 64) dropout masks
    of training mode (torch.nn.Dropout: kept units scaled by 1 / (1 - p)), None = eval"""
    import torch
    B = x.shape[0]
    h = torch.relu(_lin(p, "mlp.0", x.reshape(B, -1)))
    if masks is not None:
        h = h * masks[0] / (1.0 - drop)
    h = torch.relu(_lin(p, "mlp.3", h))
    if masks is not None:
        h = h * masks[1] / (1.0 - drop)
    h = torch.relu(_lin(p, "mlp.6", h))
    return torch.tanh(_lin(p, "mlp.8", h)).reshape(B, -1, 2)


def world_forward(kind, p, x, **kw):
    return mlp_forward(p, x, **kw) if kind == "mlp" else attention_forward(p, x)


def _params(world, dtype=None, device=None):
    return {k: v.detach().clone().to(dtype=dtype or v.dtype, device=device or v.device).requires_grad_()
            for k, v in world.state_dict().items()}


@pytest.mark.parametrize("name", MODEL_WORLD_NAMES)
def test_restatement_matches_reference(name):
    """The torch restatement above reproduces the velocities the REFERENCE's modules predicted (new_v of every
    model_world_*.npz) within 2e-6, so autograd of it is the gradient of the reference's forward."""
    import torch
    from modelcrowdnav_b200.world_model import AttentionWorld, MlpWorld
    g = load_model_world(name)
    kind = "mlp" if str(g["world"]) == "mlp" else "attention"
    world = MlpWorld(int(g["H"])) if kind == "mlp" else AttentionWorld()
    off = 0
    p = {}
    for k, v in world.state_dict().items():
        p[k] = torch.from_numpy(g["world_weights"][off:off + v.numel()].reshape(tuple(v.shape)).astype(np.float64))
        off += v.numel()
    T = len(g["reward"])
    x = torch.from_numpy(np.stack([g["agents"][t][1:, :4] for t in range(T)]).astype(np.float32).astype(np.float64))
    got = world_forward(kind, p, x).numpy()
    assert np.max(np.abs(got - g["new_v"][:T])) <= 2e-6


def test_early_stopping_rule():
    """pytorchtools.EarlyStopping: val <= best - delta improves (the first always does), otherwise the counter grows until
    patience; delta = 0 counts an equal loss as an improvement, delta > 0 does not count a smaller step."""
    from modelcrowdnav_b200.world_trainer import EarlyStopping
    es = EarlyStopping(patience=2)
    assert [es.update(v) for v in (1.0, 0.5, 0.5, 0.6, 0.7)] == [(True, False), (True, False), (True, False), (False, False),
                                                               (False, True)]
    es = EarlyStopping(patience=3, delta=0.1)
    assert [es.update(v) for v in (1.0, 0.9, 0.95, 0.85, 0.8)] == [(True, False), (True, False), (False, False),
                                                                 (False, False), (True, False)]
    assert es.best == 0.8 and es.counter == 0


# ---- GPU ---------------------------------------------------------------------------------------------------------------
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


def _world(kind, H, seed=0, drop=0.0):
    import torch
    from modelcrowdnav_b200.world_model import AttentionWorld, MlpWorld
    torch.manual_seed(seed)
    return MlpWorld(H, drop_rate=drop) if kind == "mlp" else AttentionWorld()


def _data(n, H, seed, dev):
    """human states like a crowd's (positions in +-4 m, velocities in +-1 m/s) and velocities to learn"""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.cat([torch.rand((n, H, 2), generator=g) * 8 - 4, torch.rand((n, H, 2), generator=g) * 2 - 1], dim=-1)
    y = torch.rand((n, H, 2), generator=g) * 2 - 1
    return x.to(dev), y.to(dev)


def _trainer(world, dev, **kw):
    from modelcrowdnav_b200.world_trainer import WorldTrainer
    kw.setdefault("lr", 1e-3)
    kw.setdefault("max_batch", 4096)
    return WorldTrainer(world, dev, **kw)


def _grad_errors(got, ref):
    scale = np.abs(ref).max()
    assert scale > 0
    return np.max(np.abs(got - ref)) / scale


KINDS = ["attention", "mlp"]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H", [(100, 5), (37, 10), (1, 1), (64, 16), (9, 3)])
@pytest.mark.parametrize("kind", KINDS)
def test_gradient_matches_autograd(dev, no_tf32, kind, B, H):
    """One grad_out step against torch autograd of the restatement: the loss within 1e-6 relative, every gradient entry
    within 2e-5 of the largest (the value-network trainer's bars).  MlpWorld runs 8 samples per CTA, so 37 and 9 samples end
    in a partial CTA."""
    import torch
    world = _world(kind, H)
    x, y = _data(B, H, seed=B * 100 + H, dev=dev)
    p = _params(world, device=dev)
    out = world_forward(kind, p, x)
    loss = torch.nn.functional.mse_loss(out, y)
    loss.backward()
    ref_loss = float(((out.detach().double() - y.double()) ** 2).mean())
    ref = torch.cat([p[k].grad.reshape(-1) for k in p]).cpu().numpy()
    tr = _trainer(world, dev)
    got_loss = float(tr.gradient(x, y))
    got = tr.grad.cpu().numpy()
    assert got.size == ref.size == (94953 if kind == "attention" else 4 * H * 128 + 128 + 8256 + 780 + 26 * H)
    assert abs(got_loss - ref_loss) <= 1e-6 * abs(ref_loss), (got_loss, ref_loss)
    assert _grad_errors(got, ref) <= 2e-5
    tr.close()


@pytest.mark.gpu
def test_dropout_masks(dev, no_tf32):
    """MlpWorld at p = 0.5: with the masks the kernel drew applied in torch, the gradient meets the bars above; the kept
    fraction over 4096 x 192 units is within 4 sigma of 1 - p; the same (seed, step) draws the same masks and the next step
    other ones."""
    import torch
    H, B, drop = 5, 4096, 0.5
    world = _world("mlp", H, drop=drop)
    x, y = _data(B, H, seed=3, dev=dev)
    tr = _trainer(world, dev, seed=1234)
    mask = torch.zeros((B, 192), dtype=torch.uint8, device=dev)
    got_loss = float(tr.gradient(x, y, mask=mask))
    got = tr.grad.cpu().numpy()
    m = mask.float()
    p = _params(world, device=dev)
    out = mlp_forward(p, x, masks=(m[:, :128], m[:, 128:]), drop=drop)
    loss = torch.nn.functional.mse_loss(out, y)
    loss.backward()
    ref = torch.cat([p[k].grad.reshape(-1) for k in p]).cpu().numpy()
    assert abs(got_loss - float(loss.detach())) <= 1e-6 * float(loss.detach())
    assert _grad_errors(got, ref) <= 2e-5
    n = mask.numel()
    kept = float(m.mean())
    assert abs(kept - (1 - drop)) <= 4 * np.sqrt(drop * (1 - drop) / n), kept
    mask2 = torch.zeros_like(mask)
    tr.gradient(x, y, mask=mask2)                                   # step 1
    assert not torch.equal(mask, mask2)
    tr.sync(reset_optimizer=True)                                   # back to step 0
    mask3 = torch.zeros_like(mask)
    tr.gradient(x, y, mask=mask3)
    assert torch.equal(mask, mask3)
    # masks do not depend on the batch split: the first 100 samples of a 100-sample step draw what the 4096-sample one drew
    tr.sync(reset_optimizer=True)
    mask4 = torch.zeros((100, 192), dtype=torch.uint8, device=dev)
    tr.gradient(x[:100], y[:100], mask=mask4)
    assert torch.equal(mask4, mask[:100])
    tr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_adam_matches_torch(dev, kind):
    """5 steps of grad_out + apply against torch.optim.Adam(foreach=False) stepping on the same gradient: every parameter
    tensor within 1e-6 x its max |w|.  The fused step equals grad_out + apply bit for bit."""
    import torch
    H, B = 5, 64
    world = _world(kind, H)
    twin = _world(kind, H)
    x, y = _data(B, H, seed=11, dev=dev)
    tr = _trainer(world, dev, lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    fused = _trainer(twin, dev, lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    ref = {k: v.detach().clone().requires_grad_() for k, v in world.state_dict().items()}
    opt = torch.optim.Adam(list(ref.values()), lr=1e-3, betas=(0.9, 0.999), eps=1e-8, foreach=False)
    names = list(ref)
    for _ in range(5):
        tr.gradient(x, y)
        off = 0
        for k in names:
            n = ref[k].numel()
            ref[k].grad = tr.grad[off:off + n].view(ref[k].shape).clone()
            off += n
        opt.step()
        tr.apply()
        fused.step(x, y)
        got = world.state_dict()
        for k in names:
            err = float((got[k] - ref[k].detach()).abs().max())
            assert err <= 1e-6 * float(ref[k].detach().abs().max()), (k, err)
    assert torch.equal(tr.flat, fused.flat)
    tr.close(); fused.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_100_steps_match_torch(dev, no_tf32, kind):
    """100 fused steps against 100 steps of torch autograd + torch.optim.Adam on the same batches (B = 100, H = 5, lr 1e-3):
    the two loss curves agree at every step to 2e-3 relative.  Adam's m / sqrt(v) turns last-bit gradient differences near
    zero into full-size steps, so the curves drift apart slowly.  Measured on a B200: largest relative difference 3.8e-4
    (AttentionWorld) and 2.7e-7 (MlpWorld)."""
    import torch
    H, B, N = 5, 100, 1000
    world = _world(kind, H)
    X, Y = _data(N, H, seed=5, dev=dev)
    ref = _params(world, device=dev)
    opt = torch.optim.Adam(list(ref.values()), lr=1e-3, foreach=False)
    tr = _trainer(world, dev, lr=1e-3)
    g = torch.Generator().manual_seed(0)
    worst = 0.0
    for _ in range(100):
        idx = torch.randint(0, N, (B,), generator=g).to(dev)
        got = float(tr.step(X, Y, index=idx))
        opt.zero_grad()
        loss = torch.nn.functional.mse_loss(world_forward(kind, ref, X[idx]), Y[idx])
        loss.backward()
        opt.step()
        ref_loss = float(loss.detach())
        worst = max(worst, abs(got - ref_loss) / ref_loss)
    print("%s: worst relative loss difference over 100 steps %.3g" % (kind, worst))
    assert worst <= 2e-3, worst
    tr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_indexed_step_equals_gathered(dev, kind):
    """A step on the samples index of X / Y equals a step on the gathered batch X[index], bit for bit (loss and weights)."""
    import torch
    H = 5
    X, Y = _data(500, H, seed=9, dev=dev)
    idx = torch.randperm(500, generator=torch.Generator().manual_seed(1))[:77].to(dev)
    a, b = _trainer(_world(kind, H), dev), _trainer(_world(kind, H), dev)
    for _ in range(3):
        la = a.step(X, Y, index=idx)
        lb = b.step(X[idx], Y[idx])
        assert torch.equal(la, lb)
    assert torch.equal(a.flat, b.flat)
    a.close(); b.close()


@pytest.mark.gpu
def test_recorded_pairs_match_host_reads(dev):
    """cn_env_copy_world_pairs between the ORCA solve and the step, step by step on 6 envs x 3 humans: x = get_state's human
    (px, py, vx, vy) cast to fp32 and y = human_actions cast to fp32, bit for bit; frozen envs are invalid.  Then
    collect_world_transitions over whole episodes: the valid pairs are as many as the episodes' steps."""
    import torch
    import modelcrowdnav_b200 as mcn
    from modelcrowdnav_b200.world_trainer import collect_world_transitions
    E, H = 6, 3
    env = mcn.BatchedCrowdSim(E, H, seed=4)
    env.reset_device()
    lib = env.lib
    x = torch.empty((E, H, 4), dtype=torch.float32, device=dev)
    y = torch.empty((E, H, 2), dtype=torch.float32, device=dev)
    v = torch.empty(E, dtype=torch.uint8, device=dev)
    from modelcrowdnav_b200._capi import CrowdNavError
    with pytest.raises(CrowdNavError, match="no cached ORCA"):
        mcn._capi.check(lib.cn_env_copy_world_pairs(env.handle, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), None, None))
    saw_frozen = False
    for t in range(60):
        env.orca()
        mcn._capi.check(lib.cn_env_copy_world_pairs(env.handle, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()),
                                                    C.c_void_p(v.data_ptr()), None))
        agents, _ = env.get_state()
        frozen = env.episode_table()["frozen"]
        assert np.array_equal(x.cpu().numpy(), agents[:, 1:, :4].astype(np.float32)), t
        assert np.array_equal(y.cpu().numpy(), env.human_actions().astype(np.float32)), t
        assert np.array_equal(v.cpu().numpy(), 1 - frozen), t
        saw_frozen |= bool(frozen.any())
        env.robot_orca(0.1)
        env.step(read=False)
    assert saw_frozen
    env.close()
    env = mcn.BatchedCrowdSim(64, 5, seed=8)
    env.reset_device()
    X, Y, ids = collect_world_transitions(env, robot="orca", safety_space=0.1)
    table = env.episode_table()
    assert table["frozen"].all()
    assert X.shape[0] == Y.shape[0] == ids.shape[0] == int(table["steps"].sum())
    assert np.array_equal(np.bincount(ids.cpu().numpy(), minlength=64), table["steps"])
    env.close()


@pytest.mark.gpu
def test_end_to_end(dev, weights0):
    """ORCA transitions of 2,048 circle-crossing episodes (H = 5), split by episode (every fifth env held out); an
    AttentionWorld and an MlpWorld(5) (dropout 0.5) trained for 4 epochs with early stopping.  The validation MSE falls to
    at most half its initial value (measured on a B200: AttentionWorld 0.031x, MlpWorld 0.21x).  Then, with no explicit
    reload, predict_into on held-out states equals the torch restatement of the trained block within 1e-5, and its MSE the
    trainer's own validation forward (cn_world_trainer_eval); an Explorer run over ModelCrowdSim with the trained model
    completes; the saved state dict predicts the same in a fresh container and in the float64 restatement."""
    import io
    import torch
    import modelcrowdnav_b200 as mcn
    from modelcrowdnav_b200.world_trainer import collect_world_transitions
    E, H = 2048, 5
    env = mcn.BatchedCrowdSim(E, H, seed=21)
    env.reset_device()
    X, Y, ids = collect_world_transitions(env, robot="orca", safety_space=0.1)
    env.close()
    val = ids % 5 == 0
    Xt, Yt, Xv, Yv = X[~val], Y[~val], X[val], Y[val]
    for kind in KINDS:
        world = _world(kind, H, seed=3, drop=0.5)
        tr = _trainer(world, dev, lr=1e-3, max_batch=1024)
        v0 = float(tr.evaluate(Xv, Yv))
        hist = tr.optimize_epoch(Xt, Yt, batch_size=1024, num_epochs=4, val=(Xv, Yv), patience=2,
                                 generator=torch.Generator().manual_seed(0))
        best = min(h["val"] for h in hist)
        print("%s: %d train / %d val pairs, val MSE %.4g -> %s (%.3gx)" % (
            kind, Xt.shape[0], Xv.shape[0], v0, [round(h["val"], 5) for h in hist], best / v0))
        assert best <= 0.5 * v0, (v0, hist)
        # predict_into on held-out states, through the model's own handle (no explicit reload)
        n = 256
        xs = Xv[:n]
        agents = np.zeros((n, H + 1, 8))
        agents[:, 1:, :4] = xs.cpu().numpy()
        agents[:, :, 6] = 0.3; agents[:, :, 7] = 1.0
        b = mcn.BatchedCrowdSim(n, H)
        b.set_state(agents)
        world.predict_into(b)
        pred = b.human_actions()
        b.close()
        p = {k: v.detach() for k, v in world.state_dict().items()}
        with torch.no_grad():
            ref = world_forward(kind, p, xs).cpu().numpy()
        assert np.max(np.abs(pred - ref)) <= 1e-5
        mse = float(((torch.from_numpy(pred).to(dev).float() - Yv[:n]) ** 2).mean())
        ev = float(tr.evaluate(xs, Yv[:n]))
        assert abs(mse - ev) <= 1e-5 * ev, (mse, ev)
        # the saved state dict, in a fresh container and in float64
        buf = io.BytesIO()
        torch.save(world.state_dict(), buf)
        buf.seek(0)
        fresh = _world(kind, H, seed=99)
        fresh.load_state_dict(torch.load(buf))
        b = mcn.BatchedCrowdSim(n, H)
        b.set_state(agents)
        fresh.predict_into(b)
        assert np.array_equal(b.human_actions(), pred)
        b.close()
        p64 = {k: v.detach().double().cpu() for k, v in fresh.state_dict().items()}
        ref64 = world_forward(kind, p64, xs.double().cpu()).numpy()
        assert np.max(np.abs(pred - ref64)) <= 1e-5
        tr.close()
    # Explorer over ModelCrowdSim driven by the last trained model
    import modelcrowdnav_b200.compat as compat
    from test_gpu_facade import ENV_INI, _cfg, _setup
    _, robot, policy, _ = _setup(weights0, "f32", human_num=5)
    menv = compat.make("ModelCrowdSim-v0")
    menv.configure(_cfg(ENV_INI))
    menv.set_robot(robot)
    policy.set_env(menv)
    menv.sim_world, menv.device = world, dev
    explorer = mcn.Explorer(menv, robot, dev, gamma=0.9)
    explorer.run_k_episodes(8, "test")
    assert len(explorer.last_run["steps"]) == 8


@pytest.mark.gpu
def test_early_stopping_restores_best(dev, monkeypatch):
    """optimize_epoch with a scripted validation sequence: it stops at the epoch the EarlyStopping rule says and leaves the
    block of the best epoch (the first of two equal losses with delta > 0)."""
    import torch
    H = 5
    X, Y = _data(300, H, seed=2, dev=dev)
    tr = _trainer(_world("attention", H), dev, lr=1e-3)
    script = iter([1.0, 0.8, 0.75, 0.9, 0.8, 0.5])          # delta 0.1: 0.75 does not improve on 0.8; stop after 0.8 (3rd miss)
    blocks = []

    def scripted(Xv, Yv):
        blocks.append(tr.flat.clone())
        return torch.tensor(next(script), device=dev)
    monkeypatch.setattr(tr, "_validate", scripted)
    hist = tr.optimize_epoch(X, Y, batch_size=64, num_epochs=6, val=(X, Y), patience=3, delta=0.1)
    assert [h["val"] for h in hist] == pytest.approx([1.0, 0.8, 0.75, 0.9, 0.8])
    assert torch.equal(tr.flat, blocks[1])
    assert not torch.equal(tr.flat, blocks[-1])
    tr.close()


@pytest.mark.gpu
def test_refusals(dev):
    """Every limit returns its code and message and writes nothing."""
    import torch
    from modelcrowdnav_b200 import _capi
    from modelcrowdnav_b200._capi import CN_EINVAL, CN_EUNSUPPORTED
    lib = _capi.load()
    h = C.c_void_p()

    def create(kind, H, drop=0.0, max_batch=16):
        h.value = None
        rc = lib.cn_world_trainer_create(kind, H, 0, max_batch, drop, C.byref(h))
        return rc, lib.cn_last_error().decode()
    for drop in (-0.1, 1.0, float("nan")):
        rc, msg = create(_capi.WORLD_MLP, 5, drop)
        assert (rc, h.value) == (CN_EINVAL, None) and "drop_rate" in msg
    rc, msg = create(_capi.WORLD_ATTENTION, 5, 0.5)
    assert (rc, h.value) == (CN_EINVAL, None) and "no dropout" in msg
    rc, msg = create(_capi.WORLD_ATTENTION, 24)
    assert (rc, h.value) == (CN_EUNSUPPORTED, None) and "shared-memory plan" in msg
    assert create(_capi.WORLD_ATTENTION, 23)[0] == 0
    lib.cn_world_trainer_destroy(h)
    assert create(_capi.WORLD_MLP, 5)[0] == 0
    n = int(lib.cn_world_trainer_param_count(h))
    w = torch.randn(n, device=dev)
    w0 = w.clone()
    x, y = _data(32, 5, seed=0, dev=dev)
    loss = torch.zeros((), device=dev)

    def step(batch, H):
        rc = lib.cn_world_trainer_step(h, C.c_void_p(w.data_ptr()), C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), None,
                                       batch, H, 1e-3, 0.9, 0.999, 1e-8, 0, None, C.c_void_p(loss.data_ptr()), None, None)
        torch.cuda.synchronize()
        return rc, lib.cn_last_error().decode()
    rc, msg = step(8, 5)
    assert rc == CN_EINVAL and "sync_weights" in msg
    assert lib.cn_world_trainer_sync_weights(h, C.c_void_p(w.data_ptr()), 1, None) == 0
    rc, msg = step(17, 5)
    assert rc == CN_EINVAL and "max_batch" in msg
    rc, msg = step(8, 4)
    assert rc == CN_EINVAL and "MlpWorld was built for 5 humans, the data has 4" in msg
    assert torch.equal(w, w0) and float(loss) == 0.0
    assert step(8, 5)[0] == 0
    assert not torch.equal(w, w0) and float(loss) > 0
    lib.cn_world_trainer_destroy(h)
