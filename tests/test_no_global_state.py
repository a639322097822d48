"""SARL without the global state ([sarl] with_global_state = false, sarl.py:40-47): attention.0 sees e_i alone.

Ground truth is the torch ValueNetwork of policy.py (make_value_network(..., with_global_state=False)), which restates
sarl.py:28-65 with the switch.  The CPU oracle evaluates the global-state network only; given attention.0 weights whose
group-mean columns are ZERO it computes exactly the network without the global state (every mean term adds 0 * mean = 0),
so the oracle runs unmodified on that zero-padded layout.  test_oracle_pinned_to_torch_module checks this first."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, TIE_GAP, check_argmax, value_errors

E1 = 100                                  # mlp1_dims[-1] at the default [sarl] dims
OM_DIM = 48                               # [om] cell_num 4, om_channel_size 3
OM_KW = dict(input_dim=13 + OM_DIM, with_om=1, cell_num=4, cell_size=1.0, om_channel_size=3)
NOGS = dict(without_global_state=1)


@pytest.fixture(scope="module")
def mcn():
    import modelcrowdnav_b200 as m
    return m


@pytest.fixture(scope="module")
def gpu(mcn):
    assert mcn._capi.load().cn_device_count() > 0, "GPU tests need a CUDA device"
    return mcn


# ---- weights ---------------------------------------------------------------------------------------------------------
def _net(input_dim=13, with_global_state=False):
    from modelcrowdnav_b200.policy import make_value_network
    return make_value_network(input_dim, 6, [150, 100], [100, 50], [150, 100, 100, 1], [100, 100, 1], with_global_state)


def _flat(model):
    return np.concatenate([v.detach().cpu().numpy().ravel() for v in model.state_dict().values()]).astype(np.float32)


def _load(model, flat):
    import torch
    sd, off = {}, 0
    for k, v in model.state_dict().items():
        sd[k] = torch.from_numpy(np.ascontiguousarray(flat[off:off + v.numel()]).reshape(tuple(v.shape)))
        off += v.numel()
    assert off == flat.size
    model.load_state_dict(sd)
    return model


def seeded_weights(seed=0, input_dim=13):
    """nn.Linear's default init of the network without the global state under torch.manual_seed(seed)."""
    import torch
    torch.manual_seed(seed)
    return _flat(_net(input_dim))


def trained_weights(input_dim=13):
    """Realistic magnitudes: the GPU-trained SARL with attention.0 cut to its 100 mlp1_out columns.  With occupancy maps,
    mlp1.0's 48 map columns are a seeded default init (the trained network has none)."""
    import torch
    sd = _load(_net(13, True), np.load(os.path.join(GOLDEN, "sarl_weights_trained.npy"))).state_dict()
    sd["attention.0.weight"] = sd["attention.0.weight"][:, :E1].clone()
    if input_dim != 13:
        torch.manual_seed(7)
        extra = _net(input_dim).state_dict()["mlp1.0.weight"][:, 13:]
        sd["mlp1.0.weight"] = torch.cat([sd["mlp1.0.weight"], extra], dim=1)
    m = _net(input_dim)
    m.load_state_dict(sd)
    return _flat(m)


def oracle_layout(w, input_dim=13):
    """The same network in the global-state layout with zero group-mean columns in attention.0 (what the oracle reads)."""
    import torch
    sd = _load(_net(input_dim), w).state_dict()
    wa = sd["attention.0.weight"]
    sd["attention.0.weight"] = torch.cat([wa, torch.zeros_like(wa)], dim=1)
    m = _net(input_dim, True)
    m.load_state_dict(sd)
    return _flat(m)


WSETS = {"seed": lambda input_dim=13: seeded_weights(3, input_dim), "trained": trained_weights}


def _oracle_cfg(o, om):
    scfg = o.SarlCfg.default()
    if om:
        scfg.input_dim = 13 + OM_DIM
    return scfg


def _random_rows(o, rng, B, H):
    """B x H x 13 rotated joint states of random scenes (oracle.transform)."""
    out = np.empty((B, H, 13), np.float32)
    for b in range(B):
        a = np.zeros((H + 1, 8))
        a[:, 0:2] = rng.uniform(-5, 5, (H + 1, 2))
        a[:, 2:4] = rng.uniform(-1, 1, (H + 1, 2))
        a[:, 4:6] = rng.uniform(-5, 5, (H + 1, 2))
        a[:, 6] = rng.uniform(0.3, 0.5, H + 1)
        a[:, 7] = rng.uniform(0.5, 1.5, H + 1)
        out[b] = o.transform(a)
    return out


# ---- CPU -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("wset", ["seed", "trained"])
@pytest.mark.parametrize("H", [1, 5, 10, 50])
def test_oracle_pinned_to_torch_module(oracle_mod, wset, H):
    """The oracle on the zero-padded layout == make_value_network(..., with_global_state=False), 1e-5 relative."""
    import torch
    o = oracle_mod
    w = WSETS[wset]()
    model = _load(_net(), w)
    x = _random_rows(o, np.random.default_rng(H), 16, H)
    with torch.no_grad():
        ref = model(torch.from_numpy(x)).numpy().reshape(-1)
    wo = oracle_layout(w)
    got = np.array([o.sarl_forward(o.SarlCfg.default(), wo, x[b]) for b in range(x.shape[0])])
    assert value_errors(got, ref, "f32") <= 1.0
    # and the global-state module with those padded weights is the same function
    with torch.no_grad():
        ref_gs = _load(_net(13, True), wo)(torch.from_numpy(x)).numpy().reshape(-1)
    assert value_errors(ref_gs, ref, "f32") <= 1.0


def test_param_counts(mcn):
    lib = mcn._capi.load()
    count = lambda **kw: int(lib.cn_policy_param_count(C.byref(mcn._capi.default_sarl_cfg(**kw))))
    n_torch = lambda input_dim, gs: sum(p.numel() for p in _net(input_dim, gs).parameters())
    assert count() == n_torch(13, True) == 96502
    assert count(**NOGS) == n_torch(13, False) == 86502
    assert count(**OM_KW, **NOGS) == n_torch(13 + OM_DIM, False) == 93702
    assert len(seeded_weights()) == 86502 and len(trained_weights()) == 86502 and len(oracle_layout(trained_weights())) == 96502
    assert C.sizeof(mcn._capi.SarlCfg) == 136 and mcn._capi.default_sarl_cfg().without_global_state == 0


def test_configure_and_refusals(mcn):
    """SARL.configure with with_global_state = false builds the smaller attention and asks the library for it; the flag is
    refused for CADRL and LSTM-RL before any device is touched."""
    import configparser
    from test_gpu_facade import POLICY_INI
    cp = configparser.RawConfigParser()
    cp.read_string(POLICY_INI)
    cp.set("sarl", "with_global_state", "false")
    pol = mcn.policy_factory["sarl"]()
    pol.configure(cp)
    assert tuple(pol.get_model().attention[0].weight.shape) == (100, 100)
    assert pol._net_kwargs["without_global_state"] == 1 and pol.precision == "f16_tc"
    lib = mcn._capi.load()
    for net in (mcn._capi.NET_CADRL, mcn._capi.NET_LSTM_RL):
        h = C.c_void_p()
        cfg = mcn._capi.default_sarl_cfg(network=net, without_global_state=1)
        assert lib.cn_policy_create(C.byref(cfg), 0, C.byref(h)) == mcn._capi.CN_EINVAL
        assert b"global state" in lib.cn_last_error()


# ---- GPU: FP32 lookahead -------------------------------------------------------------------------------------------------
def _scenes(o, n, H, start=0):
    rule, width = ("circle_crossing", 10.0) if H <= 10 else ("square_crossing", 16.0)
    return np.stack([o.generate_scene("val", start + c, human_num=H, rule=rule, square_width=width) for c in range(n)])


@pytest.mark.gpu
@pytest.mark.parametrize("H,query_env,om,kin", [(1, 0, 0, 0), (5, 1, 0, 1), (5, 0, 1, 0), (10, 1, 1, 1), (13, 0, 0, 0),
                                                (13, 1, 1, 0), (50, 1, 0, 0), (50, 0, 1, 1), (64, 0, 0, 1)])
def test_f32_lookahead_vs_oracle(gpu, oracle_mod, H, query_env, om, kin):
    """FP32 lookahead: every value within 1e-5 relative, the choice optimal up to the tie gap, the step outcome exact, over
    three evolving steps; holonomic and unicycle robots, with and without occupancy maps, both query_env modes."""
    o, mcn = oracle_mod, gpu
    E = 8 if H <= 13 else 3
    input_dim = 13 + (OM_DIM if om else 0)
    w = trained_weights(input_dim) if H % 2 else seeded_weights(H, input_dim)
    wo = oracle_layout(w, input_dim)
    ecfg, scfg, omc = o.EnvCfg.default(), _oracle_cfg(o, om), o.OmCfg.default()
    env = mcn.BatchedCrowdSim(E, H, robot_kinematics=kin)
    pol = mcn.BatchedSARL(precision="f32", kinematics=kin, **NOGS, **(OM_KW if om else {}))
    assert pol.n_params == w.size
    pol.load_weights(w)
    env.set_state(_scenes(o, E, H))
    for step in range(3):
        env.orca()
        hv = env.human_actions()
        cur, times = env.get_state()
        theta = env.get_theta() if kin else np.zeros(E)
        pol.lookahead(env, query_env=query_env)
        best, values = pol.read(env)
        ovals = []
        for e in range(E):
            if om:
                _, ov, _ = o.lookahead_om(ecfg, scfg, omc, wo, cur[e], times[e], pol.action_table, query_env, hv[e],
                                          kinematics=kin, theta=theta[e])
            else:
                _, ov, _ = o.lookahead(ecfg, scfg, wo, cur[e], times[e], pol.action_table, query_env, hv[e], kinematics=kin,
                                       theta=theta[e])
            assert value_errors(values[e], ov, "f32") <= 1.0, (step, e)
            ovals.append(ov)
        ovals = np.stack(ovals)
        regret = ovals.max(axis=1) - ovals[np.arange(E), best]
        assert np.all(regret <= TIE_GAP["f32"]), regret.max()
        reward, done, info, _ = env.step(update=True)
        for e in range(E):
            r, d, i, _ = o.step_outcome(ecfg, cur[e], times[e], pol.action_table[best[e]], kin, theta[e])
            assert (reward[e], bool(done[e]), int(info[e])) == (r, bool(d), int(i)), (step, e)
    env.close(); pol.close()


# ---- GPU: tensor-core lookahead ------------------------------------------------------------------------------------------
def _tc_pair(mcn, om, **kw):
    cfg = dict(NOGS, **(OM_KW if om else {}), **kw)
    w = trained_weights(13 + (OM_DIM if om else 0))
    p32, p16 = mcn.BatchedSARL(precision="f32", **cfg), mcn.BatchedSARL(precision="f16_tc", **cfg)
    p32.load_weights(w); p16.load_weights(w)
    return p32, p16, w


def _tc_vs_f32(p32, p16, env, query_env=0):
    p32.lookahead(env, query_env); b32, v32 = p32.read(env)
    p16.lookahead(env, query_env); b16, v16 = p16.read(env)
    assert v16.shape == v32.shape
    assert value_errors(v16, v32, "f16_tc") <= 1.0
    regret = v32.max(axis=1) - v32[np.arange(len(b16)), b16]
    assert np.all(regret <= TIE_GAP["f16_tc"]), regret.max()
    return b32, v32, b16, v16


@pytest.mark.gpu
@pytest.mark.parametrize("om", [0, 1])
@pytest.mark.parametrize("E,H,speeds,rots", [(1000, 4, 3, 8), (777, 6, 5, 16), (130, 13, 2, 5)])
def test_tc_matches_f32_odd_shapes(gpu, E, H, speeds, rots, om):
    """Sizes that divide nothing (env count, humans per group, action count) on evolving auto-reset states: the tensor-core
    values against the FP32 path (itself pinned to the oracle above), and the argmax on the decidable states."""
    mcn = gpu
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=5, sim_rule=1)
    p32, p16, _ = _tc_pair(mcn, om, speed_samples=speeds, rotation_samples=rots)
    assert p16.A == speeds * rots + 1
    env.reset_device()
    b32s, v32s, b16s = [], [], []
    for step in range(4):
        env.orca()
        b32, v32, b16, _ = _tc_vs_f32(p32, p16, env)
        b32s.append(b32); v32s.append(v32); b16s.append(b16)
        env.step(update=True, read=False)
    check_argmax(np.concatenate(b16s), np.concatenate(b32s), np.concatenate(v32s), "f16_tc", min_decidable=E // 4)
    env.close(); p32.close(); p16.close()


@pytest.mark.gpu
@pytest.mark.parametrize("om", [0, 1])
@pytest.mark.parametrize("E,H", [(8192, 5), (8192, 10), (4096, 50)])
def test_tc_at_benchmark_sizes(gpu, oracle_mod, E, H, om):
    """The compile-time-H row kernels (5, 10 humans) and the run-time-H one (50 humans) at benchmark sizes: against FP32 on
    every env, against the oracle on a sample."""
    o, mcn = oracle_mod, gpu
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=13, sim_rule=1 if H == 50 else 0)
    p32, p16, w = _tc_pair(mcn, om)
    env.reset_device()
    for _ in range(6):                      # evolved states, not only fresh scenes
        env.orca()
        env.robot_orca(0.0)
        env.step(update=True, read=False)
    env.orca()
    b32, v32, b16, v16 = _tc_vs_f32(p32, p16, env)
    check_argmax(b16, b32, v32, "f16_tc", min_decidable=E // 4)
    ecfg, scfg, omc = o.EnvCfg.default(), _oracle_cfg(o, om), o.OmCfg.default()
    wo = oracle_layout(w, 13 + (OM_DIM if om else 0))
    cur, times = env.get_state()
    hv = env.human_actions()
    for e in np.random.default_rng(E + H).choice(E, 12 if H == 50 else 32, replace=False):
        if om:
            _, ov, _ = o.lookahead_om(ecfg, scfg, omc, wo, cur[e], times[e], p16.action_table, False, hv[e])
        else:
            _, ov, _ = o.lookahead(ecfg, scfg, wo, cur[e], times[e], p16.action_table, False, hv[e])
        assert value_errors(v32[e], ov, "f32") <= 1.0, e
        assert value_errors(v16[e], ov, "f16_tc") <= 1.0, e
        assert ov.max() - ov[b16[e]] <= TIE_GAP["f16_tc"], e
    env.close(); p32.close(); p16.close()


# ---- GPU: TD-target forward and the fused trainer ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("wset", ["seed", "trained"])
@pytest.mark.parametrize("H", [1, 5])
def test_policy_forward_vs_torch(gpu, oracle_mod, H, wset):
    """cn_policy_forward (TD targets) against the torch module on a random batch of 100, 1e-5 relative."""
    import torch
    w = WSETS[wset]()
    x = torch.from_numpy(_random_rows(oracle_mod, np.random.default_rng(100 + H), 100, H))
    with torch.no_grad():
        ref = _load(_net(), w)(x).numpy().reshape(-1)
    pol = gpu.BatchedSARL(precision="f32", **NOGS)
    pol.load_weights(w)
    got = pol.forward(x.cuda()).cpu().numpy()
    assert value_errors(got, ref, "f32") <= 1.0
    pol.close()


def _memory(mcn, o, dev, n=600, H=5):
    import torch
    rng = np.random.default_rng(1)
    memory = mcn.ReplayMemory(100000, device=dev)
    states = torch.from_numpy(_random_rows(o, rng, n, H)).to(dev)
    values = torch.from_numpy(rng.uniform(-0.25, 1.0, (n, 1)).astype(np.float32)).to(dev)
    memory.push_batch(states, values)
    return memory


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fused", "graph"])
def test_trainer_matches_eager_sgd(gpu, oracle_mod, mode):
    """Trainer(mode) against Trainer(mode="eager") (torch SGD with momentum): 100 steps on the same batches from the same
    start weights after one set_learning_rate, weights within 1e-5; and one fused step's gradient against autograd."""
    import torch
    from modelcrowdnav_b200.trainer import Trainer
    mcn, dev = gpu, torch.device("cuda:0")
    memory = _memory(mcn, oracle_mod, dev)
    w0 = trained_weights()
    idx = torch.randint(len(memory), (100, 100), generator=torch.Generator().manual_seed(2)).to(dev)
    out = {}
    for m in ("eager", mode):
        model = _load(_net(), w0).to(dev)
        tr = Trainer(model, memory, dev, 100, mode=m)
        tr.set_learning_rate(0.01)
        for i in range(idx.shape[0]):
            tr._step(idx[i])
        tr._after()
        out[m] = _flat(model)
    assert np.max(np.abs(out[mode] - out["eager"])) <= 1e-5, np.max(np.abs(out[mode] - out["eager"]))
    assert np.max(np.abs(out["eager"] - w0)) > 1e-3                    # the steps moved the weights
    if mode != "fused":
        return
    from modelcrowdnav_b200._capi import check
    from modelcrowdnav_b200.fused_trainer import FusedSarlTrainer
    model = _load(_net(), w0).to(dev)
    x, y = memory.states[idx[0]].contiguous(), memory.values[idx[0]].contiguous()
    torch.nn.functional.mse_loss(model(x), y).backward()
    ref = torch.cat([p.grad.reshape(-1) for p in model.parameters()]).cpu().numpy()
    ft = FusedSarlTrainer(model, dev)
    assert ft.cfg.without_global_state == 1
    ft.sync_from_model()
    loss = torch.zeros((), device=dev)
    check(ft.lib.cn_trainer_step(ft.handle, C.c_void_p(ft.flat.data_ptr()), C.c_void_p(x.data_ptr()),
                                 C.c_void_p(y.reshape(-1).contiguous().data_ptr()), x.shape[0], x.shape[1], 0.01, 0.9,
                                 C.c_void_p(ft.grad.data_ptr()), C.c_void_p(loss.data_ptr()), None))
    torch.cuda.synchronize()
    got = ft.grad.cpu().numpy()
    assert got.size == ref.size == 86502
    assert np.max(np.abs(got - ref)) <= 2e-5 * np.abs(ref).max(), (np.max(np.abs(got - ref)), np.abs(ref).max())
    ft.close()


# ---- GPU: pipelined rollout, CUDA graphs ---------------------------------------------------------------------------------
@pytest.mark.gpu
def test_pipelined_rollout_and_graph_capture(gpu):
    """PipelinedHostRollout (2 shards, CUDA graphs) returns bit for bit what the single device-resident handle computes over
    20 auto-reset steps; cn_rollout_step captured into a CUDA graph walks the same trajectory as eager launches."""
    import torch
    mcn = gpu
    E, H = 256, 5
    w = trained_weights()
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=3)
    pol = mcn.BatchedSARL(precision="f16_tc", **NOGS); pol.load_weights(w)
    env.reset_device()
    pipe = mcn.PipelinedHostRollout(E, H, w, shards=2, precision="f16_tc", auto_reset=1, seed=3, policy_cfg=dict(NOGS),
                                    use_graphs=True)
    pipe.reset_device()
    for _ in range(20):
        mcn.rollout_step(pol, env)
        pipe.step()
    pipe.sync()
    sa, ta = env.get_state()
    r, d, i, _ = env.read_outputs()
    agents, times, reward, action_idx, done, info = pipe.results()
    assert np.array_equal(sa, agents) and np.array_equal(ta, times)
    assert np.array_equal(r, reward) and np.array_equal(d, done) and np.array_equal(i, info)
    pipe.close(); env.close(); pol.close()

    E = 512
    envs = [mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=9) for _ in range(2)]
    pols = [mcn.BatchedSARL(precision="f16_tc", **NOGS) for _ in range(2)]
    for p in pols:
        p.load_weights(w)
    for e in envs:
        e.reset_device()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            mcn.rollout_step(pols[1], envs[1], stream=side.cuda_stream)
    side.synchronize()
    for _ in range(3):
        mcn.rollout_step(pols[0], envs[0])
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        mcn.rollout_step(pols[1], envs[1], stream=torch.cuda.current_stream().cuda_stream)
    mcn.rollout_step(pols[0], envs[0])
    for _ in range(40):
        graph.replay()
    torch.cuda.synchronize()
    for _ in range(39):
        mcn.rollout_step(pols[0], envs[0])
    a0, t0 = envs[0].get_state()
    a1, t1 = envs[1].get_state()
    assert np.array_equal(a0, a1) and np.array_equal(t0, t1)
    for x in envs + pols:
        x.close()


# ---- GPU: the reference-facing façade ------------------------------------------------------------------------------------
def _facade(w, precision):
    """env, robot, SARL (with_global_state = false), explorer wired as crowd_nav/test.py:52-87 does."""
    import torch
    import modelcrowdnav_b200 as mcn
    from test_gpu_facade import ENV_INI, POLICY_INI, _cfg
    policy = mcn.policy_factory["sarl"]()
    policy.configure(_cfg(POLICY_INI, sarl__with_global_state="false"))
    policy.precision = precision
    _load(policy.get_model(), w)
    env = mcn.CrowdSim()
    env.configure(_cfg(ENV_INI))
    robot = mcn.Robot(_cfg(ENV_INI), "robot")
    robot.set_policy(policy)
    env.set_robot(robot)
    device = torch.device("cuda:0")
    explorer = mcn.Explorer(env, robot, device, gamma=0.9)
    policy.set_phase("test")
    policy.set_device(device)
    policy.set_env(env)
    return env, policy, explorer


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f16_tc"])
def test_facade_episodes(gpu, oracle_mod, precision):
    """run_k_episodes on 20 test cases: at f32 the per-episode outcomes equal an oracle-driven roll-out of the same cases;
    at f16_tc the episodes run to completion."""
    o = oracle_mod
    w = trained_weights()
    env, policy, explorer = _facade(w, precision)
    explorer.run_k_episodes(20, "test")
    run = explorer.last_run
    cases = [int(c) for c in run["cases"]]
    assert len(cases) == 20 and np.all(np.isin(run["info"], (2, 3, 4)))
    if precision != "f32":
        return
    agents = np.ascontiguousarray(np.stack([o.generate_scene("test", c, human_num=5) for c in cases]))
    times, done = np.zeros(20), np.zeros(20, np.uint8)
    info, steps = np.zeros(20, np.int64), np.zeros(20, np.int64)
    actions = o.action_space()
    for t in range(200):
        before = done.copy()
        _, _, inf = o.batch_lookahead_step(o.EnvCfg.default(), o.SarlCfg.default(), oracle_layout(w), agents, times, actions,
                                           False, done)
        new = (done != 0) & (before == 0)
        info[new], steps[new] = inf[new], t + 1
        if done.all():
            break
    assert done.all()
    assert np.array_equal(run["info"], info), (run["info"], info)
    assert np.array_equal(run["steps"], steps), (run["steps"], steps)
