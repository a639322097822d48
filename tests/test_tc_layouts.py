"""Human-count layouts of the tensor-core CADRL / LSTM-RL lookaheads and of the world-model kernels.

Tensor cores (CN_PREC_F16_TC, the default for both networks): cn_lookahead_tc packs G = min(64, 128 // H) groups of
(env, action) rows into each 128-row X tile.  CADRL runs its whole network on those tiles (tc_mlp3_pair_kernel<1>) and
cadrl_min_kernel finds a group's rows at (g / G) * 128 + (g % G) * H; LSTM-RL writes H X_t tiles per (env, action) tile
(tc_features_lstm_kernel) and runs H dependent UMMA stages per tile (tc_lstm_pair_kernel: no W_hh product on a tile's first
step, h_n into J on its last).  HS reaches every G transition and both ends of the range:

    H   1   2   3   7   8   32  33  42  43  50  64
    G   64  64  42  18  16  4   3   3   2   2   2

World models (csrc/world_model.cu): attention_world_kernel packs 32 // H envs per CTA (one env per CTA from 17 humans on,
refused above 32), mlp_world_kernel 16 envs per CTA with an input width of 4H; both leave frozen envs alone.  The reference
for them is a float64 numpy transcription of world_model.py:20-106, itself pinned to the reference's own outputs on the CPU.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import MODEL_WORLD_NAMES, TIE_GAP, check_argmax, load_model_world, value_errors
from test_network_shapes import random_agents, scaled_errors

HS = (1, 2, 3, 7, 8, 32, 33, 42, 43, 50, 64)
NETS = ("cadrl", "lstm")
# The scaled weight sets: every parameter times the factor of test_network_shapes.weights (CADRL x4, LSTM-RL x2), which spreads
# the 81 values of a state, then the output Linear divided by X_OUT so that the values come back to the reward scale on which
# the fp16 bars of conftest.py are absolute (|dv| <= 1e-3).  Without that division CADRL's values reach ~50 and the fp16
# rounding of its weights alone moves them by 0.02 - 0.04 (measured on the B200 and reproduced by the oracle with fp16 weights);
# LSTM-RL's mlp runs on 16x the activations the bar was measured with and misses it by up to 15 % at any H from 3 to 64, of
# which the fp16 W_ih / W_hh contribute at most 1.7e-4 even over 64 recurrent steps (the mlp weights alone 8e-4).
X_SCALE = {"cadrl": 4.0, "lstm": 2.0}
X_OUT = {"cadrl": 256.0, "lstm": 4.0}


@pytest.fixture(scope="module")
def mcn():
    import modelcrowdnav_b200 as m
    assert m._capi.load().cn_device_count() > 0, "GPU tests need a CUDA device"
    return m


def _net_kw(net):
    """BatchedSARL arguments of the reference's [cadrl] / [lstm_rl] (ValueNetwork1) networks"""
    if net == "cadrl":
        return dict(network="cadrl", mlp3_dims=[150, 100, 100, 1])
    return dict(network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50)


def _net_weights(units_nets, net, wset):
    """the reference's seeded init (tests/golden/units_nets.npz) or its scaled set; the output Linear (value_network.6 /
    mlp.6, 100 weights and a bias) follows the three hidden Linears of 13 (CADRL) or 6 + 50 (LSTM-RL) inputs"""
    w = units_nets[net + "_weights"]
    if wset == "seed":
        return w
    w = (w * np.float32(X_SCALE[net])).astype(np.float32)
    out = (13 if net == "cadrl" else 56) * 150 + 150 + 150 * 100 + 100 + 100 * 100 + 100
    w[out:out + 101] /= np.float32(X_OUT[net])
    return w


def _ocfg(o, net):
    return o.NetCfg.cadrl() if net == "cadrl" else o.NetCfg.lstm_rl()


def _scenes(o, n, H, randomize=False, start=0):
    rule, width = ("circle_crossing", 10.0) if H <= 10 else ("square_crossing", 16.0)
    return np.stack([o.generate_scene("val", start + c, human_num=H, rule=rule, square_width=width, randomize=randomize)
                     for c in range(n)])


# ---- A1: tensor cores against the oracle at every layout ---------------------------------------------------------------------
def _oracle_cases():
    """(net, H, E, weight set, kinematics, randomize): every H with 1, 2 and 5 envs and both weight sets (query_env with 2
    envs), plus a unicycle robot and heterogeneous humans (randomize_attributes) per network"""
    cases = [pytest.param(net, H, E, ws, 0, False, id="%s-H%d-E%d-%s" % (net, H, E, ws))
             for net in NETS for H in HS for E in (1, 2, 5) for ws in ("seed", "scaled")]
    for net in NETS:
        cases.append(pytest.param(net, 43, 5, "scaled", 1, False, id="%s-H43-E5-scaled-unicycle" % net))
        cases.append(pytest.param(net, 7, 5, "scaled", 0, True, id="%s-H7-E5-scaled-random" % net))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("net,H,E,wset,kin,randomize", _oracle_cases())
def test_tc_lookahead_vs_oracle(mcn, oracle_mod, units_nets, net, H, E, wset, kin, randomize):
    """The tensor-core lookahead over three evolving steps against oracle.lookahead_net: the fp16 value bars on every state,
    the chosen action optimal up to the fp16 tie gap, the argmax bar, and the step that follows (reward / done / info) exact."""
    o = oracle_mod
    query_env = int(E == 2)
    w = _net_weights(units_nets, net, wset)
    ncfg, ecfg = _ocfg(o, net), o.EnvCfg.default()
    env = mcn.BatchedCrowdSim(E, H, robot_kinematics=kin)
    pol = mcn.BatchedSARL(precision="f16_tc", kinematics=kin, **_net_kw(net))
    assert pol.n_params == w.size
    pol.load_weights(w)
    env.set_state(_scenes(o, E, H, randomize))
    alive = np.ones(E, bool)                # a finished env is frozen: the lookahead leaves its values alone
    bests, obests, ovs = [], [], []
    worst = 0.0
    for step in range(3):
        env.orca()
        hv = env.human_actions()
        cur, times = env.get_state()
        theta = env.get_theta() if kin else np.zeros(E)
        pol.lookahead(env, query_env=query_env)
        best, values = pol.read(env)
        live = np.flatnonzero(alive)
        ref = [o.lookahead_net(ecfg, ncfg, w, cur[e], times[e], pol.action_table, query_env, hv[e], kinematics=kin,
                               theta=theta[e]) for e in live]
        ovals = np.stack([r[1] for r in ref])
        for k, e in enumerate(live):
            err = value_errors(values[e], ovals[k], "f16_tc")
            worst = max(worst, err)
            assert err <= 1.0, (step, e, np.abs(values[e] - ovals[k]).max())
        regret = ovals.max(axis=1) - ovals[np.arange(len(live)), best[live]]
        assert np.all(regret <= TIE_GAP["f16_tc"]), (step, regret.max())
        bests.append(best[live]); obests.append([r[0] for r in ref]); ovs.append(ovals)
        reward, done, info, _ = env.step(update=True)
        for e in live:
            r, d, i, _ = o.step_outcome(ecfg, cur[e], times[e], pol.action_table[best[e]], kin, theta[e])
            assert (reward[e], bool(done[e]), int(info[e])) == (r, bool(d), int(i)), (step, e)
        alive &= ~done.astype(bool)
        if not alive.any():
            break
    n = sum(len(b) for b in bests)
    # at least one decidable state; a single env's three states can all be ties (LSTM-RL's scaled set at 2 and 3 humans), where
    # the regret bar above still holds every choice to the oracle's optimum
    agree, total = check_argmax(np.concatenate(bests), np.concatenate(obests), np.concatenate(ovs), "f16_tc",
                                min_decidable=1 if E > 1 else 0)
    print("tc-vs-oracle %s H=%d E=%d %s: worst value_errors %.3f, %d / %d decidable states agree (of %d)" % (
        net, H, E, wset, worst, agree, total, n))
    env.close(); pol.close()


# ---- A3: BASELINE's sizes ------------------------------------------------------------------------------------------------------
# BASELINE.json configs[1], [2] (per GPU) and [4]: (envs, humans, sim rule, query_env, oracle sample size)
SIZES = [(8192, 5, 0, 0, 512), (8192, 10, 1, 1, 512), (4096, 50, 1, 0, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("net", NETS)
@pytest.mark.parametrize("E,H,rule,query_env,n_sample", SIZES)
def test_tc_benchmark_sizes_vs_oracle(mcn, oracle_mod, units_nets, net, E, H, rule, query_env, n_sample):
    """CADRL and LSTM-RL at BASELINE's configurations after three evolved steps: tensor cores against FP32 on every env,
    both against the oracle on a random sample, and the step that follows exact on the sample."""
    o = oracle_mod
    w = units_nets[net + "_weights"]
    ncfg, ecfg = _ocfg(o, net), o.EnvCfg.default()
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=11, sim_rule=rule)
    p16 = mcn.BatchedSARL(precision="f16_tc", **_net_kw(net))
    p32 = mcn.BatchedSARL(precision="f32", **_net_kw(net))
    p16.load_weights(w); p32.load_weights(w)
    env.reset_device()
    for _ in range(3):
        mcn.rollout_step(p16, env, query_env)
    state, times = env.get_state()
    env.orca()
    hv = env.human_actions()
    p32.lookahead(env, query_env); b32, v32 = p32.read(env)
    p16.lookahead(env, query_env); b16, v16 = p16.read(env)
    # (1) every env: tensor cores against FP32
    worst = value_errors(v16, v32, "f16_tc")
    assert worst <= 1.0, np.abs(v16 - v32).max()
    regret = v32.max(axis=1) - v32[np.arange(E), b16]
    assert np.all(regret <= TIE_GAP["f16_tc"]), regret.max()
    agree, total = check_argmax(b16, b32, v32, "f16_tc", min_decidable=E // 4)      # measured 47 - 82 %
    # (2) a random sample against the oracle, both precisions
    sample = np.sort(np.random.RandomState(E + H).choice(E, n_sample, replace=False))
    ref = [o.lookahead_net(ecfg, ncfg, w, state[e], times[e], p16.action_table, query_env, hv[e]) for e in sample]
    ov = np.stack([r[1] for r in ref])
    assert value_errors(v32[sample], ov, "f32") <= 1.0
    assert value_errors(v16[sample], ov, "f16_tc") <= 1.0
    for b, prec in ((b32, "f32"), (b16, "f16_tc")):
        assert np.all(ov.max(axis=1) - ov[np.arange(n_sample), b[sample]] <= TIE_GAP[prec]), prec
        check_argmax(b[sample], [r[0] for r in ref], ov, prec, min_decidable=n_sample // 4)
    # (3) the step that follows (the tensor-core path's pending actions) on the sample
    reward, done, info, _ = env.step(update=True)
    for e in sample:
        r, d, i, _ = o.step_outcome(ecfg, state[e], times[e], p16.action_table[b16[e]])
        assert (reward[e], bool(done[e]), int(info[e])) == (r, bool(d), int(i)), e
    print("tc-benchmark %s E=%d H=%d: worst value_errors vs f32 %.3f, %d / %d decidable states agree" % (
        net, E, H, worst, agree, total))
    env.close(); p16.close(); p32.close()


# ---- B1: the world models in float64 (CPU) -------------------------------------------------------------------------------------
def _lin(p, name, x):
    return x @ p[name + ".weight"].T + p[name + ".bias"]


def _relu(x):
    return np.maximum(x, 0.0)


def attention_world_ref(p, x):
    """AttentionWorld.forward (world_model.py:53-106) in float64: x (B, H, 4) -> (B, H, 2).  ReLU after every hidden Linear,
    none after mlp2.2, the score or the output; the reference's masked softmax exp(s) * (s != 0) without max subtraction;
    mlp3 on [state_i | the env's attention-weighted feature]."""
    e = _relu(_lin(p, "mlp1.2", _relu(_lin(p, "mlp1.0", x))))
    f = _lin(p, "mlp2.2", _relu(_lin(p, "mlp2.0", e)))
    u = np.concatenate([e, np.broadcast_to(e.mean(axis=1, keepdims=True), e.shape)], axis=-1)
    s = _lin(p, "attention.4", _relu(_lin(p, "attention.2", _relu(_lin(p, "attention.0", u)))))[..., 0]
    ex = np.exp(s) * (s != 0)
    wgt = ex / ex.sum(axis=1, keepdims=True)
    feat = np.einsum("bh,bhk->bk", wgt, f)
    j = np.concatenate([x, np.broadcast_to(feat[:, None, :], f.shape)], axis=-1)
    g = _relu(_lin(p, "mlp3.4", _relu(_lin(p, "mlp3.2", _relu(_lin(p, "mlp3.0", j))))))
    return _lin(p, "mlp3.6", g)


def mlp_world_ref(p, x):
    """MlpWorld.forward (world_model.py:20-50) in float64, dropout the identity: x (B, H * 4) -> (B, H * 2)"""
    h = _relu(_lin(p, "mlp.6", _relu(_lin(p, "mlp.3", _relu(_lin(p, "mlp.0", x))))))
    return np.tanh(_lin(p, "mlp.8", h))


def world_ref(world, x):
    """float64 prediction of a world-model container for human states x (B, H, 4) (cast to float32 first, as the reference's
    torch.Tensor and the kernel do): (B, H, 2)"""
    p = {k: v.detach().cpu().double().numpy() for k, v in world.state_dict().items()}
    x = np.asarray(x, np.float32).astype(np.float64)
    B, H = x.shape[:2]
    if type(world).__name__ == "MlpWorld":
        return mlp_world_ref(p, x.reshape(B, H * 4)).reshape(B, H, 2)
    return attention_world_ref(p, x)


def _golden_world(g):
    import torch
    from modelcrowdnav_b200.world_model import AttentionWorld, MlpWorld
    world = MlpWorld(int(g["H"])) if str(g["world"]) == "mlp" else AttentionWorld()
    off, new = 0, {}
    for k, v in world.state_dict().items():
        new[k] = torch.from_numpy(g["world_weights"][off:off + v.numel()].reshape(tuple(v.shape)).copy())
        off += v.numel()
    world.load_state_dict(new)
    return world


@pytest.mark.parametrize("name", MODEL_WORLD_NAMES)
def test_world_transcription_matches_reference(name):
    """The float64 transcriptions above reproduce the velocities the REFERENCE's AttentionWorld / MlpWorld predicted on every
    recorded step (tests/golden/model_world_*.npz) within the bar the kernel is held to there (2e-6)."""
    g = load_model_world(name)
    T = len(g["reward"])
    x = np.stack([g["agents"][t][1:, :4] for t in range(T)])
    got = world_ref(_golden_world(g), x)
    assert np.max(np.abs(got - g["new_v"][:T])) <= 2e-6, np.max(np.abs(got - g["new_v"][:T]))


# ---- B2: the world-model kernels at every layout (GPU) -------------------------------------------------------------------------
# the scaled sets: AttentionWorld x3 (its scores then reach ~17, far from the float32 overflow of exp at 88); MlpWorld x2 --
# at x3 its tanh-bounded outputs come from pre-activations of several hundred, where torch's own float32 forward is 9.4e-6 off
# at 64 humans, at the 1e-5 bar
W_SCALE = {"attention": 3.0, "mlp": 2.0}


def _world(kind, H, wset):
    """seeded default init (torch.manual_seed(H)) or the same times W_SCALE"""
    import torch
    from modelcrowdnav_b200.world_model import AttentionWorld, MlpWorld
    torch.manual_seed(H)
    world = MlpWorld(H) if kind == "mlp" else AttentionWorld()
    if wset == "scaled":
        with torch.no_grad():
            for prm in world.parameters():
                prm.mul_(W_SCALE[kind])
    return world


def _world_errors(got, ref, wset):
    """every value within 1e-5 * max(|v|, 0.1) for the seeded weights.  The scaled AttentionWorld gives velocities of up to
    ~50 from hidden activations of several hundred, where float32 itself (numpy's float32 forward on the same inputs) is off
    by up to 17x that per-value bar on the components near zero: there the bar is 1e-5 of the largest |value| compared
    (test_network_shapes.scaled_errors, the bar of every scaled-weight FP32 comparison)."""
    return scaled_errors(got, ref, 1.0 if wset == "seed" else wset)


def _world_cases():
    cases = []
    for H in (1, 2, 3, 7, 11, 16, 17, 31, 32):
        epc = max(1, 32 // H)
        for E in (1, 3 * epc + 1):
            cases += [pytest.param("attention", H, E, ws, id="attention-H%d-E%d-%s" % (H, E, ws)) for ws in ("seed", "scaled")]
    for H in (1, 7, 33, 64):
        for E in (1, 17, 1000):
            cases += [pytest.param("mlp", H, E, ws, id="mlp-H%d-E%d-%s" % (H, E, ws)) for ws in ("seed", "scaled")]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("kind,H,E,wset", _world_cases())
def test_world_kernel_vs_float64(mcn, kind, H, E, wset):
    """world.predict_into(env) and world(x) against the float64 transcription: AttentionWorld from 32 envs per CTA (H = 1)
    through H that do not divide 32 to one env per CTA (17 .. 32), with a partial last CTA; MlpWorld up to 64 humans
    (input width 256) with 1, 17 (a partial second CTA) and 1000 envs."""
    import torch
    world = _world(kind, H, wset)
    rng = np.random.default_rng(1000 * H + E)
    agents = np.stack([random_agents(rng, H) for _ in range(E)])
    ref = world_ref(world, agents[:, 1:, :4])
    env = mcn.BatchedCrowdSim(E, H)
    env.set_state(agents)
    world.predict_into(env)
    got = env.human_actions()
    err = _world_errors(got, ref, wset)
    assert err <= 1.0, (err, np.abs(got - ref).max())
    x = torch.tensor(agents[:, 1:, :4].reshape(E, H * 4), dtype=torch.float32, device="cuda")
    out = world(x).cpu().numpy().reshape(E, H, 2)
    assert _world_errors(out, ref, wset) <= 1.0
    print("world %s H=%d E=%d %s: max |dv| %.3g (bar ratio %.3f, max |v| %.3g)" % (
        kind, H, E, wset, np.abs(got - ref).max(), err, np.abs(ref).max()))
    env.close()


# ---- B3: edges -----------------------------------------------------------------------------------------------------------------
def _masking_world():
    """AttentionWorld with hand-set weights, all biases zero: score_i = relu(px_i) (px -> mlp1.0 -> mlp1.2 -> attention.0's
    e_i half -> attention.2 -> attention.4, unit weights on one lane each), feature_i = py_i (mlp1.0 lane 1 -> mlp1.2 ->
    mlp2.0 -> mlp2.2), and every human's predicted vx = the env's attention-weighted sum of py (mlp3.0 on the feature column
    -> mlp3.2 -> mlp3.4 -> mlp3.6 row 0); vy = 0."""
    import torch
    from modelcrowdnav_b200.world_model import AttentionWorld
    world = AttentionWorld()
    sd = {k: torch.zeros_like(v) for k, v in world.state_dict().items()}
    sd["mlp1.0.weight"][0, 0] = 1.0; sd["mlp1.0.weight"][1, 1] = 1.0
    sd["mlp1.2.weight"][0, 0] = 1.0; sd["mlp1.2.weight"][1, 1] = 1.0
    sd["attention.0.weight"][0, 0] = 1.0
    sd["attention.2.weight"][0, 0] = 1.0
    sd["attention.4.weight"][0, 0] = 1.0
    sd["mlp2.0.weight"][0, 1] = 1.0
    sd["mlp2.2.weight"][0, 0] = 1.0
    sd["mlp3.0.weight"][0, 4] = 1.0
    sd["mlp3.2.weight"][0, 0] = 1.0
    sd["mlp3.4.weight"][0, 0] = 1.0
    sd["mlp3.6.weight"][0, 0] = 1.0
    world.load_state_dict(sd)
    return world


@pytest.mark.gpu
def test_world_masked_softmax_exact_zero_scores(mcn):
    """The reference's softmax weighs a human by exp(s) * (s != 0): a human whose score is exactly 0 gets weight exactly 0,
    not exp(0) / z.  Scores relu(px) are 0 for the humans at px <= 0; they stand at py = 1000, so any weight they received
    would show in vx = sum_i w_i py_i.  Envs of 1 to 32 humans, every one with at least one human at px > 0."""
    world = _masking_world()
    rng = np.random.default_rng(5)
    for H in (2, 3, 7, 17, 32):
        E = 2 * max(1, 32 // H) + 1
        agents = np.stack([random_agents(rng, H) for _ in range(E)])
        agents[:, 1:, 0] = rng.uniform(0.5, 2.0, (E, H)) * rng.choice([-1.0, 1.0], (E, H))
        agents[:, 1:, 0][rng.random((E, H)) < 0.2] = 0.0                   # score relu(0) = 0 as well
        agents[:, 1, 0] = 1.5                                              # never all masked (z = 0)
        agents[:, 1:, 1] = np.where(agents[:, 1:, 0] > 0, rng.uniform(0.5, 2.0, (E, H)), 1000.0)
        px, py = agents[:, 1:, 0].astype(np.float32), agents[:, 1:, 1].astype(np.float32).astype(np.float64)
        ex = np.where(px > 0, np.exp(np.maximum(px, 0).astype(np.float64)), 0.0)
        want = (ex * py).sum(axis=1) / ex.sum(axis=1)
        ref = world_ref(world, agents[:, 1:, :4])
        assert np.allclose(ref[:, :, 0], want[:, None], rtol=1e-12, atol=0) and np.all(ref[:, :, 1] == 0)
        assert np.all(want < 2.0)                                          # no weight on a py = 1000 human
        env = mcn.BatchedCrowdSim(E, H)
        env.set_state(agents)
        world.predict_into(env)
        got = env.human_actions()
        assert value_errors(got, ref, "f32") <= 1.0, (H, np.abs(got - ref).max())
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,H", [("attention", 5), ("attention", 20), ("mlp", 3), ("mlp", 40)])
def test_world_predict_skips_frozen_envs(mcn, oracle_mod, kind, H):
    """Envs that finished an episode (auto_reset off: a collision on the first step) are frozen: after predict_into they
    still hold the velocities written before it, and every other env holds the prediction."""
    o = oracle_mod
    E = 40
    world = _world(kind, H, "seed")
    rule = "circle_crossing" if H <= 5 else "square_crossing"
    agents = np.stack([o.generate_scene("test", c, human_num=H, rule=rule, square_width=16.0) for c in range(E)])
    hit = np.arange(E) % 3 == 1
    agents[hit, 1, :2] = agents[hit, 0, :2] + [0.5, 0.0]                    # human 1 overlaps the robot: Collision
    env = mcn.BatchedCrowdSim(E, H)
    env.set_state(agents)
    env.orca()
    _, done, info, _ = env.step(np.zeros((E, 2)), update=True)
    assert np.array_equal(done.astype(bool), hit) and np.all(info[hit] == o.COLLISION)
    frozen = env.episode_table()["frozen"].astype(bool)
    assert np.array_equal(frozen, hit)
    sentinel = np.full((E, H, 2), -123.25)
    env.set_human_actions(sentinel)
    world.predict_into(env)
    got = env.human_actions()
    cur, _ = env.get_state()
    ref = world_ref(world, cur[:, 1:, :4])
    assert np.all(got[frozen] == -123.25)
    assert value_errors(got[~frozen], ref[~frozen], "f32") <= 1.0
    env.close()


@pytest.mark.gpu
def test_world_refusals(mcn):
    """cn_world_predict refuses, with CN_EUNSUPPORTED / CN_EINVAL and a message, and writes nothing: AttentionWorld above
    32 humans, an MlpWorld built for another human count than the env's, and a model whose weights were never loaded."""
    from modelcrowdnav_b200 import _capi
    lib = _capi.load()

    def predict(kind, h_model, h_env, load=True):
        w = C.c_void_p()
        _capi.check(lib.cn_world_create(kind, h_model, 0, C.byref(w)))
        if load:
            flat = np.zeros(int(lib.cn_world_param_count(w)), np.float32)
            _capi.check(lib.cn_world_load_weights(w, flat.ctypes.data_as(C.c_void_p), flat.size, None))
        env = mcn.BatchedCrowdSim(3, h_env)
        env.set_human_actions(np.full((3, h_env, 2), 7.5))
        rc = lib.cn_world_predict(w, env.handle, None)
        msg = lib.cn_last_error()
        untouched = bool(np.all(env.human_actions() == 7.5))
        env.close()
        lib.cn_world_destroy(w)
        return rc, msg, untouched

    for args, code, text in (((_capi.WORLD_ATTENTION, 0, 33), _capi.CN_EUNSUPPORTED, b"32"),
                             ((_capi.WORLD_MLP, 5, 6), _capi.CN_EINVAL, b"5 humans"),
                             ((_capi.WORLD_MLP, 5, 5, False), _capi.CN_EINVAL, b"load_weights"),
                             ((_capi.WORLD_ATTENTION, 0, 5, False), _capi.CN_EINVAL, b"load_weights")):
        rc, msg, untouched = predict(*args)
        assert rc == code and msg and text in msg, (args, rc, msg)
        assert untouched, args
    ok = predict(_capi.WORLD_ATTENTION, 0, 32)                             # the largest AttentionWorld layout runs
    assert ok[0] == _capi.CN_OK and not ok[2]
