"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference goldens."""
import numpy as np
import pytest

from conftest import (TIE_GAP, TRAJ_NAMES, TRAJ_NAMES_KIN, TRAJ_NAMES_MIXED, TRAJ_NAMES_NETS, TRAJ_NAMES_OM, check_argmax,
                      load_traj, net_tag, value_errors, weights_for)

pytestmark = pytest.mark.gpu


def check_choice(best, ref_best, ref_values, precision, min_decidable=0):
    """The two argmax bars of every lookahead test.  (1) On the DECIDABLE states (reference top-2 gap above the tie
    threshold) the action index matches on >= 99.9 %, and there are at least `min_decidable` such states.  (2) On EVERY
    state, decidable or not, the chosen action is optimal under the REFERENCE's values up to the tie threshold -- never
    vacuous, even for random-init weights whose 81 values lie within 1e-4 of each other."""
    ref_values = np.asarray(ref_values, np.float64)
    best = np.asarray(best)
    check_argmax(best, ref_best, ref_values, precision, min_decidable)
    regret = ref_values.max(axis=1) - ref_values[np.arange(len(best)), best]
    assert np.all(regret <= TIE_GAP[precision]), "chosen action worse than the reference optimum by %.3g" % regret.max()


@pytest.fixture(scope="module")
def mcn():
    import modelcrowdnav_b200 as m
    assert m._capi.load().cn_device_count() > 0, "GPU tests need a CUDA device"
    return m


def _scenes(oracle_mod, n, H, rule="circle_crossing", phase="test", start=0):
    return np.stack([oracle_mod.generate_scene(phase, start + c, human_num=H, rule=rule) for c in range(n)])


@pytest.mark.parametrize("H,rule,visible", [(5, "circle_crossing", 0), (10, "square_crossing", 0),
                                            (5, "circle_crossing", 1), (20, "square_crossing", 0)])
def test_orca_and_step_bit_exact(mcn, oracle_mod, H, rule, visible):
    """ORCA velocities, reward/done/info codes and the updated state are bit-exact over 30 steps."""
    o = oracle_mod
    E = 96
    ecfg = o.EnvCfg.default(robot_visible=visible)
    env = mcn.BatchedCrowdSim(E, H, robot_visible=visible)
    agents = _scenes(o, E, H, rule)
    env.set_state(agents)
    rs = np.random.RandomState(0)
    table = o.action_space()
    times = np.zeros(E)
    infos = set()
    for step in range(30):
        env.orca()
        hv = env.human_actions()
        acts = table[rs.randint(0, 81, E)]
        reward, done, info, dmin = env.step(acts, update=True)
        got, gtimes = env.get_state()
        for e in range(E):
            if step > 0 and frozen[e]:
                continue
            ohv = o.human_actions(ecfg, agents[e])
            assert np.array_equal(ohv, hv[e]), (step, e)
            r, d, i, dm = o.step_outcome(ecfg, agents[e], times[e], acts[e])
            assert (r, d, i) == (reward[e], bool(done[e]), int(info[e])), (step, e)
            if i == o.DANGER:
                assert dm == dmin[e]
            times[e] = o.apply_step(ecfg, agents[e], times[e], acts[e], ohv)
            infos.add(i)
        frozen = done.astype(bool) if step == 0 else (frozen | done.astype(bool))
        live = ~frozen | done.astype(bool)
        assert np.array_equal(got[live], agents[live]) and np.array_equal(gtimes[live], times[live])
    assert {o.NOTHING, o.DANGER} <= infos
    env.close()


def test_step_ladder_edge_cases(mcn, oracle_mod):
    """Timeout > Collision > ReachGoal > Danger > Nothing priority, degenerate segment, update=False."""
    o = oracle_mod
    ecfg = o.EnvCfg.default()
    base = o.generate_scene("test", 0)
    cases, times, acts = [], [], []
    a = base.copy(); cases.append(a); times.append(24.0); acts.append([0.0, 1.0])                 # timeout
    a = base.copy(); a[1, :2] = a[0, :2] + [0.5, 0.0]; cases.append(a); times.append(0.0); acts.append([1.0, 0.0])  # collision
    a = base.copy(); a[0, :2] = [0.0, 3.9]; cases.append(a); times.append(3.0); acts.append([0.0, 0.4])  # reach goal
    a = base.copy(); a[1, :2] = a[0, :2] + [0.75, 0.0]; cases.append(a); times.append(0.0); acts.append([0.0, 0.0])  # danger, static
    a = base.copy(); a[0, :2] = [0.0, 3.9]; a[1, :2] = a[0, :2] + [0.3, 0]; cases.append(a); times.append(24.0); acts.append([0.0, 0.4])  # all at once
    a = base.copy(); cases.append(a); times.append(0.0); acts.append([0.0, 0.0])                  # nothing
    E = len(cases)
    env = mcn.BatchedCrowdSim(E, 5)
    agents = np.stack(cases); times = np.array(times); acts = np.array(acts)
    env.set_state(agents, times)
    env.orca()
    reward, done, info, dmin = env.step(acts, update=False)
    obs = env.next_obs()
    got, gt = env.get_state()
    assert np.array_equal(got, agents) and np.array_equal(gt, times)       # update=False does not mutate
    hv = env.human_actions()
    for e in range(E):
        r, d, i, dm = o.step_outcome(ecfg, agents[e], times[e], acts[e])
        assert (r, d, i) == (reward[e], bool(done[e]), int(info[e])), e
        # crowd_sim.py:428-430 / agent.py:63-74
        assert np.array_equal(obs[e, :, 0:2], agents[e, 1:, 0:2] + hv[e] * 0.25)
        assert np.array_equal(obs[e, :, 2:4], hv[e]) and np.array_equal(obs[e, :, 4], agents[e, 1:, 6])
    assert list(info) == [o.TIMEOUT, o.COLLISION, o.REACHGOAL, o.DANGER, o.TIMEOUT, o.NOTHING]
    env.close()


@pytest.mark.parametrize("precision", ["f32", "f16_tc"])
@pytest.mark.parametrize("name", TRAJ_NAMES + TRAJ_NAMES_MIXED)
def test_golden_trajectories(mcn, oracle_mod, weights0, name, precision):
    """Teacher-forced replay of the reference's own episodes (tests/golden, scripts/gen_golden.py)."""
    tr = load_traj(name)
    weights0 = weights_for(name)
    H = tr["H"]
    states, times, recs = [], [], []
    for case, rec in tr["cases"].items():
        for t in range(len(rec["time"])):
            states.append(rec["agents"][t]); times.append(rec["time"][t]); recs.append((rec, t))
    E = len(states)
    env = mcn.BatchedCrowdSim(E, H, robot_visible=tr["robot_visible"])
    pol = mcn.BatchedSARL(precision=precision)
    pol.load_weights(weights0)
    assert np.array_equal(pol.action_table, recs[0][0]["table"])            # bit-exact action table
    env.set_state(np.stack(states), np.array(times))
    env.orca()
    hv = env.human_actions()
    pol.lookahead(env, query_env=tr["query_env"])
    best, values = pol.read(env)
    # step with the REFERENCE's action so the state transition is compared like for like
    acts = np.stack([rec["action"][t] for rec, t in recs])
    reward, done, info, dmin = env.step(acts, update=True)
    got, gt = env.get_state()
    for e, (rec, t) in enumerate(recs):
        assert np.array_equal(hv[e], rec["human_v"][t]), (name, e)
        assert value_errors(values[e], rec["values"][t], precision) <= 1.0, (name, e)
        assert (reward[e], bool(done[e]), int(info[e])) == (rec["reward"][t], bool(rec["done"][t]), int(rec["info"][t]))
        if t + 1 < len(rec["time"]):
            assert np.array_equal(got[e], rec["agents"][t + 1]) and gt[e] == rec["time"][t + 1]
    ref_values = np.stack([rec["values"][t] for rec, t in recs])
    # the trained-weight fixtures must decide (>= 70 % of their states have a clear winner); seed-0 weights barely do
    check_choice(best, [rec["best"][t] for rec, t in recs], ref_values, precision,
                 min_decidable=int(0.7 * E) if name.endswith("trained") else 0)
    env.close(); pol.close()


@pytest.mark.parametrize("precision", ["f32", "f16_tc"])
@pytest.mark.parametrize("H,rule,query_env", [(5, "circle_crossing", 0), (5, "circle_crossing", 1),
                                              (10, "square_crossing", 0), (3, "circle_crossing", 0),
                                              (1, "circle_crossing", 0), (2, "circle_crossing", 1),
                                              (7, "square_crossing", 1), (20, "square_crossing", 0)])
def test_lookahead_vs_oracle(mcn, oracle_mod, weights0, H, rule, query_env, precision):
    """81 action values and the argmax against the oracle on evolving states (not only reset states)."""
    o = oracle_mod
    E = 48
    ecfg, scfg = o.EnvCfg.default(), o.SarlCfg.default()
    env = mcn.BatchedCrowdSim(E, H)
    pol = mcn.BatchedSARL(precision=precision)
    pol.load_weights(weights0)
    agents = _scenes(o, E, H, rule, phase="val")
    env.set_state(agents)
    for step in range(6):
        env.orca()
        pol.lookahead(env, query_env=query_env)
        best, values = pol.read(env)
        hv = env.human_actions()
        state, times = env.get_state()
        obests, ovalues = [], []
        for e in range(E):
            obest, ovals, reached = o.lookahead(ecfg, scfg, weights0, state[e], times[e], pol.action_table,
                                                query_env, hv[e])
            assert value_errors(values[e], ovals, precision) <= 1.0, (step, e)
            obests.append(obest); ovalues.append(ovals)
        check_choice(best, obests, np.stack(ovalues), precision)
        env.step(update=True, read=False)      # advance with the GPU's own chosen actions
    env.close(); pol.close()


def test_reach_destination_and_untrained(mcn, oracle_mod, weights0):
    """policy.py:43-49 early exit (action 0) and the all-NaN ValueError (multi_human_rl.py:57-58)."""
    o = oracle_mod
    agents = _scenes(o, 4, 5)
    agents[1, 0, :2] = [0.05, 3.9]            # robot already within its radius of the goal
    env = mcn.BatchedCrowdSim(4, 5)
    pol = mcn.BatchedSARL()
    pol.load_weights(weights0)
    env.set_state(agents)
    pol.lookahead(env)
    best, _ = pol.read(env)
    assert best[1] == 0
    w = weights0.copy(); w[-1] = np.nan       # mlp3.6.bias = NaN -> every value NaN
    pol.load_weights(w)
    pol.lookahead(env)
    with pytest.raises(mcn.CrowdNavError) as ei:
        pol.read(env)
    assert ei.value.code == mcn._capi.CN_EVALUE and "not well trained" in str(ei.value)
    env.close(); pol.close()


def test_transform_and_forward(mcn, oracle_mod, weights0, units):
    """MultiHumanRL.transform and ValueNetwork.forward on device tensors vs reference fixtures."""
    import torch
    o = oracle_mod
    pol = mcn.BatchedSARL()
    pol.load_weights(weights0)
    for H in (5, 10):
        x = torch.from_numpy(units["vnet_in_h%d" % H]).cuda()
        v = pol.forward(x).cpu().numpy()
        ref = units["vnet_out_h%d" % H]
        assert value_errors(v, ref, "f32") <= 1.0
    E, H = 32, 5
    env = mcn.BatchedCrowdSim(E, H)
    agents = _scenes(o, E, H)
    agents[:, :, 2:4] = np.random.RandomState(1).uniform(-1, 1, (E, H + 1, 2))
    env.set_state(agents)
    t = pol.transform(env).cpu().numpy()
    for e in range(E):
        assert np.max(np.abs(t[e] - o.transform(agents[e]))) < 5e-6
    env.close(); pol.close()


def test_robot_orca_il(mcn, oracle_mod):
    """Robot driven by ORCA with safety_space 0.15 (imitation learning, train.py:157-166)."""
    o = oracle_mod
    E, H = 64, 5
    ecfg = o.EnvCfg.default()
    env = mcn.BatchedCrowdSim(E, H)
    agents = _scenes(o, E, H, phase="train")
    env.set_state(agents)
    for step in range(10):
        env.orca(); env.robot_orca(0.15)
        env.step(update=True, read=False)
        for e in range(E):
            hv = o.human_actions(ecfg, agents[e])
            ra = o.robot_orca_action(ecfg, agents[e], 0.15)
            o.apply_step(ecfg, agents[e], 0.0, ra, hv)
        got, _ = env.get_state()
        assert np.array_equal(got, agents), step
    env.close()


def test_episode_stats_and_freeze(mcn, oracle_mod, weights0):
    """Explorer counters accumulated on the device (explorer.py:41-51,92-141); finished envs freeze."""
    o = oracle_mod
    E, H = 64, 5
    ecfg, scfg = o.EnvCfg.default(), o.SarlCfg.default()
    env = mcn.BatchedCrowdSim(E, H)
    pol = mcn.BatchedSARL()
    pol.load_weights(weights0)
    agents = _scenes(o, E, H)
    agents[:8, 0, :2] = [0.0, 3.0]             # some robots close to the goal -> ReachGoal quickly
    env.set_state(agents)
    ref = dict(episodes=0, success=0, collision=0, timeout=0, steps=0, too_close=0, sum_min_dist=0.0,
               sum_success_time=0.0, sum_collision_time=0.0, sum_timeout_time=0.0, sum_return=0.0)
    times = np.zeros(E); done_flags = np.zeros(E, bool); ep_ret = np.zeros(E); ep_steps = np.zeros(E, int)
    for step in range(12):
        mcn.rollout_step(pol, env, query_env=False)
        best, _ = pol.read(env, values=False)
        for e in range(E):
            if done_flags[e]:
                continue
            hv = o.human_actions(ecfg, agents[e])
            act = pol.action_table[best[e]]
            r, d, i, dm = o.step_outcome(ecfg, agents[e], times[e], act)
            times[e] = o.apply_step(ecfg, agents[e], times[e], act, hv)
            ep_ret[e] += pow(0.9, ep_steps[e] * 0.25 * 1.0) * r; ep_steps[e] += 1
            ref["steps"] += 1
            if i == o.DANGER:
                ref["too_close"] += 1; ref["sum_min_dist"] += dm
            if d:
                done_flags[e] = True; ref["episodes"] += 1; ref["sum_return"] += ep_ret[e]
                key = {o.REACHGOAL: "success", o.COLLISION: "collision", o.TIMEOUT: "timeout"}[i]
                ref[key] += 1
                ref["sum_%s_time" % key] += 25.0 if i == o.TIMEOUT else times[e]
    st = env.stats()
    got, _ = env.get_state()
    assert np.array_equal(got, agents)
    for k, v in ref.items():
        assert st[k] == pytest.approx(v, rel=1e-12, abs=1e-12), k
    assert st["success"] >= 1
    env.close(); pol.close()


@pytest.mark.parametrize("robot", ["policy", "orca", "keep"])
def test_native_episode_loop_equals_stepwise(mcn, oracle_mod, weights_trained, robot):
    """cn_rollout_episodes (explorer.py:53-69 enqueued natively, with the replay records) leaves exactly what the same steps
    issued one call at a time leave: final state, per-env episode table, per-step transformed states / rewards / done flags."""
    import torch
    from modelcrowdnav_b200 import _capi
    o = oracle_mod
    E, H, T = 96, 5, 102
    agents = _scenes(o, E, H)
    agents[:8, 0, :2] = [0.0, 3.0]
    pol = mcn.BatchedSARL(precision="f32")
    pol.load_weights(weights_trained)
    mode = dict(policy=_capi.ROBOT_POLICY, orca=_capi.ROBOT_ORCA, keep=_capi.ROBOT_KEEP)[robot]

    ref = mcn.BatchedCrowdSim(E, H)
    ref.set_state(agents)
    if robot == "keep":
        ref.set_actions(np.zeros((E, 2)))
    S_ref, R_ref, D_ref = [], [], []
    for t in range(T):
        S_ref.append(pol.transform(ref))
        ref.orca()
        if robot == "policy":
            pol.lookahead(ref, query_env=True, epsilon=0.0)
        elif robot == "orca":
            ref.robot_orca(0.0)
        r, d, _, _ = ref.step(update=True)
        R_ref.append(r); D_ref.append(d)
        if ref.all_done():
            break
    n_ref = len(R_ref)

    env = mcn.BatchedCrowdSim(E, H)
    env.set_state(agents)
    if robot == "keep":
        env.set_actions(np.zeros((E, 2)))
    n, S, R, D = env.run_episodes(T, policy=pol if robot == "policy" else None, robot_mode=mode, query_env=True,
                                  check_every=4, record=(pol, False))
    assert n_ref <= n <= min(T, n_ref + 8)               # stops at most two check intervals after the last episode ended
    assert S.shape == (n, E, H, 13) and R.shape == (n, E) and D.shape == (n, E)
    assert torch.equal(S[:n_ref], torch.stack(S_ref))
    assert np.array_equal(R[:n_ref].cpu().numpy(), np.stack(R_ref))
    assert np.array_equal(D[:n_ref].cpu().numpy(), np.stack(D_ref))
    assert (D[n_ref:] == 1).all() and (R[n_ref:] == 0).all()     # steps after the last episode: everything frozen
    a, b = env.episode_table(), ref.episode_table()
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    assert a["frozen"].all() and (a["episodes"] == 1).all()
    assert np.array_equal(env.get_state()[0], ref.get_state()[0])
    env.close(); ref.close(); pol.close()


@pytest.mark.parametrize("H", [5, 20])
def test_device_reset_properties(mcn, H):
    """Device-side reset: scene invariants of crowd_sim.py:165-217 and shard invariance (global env id).  H = 20 takes the
    warp-per-env generator (reset_env_warp), H = 5 the thread-per-env one."""
    E = 512
    for rule, name in ((0, "circle"), (1, "square")):
        if H > 5 and rule == 0:
            continue                                    # 20 humans do not fit the radius-4 circle under the separation rule
        env = mcn.BatchedCrowdSim(E, H, sim_rule=rule, seed=7)
        env.reset_device()
        a, t = env.get_state()
        assert np.all(t == 0) and np.all(a[:, :, 2:4] == 0)
        assert np.all(a[:, 0, :2] == [0, -4]) and np.all(a[:, 0, 4:6] == [0, 4])
        if rule == 0:
            assert np.array_equal(a[:, 1:, 4:6], -a[:, 1:, 0:2])
            r = np.hypot(a[:, 1:, 0], a[:, 1:, 1])
            assert np.all(r > 4 - 0.75) and np.all(r < 4 + 0.75)
        else:
            assert np.all(np.abs(a[:, 1:, 0]) <= 5) and np.all(np.abs(a[:, 1:, 1]) <= 5)
            assert np.all(a[:, 1:, 0] * a[:, 1:, 4] <= 0)          # goal on the other side
        for i in range(1, H + 1):                                   # min separation 0.8 vs earlier agents
            for j in range(i):
                d = np.hypot(a[:, i, 0] - a[:, j, 0], a[:, i, 1] - a[:, j, 1])
                assert np.all(d >= 0.8)
        # shard invariance: envs [256, 512) generated alone equal the second half
        env2 = mcn.BatchedCrowdSim(E // 2, H, sim_rule=rule, seed=7, env_id_offset=E // 2)
        env2.reset_device()
        b, _ = env2.get_state()
        assert np.array_equal(b, a[E // 2:])
        env.close(); env2.close()


def test_auto_reset_rollout_runs(mcn, weights0):
    """Throughput mode: auto_reset keeps every env alive; counters add up."""
    E, H = 256, 5
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=3)
    pol = mcn.BatchedSARL()
    pol.load_weights(weights0)
    env.reset_device()
    n = 110
    for _ in range(n):
        mcn.rollout_step(pol, env)
    st = env.stats()
    assert st["steps"] == E * n
    assert st["episodes"] == st["success"] + st["collision"] + st["timeout"] >= E   # >= 1 timeout each (97 steps)
    a, t = env.get_state()
    assert np.all(np.isfinite(a)) and np.all(t <= 25.0)
    env.close(); pol.close()


def test_host_step_matches_device_step(mcn, oracle_mod, weights0):
    """cn_rollout_step_host (HOST buffers, e2e path) == device-resident rollout."""
    o = oracle_mod
    E, H = 128, 5
    agents = _scenes(o, E, H)
    env_a = mcn.BatchedCrowdSim(E, H); env_b = mcn.BatchedCrowdSim(E, H)
    pol = mcn.BatchedSARL(); pol.load_weights(weights0)
    env_a.set_state(agents); env_b.set_state(agents)
    buf = mcn.HostStepBuffers(env_b)
    buf.agents_in[...] = agents; buf.times_in[...] = 0
    for step in range(5):
        mcn.rollout_step(pol, env_a)
        ra, da, ia, _ = env_a.read_outputs()
        mcn.rollout_step_host(pol, env_b, buf)
        sa, ta = env_a.get_state()
        assert np.array_equal(sa, buf.agents_out) and np.array_equal(ta, buf.times_out)
        assert np.array_equal(ra, buf.reward) and np.array_equal(da, buf.done) and np.array_equal(ia, buf.info)
        buf.agents_in[...] = buf.agents_out; buf.times_in[...] = buf.times_out
    env_a.close(); env_b.close(); pol.close()


@pytest.mark.parametrize("N,K,bmn", [(16, 16, 0), (64, 112, 0), (112, 112, 0), (160, 32, 0), (112, 224, 0), (160, 80, 0),
                                     (256, 64, 0), (64, 128, 1), (112, 128, 1), (16, 16, 1), (64, 48, 1),
                                     (112, 160, 2), (112, 112, 2), (64, 32, 2)])
def test_umma_selftest(mcn, N, K, bmn):
    """tcgen05.mma building block (descriptor / chunked K-major layout / TMEM read-back) vs fp32 matmul."""
    import ctypes as C
    rs = np.random.RandomState(N * 1000 + K)
    a = rs.uniform(-1, 1, (128, K)).astype(np.float16).astype(np.float32)
    b = rs.uniform(-1, 1, (N, K)).astype(np.float16).astype(np.float32)
    d = np.zeros((128, N), np.float32)
    lib = mcn._capi.load()
    fn = {0: lib.cn_selftest_umma, 1: lib.cn_selftest_umma_bmn, 2: lib.cn_selftest_umma_ts}[bmn]   # SS, MN-major B, A in TMEM
    mcn._capi.check(fn(N, K, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p),
                                         d.ctypes.data_as(C.c_void_p), 0))
    ref = a.astype(np.float64) @ b.astype(np.float64).T
    assert np.max(np.abs(d - ref)) < 1e-4 * K


@pytest.mark.parametrize("N,K", [(32, 16), (64, 112), (112, 112), (160, 32), (112, 160), (224, 112), (256, 64)])
def test_umma_pair_selftest(mcn, N, K):
    """cta_group::2 building block: M = 256 over a 2-CTA cluster, B split in N halves, remote operand-ready
    arrivals and multicast completion, vs fp32 matmul."""
    import ctypes as C
    rs = np.random.RandomState(N * 1000 + K + 7)
    a = rs.uniform(-1, 1, (256, K)).astype(np.float16).astype(np.float32)
    b = rs.uniform(-1, 1, (N, K)).astype(np.float16).astype(np.float32)
    d = np.zeros((256, N), np.float32)
    lib = mcn._capi.load()
    mcn._capi.check(lib.cn_selftest_umma_pair(N, K, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p),
                                              d.ctypes.data_as(C.c_void_p), 3, None, 0))
    ref = a.astype(np.float64) @ b.astype(np.float64).T
    assert np.max(np.abs(d - ref)) < 1e-4 * K


@pytest.mark.parametrize("rule", [0, 1])
def test_device_reset_randomize_attributes(mcn, rule):
    """[env] randomize_attributes on the device generator: v_pref in [0.5, 1.5], radius in [0.3, 0.5], heterogeneous,
    and the reference's separation rule holds with the per-human radii (crowd_sim.py:167-186, agent.py:39-45)."""
    E, H = 512, 5
    env = mcn.BatchedCrowdSim(E, H, seed=3, sim_rule=rule, randomize_attributes=1)
    env.reset_device()
    a, t = env.get_state()
    r, vp = a[:, 1:, 6], a[:, 1:, 7]
    assert np.all((r >= 0.3) & (r <= 0.5)) and np.all((vp >= 0.5) & (vp <= 1.5))
    assert r.std() > 0.03 and vp.std() > 0.15
    assert np.all(a[:, 0, 6] == 0.3) and np.all(a[:, 0, 7] == 1.0)          # the robot keeps its configured attributes
    for i in range(1, H + 1):
        for j in range(i):
            dmin = a[:, i, 6] + a[:, j, 6] + 0.2
            assert np.all(np.hypot(a[:, i, 0] - a[:, j, 0], a[:, i, 1] - a[:, j, 1]) >= dmin)
            if rule == 1 or j > 0:
                assert np.all(np.hypot(a[:, i, 4] - a[:, j, 4], a[:, i, 5] - a[:, j, 5]) >= dmin)
    env.close()


@pytest.mark.parametrize("E,H,speeds,rots", [(1000, 4, 3, 8), (777, 6, 5, 16), (130, 13, 2, 5)])
def test_tc_matches_f32_odd_shapes(mcn, weights0, E, H, speeds, rots):
    """Tile bookkeeping of the CTA-pair kernels on sizes that divide nothing (env count, humans per group, action
    count): the tensor-core values against the FP32 CUDA-core path (itself checked against the oracle) on evolving
    device-generated states."""
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=5, sim_rule=1)
    p32 = mcn.BatchedSARL(precision="f32", speed_samples=speeds, rotation_samples=rots)
    p16 = mcn.BatchedSARL(precision="f16_tc", speed_samples=speeds, rotation_samples=rots)
    p32.load_weights(weights0); p16.load_weights(weights0)
    assert p16.A == speeds * rots + 1
    env.reset_device()
    for step in range(4):
        env.orca()
        p32.lookahead(env, 0); b32, v32 = p32.read(env)
        p16.lookahead(env, 0); b16, v16 = p16.read(env)
        assert v16.shape == (E, p16.A)
        assert value_errors(v16, v32, "f16_tc") <= 1.0
        check_choice(b16, b32, v32, "f16_tc")
        env.step(update=True, read=False)
    env.close(); p32.close(); p16.close()


@pytest.mark.parametrize("net", ["cadrl", "lstm", "om_sarl"])
@pytest.mark.parametrize("E,H,query_env", [(1000, 4, 0), (777, 6, 1), (130, 13, 0), (3000, 5, 0)])
def test_tc_other_networks_match_f32_at_size(mcn, units_nets, units_om, net, E, H, query_env):
    """The tensor-core forms of CADRL (tc_mlp3_pair_kernel<1>), LSTM-RL (tc_lstm_pair_kernel: several rounds per slot, every
    step count) and OM-SARL (tc_om_bias_kernel + the row kernel's bias epilogue) against their FP32 kernels (themselves pinned
    to the reference's episodes) on sizes that divide nothing, over evolving device-generated states."""
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=11, sim_rule=1)
    if net == "om_sarl":
        p32, p16 = _om_policy(mcn, "sarl", "f32"), _om_policy(mcn, "sarl", "f16_tc")
        w = units_om["om_sarl_weights"]
    else:
        p32, p16 = _net_policy(mcn, net, precision="f32"), _net_policy(mcn, net, precision="f16_tc")
        w = units_nets[net + "_weights"]
    p32.load_weights(w); p16.load_weights(w)
    env.reset_device()
    for step in range(3):
        env.orca()
        p32.lookahead(env, query_env); b32, v32 = p32.read(env)
        p16.lookahead(env, query_env); b16, v16 = p16.read(env)
        assert value_errors(v16, v32, "f16_tc") <= 1.0
        check_choice(b16, b32, v32, "f16_tc")
        env.step(update=True, read=False)
    env.close(); p32.close(); p16.close()


def test_packed_host_step_matches_device_step(mcn, oracle_mod, weights0):
    """cn_rollout_step_host_packed (one H2D + one D2H per step, ping-ponged pinned blocks) == the device-resident step."""
    E, H = 40, 5
    agents = _scenes(oracle_mod, E, H, "circle_crossing", phase="val")
    env_a = mcn.BatchedCrowdSim(E, H); env_b = mcn.BatchedCrowdSim(E, H)
    pol = mcn.BatchedSARL(precision="f32"); pol.load_weights(weights0)
    env_a.set_state(agents)
    env_b.set_state(agents)            # initialises env_b's episode bookkeeping like a reset would
    buf = mcn.PackedHostStepBuffers(env_b)
    assert buf.in_bytes == 8 * (E * (H + 1) * 8 + E) and buf.out_bytes == buf.in_bytes + 14 * E
    buf.agents_in[...] = agents; buf.times_in[...] = 0
    for step in range(5):
        mcn.rollout_step(pol, env_a)
        ra, da, ia, _ = env_a.read_outputs()
        ba = env_a.read_actions()[0] if hasattr(env_a, "read_actions") else None
        mcn.rollout_step_host_packed(pol, env_b, buf)
        sa, ta = env_a.get_state()
        assert np.array_equal(sa, buf.agents_out) and np.array_equal(ta, buf.times_out)
        assert np.array_equal(ra, buf.reward) and np.array_equal(da, buf.done) and np.array_equal(ia, buf.info)
        if ba is not None:
            assert np.array_equal(np.asarray(ba).reshape(-1), buf.action_idx)
        buf.swap()
    env_a.close(); env_b.close(); pol.close()


@pytest.mark.parametrize("net,shards,graphs", [("sarl", 2, False), ("sarl", 4, True), ("sarl", 2, True), ("cadrl", 2, True),
                                               ("lstm", 2, True), ("om_sarl", 2, True)])
def test_pipelined_host_rollout_matches_device_step(mcn, oracle_mod, weights0, units_nets, units_om, net, shards, graphs):
    """PipelinedHostRollout (env shards on their own streams, cn_rollout_step_host_packed_async: the copies of one
    shard overlap the kernels of another) returns bit for bit what the single device-resident handle computes,
    including the episodes that finish and are re-seeded on the device (global env ids key the Philox streams).
    Every tensor-core network: each hands its scoring stage and argmax over to the shard's tail stream."""
    E, H = 256, 5
    if net == "sarl":
        cfg, w = {}, weights0
    elif net == "om_sarl":
        cfg, w = _om_kw("sarl"), units_om["om_sarl_weights"]
    else:
        cfg, w = _net_kw(net), units_nets[net + "_weights"]
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=3)
    pol = mcn.BatchedSARL(precision="f16_tc", **cfg); pol.load_weights(w)
    env.reset_device()
    a0, t0 = env.get_state()
    pipe = mcn.PipelinedHostRollout(E, H, w, shards=shards, precision="f16_tc", auto_reset=1, seed=3, policy_cfg=cfg,
                                    use_graphs=graphs)                    # graphs: one captured launch per shard and step
    pipe.reset_device()
    b = [x for x in pipe.bufs]
    assert np.array_equal(np.concatenate([x.agents_in for x in b]), a0)   # same scenes whatever the sharding
    for step in range(110):                                          # past the 100-step time limit: episodes end
        mcn.rollout_step(pol, env)
        pipe.step()
    pipe.sync()
    sa, ta = env.get_state()
    r, d, i, _ = env.read_outputs()
    agents, times, reward, action_idx, done, info = pipe.results()
    assert np.array_equal(sa, agents) and np.array_equal(ta, times)
    assert np.array_equal(r, reward) and np.array_equal(d, done) and np.array_equal(i, info)
    st = env.stats()
    assert st["episodes"] > 0                                       # some episodes ended and were re-seeded
    assert sum(e.stats()["episodes"] for e in pipe.envs) == st["episodes"]
    pipe.close()
    # the device-resident form of the same sharding (cn_rollout_step_sharded: no copies, no host sync between steps)
    dev = mcn.PipelinedHostRollout(E, H, w, shards=shards, precision="f16_tc", auto_reset=1, seed=3, policy_cfg=cfg)
    dev.reset_device()
    for step in range(110):
        dev.step_device()
    dev.sync_device()
    got = [e.get_state() for e in dev.envs]
    assert np.array_equal(np.concatenate([g[0] for g in got]), sa) and np.array_equal(np.concatenate([g[1] for g in got]), ta)
    dev.close(); env.close(); pol.close()


@pytest.mark.parametrize("precision", ["f32", "f16_tc"])
@pytest.mark.parametrize("name", TRAJ_NAMES_KIN)
def test_golden_trajectories_kinematics(mcn, weights0, name, precision):
    """Robot kinematics None (the fork exactly as shipped: ActionRot dynamics, heading feature zero) and unicycle:
    teacher-forced replay of the reference's own episodes.  Action table bit-exact; values / argmax to the same bars as
    the holonomic fixtures; integer outputs exact; positions, velocities and heading to 1e-12 (the non-holonomic step
    goes through double cos / sin, where CUDA and glibc agree to 1-2 ulp, not bit for bit)."""
    tr = load_traj(name)
    H, kin = tr["H"], tr["kinematics"]
    states, times, thetas, recs = [], [], [], []
    for case, rec in tr["cases"].items():
        for t in range(len(rec["time"])):
            states.append(rec["agents"][t]); times.append(rec["time"][t]); thetas.append(rec["theta"][t])
            recs.append((rec, t))
    E = len(states)
    env = mcn.BatchedCrowdSim(E, H, robot_visible=tr["robot_visible"], robot_kinematics=kin)
    pol = mcn.BatchedSARL(precision=precision, kinematics=kin)
    pol.load_weights(weights0)
    assert np.array_equal(pol.action_table, recs[0][0]["table"])            # bit-exact (v, r) table
    env.set_state(np.stack(states), np.array(times))
    assert np.all(env.get_theta() == np.pi / 2)                             # a host scene is a reset
    env.set_theta(np.array(thetas))
    env.orca()
    hv = env.human_actions()
    pol.lookahead(env, query_env=tr["query_env"])
    best, values = pol.read(env)
    acts = np.stack([rec["action"][t] for rec, t in recs])                  # the REFERENCE's (v, r) actions
    reward, done, info, dmin = env.step(acts, update=True)
    got, gt = env.get_state()
    th = env.get_theta()
    for e, (rec, t) in enumerate(recs):
        assert np.array_equal(hv[e], rec["human_v"][t]), (name, e)
        assert value_errors(values[e], rec["values"][t], precision) <= 1.0, (name, e)
        assert (reward[e], bool(done[e]), int(info[e])) == (rec["reward"][t], bool(rec["done"][t]), int(rec["info"][t]))
        if t + 1 < len(rec["time"]):
            assert np.allclose(got[e], rec["agents"][t + 1], rtol=0, atol=1e-12) and gt[e] == rec["time"][t + 1]
            assert np.array_equal(got[e][1:], rec["agents"][t + 1][1:])    # humans never touch cos / sin: bit-exact
            assert abs(th[e] - rec["theta"][t + 1]) <= 1e-12
    check_choice(best, [rec["best"][t] for rec, t in recs], np.stack([rec["values"][t] for rec, t in recs]), precision)
    env.close(); pol.close()


def _net_kw(tag):
    """BatchedSARL arguments of the reference's CADRL / LSTM-RL ([cadrl], [lstm_rl] of policy.config)."""
    if tag == "cadrl":
        return dict(network="cadrl", mlp3_dims=[150, 100, 100, 1])
    m1 = [150, 100, 100, 50] if tag == "lstm2" else [0, 0, 0, 0]
    return dict(network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50, lstm_mlp1_dims=m1)


def _net_policy(mcn, tag, **kw):
    kw = {k: v for k, v in kw.items() if v is not None}
    return mcn.BatchedSARL(precision=kw.pop("precision", "f32"), **_net_kw(tag), **kw)


@pytest.mark.parametrize("tag", ["cadrl", "lstm", "lstm2"])
def test_other_value_networks_forward(mcn, units_nets, tag):
    """cn_policy_forward for the CADRL mlp (min over the rows of an item) and both LSTM-RL networks against the outputs of
    the reference's torch modules (tests/golden/units_nets.npz)."""
    import torch
    pol = _net_policy(mcn, tag)
    w = units_nets[tag + "_weights"]
    assert pol.n_params == w.size
    pol.load_weights(w)
    for H in (1, 5):
        x, ref = units_nets["%s_in_h%d" % (tag, H)], units_nets["%s_out_h%d" % (tag, H)]
        got = pol.forward(torch.from_numpy(x).cuda()).cpu().numpy()
        want = ref.min(axis=1) if tag == "cadrl" else ref
        assert value_errors(got, want, "f32") <= 1.0
    with pytest.raises(mcn.CrowdNavError):                             # tensor-core LSTM-RL is ValueNetwork1 only: no silent fallback
        mcn.BatchedSARL(precision="f16_tc", network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50,
                        lstm_mlp1_dims=[150, 100, 100, 50])
    with pytest.raises(mcn.CrowdNavError):
        mcn.BatchedSARL(precision="f16_tc", network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=64)
    with pytest.raises(mcn.CrowdNavError):                             # tensor-core CADRL is the default [cadrl] shape only
        mcn.BatchedSARL(precision="f16_tc", network="cadrl", mlp3_dims=[128, 100, 100, 1])
    pol.close()


@pytest.mark.parametrize("precision", ["f32", "f16_tc"])
@pytest.mark.parametrize("name", TRAJ_NAMES_NETS)
def test_golden_trajectories_other_networks(mcn, oracle_mod, units_nets, name, precision):
    """CADRL.predict (value = reward + gamma_bar * min over humans) and LstmRL.predict (humans sorted by decreasing
    distance unless query_env) on the GPU: teacher-forced replay of the reference's own episodes, same bars as SARL.
    CADRL also runs on the tensor cores (its mlp is the three UMMA stages of the mlp3 kernel), and so does LSTM-RL's
    ValueNetwork1 (tc_lstm_pair_kernel: one UMMA stage per human, then the mlp3 kernel); ValueNetwork2 is FP32 only."""
    tr = load_traj(name)
    tag = net_tag(tr)
    if precision == "f16_tc" and tag == "lstm2":
        pytest.skip("LSTM-RL with the interaction module has no tensor-core path (refused by cn_policy_create)")
    H = tr["H"]
    states, times, recs = [], [], []
    for case, rec in tr["cases"].items():
        for t in range(len(rec["time"])):
            states.append(rec["agents"][t]); times.append(rec["time"][t]); recs.append((rec, t))
    E = len(states)
    kin = tr["kinematics"]
    env = mcn.BatchedCrowdSim(E, H, robot_kinematics=kin)
    pol = _net_policy(mcn, tag, kinematics=kin, precision=precision)
    pol.load_weights(units_nets[tag + "_weights"])
    assert np.array_equal(pol.action_table, recs[0][0]["table"])
    env.set_state(np.stack(states), np.array(times))
    if kin != 0:
        env.set_theta(np.array([rec["theta"][t] for rec, t in recs]))
    env.orca()
    pol.lookahead(env, query_env=tr["query_env"])
    best, values = pol.read(env)
    acts = np.stack([rec["action"][t] for rec, t in recs])
    reward, done, info, dmin = env.step(acts, update=True)
    got, gt = env.get_state()
    agree = total = 0
    for e, (rec, t) in enumerate(recs):
        ref_v = rec["values"][t]
        assert value_errors(values[e], ref_v, precision) <= 1.0, (name, e)
        assert ref_v.max() - ref_v[best[e]] <= TIE_GAP[precision], (name, e)       # the chosen action is optimal for the reference
        top2 = np.sort(ref_v)[-2:]
        if top2[1] - top2[0] > TIE_GAP[precision]:
            total += 1
            agree += int(best[e] == rec["best"][t])
        assert (reward[e], bool(done[e]), int(info[e])) == (rec["reward"][t], bool(rec["done"][t]), int(rec["info"][t]))
        if t + 1 < len(rec["time"]):
            if kin == 0:
                assert np.array_equal(got[e], rec["agents"][t + 1])
            else:                                            # double cos / sin in the robot update: 1-2 ulp, humans exact
                assert np.allclose(got[e], rec["agents"][t + 1], rtol=0, atol=1e-12)
                assert np.array_equal(got[e][1:], rec["agents"][t + 1][1:])
            assert gt[e] == rec["time"][t + 1]
    assert (total > 0 or precision == "f16_tc") and agree >= 0.999 * total, (agree, total)
    env.close(); pol.close()


def test_lstm_last_state_is_sorted(mcn, oracle_mod, units_nets):
    """cn_policy_last_state: LSTM-RL's last_state rows follow predict()'s human order (decreasing distance, stable);
    cn_policy_transform keeps the env order (MultiHumanRL.transform never sorts)."""
    o = oracle_mod
    E, H = 32, 5
    agents = _scenes(o, E, H, "square_crossing", phase="val")
    agents[3, 2, :2] = agents[3, 0, :2] + [1.0, 2.0]; agents[3, 4, :2] = agents[3, 0, :2] + [-2.0, 1.0]   # a tie
    env = mcn.BatchedCrowdSim(E, H)
    pol = _net_policy(mcn, "lstm")
    pol.load_weights(units_nets["lstm_weights"])
    env.set_state(agents)
    plain = pol.transform(env).cpu().numpy()
    last = pol.transform(env, last_state=True).cpu().numpy()
    for e in range(E):
        want = o.transform(agents[e])
        assert np.max(np.abs(plain[e] - want)) <= 1e-6
        assert np.array_equal(last[e], plain[e][o.lstm_human_order(agents[e])])
    env.close(); pol.close()


def _om_kw(policy):
    kw = dict(input_dim=61, with_om=1, cell_num=4, cell_size=1.0, om_channel_size=3)
    if policy == "sarl":
        return kw
    return dict(network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50, **kw)


def _om_policy(mcn, policy, precision="f32"):
    return mcn.BatchedSARL(precision=precision, **_om_kw(policy))


@pytest.mark.parametrize("H", [2, 5, 10])
def test_transform_with_occupancy_maps(mcn, units_om, H):
    """cn_policy_transform with_om: rotated rows + occupancy maps of the current human states against the reference's
    MultiHumanRL.transform (multi_human_rl.py:90-163); the occupancy channel must be exact."""
    agents, trs = units_om["om_agents_h%d" % H], units_om["om_transform_h%d" % H]
    E = agents.shape[0]
    env = mcn.BatchedCrowdSim(E, H)
    pol = _om_policy(mcn, "sarl")
    pol.load_weights(units_om["om_sarl_weights"])
    env.set_state(np.ascontiguousarray(agents))
    got = pol.transform(env).cpu().numpy()
    assert got.shape == trs.shape == (E, H, 61)
    assert np.max(np.abs(got - trs)) <= 1e-5
    assert np.array_equal(got[:, :, 13::3], trs[:, :, 13::3])
    with pytest.raises(mcn.CrowdNavError):                               # OM-LSTM-RL is FP32 only: refused, no silent fallback
        mcn.BatchedSARL(network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50, precision="f16_tc", input_dim=61, with_om=1)
    with pytest.raises(mcn.CrowdNavError):                               # the map size must match input_dim
        mcn.BatchedSARL(precision="f16_tc", input_dim=61, with_om=1, cell_num=5)
    env.close(); pol.close()


@pytest.mark.parametrize("precision", ["f32", "f16_tc"])
@pytest.mark.parametrize("name", TRAJ_NAMES_OM)
def test_golden_trajectories_with_occupancy_maps(mcn, units_om, name, precision):
    """OM-SARL / OM-LSTM-RL lookahead on the GPU against the reference's own episodes (values 1e-5 / the fp16 bars, argmax,
    transition).  On the tensor-core path the map enters mlp1.0 as an fp32 row bias per (env, human) (tc_om_bias_kernel)."""
    tr = load_traj(name)
    if precision == "f16_tc" and tr["policy"] != "sarl":
        from modelcrowdnav_b200 import _capi
        with pytest.raises(_capi.CrowdNavError):                  # OM-LSTM-RL stays FP32: refused, not silently rerouted
            _om_policy(mcn, tr["policy"], precision)
        return
    H = tr["H"]
    states, times, recs = [], [], []
    for case, rec in tr["cases"].items():
        for t in range(len(rec["time"])):
            states.append(rec["agents"][t]); times.append(rec["time"][t]); recs.append((rec, t))
    E = len(states)
    env = mcn.BatchedCrowdSim(E, H)
    pol = _om_policy(mcn, tr["policy"], precision)
    pol.load_weights(units_om[("om_sarl" if tr["policy"] == "sarl" else "om_lstm") + "_weights"])
    env.set_state(np.stack(states), np.array(times))
    env.orca()
    pol.lookahead(env, query_env=tr["query_env"])
    best, values = pol.read(env)
    acts = np.stack([rec["action"][t] for rec, t in recs])
    reward, done, info, dmin = env.step(acts, update=True)
    agree = total = 0
    for e, (rec, t) in enumerate(recs):
        ref_v = rec["values"][t]
        assert value_errors(values[e], ref_v, precision) <= 1.0, (name, e)
        top2 = np.sort(ref_v)[-2:]
        if top2[1] - top2[0] > TIE_GAP[precision]:
            total += 1
            agree += int(best[e] == rec["best"][t])
        assert ref_v.max() - ref_v[best[e]] <= TIE_GAP[precision]          # never vacuous: the choice is optimal up to a tie
        assert (reward[e], bool(done[e]), int(info[e])) == (rec["reward"][t], bool(rec["done"][t]), int(rec["info"][t]))
    assert (total > 0 or precision == "f16_tc") and (total == 0 or agree / total >= 0.999), (agree, total)
    env.close(); pol.close()


def test_rollout_step_is_cuda_graph_capturable(mcn, weights0):
    """include/crowdnav_b200.h promises a capturable step: cn_rollout_step (ORCA forked on a side stream, lookahead, step,
    auto-reset) captured once into a CUDA graph and replayed must walk the same trajectory as eager launches."""
    import torch
    E, H = 512, 5
    envs = [mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=9) for _ in range(2)]
    pols = [mcn.BatchedSARL(precision="f16_tc") for _ in range(2)]
    for p in pols:
        p.load_weights(weights0)
    for e in envs:
        e.reset_device()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):                                    # warm-up: allocates the workspaces outside the capture
            mcn.rollout_step(pols[1], envs[1], stream=side.cuda_stream)
    side.synchronize()
    for _ in range(3):
        mcn.rollout_step(pols[0], envs[0])
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        mcn.rollout_step(pols[1], envs[1], stream=torch.cuda.current_stream().cuda_stream)
    mcn.rollout_step(pols[0], envs[0])                        # the captured launch did not execute: replay it once below
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


@pytest.mark.parametrize("H", [13, 50])
def test_tc_large_groups_vs_oracle(mcn, oracle_mod, weights0, H):
    """Run-time-H path of the CTA-pair kernel with few, large groups (H = 50: BASELINE's dense-crowd configuration, 2 groups
    of 50 rows per tile; H = 13: 9 groups): split group mean, single-exp softmax and split weighted-feature sums against
    the oracle and the FP32 path."""
    o = oracle_mod
    E = 6
    ecfg, scfg = o.EnvCfg.default(), o.SarlCfg.default()
    env = mcn.BatchedCrowdSim(E, H, square_width=14.0)
    p16 = mcn.BatchedSARL(precision="f16_tc"); p16.load_weights(weights0)
    p32 = mcn.BatchedSARL(precision="f32"); p32.load_weights(weights0)
    agents = np.stack([o.generate_scene("val", c, human_num=H, rule="square_crossing", square_width=14.0) for c in range(E)])
    env.set_state(agents)
    for step in range(2):
        env.orca()
        hv = env.human_actions()
        p32.lookahead(env, 0); b32, v32 = p32.read(env)
        p16.lookahead(env, 0); b16, v16 = p16.read(env)
        cur, times = env.get_state()
        for e in range(E):
            obest, ovals, _ = o.lookahead(ecfg, scfg, weights0, cur[e], times[e], p16.action_table, False, hv[e])
            assert value_errors(v32[e], ovals, "f32") <= 1.0
            assert value_errors(v16[e], ovals, "f16_tc") <= 1.0
        env.step(update=True, read=False)
    env.close(); p16.close(); p32.close()


@pytest.mark.parametrize("E,H", [(1, 1), (2, 1), (1, 5), (3, 2), (2, 64)])
def test_smallest_and_largest_shapes_vs_oracle(mcn, oracle_mod, weights_trained, E, H):
    """The ends of the supported range: one env, one human (the group mean and the softmax degenerate to the row itself,
    sarl.py:47-58), a tile that is almost empty, and CN_MAX_HUMANS = 64 humans (2 groups per tile).  ORCA velocities and
    the step bit-exact against the oracle, lookahead values to the bars of both precisions, three evolved steps."""
    o = oracle_mod
    ecfg, scfg = o.EnvCfg.default(), o.SarlCfg.default()
    rule, width = ("circle_crossing", 10.0) if H <= 5 else ("square_crossing", 16.0)
    env = mcn.BatchedCrowdSim(E, H, square_width=width)
    p16 = mcn.BatchedSARL(precision="f16_tc"); p16.load_weights(weights_trained)
    p32 = mcn.BatchedSARL(precision="f32"); p32.load_weights(weights_trained)
    agents = np.stack([o.generate_scene("test", 40 + c, human_num=H, rule=rule, square_width=width) for c in range(E)])
    env.set_state(agents)
    times = np.zeros(E)
    for step in range(3):
        env.orca()
        hv = env.human_actions()
        p16.lookahead(env, 1); b16, v16 = p16.read(env)
        p32.lookahead(env, 1); b32, v32 = p32.read(env)
        ref_vals = []
        for e in range(E):
            ohv = o.human_actions(ecfg, agents[e])
            assert np.array_equal(hv[e], ohv)
            obest, ovals, _ = o.lookahead(ecfg, scfg, weights_trained, agents[e], times[e], p32.action_table, True, ohv)
            assert value_errors(v32[e], ovals, "f32") <= 1.0
            assert value_errors(v16[e], ovals, "f16_tc") <= 1.0
            ref_vals.append(ovals)
        ref_vals = np.stack(ref_vals)
        for best, prec in ((b32, "f32"), (b16, "f16_tc")):
            regret = ref_vals.max(axis=1) - ref_vals[np.arange(E), best]
            assert np.all(regret <= TIE_GAP[prec])
        reward, done, info, dmin = env.step(update=True)          # the pending action is the FP32 path's choice
        for e in range(E):
            act = p32.action_table[b32[e]]
            r, d, i, dm = o.step_outcome(ecfg, agents[e], times[e], act)
            assert (reward[e], bool(done[e]), int(info[e])) == (r, bool(d), int(i))
            times[e] = o.apply_step(ecfg, agents[e], times[e], act, o.human_actions(ecfg, agents[e]))
        got, gt = env.get_state()
        assert np.array_equal(got, agents) and np.array_equal(gt, times)
    env.close(); p16.close(); p32.close()


def test_shape_limits_are_refused(mcn):
    """Out-of-range shapes fail loudly at handle creation (CN_EINVAL with a message), never silently clamp."""
    from modelcrowdnav_b200 import _capi
    for kw in (dict(num_envs=0, human_num=5), dict(num_envs=4, human_num=0), dict(num_envs=4, human_num=65)):
        with pytest.raises(_capi.CrowdNavError) as ei:
            mcn.BatchedCrowdSim(kw["num_envs"], kw["human_num"])
        assert ei.value.code == _capi.CN_EINVAL
