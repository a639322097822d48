"""Value networks at non-default layer widths and occupancy-map settings.

cn_policy_create accepts any layer width in [1, 256], lstm_hidden in [1, 64], cell_num 1..8, om_channel_size 1..3 and any
cell_size > 0; every FP32 kernel sizes its buffers from the layer list (pad4 strides, shared-memory plans, the 16 / 4 / 1 K-tails
of dense_t).  The widths below divide nothing and reach both ends of that range, so a stride that assumes a multiple of 4, an
off-by-one in a K-tail or a map-channel branch that only the default [om] exercises shows up here.

References: the torch modules of policy.py in float64 for the networks, a float64 numpy transcription of
build_occupancy_maps (multi_human_rl.py:109-163) for the maps, and the C oracle (itself pinned to both on the CPU below) for
the lookahead.  The oracle computes SARL with the global state only; without it, the oracle gets an attention.0 whose
group-mean columns are zero, which is the same function (tests/test_no_global_state.py)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, TIE_GAP, VALUE_FLOOR, check_argmax, value_errors

SARL_DEFAULT = dict(m1=[150, 100], m2=[100, 50], at=[100, 100, 1], m3=[150, 100, 100, 1])
ODD = dict(m1=[37, 23], m2=[19, 7], at=[13, 5, 1], m3=[29, 11, 3, 1])
SHAPES = {
    "sarl_odd": dict(net="sarl", **ODD),
    "sarl_odd_nogs": dict(net="sarl", gs=False, **ODD),
    "sarl_tiny": dict(net="sarl", m1=[2, 1], m2=[1, 2], at=[1, 1, 1], m3=[2, 1, 2, 1]),
    "sarl_wide": dict(net="sarl", m1=[256, 256], m2=[256, 256], at=[256, 256, 1], m3=[256, 256, 256, 1]),
    "sarl_default": dict(net="sarl", **SARL_DEFAULT),
    "sarl_default_nogs": dict(net="sarl", gs=False, **SARL_DEFAULT),
    "cadrl_odd": dict(net="cadrl", m3=[37, 23, 5, 1]),
    "cadrl_wide": dict(net="cadrl", m3=[256, 256, 256, 1]),
    "cadrl_tiny": dict(net="cadrl", m3=[1, 1, 1, 1]),
    "lstm_h1": dict(net="lstm", hidden=1, m3=[29, 11, 3, 1]),
    "lstm_h7": dict(net="lstm", hidden=7, m3=[29, 11, 3, 1]),
    "lstm_h64": dict(net="lstm", hidden=64, m3=[29, 11, 3, 1]),
    "lstm_vn2_odd": dict(net="lstm", lm1=[37, 23, 11, 9], hidden=13, m3=[29, 11, 3, 1]),
    "lstm_default": dict(net="lstm", hidden=50, m3=[150, 100, 100, 1]),
}
# (cell_num, om_channel_size, cell_size)
MAPS = [(1, 1, 1.0), (2, 2, 0.5), (3, 3, 1.7), (5, 1, 0.25), (8, 3, 1.0), (8, 2, 2.0)]

# (shape, map or None): the non-default widths without maps, the map matrix on the default SARL (with and without the global
# state) and LSTM-RL ValueNetwork1, and one odd-width SARL with maps
CONFIGS = ([(s, None) for s in SHAPES if not s.endswith("default") and not s.endswith("default_nogs")] +
           [(s, m) for s in ("sarl_default", "sarl_default_nogs", "lstm_default") for m in MAPS] + [("sarl_odd", (3, 3, 1.7))])


def cfg_id(c):
    s, m = c
    return s if m is None else "%s-om%dx%dx%g" % (s, *m)


def om_dim(m):
    return 0 if m is None else m[0] * m[0] * m[1]


# ---- the network of a configuration in each of its forms -------------------------------------------------------------------
def torch_model(c):
    from modelcrowdnav_b200.policy import make_cadrl_network, make_lstm_network, make_value_network
    sp, in_dim = SHAPES[c[0]], 13 + om_dim(c[1])
    if sp["net"] == "sarl":
        return make_value_network(in_dim, 6, sp["m1"], sp["m2"], sp["m3"], sp["at"], sp.get("gs", True))
    if sp["net"] == "cadrl":
        return make_cadrl_network(in_dim, sp["m3"])
    return make_lstm_network(in_dim, 6, sp.get("lm1"), sp["m3"], sp["hidden"])


def policy_kwargs(c):
    """BatchedSARL / cn_sarl_cfg fields of a configuration"""
    sp, m = SHAPES[c[0]], c[1]
    kw = {} if m is None else dict(input_dim=13 + om_dim(m), with_om=1, cell_num=m[0], om_channel_size=m[1], cell_size=m[2])
    if sp["net"] == "sarl":
        kw.update(mlp1_dims=sp["m1"], mlp2_dims=sp["m2"], attn_dims=sp["at"], mlp3_dims=sp["m3"])
        if not sp.get("gs", True):
            kw["without_global_state"] = 1
    elif sp["net"] == "cadrl":
        kw.update(network="cadrl", mlp3_dims=sp["m3"])
    else:
        kw.update(network="lstm_rl", mlp3_dims=sp["m3"], lstm_hidden=sp["hidden"], lstm_mlp1_dims=sp.get("lm1", [0, 0, 0, 0]))
    return kw


def capi_cfg(mcn, c, **kw):
    kw = dict(policy_kwargs(c), **kw)
    if isinstance(kw.get("network"), str):
        kw["network"] = {"cadrl": mcn._capi.NET_CADRL, "lstm_rl": mcn._capi.NET_LSTM_RL}[kw["network"]]
    return mcn._capi.default_sarl_cfg(**kw)


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


def weights(c, scale=1.0, seed=0):
    """nn.Linear's default init under torch.manual_seed(seed), times `scale` (scale "x4": the scaled set of the shape).  At
    default init the 81 action values of a state lie within ~1e-4 of each other; x4 spreads them (median top-2 gap ~1) so that
    the argmax checks decide something.  SARL and LSTM-RL take x2 (median top-2 gap ~5e-3): at x4 SARL's attention scores reach
    the float32 overflow of the reference's un-stabilised softmax (exp(score) = inf, then inf / inf = NaN in the torch float32
    module too), and LSTM-RL's saturated gates carry float32 rounding through 64 recurrent steps to ~3e-5 of the values."""
    import torch
    if scale == "x4":
        scale = 4.0 if SHAPES[c[0]]["net"] == "cadrl" else 2.0
    torch.manual_seed(seed)
    return _flat(torch_model(c)) * np.float32(scale)


def trained_weights(c):
    """The GPU-trained default SARL (tests/golden/sarl_weights_trained.npy) in configuration c: without the global state
    attention.0 keeps its e_i columns, and mlp1.0's map columns are a seeded default init (the trained network has none)."""
    import torch
    sd = _load(torch_model(("sarl_default", None)), np.load(os.path.join(GOLDEN, "sarl_weights_trained.npy"))).state_dict()
    if not SHAPES[c[0]].get("gs", True):
        sd["attention.0.weight"] = sd["attention.0.weight"][:, :SARL_DEFAULT["m1"][1]].clone()
    torch.manual_seed(7)
    model = torch_model(c)
    sd["mlp1.0.weight"] = torch.cat([sd["mlp1.0.weight"], model.state_dict()["mlp1.0.weight"][:, 13:]], dim=1)
    model.load_state_dict(sd)
    return _flat(model)


def oracle_net(o, c, w):
    """(oracle config, weights in the oracle's layout) of a configuration"""
    sp, in_dim = SHAPES[c[0]], 13 + om_dim(c[1])
    if sp["net"] == "sarl":
        cfg = o.SarlCfg(in_dim, 6, (C.c_int * 2)(*sp["m1"]), (C.c_int * 2)(*sp["m2"]), (C.c_int * 3)(*sp["at"]),
                        (C.c_int * 4)(*sp["m3"]))
        if not sp.get("gs", True):             # attention.0 with zero group-mean columns
            import torch
            sd = _load(torch_model(c), w).state_dict()
            wa = sd["attention.0.weight"]
            sd["attention.0.weight"] = torch.cat([wa, torch.zeros_like(wa)], dim=1)
            w = np.concatenate([v.numpy().ravel() for v in sd.values()]).astype(np.float32)
        return cfg, w
    if sp["net"] == "cadrl":
        return o.NetCfg(o.NET_CADRL, in_dim, 6, (C.c_int * 4)(*sp["m3"]), 0, (C.c_int * 4)(0, 0, 0, 0)), w
    return o.NetCfg(o.NET_LSTM_RL, in_dim, 6, (C.c_int * 4)(*sp["m3"]), sp["hidden"],
                    (C.c_int * 4)(*sp.get("lm1", [0, 0, 0, 0]))), w


def oracle_forward(o, c, ocfg, wo, x):
    """the value network on one joint state x (H, D): SARL / LSTM-RL -> scalar, CADRL -> one value per row"""
    if SHAPES[c[0]]["net"] == "sarl":
        return o.sarl_forward(ocfg, wo, x)
    return o.net_forward(ocfg, wo, x)


def oracle_lookahead(o, c, ocfg, wo, agents, t, actions, query_env, hv, kin, theta):
    ecfg = o.EnvCfg.default()
    if c[1] is not None:
        return o.lookahead_om(ecfg, ocfg, o.OmCfg(c[1][0], c[1][2], c[1][1]), wo, agents, t, actions, query_env, hv,
                              kinematics=kin, theta=theta)
    fn = o.lookahead if SHAPES[c[0]]["net"] == "sarl" else o.lookahead_net
    return fn(ecfg, ocfg, wo, agents, t, actions, query_env, hv, kinematics=kin, theta=theta)


def om_cfg(o, m):
    return o.OmCfg(m[0], m[2], m[1])


# ---- scenes ----------------------------------------------------------------------------------------------------------------
def random_agents(rng, H):
    """(H+1, 8) agents at random positions with random velocities (every map cell and channel can be hit)"""
    a = np.zeros((H + 1, 8))
    a[:, 0:2] = rng.uniform(-4, 4, (H + 1, 2))
    a[:, 2:4] = rng.uniform(-1, 1, (H + 1, 2))
    a[:, 4:6] = rng.uniform(-5, 5, (H + 1, 2))
    a[:, 6] = rng.uniform(0.3, 0.5, H + 1)
    a[:, 7] = rng.uniform(0.5, 1.5, H + 1)
    return a


def edge_agents(cn, cs):
    """Humans whose coordinates relative to human 1 (at the origin, heading +x) are exact in binary: on cell edges at
    +-k * cs / 2 along both axes, on the map's outer edges at cn/2 * cs (outside) and -cn/2 * cs (inside), two at the same
    point, and one standing still.  Velocities are axis-aligned.  Only human 1's map is an edge case: the other humans see
    the same points rotated by angles such as atan2(1, 2), where a point can fall on a cell edge up to the last bit of a
    float64 cos / sin, and two correct math libraries may round it to either side."""
    h = cs / 2
    humans = [(0, 0, 1, 0)]
    humans += [(k * h, 0, (0, 1, -1, 0)[i % 4], (1, 0, 0, -0.5)[i % 4]) for i, k in enumerate((-cn, -2, -1, 1, 2, cn))]
    humans += [(0, k * h, (1, 0)[i % 2], (0, -1)[i % 2]) for i, k in enumerate((-cn, -1, 1, cn))]
    humans += [(2 * h, 2 * h, 0, 1), (2 * h, 2 * h, -1, 0), (-h, h, 0, 0)]
    a = np.zeros((len(humans) + 1, 8))
    a[0] = [0, -20, 0.5, 0, 0, 20, 0.3, 1.0]
    for i, (px, py, vx, vy) in enumerate(humans):
        a[i + 1] = [px, py, vx, vy, px, py, 0.3, 1.0]
    return a


def ref_occupancy_maps(humans, cell_num, cell_size, om_channel_size):
    """build_occupancy_maps (multi_human_rl.py:109-163) restated in numpy float64: humans (H, 4) = px py vx vy, H >= 2."""
    occupancy_maps = []
    for i in range(len(humans)):
        human = humans[i]
        other_humans = np.concatenate([humans[j:j + 1] for j in range(len(humans)) if j != i], axis=0)
        other_px = other_humans[:, 0] - human[0]
        other_py = other_humans[:, 1] - human[1]
        human_velocity_angle = np.arctan2(human[3], human[2])
        other_human_orientation = np.arctan2(other_py, other_px)
        rotation = other_human_orientation - human_velocity_angle
        distance = np.linalg.norm([other_px, other_py], axis=0)
        other_px = np.cos(rotation) * distance
        other_py = np.sin(rotation) * distance
        other_x_index = np.floor(other_px / cell_size + cell_num / 2)
        other_y_index = np.floor(other_py / cell_size + cell_num / 2)
        other_x_index[other_x_index < 0] = float("-inf")
        other_x_index[other_x_index >= cell_num] = float("-inf")
        other_y_index[other_y_index < 0] = float("-inf")
        other_y_index[other_y_index >= cell_num] = float("-inf")
        grid_indices = cell_num * other_y_index + other_x_index
        occupancy_map = np.isin(range(cell_num ** 2), grid_indices)
        if om_channel_size == 1:
            occupancy_maps.append([occupancy_map.astype(int)])
            continue
        other_human_velocity_angles = np.arctan2(other_humans[:, 3], other_humans[:, 2])
        rotation = other_human_velocity_angles - human_velocity_angle
        speed = np.linalg.norm(other_humans[:, 2:4], axis=1)
        other_vx = np.cos(rotation) * speed
        other_vy = np.sin(rotation) * speed
        dm = [list() for _ in range(cell_num ** 2 * om_channel_size)]
        for k, index in np.ndenumerate(grid_indices):
            if index in range(cell_num ** 2):
                if om_channel_size == 2:
                    dm[2 * int(index)].append(other_vx[k])
                    dm[2 * int(index) + 1].append(other_vy[k])
                else:
                    dm[3 * int(index)].append(1)
                    dm[3 * int(index) + 1].append(other_vx[k])
                    dm[3 * int(index) + 2].append(other_vy[k])
        for k, cell in enumerate(dm):
            dm[k] = sum(dm[k]) / len(dm[k]) if len(dm[k]) != 0 else 0
        occupancy_maps.append([dm])
    return np.concatenate(occupancy_maps, axis=0).astype(np.float32)        # torch.from_numpy(...).float()


def scaled_errors(got, ref, scale):
    """value_errors(..., "f32") for the seeded weights.  The x4 weights give values of up to ~100 from activations of that
    size, and float32 rounds relative to the activations, not to a value near zero: there the bar is 1e-5 of the largest
    |value| compared (the same bar where the values span the unit reward scale)."""
    if scale == 1.0:
        return value_errors(got, ref, "f32")
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    dv = np.where(np.isnan(got - ref), np.inf, np.abs(got - ref))
    return float(dv.max() / (1e-5 * max(np.abs(ref).max(), VALUE_FLOOR)))


# ---- CPU: the oracle against float64 torch ---------------------------------------------------------------------------------
@pytest.mark.parametrize("c", CONFIGS, ids=cfg_id)
def test_oracle_pinned_to_torch_float64(oracle_mod, c):
    """oracle.sarl_forward / net_forward == the torch module in float64 within 1e-5 relative (floor VALUE_FLOOR), on random
    joint states of 1, 7, 33 and 64 humans with the oracle's own maps, seeded and x4 weights."""
    import torch
    o = oracle_mod
    for scale in (1.0, "x4"):
        w = weights(c, scale)
        model = _load(torch_model(c), w).double()
        ocfg, wo = oracle_net(o, c, w)
        rng = np.random.default_rng(len(cfg_id(c)))
        for H in (1, 7, 33, 64):
            xs = []
            for _ in range(3):
                a = random_agents(rng, H)
                xs.append(o.transform(a) if c[1] is None else o.transform_om(om_cfg(o, c[1]), a))
            x = np.stack(xs)
            got = np.array([oracle_forward(o, c, ocfg, wo, xb) for xb in x], np.float64)
            with torch.no_grad():
                if SHAPES[c[0]]["net"] == "cadrl":
                    ref = model(torch.from_numpy(x.reshape(-1, x.shape[2])).double()).numpy().reshape(got.shape)
                else:
                    ref = model(torch.from_numpy(x).double()).numpy().reshape(-1)
            assert scaled_errors(got, ref, scale) <= 1.0, (scale, H, np.abs(got - ref).max())


# ---- CPU: the occupancy-map builder ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", MAPS, ids=lambda m: "%dx%dx%g" % m)
def test_oracle_occupancy_maps(oracle_mod, m):
    """oracle.occupancy_maps == the numpy transcription of build_occupancy_maps bit for bit after the float32 cast: seeded
    random crowds of 2 to 64 humans, and the edge scene (cell edges, outer edges, coincident and standing humans)."""
    o = oracle_mod
    rng = np.random.default_rng(m[0] * 10 + m[1])
    scenes = [random_agents(rng, H)[1:, :4] for H in (2, 3, 13, 64) for _ in range(3)]
    scenes += [rng.uniform(-m[0] * m[2] / 2, m[0] * m[2] / 2, (20, 4))]       # a crowd inside one human's map
    n_random = len(scenes)
    for cs in sorted({m[2], 1.0, 0.5}):
        scenes.append(edge_agents(m[0], cs)[1:, :4])
    hit = 0
    for k, humans in enumerate(scenes):
        ref = ref_occupancy_maps(humans, m[0], m[2], m[1])
        got = o.occupancy_maps(o.OmCfg(m[0], m[2], m[1]), humans)
        assert got.shape == ref.shape == (len(humans), om_dim(m))
        if k >= n_random:           # the edge scenes are built around human 1's map
            got, ref = got[:1], ref[:1]
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), np.argwhere(got != ref)[:5]
        hit += int(np.count_nonzero(ref))
    assert hit > 0


def test_edge_scene_is_on_the_edges():
    """The edge scene's relative coordinates are what its docstring claims: on the outer edge at +cn/2 * cs the human is
    outside human 1's map, at -cn/2 * cs inside it."""
    for cn, cs in ((1, 1.0), (8, 2.0), (5, 0.25)):
        ref = ref_occupancy_maps(edge_agents(cn, cs)[1:, :4], cn, cs, 1)[0].reshape(cn, cn)
        assert ref[cn // 2, 0] == 1                     # (-cn/2 * cs, 0): column 0 of the middle row
        assert ref.sum() >= min(3, cn * cn)


# ---- CPU: configuration ----------------------------------------------------------------------------------------------------
def _policy_config(**sarl):
    from modelcrowdnav_b200.train_loop import POLICY_DEFAULT, make_config
    cp = make_config(POLICY_DEFAULT)
    for k, v in sarl.items():
        sect, key = k.split("__") if "__" in k else ("sarl", k)
        cp.set(sect, key, v)
    return cp


@pytest.mark.parametrize("sarl,precision", [
    ({}, "f16_tc"), (dict(with_global_state="false"), "f16_tc"), (dict(with_om="true"), "f16_tc"),
    (dict(with_om="true", om__cell_num="8", om__om_channel_size="2"), "f16_tc"),
    (dict(mlp1_dims="128, 64"), "f32"), (dict(mlp2_dims="100, 49"), "f32"), (dict(attention_dims="100, 99, 1"), "f32"),
    (dict(mlp3_dims="29, 11, 3, 1", with_global_state="false"), "f32"),
    (dict(mlp1_dims="37, 23", with_om="true"), "f32")])
def test_sarl_configure_precision(sarl, precision):
    """SARL.configure keeps the tensor cores for the widths cn_tc_init runs (the default [sarl] widths with any [om] and either
    global-state setting) and picks FP32 for every other shape."""
    import modelcrowdnav_b200 as mcn
    pol = mcn.policy_factory["sarl"]()
    pol.configure(_policy_config(**sarl))
    assert pol.precision == precision
    n = sum(p.numel() for p in pol.get_model().parameters())
    assert n == sum(np.prod(v.shape) for v in pol.get_model().state_dict().values())


@pytest.mark.parametrize("key,value", [("mlp1_dims", "150"), ("mlp1_dims", "150, 100, 50"), ("mlp2_dims", "100"),
                                       ("attention_dims", "100, 1"), ("attention_dims", "100, 100, 100, 1"),
                                       ("mlp3_dims", "150, 100, 1"), ("mlp3_dims", "150, 100, 100, 100, 1"),
                                       ("attention_dims", "100, 100, 2"), ("mlp3_dims", "150, 100, 100, 3")])
def test_sarl_configure_refuses_bad_lists(key, value):
    """A width list of the wrong length, or an attention / mlp3 that does not end in one unit, is refused by name."""
    import modelcrowdnav_b200 as mcn
    pol = mcn.policy_factory["sarl"]()
    with pytest.raises((ValueError, NotImplementedError), match=key):
        pol.configure(_policy_config(**{key: value}))


def test_default_sarl_cfg_refuses_wrong_lengths():
    from modelcrowdnav_b200 import _capi
    for k, n in (("mlp1_dims", 2), ("mlp2_dims", 2), ("attn_dims", 3), ("mlp3_dims", 4), ("lstm_mlp1_dims", 4)):
        assert list(getattr(_capi.default_sarl_cfg(**{k: list(range(1, n + 1))}), k)) == list(range(1, n + 1))
        for m in (n - 1, n + 1):
            with pytest.raises(ValueError, match=k):
                _capi.default_sarl_cfg(**{k: list(range(1, m + 1))})


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mcn():
    import modelcrowdnav_b200 as m
    assert m._capi.load().cn_device_count() > 0, "GPU tests need a CUDA device"
    return m


@pytest.fixture
def no_tf32():
    import torch
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


# shapes the fused trainer refuses at cn_trainer_create (max_humans 16, CADRL 1)
TRAINER_REFUSALS = {
    "sarl_wide",                  # 16 humans x 256-wide activations and weight blocks: more than 227 kB of shared memory
    "cadrl_wide",                 # 8 samples per CTA with the 256 x 256 weight blocks staged
    "lstm_default-om8x3x1",       # 16 humans x 205 input floats with the LSTM's gates and states
}


def _scenes(o, n, H, start=0):
    rule, width = ("circle_crossing", 10.0) if H <= 10 else ("square_crossing", 16.0)
    return np.stack([o.generate_scene("val", start + c, human_num=H, rule=rule, square_width=width) for c in range(n)])


def _lookahead_cases():
    """three (humans, query_env, kinematics, weight scale) per configuration; 1 and 64 humans and a unicycle robot at least
    once per network"""
    Hs = {"sarl_odd": (1, 13, 64), "sarl_odd_nogs": (2, 7, 33), "sarl_tiny": (1, 7, 64), "sarl_wide": (1, 2, 13),
          "cadrl_odd": (1, 13, 64), "cadrl_wide": (2, 7, 33), "cadrl_tiny": (1, 7, 64), "lstm_h1": (1, 7, 64),
          "lstm_h7": (2, 13, 33), "lstm_h64": (1, 7, 64), "lstm_vn2_odd": (2, 13, 64)}
    unicycle = {"sarl_odd", "cadrl_odd", "lstm_h7", "sarl_default"}
    cases = []
    for i, c in enumerate(CONFIGS):
        hs = Hs.get(c[0]) if c[1] is None else ((1, 7, 33), (2, 13, 64))[i % 2]
        if c[1] is not None and c[0] == "sarl_odd":
            hs = (2, 13, 64)
        for j, H in enumerate(hs):
            kin = int(j == 2 and c[0] in unicycle and (c[1] is None or c[1] == MAPS[0]))
            cases.append(pytest.param(c, H, j == 1, kin, 1.0 if j == 0 else "x4", id="%s-H%d-q%d-k%d-%s" % (
                cfg_id(c), H, j == 1, kin, "seed" if j == 0 else "x4")))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("c,H,query_env,kin,scale", _lookahead_cases())
def test_f32_lookahead_vs_oracle(mcn, oracle_mod, c, H, query_env, kin, scale):
    """FP32 lookahead over three evolving steps: every value within 1e-5 relative of the oracle, the choice optimal up to the
    tie gap (and the argmax bar on the x4 weights), reward / done / info exact."""
    o = oracle_mod
    E = 4 if H <= 13 else 2
    if SHAPES[c[0]]["m3"][0] == 256:
        E = min(E, 2)
    w = weights(c, scale, seed=H)
    ocfg, wo = oracle_net(o, c, w)
    ecfg = o.EnvCfg.default()
    env = mcn.BatchedCrowdSim(E, H, robot_kinematics=kin)
    pol = mcn.BatchedSARL(precision="f32", kinematics=kin, **policy_kwargs(c))
    assert pol.n_params == w.size
    pol.load_weights(w)
    env.set_state(_scenes(o, E, H))
    bests, orefs, ovs = [], [], []
    alive = np.ones(E, bool)              # a finished env is frozen: the lookahead leaves its values alone
    for step in range(3):
        env.orca()
        hv = env.human_actions()
        cur, times = env.get_state()
        theta = env.get_theta() if kin else np.zeros(E)
        pol.lookahead(env, query_env=query_env)
        best, values = pol.read(env)
        best, values = best[alive], values[alive]
        ovals = np.stack([oracle_lookahead(o, c, ocfg, wo, cur[e], times[e], pol.action_table, query_env, hv[e], kin,
                                           theta[e])[1] for e in np.flatnonzero(alive)])
        for e in range(len(best)):
            assert scaled_errors(values[e], ovals[e], scale) <= 1.0, (step, e, np.abs(values[e] - ovals[e]).max())
        regret = ovals.max(axis=1) - ovals[np.arange(len(best)), best]
        assert np.all(regret <= TIE_GAP["f32"]), regret.max()
        bests.append(best); orefs.append(ovals.argmax(axis=1)); ovs.append(ovals)
        full_best = np.zeros(E, np.int64)
        full_best[alive] = best
        reward, done, info, _ = env.step(update=True)
        for e in np.flatnonzero(alive):
            r, d, i, _ = o.step_outcome(ecfg, cur[e], times[e], pol.action_table[full_best[e]], kin, theta[e])
            assert (reward[e], bool(done[e]), int(info[e])) == (r, bool(d), int(i)), (step, e)
        alive &= ~done.astype(bool)
    if scale != 1.0 and bests:
        # per-state regret above is the stronger check; tiny widths can leave every value tied, so no decidable minimum here
        check_argmax(np.concatenate(bests), np.concatenate(orefs), np.concatenate(ovs), "f32", min_decidable=0)
    env.close(); pol.close()


@pytest.mark.gpu
@pytest.mark.parametrize("m", MAPS, ids=lambda m: "%dx%dx%g" % m)
def test_transform_vs_oracle(mcn, oracle_mod, m):
    """cn_policy_transform (SARL) and cn_policy_last_state (LSTM-RL, humans sorted by decreasing distance) == the oracle's
    rows and maps bit for bit: random scenes of 1, 2, 13 and 64 humans and the edge scenes."""
    o = oracle_mod
    omc = om_cfg(o, m)
    rng = np.random.default_rng(m[0] + 7 * m[1])
    groups = [np.stack([random_agents(rng, H) for _ in range(6)]) for H in (1, 2, 13, 64)]
    groups.append(np.stack([edge_agents(m[0], cs) for cs in sorted({m[2], 1.0, 0.5})]))
    for name in ("sarl_default", "lstm_default"):
        c = (name, m)
        pol = mcn.BatchedSARL(precision="f32", **policy_kwargs(c))
        for agents in groups:
            E, H = agents.shape[0], agents.shape[1] - 1
            env = mcn.BatchedCrowdSim(E, H)
            env.set_state(agents)
            lstm = name.startswith("lstm")
            got = pol.transform(env, last_state=lstm).cpu().numpy()
            for e in range(E):
                order = o.lstm_human_order(agents[e]) if lstm else np.arange(H)
                ref = o.transform_om(omc, agents[e], order=order if lstm else None)
                # the 13 rotated features to float32 trigonometry (5e-6, as test_gpu_parity), the maps bit for bit
                assert np.max(np.abs(got[e][:, :13] - ref[:, :13])) < 5e-6, (name, H, e)
                rows = order == 0 if agents is groups[-1] else slice(None)      # edge scenes: human 1's map
                gm, rm = got[e][rows, 13:], ref[rows, 13:]
                assert np.array_equal(gm.view(np.uint32), rm.view(np.uint32)), (name, H, e, np.argwhere(gm != rm)[:5])
            env.close()
        pol.close()


def _forward_cases(c):
    """(humans, batch) pairs: batches that leave a partial last chunk of the 64 // H samples per CTA"""
    out = []
    for H in (1, 5, 13, 64):
        if SHAPES[c[0]]["net"] == "cadrl" and H not in (1, 5, 13):
            continue
        ca = 64 // H
        out += [(H, B) for B in sorted({1, ca - 1, ca + 1, 1001}) if B > 0]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("c", CONFIGS, ids=cfg_id)
def test_policy_forward_vs_torch_float64(mcn, c):
    """cn_policy_forward (the TD targets) against the torch module in float64 within 1e-5 relative, for batches that fill
    the per-CTA sample chunks and leave a partial one; CADRL with several humans against torch's min over the rows."""
    import torch
    w = weights(c, "x4")
    pol = mcn.BatchedSARL(precision="f32", **policy_kwargs(c))
    pol.load_weights(w)
    model = _load(torch_model(c), w).double().cuda()
    g = torch.Generator().manual_seed(11)
    D = 13 + om_dim(c[1])
    for H, B in _forward_cases(c):
        x = torch.rand((B, H, D), generator=g) * 4 - 2
        x[..., 2] = 0.0
        if c[1] is not None and c[1][1] != 2:
            x[..., 13::c[1][1]] = (x[..., 13::c[1][1]] > 0).float()        # occupancy flags
        x = x.cuda()
        out = pol.forward(x)
        with torch.no_grad():
            if SHAPES[c[0]]["net"] == "cadrl":
                ref = model(x.double().reshape(-1, D)).reshape(B, H).min(dim=1).values
            else:
                ref = model(x.double()).reshape(-1)
        assert scaled_errors(out.cpu().numpy(), ref.cpu().numpy(), "x4") <= 1.0, (H, B)
    pol.close()


@pytest.mark.gpu
@pytest.mark.parametrize("c", CONFIGS, ids=cfg_id)
def test_param_counts_and_trainer_shapes(mcn, c):
    """cn_policy_param_count = cn_trainer_param_count = the torch module's count; the trainer refuses exactly the shapes
    TRAINER_REFUSALS lists, with CN_EUNSUPPORTED and a message."""
    lib = mcn._capi.load()
    cfg = capi_cfg(mcn, c)
    n = sum(p.numel() for p in torch_model(c).parameters())
    assert int(lib.cn_policy_param_count(C.byref(cfg))) == n
    h = C.c_void_p()
    rc = lib.cn_trainer_create(C.byref(cfg), 0, 128, 1 if SHAPES[c[0]]["net"] == "cadrl" else 16, C.byref(h))
    if cfg_id(c) in TRAINER_REFUSALS:
        assert rc == mcn._capi.CN_EUNSUPPORTED and lib.cn_last_error(), rc
        return
    mcn._capi.check(rc)
    assert int(lib.cn_trainer_param_count(h)) == n
    lib.cn_trainer_destroy(h)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [c for c in CONFIGS if cfg_id(c) not in TRAINER_REFUSALS], ids=cfg_id)
def test_fused_trainer_vs_autograd_float64(mcn, no_tf32, c):
    """One cn_trainer_step with grad_out against autograd on model.double() (loss within 1e-6 relative, every gradient entry
    within 2e-5 of the largest), for 1, 37 and 128 samples of 1, 3 and 16 humans; then 20 Trainer(mode="fused") steps
    against mode="eager", weights within 1e-5."""
    import torch
    from modelcrowdnav_b200._capi import check
    from modelcrowdnav_b200.fused_trainer import FusedTrainer
    from modelcrowdnav_b200.trainer import Trainer
    dev = torch.device("cuda:0")
    cadrl = SHAPES[c[0]]["net"] == "cadrl"
    D = 13 + om_dim(c[1])
    w0 = weights(c, 1.0, seed=5)
    g = torch.Generator().manual_seed(3)

    def batch(B, H):
        x = torch.rand((B, D) if cadrl else (B, H, D), generator=g) * 4 - 2
        x[..., 2] = 0.0
        return x.to(dev).contiguous(), (torch.rand((B, 1), generator=g) - 0.25).to(dev)

    ft = FusedTrainer(_load(torch_model(c), w0).to(dev), dev)
    for B, H in ((1, 1), (37, 3), (128, 16)):
        H = 1 if cadrl else H
        x, y = batch(B, H)
        ft.sync_from_model()
        loss = torch.zeros((), device=dev)
        check(ft.lib.cn_trainer_step(ft.handle, C.c_void_p(ft.flat.data_ptr()), C.c_void_p(x.data_ptr()),
                                     C.c_void_p(y.reshape(-1).contiguous().data_ptr()), B, H, 0.01, 0.9,
                                     C.c_void_p(ft.grad.data_ptr()), C.c_void_p(loss.data_ptr()), ft._stream()))
        torch.cuda.synchronize()
        ref_model = _load(torch_model(c), w0).double().to(dev)
        torch.nn.functional.mse_loss(ref_model(x.double()), y.double()).backward()
        ref = torch.cat([p.grad.reshape(-1) for p in ref_model.parameters()]).cpu().numpy()
        got = ft.grad.cpu().numpy()
        with torch.no_grad():
            ref_loss = ((ref_model(x.double()) - y.double()) ** 2).mean()
        # relative to the larger of the loss and the targets' mean square: one sample's (value - target) can cancel
        assert abs(float(loss) - float(ref_loss)) <= 1e-6 * max(float(ref_loss), float((y.double() ** 2).mean())), (
            B, H, float(loss), float(ref_loss))
        assert np.max(np.abs(got - ref)) <= 2e-5 * np.abs(ref).max(), (B, H, np.max(np.abs(got - ref)), np.abs(ref).max())
    ft.close()

    memory = mcn.ReplayMemory(100000, device=dev)
    x, y = batch(600, 5)
    memory.push_batch(x, y)
    idx = torch.randint(len(memory), (20, 100), generator=torch.Generator().manual_seed(2)).to(dev)
    out = {}
    for mode in ("eager", "fused"):
        model = _load(torch_model(c), w0).to(dev)
        tr = Trainer(model, memory, dev, 100, mode=mode)
        tr.set_learning_rate(0.01)
        for i in range(idx.shape[0]):
            tr._step(idx[i])
        tr._after()
        out[mode] = _flat(model)
    assert np.max(np.abs(out["fused"] - out["eager"])) <= 1e-5, np.max(np.abs(out["fused"] - out["eager"]))
    assert np.max(np.abs(out["eager"] - w0)) > 0


def _tc_cases():
    return [pytest.param(m, gs, id="%dx%dx%g-%s" % (*m, "gs" if gs else "nogs")) for m in MAPS for gs in (True, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("m,gs", _tc_cases())
def test_tc_om_sarl_map_shapes(mcn, oracle_mod, m, gs):
    """OM-SARL on the tensor cores at every map shape (tc_om_bias_kernel over om_dim 1 .. 192), for 1, 5, 10, 13 and 50 humans
    (the compile-time H = 5 and 10 row kernels and the run-time-H one): against FP32 on ~500 auto-reset envs with the fp16
    bars and the argmax bar, and against the oracle on 16 of them.  The trained weights the fp16 bars were measured on
    (conftest.py): seeded weights leave most states tied, and scaled ones give fp16 rounding of activations ~10x larger than
    the values, which the 1e-3-relative bar does not allow for."""
    o = oracle_mod
    c = ("sarl_default" if gs else "sarl_default_nogs", m)
    w = trained_weights(c)
    ocfg, wo = oracle_net(o, c, w)
    kw = policy_kwargs(c)
    p32, p16 = mcn.BatchedSARL(precision="f32", **kw), mcn.BatchedSARL(precision="f16_tc", **kw)
    p32.load_weights(w); p16.load_weights(w)
    for H in (1, 5, 10, 13, 50):
        E = 500 if H <= 13 else 200
        env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=H, sim_rule=1 if H > 10 else 0)
        env.reset_device()
        for _ in range(3):
            env.orca(); env.robot_orca(0.0); env.step(update=True, read=False)
        env.orca()
        p32.lookahead(env); b32, v32 = p32.read(env)
        p16.lookahead(env); b16, v16 = p16.read(env)
        assert value_errors(v16, v32, "f16_tc") <= 1.0, (H, np.abs(v16 - v32).max())
        regret = v32.max(axis=1) - v32[np.arange(E), b16]
        assert np.all(regret <= TIE_GAP["f16_tc"]), (H, regret.max())
        check_argmax(b16, b32, v32, "f16_tc", min_decidable=E // 4)
        cur, times = env.get_state()
        hv = env.human_actions()
        for e in np.random.default_rng(H).choice(E, 16, replace=False):
            ov = oracle_lookahead(o, c, ocfg, wo, cur[e], times[e], p16.action_table, False, hv[e], 0, 0.0)[1]
            assert value_errors(v32[e], ov, "f32") <= 1.0, (H, e)
            assert value_errors(v16[e], ov, "f16_tc") <= 1.0, (H, e)
        env.close()
    p32.close(); p16.close()


@pytest.mark.gpu
@pytest.mark.parametrize("extra", ["[sarl]\nmlp1_dims = 37, 23\nmlp2_dims = 19, 7\nattention_dims = 13, 5, 1\n"
                                   "mlp3_dims = 29, 11, 3, 1\n",
                                   "[sarl]\nwith_om = true\n[om]\ncell_num = 2\nom_channel_size = 2\ncell_size = 0.5\n"],
                         ids=["sarl_odd", "om2x2x0.5"])
def test_training_loop_non_default_shapes(mcn, no_tf32, tmp_path, extra):
    """TrainingLoop(policy_name="sarl", trainer_mode="fused") with non-default [sarl] widths or [om] settings: imitation
    learning and one RL iteration run (the explorer's lookahead included), the losses are finite, and the FP32 lookahead
    network of the trained model computes the torch model's values within 1e-5."""
    import torch
    from modelcrowdnav_b200.train_loop import TrainingLoop
    cfg = tmp_path / "policy.config"
    cfg.write_text(extra)
    loop = TrainingLoop(torch.device("cuda:0"), policy_name="sarl", trainer_mode="fused", sample_episodes=8,
                        policy_config=str(cfg))
    il_loss = loop.imitation_learning(il_episodes=16, il_epochs=2)
    assert loop.trainer._fused is not None
    loop.start_rl()
    loss = loop.rl_iteration(0.5, train_batches=10)
    assert np.isfinite(il_loss) and np.isfinite(loss), (il_loss, loss)
    x = loop.memory.states[:min(len(loop.memory), 256)].contiguous()
    got = loop.policy.handle(1.0, precision="f32").forward(x).cpu().numpy()
    with torch.no_grad():
        ref = loop.model(x).reshape(-1).cpu().numpy()
    assert value_errors(got, ref, "f32") <= 1.0


@pytest.mark.gpu
def test_shared_memory_refusal(mcn, oracle_mod):
    """All-256 SARL layers with 8 x 8 x 3 maps: 64 humans need 64 rows of 205 + 3 x 256 floats for ONE action (308 kB of
    shared memory), which the FP32 lookahead and forward refuse with CN_EUNSUPPORTED and a message; at 13 humans the same
    handle runs (fewer actions per CTA) and matches the oracle and float64 torch."""
    import torch
    o, lib = oracle_mod, mcn._capi.load()
    c = ("sarl_wide", (8, 3, 1.0))
    w = weights(c, 1.0)
    ocfg, wo = oracle_net(o, c, w)
    pol = mcn.BatchedSARL(precision="f32", **policy_kwargs(c))
    pol.load_weights(w)
    model = _load(torch_model(c), w).double().cuda()
    for H in (13, 64):
        env = mcn.BatchedCrowdSim(1, H)
        env.set_state(_scenes(o, 1, H))
        env.orca()
        x = torch.rand((3, H, 13 + om_dim(c[1])), generator=torch.Generator().manual_seed(H)).cuda()
        out = torch.empty(3, device="cuda")
        rcs = (lib.cn_policy_lookahead(pol.handle, env.handle, 0, 0.0, None),
               lib.cn_policy_forward(pol.handle, C.c_void_p(x.data_ptr()), 3, H, C.c_void_p(out.data_ptr()), None))
        if H == 64:
            for rc in rcs:
                assert rc == mcn._capi.CN_EUNSUPPORTED and b"shared memory" in lib.cn_last_error(), rc
            env.close()
            continue
        assert rcs == (mcn._capi.CN_OK, mcn._capi.CN_OK)
        _, values = pol.read(env)
        cur, times = env.get_state()
        ov = oracle_lookahead(o, c, ocfg, wo, cur[0], times[0], pol.action_table, False, env.human_actions()[0], 0, 0.0)[1]
        assert value_errors(values[0], ov, "f32") <= 1.0
        torch.cuda.synchronize()
        with torch.no_grad():
            assert value_errors(out.cpu().numpy(), model(x.double()).reshape(-1).cpu().numpy(), "f32") <= 1.0
        env.close()
    pol.close()
