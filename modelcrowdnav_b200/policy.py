"""Host-side mirror of the reference policy interface:

    Policy                    crowd_sim/envs/policy/policy.py:5-49
    ORCA                      crowd_sim/envs/policy/orca.py:7-132      (robot in imitation learning; humans)
    CADRL.set_common_parameters / build_action_space / set_device / set_epsilon   crowd_nav/policy/cadrl.py:57-102
    MultiHumanRL.predict / transform                                             crowd_nav/policy/multi_human_rl.py:11-104
    ValueNetwork, SARL        crowd_nav/policy/sarl.py:9-89
    policy_factory            crowd_nav/policy/policy_factory.py:6-8, crowd_sim/envs/policy/policy_factory.py:9-12

`SARL.get_model()` returns a torch ValueNetwork with the reference's state-dict keys (mlp1.0.weight ...), so
`load_state_dict(torch.load('rl_model.pth'))`, optimisers and checkpoints work unchanged; the lookahead itself
(`predict`) runs on the GPU through the C ABI.  torch is used for tensor hand-off and training only.
"""
import logging

import numpy as np

from . import _capi
from .batch import BatchedCrowdSim, BatchedSARL


class Policy(object):
    def __init__(self):
        self.trainable = False
        self.phase = None
        self.model = None
        self.device = None
        self.last_state = None
        self.time_step = None
        self.env = None

    def configure(self, config):
        return

    def set_phase(self, phase):
        self.phase = phase

    def set_device(self, device):
        self.device = device

    def set_env(self, env):
        self.env = env

    def get_model(self):
        return self.model

    @staticmethod
    def reach_destination(state):
        s = state.self_state
        return bool(np.linalg.norm((s.py - s.gy, s.px - s.gx)) < s.radius)


def _cuda_index(device):
    if device is None:
        return 0
    idx = getattr(device, "index", None)
    return 0 if idx is None else int(idx)


# The unmodified fork never reads [action_space] kinematics (cadrl.py:66 is commented out), so its SARL runs with
# policy.kinematics = None: ActionRot actions with rotations in [-pi/4, pi/4], non-holonomic robot dynamics, heading
# feature zero.  False (default): honour the config key (holonomic in the shipped policy.config, the north-star scope).
# True: reproduce the fork literally.  compat.install_as_reference(literal_kinematics=True) sets it.
LITERAL_FORK_KINEMATICS = False

KIN_CODE = {"holonomic": _capi.KIN_HOLONOMIC, "unicycle": _capi.KIN_UNICYCLE, None: _capi.KIN_NONE}


def joint_state_to_agents(state):
    """JointState -> (H+1, 8) exchange rows [px py vx vy gx gy radius v_pref]; unknown human goals = position."""
    s = state.self_state
    rows = [[s.px, s.py, s.vx, s.vy, s.gx, s.gy, s.radius, s.v_pref]]
    for h in state.human_states:
        rows.append([h.px, h.py, h.vx, h.vy, h.px, h.py, h.radius, 1.0])
    return np.asarray(rows, dtype=np.float64)


class ORCA(Policy):
    """ORCA policy object (orca.py:7-132).  predict() solves one agent's ORCA problem on the GPU."""

    def __init__(self):
        super().__init__()
        self.name = "ORCA"
        self.trainable = False
        self.multiagent_training = None
        self.kinematics = "holonomic"
        self.safety_space = 0
        self.neighbor_dist = 10
        self.max_neighbors = 10
        self.time_horizon = 5
        self.time_horizon_obst = 5
        self.radius = 0.3
        self.max_speed = 1
        self._batch = None

    def predict(self, state):
        from .envs import ActionXY
        agents = joint_state_to_agents(state)
        H = agents.shape[0] - 1
        if self._batch is None or self._batch.H != H:
            self._batch = BatchedCrowdSim(1, H, device=_cuda_index(self.device), time_step=self.time_step or 0.25,
                                          neighbor_dist=self.neighbor_dist, max_neighbors=self.max_neighbors,
                                          time_horizon=self.time_horizon)
        b = self._batch
        b.set_state(agents[None])
        b.robot_orca(self.safety_space)      # self = agent 0, others in list order (orca.py:99-110)
        xy, _ = b.pending_actions()
        self.last_state = state
        return ActionXY(float(xy[0, 0]), float(xy[0, 1]))


class Linear(Policy):
    """Straight-to-goal policy (crowd_sim/envs/policy/linear.py:6-24): host arithmetic, numpy like the reference."""

    def __init__(self):
        super().__init__()
        self.name = "Linear"
        self.trainable = False
        self.kinematics = "holonomic"
        self.multiagent_training = True

    def configure(self, config):
        assert True

    def predict(self, state):
        from .envs import ActionXY
        self_state = state.self_state
        theta = np.arctan2(self_state.gy - self_state.py, self_state.gx - self_state.px)
        return ActionXY(np.cos(theta) * self_state.v_pref, np.sin(theta) * self_state.v_pref)

    @staticmethod
    def batch_actions(agents):
        """predict() for the robots of a batch: agents (E, H+1, 8) -> (E, 2)."""
        r = agents[:, 0]
        theta = np.arctan2(r[:, 5] - r[:, 1], r[:, 4] - r[:, 0])
        return np.stack([np.cos(theta) * r[:, 7], np.sin(theta) * r[:, 7]], axis=1)


def mlp(input_dim, mlp_dims, last_relu=False):
    """cadrl.py:11-19"""
    import torch.nn as nn
    layers = []
    mlp_dims = [input_dim] + list(mlp_dims)
    for i in range(len(mlp_dims) - 1):
        layers.append(nn.Linear(mlp_dims[i], mlp_dims[i + 1]))
        if i != len(mlp_dims) - 2 or last_relu:
            layers.append(nn.ReLU())
    return nn.Sequential(*layers)


def make_value_network(input_dim, self_state_dim, mlp1_dims, mlp2_dims, mlp3_dims, attention_dims,
                       with_global_state=True):
    """torch ValueNetwork with the reference's parameter names and forward (sarl.py:9-65); used for
    checkpoints, training (autograd) and as the source of the weights uploaded to the CUDA lookahead."""
    import torch
    import torch.nn as nn

    class ValueNetwork(nn.Module):
        """Parameter container (state-dict keys mlp1.* mlp2.* attention.* mlp3.*) + the autograd form of the network the
        CUDA kernels evaluate; all layers act on the last axis of (batch, humans, features) tensors."""

        def __init__(self):
            super().__init__()
            self.self_state_dim = self_state_dim
            self.global_state_dim = mlp1_dims[-1]
            self.with_global_state = with_global_state
            self.mlp1 = mlp(input_dim, mlp1_dims, last_relu=True)
            self.mlp2 = mlp(mlp1_dims[-1], mlp2_dims)
            self.attention = mlp(mlp1_dims[-1] * (2 if with_global_state else 1), attention_dims)
            self.mlp3 = mlp(mlp2_dims[-1] + self_state_dim, mlp3_dims)
            self._attn = None

        @property
        def attention_weights(self):
            """softmax weights of the first sample of the last forward (sarl.py:54), fetched from the device on demand --
            the reference copies them to the host inside every forward, i.e. one sync per training step."""
            return None if self._attn is None else self._attn.cpu().numpy()

        def forward(self, state):
            embed = self.mlp1(state)                                   # (B, H, 100): per-human embedding e_i
            feat = self.mlp2(embed)                                    # (B, H, 50):  pairwise feature h_i
            if self.with_global_state:                                 # attention sees [e_i, mean_k e_k]
                embed = torch.cat([embed, embed.mean(dim=1, keepdim=True).expand_as(embed)], dim=2)
            score = self.attention(embed).squeeze(2)                   # (B, H)
            w = torch.exp(score) * (score != 0)                        # un-stabilised softmax, exact zeros masked (sarl.py:52)
            w = w / w.sum(dim=1, keepdim=True)
            self._attn = w[0].detach()
            crowd = (w.unsqueeze(2) * feat).sum(dim=1)                 # (B, 50)
            return self.mlp3(torch.cat([state[:, 0, :self.self_state_dim], crowd], dim=1))

    return ValueNetwork()


class SARL(Policy):
    """SARL with the MultiHumanRL lookahead on the GPU (sarl.py:68-89, multi_human_rl.py:11-104)."""

    def __init__(self):
        super().__init__()
        self.name = "SARL"
        self.trainable = True
        self.multiagent_training = None
        self.kinematics = None
        self.epsilon = None
        self.gamma = None
        self.sampling = None
        self.speed_samples = None
        self.rotation_samples = None
        self.query_env = None
        self.action_space = None
        self.speeds = None
        self.rotations = None
        self.action_values = None
        self.with_om = None
        self.cell_num = self.cell_size = self.om_channel_size = None
        self.self_state_dim = 6
        self.human_state_dim = 7
        self.joint_state_dim = self.self_state_dim + self.human_state_dim
        self.precision = "f16_tc"      # lookahead arithmetic on the GPU: "f16_tc" (tcgen05) or "f32"
        self._dims = None
        self._handles = {}             # (precision, v_pref) -> BatchedSARL
        self._weights_version = None
        self._single = None            # one-env batch used by predict()

    # -- configuration (cadrl.py:64-73, sarl.py:73-86) ---------------------------------------------
    def set_common_parameters(self, config):
        self.gamma = config.getfloat("rl", "gamma")
        # policy.config:14 -- the reference fork comments this read out (cadrl.py:66); the north star specifies the
        # holonomic 81-action space, so the key is honoured unless LITERAL_FORK_KINEMATICS asks for the fork's behaviour
        self.kinematics = None if LITERAL_FORK_KINEMATICS else config.get("action_space", "kinematics")
        self.sampling = config.get("action_space", "sampling")
        self.speed_samples = config.getint("action_space", "speed_samples")
        self.rotation_samples = config.getint("action_space", "rotation_samples")
        self.query_env = config.getboolean("action_space", "query_env")
        self.cell_num = config.getint("om", "cell_num")
        self.cell_size = config.getfloat("om", "cell_size")
        self.om_channel_size = config.getint("om", "om_channel_size")

    def configure(self, config):
        self.set_common_parameters(config)
        if self.kinematics not in KIN_CODE:
            raise NotImplementedError("kinematics must be holonomic, unicycle or None (the fork's literal behaviour)")
        mlp1_dims = [int(x) for x in config.get("sarl", "mlp1_dims").split(", ")]
        mlp2_dims = [int(x) for x in config.get("sarl", "mlp2_dims").split(", ")]
        mlp3_dims = [int(x) for x in config.get("sarl", "mlp3_dims").split(", ")]
        attention_dims = [int(x) for x in config.get("sarl", "attention_dims").split(", ")]
        self.with_om = config.getboolean("sarl", "with_om")
        with_global_state = config.getboolean("sarl", "with_global_state")
        self._dims = dict(mlp1_dims=mlp1_dims, mlp2_dims=mlp2_dims, attn_dims=attention_dims, mlp3_dims=mlp3_dims)
        self._net_kwargs = dict(self._dims, **self._om_kwargs())
        if not with_global_state:
            self._net_kwargs["without_global_state"] = 1
        self.model = make_value_network(self.input_dim(), self.self_state_dim, mlp1_dims, mlp2_dims, mlp3_dims,
                                        attention_dims, with_global_state)
        self.multiagent_training = config.getboolean("sarl", "multiagent_training")
        logging.info("Policy: {} {} global state".format(self.name, "w/" if with_global_state else "w/o"))

    def set_device(self, device):
        self.device = device
        self.model.to(device)

    def set_epsilon(self, epsilon):
        self.epsilon = epsilon

    def get_attention_weights(self):
        return self.model.attention_weights

    def build_action_space(self, v_pref):
        """cadrl.py:82-102; the table itself comes from the C ABI (cn_policy_action_table): (vx, vy) pairs for
        holonomic kinematics, (v, r) pairs otherwise."""
        from .envs import ActionRot, ActionXY
        h = self.handle(v_pref)
        holonomic = self.kinematics == "holonomic"
        self.speeds = [(np.exp((i + 1) / self.speed_samples) - 1) / (np.e - 1) * v_pref
                       for i in range(self.speed_samples)]
        if holonomic:
            self.rotations = np.linspace(0, 2 * np.pi, self.rotation_samples, endpoint=False)
        else:
            self.rotations = np.linspace(-np.pi / 4, np.pi / 4, self.rotation_samples)
        cls = ActionXY if holonomic else ActionRot
        self.action_space = [cls(float(x), float(y)) for x, y in h.action_table]

    # -- GPU handles -------------------------------------------------------------------------------
    def handle(self, v_pref=1.0, precision=None):
        """BatchedSARL for (precision, v_pref) with the torch model's current weights."""
        precision = precision or self.precision
        key = (precision, float(v_pref), self.kinematics)
        if key not in self._handles:
            self._handles[key] = [BatchedSARL(device=_cuda_index(self.device), precision=precision,
                                              kinematics=KIN_CODE[self.kinematics],
                                              speed_samples=self.speed_samples, rotation_samples=self.rotation_samples,
                                              gamma=self.gamma, v_pref=float(v_pref), **self._net_kwargs), None]
        entry = self._handles[key]
        version = self._model_version()
        if entry[1] != version:
            entry[0].load_weights(self.flat_weights())
            entry[1] = version
        return entry[0]

    def _model_version(self):
        return tuple(p._version for p in self.model.parameters()) + tuple(p.data_ptr() for p in self.model.parameters())

    def flat_weights(self):
        return np.concatenate([v.detach().cpu().numpy().ravel() for v in self.model.state_dict().values()]).astype(
            np.float32)

    def sync_weights(self):
        """Force re-upload of the torch model's weights to every GPU handle (after training steps)."""
        for entry in self._handles.values():
            entry[1] = None

    # -- the reference call (multi_human_rl.py:11-63) ---------------------------------------------
    def _single_env(self, state):
        """One-env batch holding `state` (robot heading included) for predict() / transform()."""
        agents = joint_state_to_agents(state)
        H = agents.shape[0] - 1
        kin = KIN_CODE[self.kinematics]
        if self._single is None or self._single.H != H or self._single.cfg.robot_kinematics != kin:
            self._single = BatchedCrowdSim(1, H, device=_cuda_index(self.device), time_step=self.time_step or 0.25,
                                           robot_kinematics=kin)
        self._single.set_state(agents[None])
        if kin != _capi.KIN_HOLONOMIC:
            self._single.set_theta(np.array([float(state.self_state.theta)]))
        return self._single

    def predict(self, state):
        from .envs import ActionRot, ActionXY
        if self.phase is None or self.device is None:
            raise AttributeError("Phase, device attributes have to be set!")
        if self.phase == "train" and self.epsilon is None:
            raise AttributeError("Epsilon attribute has to be set in training phase")
        if self.reach_destination(state):
            return ActionXY(0, 0) if self.kinematics == "holonomic" else ActionRot(0, 0)
        v_pref = state.self_state.v_pref
        if self.action_space is None:
            self.build_action_space(v_pref)
        if self.with_om and len(state.human_states) < 2:
            raise ValueError("need at least one array to concatenate")     # build_occupancy_maps with a single human
        h = self.handle(v_pref)
        if self.query_env:
            # the env façade owns the one-env batch; its ORCA result is shared with the following step()
            b = self.env._ensure_batch()
            self.env._ensure_human_actions(b)
        else:
            b = self._single_env(state)
        eps = float(self.epsilon) if self.phase == "train" else 0.0
        h.lookahead(b, query_env=self.query_env, epsilon=eps)
        try:
            best, values = h.read(b)
        except _capi.CrowdNavError as e:
            if e.code == _capi.CN_EVALUE:      # multi_human_rl.py:57-58
                raise ValueError("Value network is not well trained. ")
            raise
        self.action_values = list(values[0])
        if self.phase == "train":
            self.last_state = self._last_state(state)
        return self.action_space[int(best[0])]

    def transform(self, state):
        """multi_human_rl.py:90-104 -> tensor (H, 13) on self.device."""
        t = self.handle(state.self_state.v_pref).transform(self._single_env(state))[0]
        return t.to(self.device) if self.device is not None else t

    def _last_state(self, state):
        """What predict() stores in last_state (multi_human_rl.py:60-61)."""
        return self.transform(state)

    def input_dim(self):
        """multi_human_rl.py:106-107"""
        return self.joint_state_dim + (self.cell_num ** 2 * self.om_channel_size if self.with_om else 0)

    def _om_kwargs(self):
        """cn_sarl_cfg fields of the occupancy maps.  OM-SARL keeps the tensor-core lookahead (the map enters mlp1.0 as a row
        bias per human, tc_om_bias_kernel); OM-LSTM-RL is FP32 like LSTM-RL itself."""
        if not self.with_om:
            return {}
        if not (1 <= self.cell_num <= 8 and self.om_channel_size in (1, 2, 3)):
            raise NotImplementedError("occupancy maps: 1 <= cell_num <= 8 and om_channel_size in {1, 2, 3}")
        return dict(input_dim=self.input_dim(), with_om=1, cell_num=self.cell_num, cell_size=self.cell_size,
                    om_channel_size=self.om_channel_size)


def make_cadrl_network(input_dim, mlp_dims):
    """torch ValueNetwork of CADRL with the reference's parameter names (cadrl.py:22-30)."""
    import torch.nn as nn

    class ValueNetwork(nn.Module):
        def __init__(self):
            super().__init__()
            self.value_network = mlp(input_dim, mlp_dims)

        def forward(self, state):
            return self.value_network(state)

    return ValueNetwork()


def make_lstm_network(input_dim, self_state_dim, mlp1_dims, mlp_dims, lstm_hidden_dim):
    """torch ValueNetwork1 (mlp1_dims None) / ValueNetwork2 of LSTM-RL with the reference's parameter names and
    registration order (lstm_rl.py:9-66); the initial LSTM state follows the input's device."""
    import torch
    import torch.nn as nn

    class ValueNetwork(nn.Module):
        def __init__(self):
            super().__init__()
            self.self_state_dim = self_state_dim
            self.lstm_hidden_dim = lstm_hidden_dim
            if mlp1_dims:
                self.mlp1 = mlp(input_dim, mlp1_dims)
            self.mlp = mlp(self_state_dim + lstm_hidden_dim, mlp_dims)
            self.lstm = nn.LSTM(mlp1_dims[-1] if mlp1_dims else input_dim, lstm_hidden_dim, batch_first=True)

        def forward(self, state):
            size = state.shape
            self_state = state[:, 0, :self.self_state_dim]
            seq = state
            if mlp1_dims:
                seq = self.mlp1(state.reshape((-1, size[2]))).reshape((size[0], size[1], -1))
            h0 = torch.zeros(1, size[0], self.lstm_hidden_dim, device=state.device)
            c0 = torch.zeros(1, size[0], self.lstm_hidden_dim, device=state.device)
            _, (hn, _) = self.lstm(seq, (h0, c0))
            return self.mlp(torch.cat([self_state, hn.squeeze(0)], dim=1))

    return ValueNetwork()


def _no_attention_weights(self):
    raise AttributeError("this policy has no attention weights")


class CADRL(SARL):
    """CADRL behind the same GPU lookahead (cadrl.py:32-216): the value network scores every (robot, human) pair and an
    action is worth reward + gamma_bar * MIN over the humans (CN_NET_CADRL).  The default [cadrl] mlp_dims run on the tensor
    cores (tc_mlp3_pair_kernel<1>), any other shape on the FP32 kernels."""

    def __init__(self):
        super().__init__()
        self.name = "CADRL"
        self.precision = "f32"

    def configure(self, config):
        self.set_common_parameters(config)
        if self.kinematics not in KIN_CODE:
            raise NotImplementedError("kinematics must be holonomic, unicycle or None (the fork's literal behaviour)")
        mlp_dims = [int(x) for x in config.get("cadrl", "mlp_dims").split(", ")]
        if len(mlp_dims) != 4 or mlp_dims[-1] != 1:
            raise NotImplementedError("the CUDA CADRL network is mlp(13 -> a, b, c, 1)")
        self.model = make_cadrl_network(self.joint_state_dim, mlp_dims)
        self.multiagent_training = config.getboolean("cadrl", "multiagent_training")
        self.with_om = False
        self._dims = dict(mlp3_dims=mlp_dims)
        self._net_kwargs = dict(network="cadrl", mlp3_dims=mlp_dims)
        self.precision = "f16_tc" if mlp_dims == [150, 100, 100, 1] else "f32"
        logging.info("Policy: CADRL without occupancy map")

    # the reference's CADRL has no get_attention_weights; CrowdSim.step probes it with hasattr (crowd_sim.py:408-411)
    get_attention_weights = property(_no_attention_weights)

    def transform(self, state):
        """cadrl.py:202-216: single-human joint state -> tensor (13,)."""
        assert len(state.human_states) == 1
        return super().transform(state)[0]


class LstmRL(SARL):
    """LSTM-RL behind the same GPU lookahead (lstm_rl.py:69-105): predict() sorts the humans by decreasing distance to the
    robot, the value network runs an LSTM over them (CN_NET_LSTM_RL).  The default network (no interaction module, no
    occupancy maps, global_state_dim 50) runs on the tensor cores (tc_lstm_pair_kernel), the others on the FP32 kernels."""

    def __init__(self):
        super().__init__()
        self.name = "LSTM-RL"
        self.precision = "f32"
        self.with_interaction_module = None
        self.interaction_module_dims = None

    def configure(self, config):
        self.set_common_parameters(config)
        if self.kinematics not in KIN_CODE:
            raise NotImplementedError("kinematics must be holonomic, unicycle or None (the fork's literal behaviour)")
        mlp_dims = [int(x) for x in config.get("lstm_rl", "mlp2_dims").split(", ")]
        global_state_dim = config.getint("lstm_rl", "global_state_dim")
        self.with_om = config.getboolean("lstm_rl", "with_om")
        with_interaction_module = config.getboolean("lstm_rl", "with_interaction_module")
        mlp1_dims = [int(x) for x in config.get("lstm_rl", "mlp1_dims").split(", ")] if with_interaction_module else None
        if len(mlp_dims) != 4 or mlp_dims[-1] != 1 or (mlp1_dims and len(mlp1_dims) != 4):
            raise NotImplementedError("the CUDA LSTM-RL network uses 4-layer mlps ending in 1 unit")
        self.with_interaction_module = with_interaction_module
        self.model = make_lstm_network(self.input_dim(), self.self_state_dim, mlp1_dims, mlp_dims, global_state_dim)
        self.multiagent_training = config.getboolean("lstm_rl", "multiagent_training")
        self._dims = dict(mlp3_dims=mlp_dims)
        self._net_kwargs = dict(network="lstm_rl", mlp3_dims=mlp_dims, lstm_hidden=global_state_dim,
                                lstm_mlp1_dims=mlp1_dims or [0, 0, 0, 0], **self._om_kwargs())
        tc_shape = (not with_interaction_module and not self.with_om and global_state_dim == 50 and
                    mlp_dims == [150, 100, 100, 1] and self.self_state_dim == 6)
        self.precision = "f16_tc" if tc_shape else "f32"
        logging.info("Policy: {}LSTM-RL {} pairwise interaction module".format(
            "OM-" if self.with_om else "", "w/" if with_interaction_module else "w/o"))

    get_attention_weights = property(_no_attention_weights)      # as for CADRL

    def _last_state(self, state):
        # predict() re-orders state.human_states in place before calling MultiHumanRL.predict (lstm_rl.py:99-105)
        def dist(human):
            return np.linalg.norm(np.array(human.position) - np.array(state.self_state.position))
        state.human_states = sorted(state.human_states, key=dist, reverse=True)
        return self.transform(state)


def _none():
    return None


# crowd_nav/policy/policy_factory.py + crowd_sim/envs/policy/policy_factory.py (hot-path policies only)
policy_factory = {"linear": Linear, "orca": ORCA, "none": _none, "sarl": SARL, "cadrl": CADRL, "lstm_rl": LstmRL}
