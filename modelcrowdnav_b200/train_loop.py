"""Value-network training loop on the B200 backend: crowd_nav/train.py:85-251 (BASELINE.json configs[3]).

  imitation learning : ORCA robot (safety_space 0.15) -> replay (return-to-go targets) -> il_epochs of SGD
  reinforcement      : epsilon-greedy roll-outs -> TD targets from the target network -> train_batches of SGD,
                       target sync every target_update_interval

One process per GPU: every rank rolls out its OWN, disjoint shard of episode cases side by side as one env batch, keeps a
rank-local replay buffer, and all-reduces value-net gradients (one 386 kB bucket per SGD step) and episode statistics over
NCCL -- never anything inside the env step / lookahead (SURVEY §8(e)).

`TrainingLoop` is shared by scripts/train_sarl.py (full runs) and `bench.py --workload train` (`bench_train`: one RL
iteration per timed step, phase split, all-reduce latency).
"""
import configparser
import json
import logging
import os
import time

import numpy as np

ENV_DEFAULT = dict(env=dict(time_limit=25, time_step=0.25, val_size=100, test_size=500, randomize_attributes="false"),
                   reward=dict(success_reward=1, collision_penalty=-0.25, discomfort_dist=0.2,
                               discomfort_penalty_factor=0.5),
                   sim=dict(train_val_sim="circle_crossing", test_sim="circle_crossing", square_width=10,
                            circle_radius=4, human_num=5),
                   humans=dict(visible="true", policy="orca", radius=0.3, v_pref=1, sensor="coordinates"),
                   robot=dict(visible="false", policy="none", radius=0.3, v_pref=1, sensor="coordinates"))
POLICY_DEFAULT = dict(rl=dict(gamma=0.9), om=dict(cell_num=4, cell_size=1, om_channel_size=3),
                      action_space=dict(kinematics="holonomic", speed_samples=5, rotation_samples=16,
                                        sampling="exponential", query_env="false"),
                      sarl=dict(mlp1_dims="150, 100", mlp2_dims="100, 50", attention_dims="100, 100, 1",
                                mlp3_dims="150, 100, 100, 1", multiagent_training="true", with_om="false",
                                with_global_state="true"),
                      cadrl=dict(mlp_dims="150, 100, 100, 1", multiagent_training="false"),
                      lstm_rl=dict(global_state_dim=50, mlp1_dims="150, 100, 100, 50", mlp2_dims="150, 100, 100, 1",
                                   multiagent_training="true", with_om="false", with_interaction_module="false"))


def make_config(default, path=None):
    cp = configparser.RawConfigParser()
    cp.read_dict({k: {kk: str(vv) for kk, vv in v.items()} for k, v in default.items()})
    if path:
        cp.read(path)
    return cp


def shard_cases(base, iteration, world, rank, k):
    """First case id of rank `rank` in roll-out `iteration`: the ranks take consecutive, disjoint blocks of k cases and every
    iteration moves all of them on by world * k, whatever happened before `base` (the imitation-learning cases)."""
    return base + (iteration * world + rank) * k


class TrainingLoop(object):
    def __init__(self, device, rank=0, world=1, group=None, policy_name="sarl", precision="f16_tc", seed=0,
                 env_config=None, policy_config=None, capacity=100000, batch_size=100, trainer_mode="graph",
                 sample_episodes=64):
        import torch
        import modelcrowdnav_b200 as mcn
        from .trainer import Trainer
        self.mcn, self.torch = mcn, torch
        self.rank, self.world, self.group, self.device = rank, world, group, device
        self.sample_episodes = sample_episodes
        env_config, policy_config = make_config(ENV_DEFAULT, env_config), make_config(POLICY_DEFAULT, policy_config)
        torch.manual_seed(seed)
        self.policy = policy = mcn.policy_factory[policy_name]()
        policy.configure(policy_config)
        if policy.precision == "f16_tc":
            policy.precision = precision          # configure() chose FP32 for the shapes the tensor cores do not run
        policy.set_device(device)
        self.env = env = mcn.CrowdSim()
        env.configure(env_config)
        env.device = device.index or 0
        self.robot = robot = mcn.Robot(env_config, "robot")
        env.set_robot(robot)
        env.case_size["train"] = np.iinfo(np.uint32).max - 2000       # upstream CrowdNav value (the fork shrank it to 100)
        self.memory = mcn.ReplayMemory(capacity)
        self.model = policy.get_model()
        self.trainer = Trainer(self.model, self.memory, device, batch_size, dist_group=group, policy=policy, mode=trainer_mode)
        self.trainer.broadcast_weights()
        self.explorer = mcn.Explorer(env, robot, device, self.memory, policy.gamma, target_policy=policy, dist_group=group)
        self.rl_base = 0                  # first train case of the RL phase (common to all ranks)
        self.iteration = 0
        self.env_steps = 0

    # ---- imitation learning (train.py:144-178) ----
    def imitation_learning(self, il_episodes=500, il_epochs=50, il_learning_rate=0.01, safety_space=0.15):
        mcn = self.mcn
        il_policy = mcn.policy_factory["orca"]()
        il_policy.multiagent_training = self.policy.multiagent_training
        il_policy.safety_space = safety_space
        il_policy.set_device(self.device)
        self.robot.set_policy(il_policy)
        per_rank = (il_episodes + self.world - 1) // self.world
        self.env.case_counter["train"] = self.rank * per_rank           # disjoint demonstrations: [r * per_rank, (r + 1) * per_rank)
        self.explorer.run_k_episodes(per_rank, "train", update_memory=True, imitation_learning=True)
        self.rl_base = self.world * per_rank
        self.trainer.set_learning_rate(il_learning_rate)
        loss = self.trainer.optimize_epoch(il_epochs)
        self.explorer.update_target_model(self.model)
        return loss

    # ---- reinforcement learning (train.py:180-246) ----
    def start_rl(self, rl_learning_rate=0.001):
        self.robot.set_policy(self.policy)
        self.policy.set_env(self.env)
        self.trainer.set_learning_rate(rl_learning_rate)
        if self.explorer.target_model is None:
            self.explorer.update_target_model(self.model)

    def rl_iteration(self, epsilon, train_batches=100, target_update_interval=50, timers=None):
        """One outer-loop iteration of train.py:196-238: roll-outs into the replay memory, train_batches SGD steps, and the
        target-network sync every target_update_interval iterations.  timers (optional dict) accumulates seconds per phase."""
        torch = self.torch
        t0 = time.perf_counter()
        self.policy.set_epsilon(epsilon)
        self.env.case_counter["train"] = shard_cases(self.rl_base, self.iteration, self.world, self.rank, self.sample_episodes)
        self.explorer.run_k_episodes(self.sample_episodes, "train", update_memory=True, episode=self.iteration, returnRate=False)
        torch.cuda.synchronize(self.device)
        t1 = time.perf_counter()
        self.env_steps += int(self.explorer.last_run["steps"].sum())
        loss = self.trainer.optimize_batch(train_batches) if len(self.memory) else float("nan")
        torch.cuda.synchronize(self.device)
        t2 = time.perf_counter()
        self.iteration += 1
        if self.iteration % target_update_interval == 0:
            self.explorer.update_target_model(self.model)
        torch.cuda.synchronize(self.device)
        t3 = time.perf_counter()
        if timers is not None:
            timers["rollout_and_targets"] = timers.get("rollout_and_targets", 0.0) + (t1 - t0)
            timers["sgd_and_allreduce"] = timers.get("sgd_and_allreduce", 0.0) + (t2 - t1)
            timers["target_sync"] = timers.get("target_sync", 0.0) + (t3 - t2)
            for k, v in getattr(self.explorer, "last_timing", {}).items():
                timers[k] = timers.get(k, 0.0) + v
        return loss


def allreduce_latency_us(group, device, numel=96502, iters=200):
    """Device time of one gradient-bucket all-reduce (fp32 x numel), CUDA events, back-to-back calls."""
    import torch
    import torch.distributed as dist
    if group is None:
        return None
    buf = torch.zeros(numel, dtype=torch.float32, device=device)
    for _ in range(20):
        dist.all_reduce(buf, group=group)
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        dist.all_reduce(buf, group=group)
    e1.record()
    torch.cuda.synchronize(device)
    return 1e3 * e0.elapsed_time(e1) / iters


def bench_train(a):
    """bench.py --workload train: BASELINE.json configs[3].  A "step" = one RL training iteration on every rank: roll out
    `--train-episodes` episodes per rank side by side (epsilon-greedy SARL lookahead + ORCA step until every episode has
    ended), TD targets from the target network, `--train-batches` SGD-momentum steps of batch 100 with the NCCL gradient
    all-reduce, target sync.  value = iterations/s (max over ranks per iteration)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    group = None
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        group = dist.group.WORLD
    device = torch.device("cuda", local)
    logging.basicConfig(level=logging.WARNING)
    loop = TrainingLoop(device, rank, world, group, precision=a.precision, trainer_mode=a.trainer,
                        sample_episodes=a.train_episodes)
    # a short imitation-learning phase so that the value network (and the roll-outs it drives) is not random-init
    t0 = time.perf_counter()
    il_loss = loop.imitation_learning(il_episodes=256 * world, il_epochs=10)
    torch.cuda.synchronize(device)
    il_s = time.perf_counter() - t0
    loop.start_rl()
    loop.explorer.profile = True

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    steps0 = 0
    for _ in range(max(a.warmup, 3)):
        loop.rl_iteration(0.5, a.train_batches)
    barrier()
    timers = {}
    steps0 = loop.env_steps
    n_iter = a.steps
    t0 = time.perf_counter()
    for _ in range(n_iter):
        loop.rl_iteration(0.5, a.train_batches, timers=timers)
    barrier()
    el = time.perf_counter() - t0
    t = torch.tensor([el, float(loop.env_steps - steps0)], dtype=torch.float64, device=device)
    if world > 1:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        el, env_steps = float(mx[0]), float(sm[1])
    else:
        env_steps = float(t[1])
    ar_us = allreduce_latency_us(group, device)
    if rank == 0:
        line = {"metric": "RL training iterations/s (roll-outs + TD targets + SGD batches + gradient all-reduce)",
                "value": n_iter / el, "unit": "iterations/s", "n_gpus": world, "steps": n_iter, "warmup": max(a.warmup, 3),
                "ms_per_step": 1e3 * el / n_iter, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16 lookahead / f32 training", "data": "synthetic",
                "config": {"workload": "SARL value-network training: %d episodes per rank and iteration (circle_crossing, 5 humans), "
                                       "%d SGD batches of 100, NCCL gradient all-reduce" % (a.train_episodes, a.train_batches),
                           "trainer": a.trainer, "episodes_per_iteration": a.train_episodes * world,
                           "sgd_batches_per_iteration": a.train_batches, "replay_size_rank0": len(loop.memory),
                           "imitation_learning_s": il_s, "il_loss": il_loss},
                "env_steps_per_s": env_steps / el,
                "phase_ms_per_iteration": {k: 1e3 * v / n_iter for k, v in timers.items()},
                "sgd_step_us": 1e6 * timers.get("sgd_and_allreduce", 0.0) / n_iter / max(a.train_batches, 1),
                "allreduce_latency_us": ar_us, "allreduce_bytes": 96502 * 4,
                "gpu_launches": int(loop.policy.handle(1.0).lib.cn_launch_count())}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
