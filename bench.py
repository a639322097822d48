#!/usr/bin/env python
"""bench.py -- env-steps/s of the hot path (ORCA step + SARL lookahead) on N B200s of one node.

A "step" = one cn_rollout_step over the whole batch resident on each GPU: ORCA for every human, the
81-action SARL lookahead, CrowdSim.step(update=True) and the auto-reset of finished episodes.
Workload at any N: BASELINE.json configs[1] per GPU -- 8192 batched envs x 5 humans (weak scaling; envs are
sharded by contiguous global id, no data-path collective).  The same JSON line carries, as `extra_configs`, the other
BASELINE.json configurations (configs[2]: square_crossing x 10 humans, 8192 envs / GPU = 65,536 envs on 8 GPUs;
configs[4]: 50 humans x 4096 envs; query_env = 1; the ORCA-only step of imitation learning), a `sustained` leg
(>= 3 s of back-to-back steps, no L2 flush, clocks and throttle reasons sampled) and a `parity_sample` (the last
state of the timed run checked against the CPU oracle).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload rollout|train]
                  [--precision f32|f16_tc] [--envs 8192] [--humans 5] [--query-env 0|1] [--sim circle|square]
                  [--no-extra] [--sustained-seconds 3] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step of the main configuration computed (rank 0's envs) as
DIR/<name>.npy, so that two builds can be compared output for output: the same arguments give the same inputs.
It covers the rollout workload of --impl ours only (--workload train and --impl reference refuse it), and with
several GPUs only rank 0's envs are written.

--impl reference times the reference's CPU algorithm (the oracle port, oracle/crowdnav_oracle.c -- the
reference itself is Python + an un-vendored rvo2 and cannot travel to the GPU box) on the host cores.
--workload train times BASELINE.json configs[3]: one RL training iteration per step (episode roll-outs over the
rank's env shard + TD targets + SGD batches with the NCCL gradient all-reduce + target-network sync).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/s (ORCA step + SARL lookahead)"
UNIT = "env-steps/s"
ROW_FLOPS = 124100          # SURVEY §8(d): FLOP per (env, action, human) row of the value network
GROUP_FLOPS = 67000         # ... per (env, action): mlp3
DRAM_BYTES_FILE = os.path.join(ROOT, "profiles", "ncu_dram_bytes.json")   # written by scripts/ncu_dram_bytes.py from an ncu --set full capture


def flops_per_env_step(H, A=81):
    """SURVEY §8(d): literal ValueNetwork formulation, 2 FLOP/MAC, 81 actions."""
    return A * (ROW_FLOPS * H + GROUP_FLOPS)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops_burst=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm_gbs=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


def load_dram_bytes(precision, E, H):
    """Per-launch dram__bytes_read.sum + dram__bytes_write.sum of the lookahead kernels from the committed ncu capture."""
    try:
        d = json.load(open(DRAM_BYTES_FILE))
        return d.get("%s:%d:%d" % (precision, E, H))
    except Exception:
        return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_mhz_min": min(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU legs (the oracle port is the checker / baseline; it is never on the measured GPU path)
# ------------------------------------------------------------------------------------------------------------------
def cpu_port_rate(E, H, sim, query_env, n_threads, target_s, max_steps=None):
    """Oracle port (C restatement of the reference algorithm) on host cores: env-steps/s over a bounded sample."""
    import oracle
    oracle.build()
    ecfg, scfg = oracle.EnvCfg.default(), oracle.SarlCfg.default()
    rule = "circle_crossing" if sim == "circle" else "square_crossing"
    agents = np.stack([oracle.generate_scene("train", c, human_num=H, rule=rule) for c in range(E)])
    w = oracle.default_sarl_weights(0)
    table = oracle.action_space()
    times = np.zeros(E); done = np.zeros(E, np.uint8)
    oracle.batch_lookahead_step(ecfg, scfg, w, agents, times, table, query_env, done, n_threads=n_threads)  # warm
    t0 = time.perf_counter(); steps = 0
    while True:
        done[:] = 0
        oracle.batch_lookahead_step(ecfg, scfg, w, agents, times, table, query_env, done, n_threads=n_threads)
        steps += 1
        el = time.perf_counter() - t0
        if el >= target_s or (max_steps and steps >= max_steps):
            break
    return steps * E / el, steps, el


def run_reference(a):
    """Reference arm: the reference's CPU implementation of the path = oracle port, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    E = min(a.envs, 64 * cores)
    rate1, _, _ = cpu_port_rate(E, a.humans, a.sim, a.query_env, cores, 1.0)     # size K steps to a few minutes
    per_step = E / rate1
    t_all = []
    import oracle
    ecfg, scfg = oracle.EnvCfg.default(), oracle.SarlCfg.default()
    rule = "circle_crossing" if a.sim == "circle" else "square_crossing"
    agents = np.stack([oracle.generate_scene("train", c, human_num=a.humans, rule=rule) for c in range(E)])
    w = oracle.default_sarl_weights(0); table = oracle.action_space()
    times = np.zeros(E); done = np.zeros(E, np.uint8)
    for i in range(a.warmup + a.steps):
        done[:] = 0
        t0 = time.perf_counter()
        oracle.batch_lookahead_step(ecfg, scfg, w, agents, times, table, a.query_env, done, n_threads=cores)
        if i >= a.warmup:
            t_all.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(t_all))
    value = E / (ms / 1e3)
    sample = "%d envs x %d humans per step (bounded sample of the %d-env workload), %d OpenMP threads" % (
        E, a.humans, a.envs, cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a.envs, a.humans, a.sim, a.query_env), "envs_per_step": E, "humans": a.humans,
                       "query_env": a.query_env, "est_ms_per_step": 1e3 * per_step},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_name(E, H, sim, query_env):
    return "SARL lookahead + ORCA step, %d batched envs x %d humans per GPU, %s_crossing, query_env=%d" % (
        E, H, sim, query_env)


def parity_sample(o, pol, env, query_env, weights, n, seed=0):
    """The CURRENT state of `env` (the one the timed loop left behind): lookahead on the GPU vs the CPU oracle on `n` randomly
    sampled envs.  max_rel = max |dv| / max(|v|, 0.1) (the bar of tests/: 1e-3 for the fp16 tensor-core path);
    argmax_agree = share of sampled envs whose chosen action is optimal under the ORACLE's values up to the tie threshold."""
    ecfg, scfg = o.EnvCfg.default(), o.SarlCfg.default()
    state, times = env.get_state()
    env.orca()
    hv = env.human_actions()
    pol.lookahead(env, query_env)
    best, values = pol.read(env)
    rs = np.random.RandomState(seed)
    sample = np.sort(rs.choice(env.E, min(n, env.E), replace=False))
    max_rel, ok, dec, dec_ok = 0.0, 0, 0, 0
    for e in sample:
        obest, ov, _ = o.lookahead(ecfg, scfg, weights, state[e], times[e], pol.action_table, query_env, hv[e])
        max_rel = max(max_rel, float(np.max(np.abs(values[e] - ov) / np.maximum(np.abs(ov), 0.1))))
        ok += int(ov.max() - ov[best[e]] <= 2e-4)
        top2 = np.sort(ov)[-2:]
        if top2[1] - top2[0] > 2e-4:
            dec += 1; dec_ok += int(best[e] == obest)
    return {"n": int(len(sample)), "max_rel": max_rel, "argmax_agree": ok / len(sample),
            "decidable": dec, "decidable_exact": dec_ok, "rel_bar": 1e-3 if pol.cfg.precision == 1 else 1e-5,
            "checker": "oracle/crowdnav_oracle.c (CPU), same state, same weights"}


DUMP_LIMIT = 64 * 10**6     # bytes written by --dump-outputs in all


def step_outputs(env, pol):
    """What a caller of cn_rollout_step receives from the last step: the next state (auto-reset envs already regenerated),
    the step's reward / done / info / dmin, the chosen action and the lookahead's action values."""
    agents, times = env.get_state()
    reward, done, info, dmin = env.read_outputs()
    action_xy, action_idx = env.pending_actions()
    _, values = pol.read(env)
    return {"agents": agents, "times": times, "reward": reward, "done": done.astype(np.float32),
            "info": info.astype(np.float32), "dmin": dmin, "action_xy": action_xy,
            "action_index": action_idx.astype(np.float32), "values": values}


def dump_outputs(path, outs, limit=DUMP_LIMIT):
    """(E, ...) arrays -> path/<name>.npy.  Above `limit` bytes, a fixed seeded sample of the envs; env_index.npy says which."""
    E = len(outs["reward"])
    per_env = sum(v.nbytes for v in outs.values()) // E + 8
    n = min(E, (limit - 4096 * (len(outs) + 1)) // per_env)
    idx = np.arange(E) if n == E else np.sort(np.random.RandomState(0).choice(E, n, replace=False))
    outs = {k: v[idx] for k, v in outs.items()}
    outs["env_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in outs.items():
        np.save(os.path.join(path, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rollout", choices=["rollout", "train"])
    ap.add_argument("--precision", default=os.environ.get("CN_BENCH_PRECISION", "f16_tc"), choices=["f32", "f16_tc"])
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--humans", type=int, default=5)
    ap.add_argument("--query-env", type=int, default=0)
    ap.add_argument("--sim", default="circle", choices=["circle", "square"])
    ap.add_argument("--e2e-shards", type=int, default=4)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra_configs / sustained (quick A/B runs)")
    ap.add_argument("--sustained-seconds", type=float, default=3.0)
    ap.add_argument("--parity-envs", type=int, default=256)
    ap.add_argument("--preroll", type=int, default=64, help="untimed steps before the warm-up (episodes out of lock step)")
    ap.add_argument("--train-episodes", type=int, default=512, help="--workload train: episodes rolled out per iteration and rank")
    ap.add_argument("--train-batches", type=int, default=100, help="--workload train: SGD batches per iteration")
    ap.add_argument("--trainer", default="fused", choices=["eager", "graph", "fused"],
                    help="--workload train: fused = csrc/trainer.cu (SARL, parity-tested against the reference Trainer), graph = CUDA-graph replay of torch autograd")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "rollout"):
        ap.error("--dump-outputs needs --impl ours --workload rollout")
    a.warmup = max(a.warmup, 3)
    if a.impl == "reference":
        return run_reference(a)
    if a.workload == "train":
        from modelcrowdnav_b200.train_loop import bench_train
        return bench_train(a)

    import torch
    import modelcrowdnav_b200 as mcn
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # host-resident legs: keep every rank's pinned buffers and launch thread on the CPUs next to its GPU (multi-GPU runs only)
    numa_cpus = mcn.pin_to_gpu_numa(local) if world > 1 else 0
    peaks = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(xs):
        t = torch.tensor(list(xs), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    wpath = os.path.join(ROOT, "tests", "golden", "sarl_weights_seed0.npy")
    weights = np.load(wpath)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    tc = a.precision == "f16_tc"

    def make(E, H, sim):
        env = mcn.BatchedCrowdSim(E, H, device=local, auto_reset=1, seed=0, env_id_offset=rank * E,
                                  sim_rule=0 if sim == "circle" else 1)
        pol = mcn.BatchedSARL(device=local, precision=a.precision)
        # SARL weights: default nn.Linear init under torch.manual_seed(0) (no trained weights ship with the reference)
        pol.load_weights(weights)
        env.reset_device()
        return env, pol

    def rooflines(E, H, A, la_ms, kms):
        """Tensor roofline of the dominant kernel (tc_rows_pair_kernel) and of the whole lookahead; the timed kernels run
        alone (L2 flushed between steps, a few ms in total), so `frac` is against the BURST peak."""
        F = flops_per_env_step(H, A)
        out = {}
        if kms:
            ach = E * A * H * ROW_FLOPS / (kms["rows"] / 1e3) / 1e12
            out = {"bound": "tensor", "kernel": "tc_rows_pair_kernel", "achieved": ach, "peak": peaks["tflops_burst"],
                   "unit": "TFLOP/s", "frac": ach / peaks["tflops_burst"], "frac_vs_sustained": ach / peaks["tflops_sustained"],
                   "kernel_ms": kms["rows"], "flops_per_launch": E * A * H * ROW_FLOPS,
                   "peak_source": peaks["source"] + ", burst bf16 (kernel timed alone)",
                   "how": "CUDA events recorded by the library around the kernel on its launching stream (cn_debug_kernel_ms)"}
        ach = E * F / (la_ms / 1e3) / 1e12
        out["lookahead"] = {"achieved": ach, "frac": ach / peaks["tflops_burst"], "frac_vs_sustained": ach / peaks["tflops_sustained"],
                            "ms": la_ms, "flops_per_env_step": F, "kernels_ms": kms}
        return out

    def measure(E, H, sim, query_env, steps, warmup, clocks=False, dump=None):
        """K timed rollout steps of one configuration (device time per step, L2 flushed between steps, max over ranks),
        then the per-phase / per-kernel breakdown of the same step.  dump: directory for the last timed step's outputs."""
        env, pol = make(E, H, sim)
        # pre-roll: the envs start in lock step (all episodes at t = 0, humans far apart, trivially feasible ORCA problems);
        # 64 untimed steps spread them over the episode (crossings, dangers, finished + re-generated episodes) before timing
        for _ in range(a.preroll + warmup):
            mcn.rollout_step(pol, env, query_env)
        barrier()
        sampler = ClockSampler(local).start() if (clocks and rank == 0) else None
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        launches0 = pol.lib.cn_launch_count()
        barrier()
        t_wall0 = time.perf_counter()
        for i in range(steps):
            flush.zero_()
            ev[i][0].record()
            mcn.rollout_step(pol, env, query_env)
            ev[i][1].record()
        barrier()
        t_wall = time.perf_counter() - t_wall0
        launches = pol.lib.cn_launch_count() - launches0
        dev_ms = sum(s.elapsed_time(e) for s, e in ev)
        clk = sampler.stop() if sampler else None
        if dump and rank == 0:                       # before the breakdown below steps the envs further
            dump_outputs(dump, step_outputs(env, pol))
        # per-phase breakdown (events around each phase) and per-kernel durations of the lookahead
        phases = {"orca": 0.0, "lookahead": 0.0, "step": 0.0}
        kms = {"features": 0.0, "rows": 0.0, "mlp3": 0.0, "argmax": 0.0} if tc else None
        nb = min(steps, 20)
        if tc:
            pol.kernel_timing(True)
        for _ in range(nb):
            flush.zero_()
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            marks[0].record(); env.orca()
            marks[1].record(); pol.lookahead(env, query_env)
            marks[2].record(); env.step(update=True, read=False)
            marks[3].record()
            torch.cuda.synchronize()
            for k, name in enumerate(("orca", "lookahead", "step")):
                phases[name] += marks[k].elapsed_time(marks[k + 1]) / nb
            if tc:
                for k, v in pol.kernel_ms().items():
                    kms[k] += v / nb
        if tc:
            pol.kernel_timing(False)
        barrier()
        dev_ms, t_wall = max_over_ranks([dev_ms, t_wall])
        ms_per_step = dev_ms / steps
        res = {"value": world * E / (ms_per_step / 1e3), "ms_per_step": ms_per_step, "phase_ms": phases,
               "kernel_ms": kms, "launches": int(launches), "wall_s": t_wall, "clocks": clk,
               "roofline": rooflines(E, H, pol.A, phases["lookahead"], kms), "bad_envs": pol.bad_count()}
        return env, pol, res

    # ---------------- main configuration (BASELINE.json configs[1]) ----------------
    E, H = a.envs, a.humans
    env, pol, main_res = measure(E, H, a.sim, a.query_env, a.steps, a.warmup, clocks=True, dump=a.dump_outputs)

    # ---- parity of what was just timed: the state the loop left behind vs the CPU oracle (rank 0) ----
    parity = None
    if rank == 0 and a.parity_envs > 0:
        import oracle
        oracle.build()
        parity = parity_sample(oracle, pol, env, a.query_env, weights, a.parity_envs)
        # the same states through the TRAINED network (|V| up to 1, decisive top-2 gaps): the argmax comparison is not vacuous
        wt_path = os.path.join(ROOT, "tests", "golden", "sarl_weights_trained.npy")
        if os.path.exists(wt_path):
            wt = np.load(wt_path)
            pol_t = mcn.BatchedSARL(device=local, precision=a.precision)
            pol_t.load_weights(wt)
            parity["trained_weights"] = parity_sample(oracle, pol_t, env, a.query_env, wt, a.parity_envs)
            pol_t.close()
    barrier()

    # ---- end to end through the C ABI with HOST buffers (pinned), copies inside the timed region ----
    # Every step, every env's state is uploaded from a pinned host block and its new state + reward + done + info +
    # action are downloaded (packed blocks: one H2D and one D2H copy per shard and step).  The E envs are served as
    # `e2e_shards` env handles on their own streams (cn_rollout_step_host_packed_async), so that the PCIe copies of
    # one shard overlap the kernels of the other; the blocking single-handle call is timed next to it.
    ne = max(5, min(a.steps, 50))
    buf = mcn.PackedHostStepBuffers(env)
    a0, t0 = env.get_state()
    buf.agents_in[...] = a0; buf.times_in[...] = t0
    for _ in range(2):
        mcn.rollout_step_host_packed(pol, env, buf, a.query_env)
        buf.swap()
    barrier()
    te0 = time.perf_counter()
    for _ in range(ne):
        mcn.rollout_step_host_packed(pol, env, buf, a.query_env)
        buf.swap()                                   # next step's input = the host state just downloaded (no host copy)
    barrier()
    e2e_blocking_s = time.perf_counter() - te0
    pipe = mcn.PipelinedHostRollout(E, H, weights, device=local, shards=a.e2e_shards, precision=a.precision,
                                    env_id_offset=rank * E, auto_reset=1, seed=0,
                                    sim_rule=0 if a.sim == "circle" else 1)
    pipe.reset_device()
    for _ in range(6):                               # 2 eager steps per shard, then one graph capture per block orientation
        pipe.step(a.query_env)
    pipe.sync()
    barrier()
    te0 = time.perf_counter()
    for _ in range(ne):
        pipe.step(a.query_env)
    pipe.sync()
    barrier()
    e2e_s = time.perf_counter() - te0
    h2d_bytes, d2h_bytes = pipe.h2d_bytes, pipe.d2h_bytes
    pipe.close()
    e2e_s, e2e_blocking_s = max_over_ranks([e2e_s, e2e_blocking_s])

    # ---------------- sustained leg: >= N seconds of back-to-back steps, no flush ----------------
    sustained = None
    if not a.no_extra and a.sustained_seconds > 0:
        barrier()
        sampler = ClockSampler(local).start() if rank == 0 else None
        chunk = 500
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total_ms, nsteps = 0.0, 0
        while total_ms < 1e3 * a.sustained_seconds:
            e0.record()
            for _ in range(chunk):
                mcn.rollout_step(pol, env, a.query_env)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if world > 1:                            # every rank runs the same number of chunks
                ms = max_over_ranks([ms])[0]
            total_ms += ms; nsteps += chunk
        clk = sampler.stop() if sampler else None
        sus_value = world * E * nsteps / (total_ms / 1e3)
        F = flops_per_env_step(H, pol.A)
        sustained = {"value": sus_value, "unit": UNIT, "seconds": total_ms / 1e3, "steps": nsteps,
                     "ms_per_step": total_ms / nsteps, "l2": "no flush, back-to-back launches", "clocks": clk,
                     "tflops_whole_step": sus_value / world * F / 1e12,
                     "frac_vs_sustained_peak": sus_value / world * F / 1e12 / peaks["tflops_sustained"],
                     "frac_vs_burst_peak": sus_value / world * F / 1e12 / peaks["tflops_burst"]}
    st = env.stats()
    env.close(); pol.close()

    # ---------------- the other BASELINE.json configurations, same line ----------------
    extras = []
    if not a.no_extra:
        xs = max(5, min(a.steps, 20))
        specs = [("configs[2] per GPU: square_crossing x 10 humans, 8192 envs / GPU (65,536 envs at 8 GPUs)", 8192, 10, "square", 0),
                 ("configs[4]: dense crowd, 50 humans (square_crossing width 10, max_neighbors 10), 4096 envs / GPU", 4096, 50, "square", 0),
                 ("configs[1] with query_env = 1 (lookahead asks the env for the humans' ORCA step)", E, H, a.sim, 1)]
        for name, xE, xH, xsim, xq in specs:
            e2, p2, r = measure(xE, xH, xsim, xq, xs, 3)
            rec = {"name": name, "workload": workload_name(xE, xH, xsim, xq), "value": r["value"], "unit": UNIT, "n_gpus": world,
                   "steps": xs, "ms_per_step": r["ms_per_step"], "phase_ms": r["phase_ms"], "roofline": r["roofline"],
                   "gpu_launches": r["launches"],
                   "orca_share_of_step": (r["phase_ms"]["orca"] + r["phase_ms"]["step"]) / max(sum(r["phase_ms"].values()), 1e-9)}
            if rank == 0 and xH != H:                # a small oracle check of these kernels at their own size
                import oracle
                rec["parity_sample"] = parity_sample(oracle, p2, e2, xq, weights, 64 if xH <= 10 else 16)
            barrier()
            extras.append(rec)
            e2.close(); p2.close()
        # ORCA-only step: robot and humans driven by ORCA (imitation-learning roll-outs, train.py:157-166): HBM roofline
        xE = E
        env2 = mcn.BatchedCrowdSim(xE, H, device=local, auto_reset=1, seed=0, env_id_offset=rank * xE)
        env2.reset_device()
        def orca_step():
            env2.orca(); env2.robot_orca(0.15); env2.step(update=True, read=False)
        for _ in range(3):
            orca_step()
        barrier()
        ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(xs)]
        for i in range(xs):
            flush.zero_()
            ev2[i][0].record(); orca_step(); ev2[i][1].record()
        barrier()
        ms = max_over_ranks([sum(s.elapsed_time(e) for s, e in ev2) / xs])[0]
        step_bytes = 48 * (H + 1) + 22
        gbs = xE * step_bytes / (ms / 1e3) / 1e9
        extras.append({"name": "step only: ORCA for the humans and the robot + CrowdSim.step (imitation-learning roll-out), no lookahead",
                       "workload": "%d envs x %d humans per GPU, circle_crossing" % (xE, H), "value": world * xE / (ms / 1e3),
                       "unit": "env-steps/s", "n_gpus": world, "steps": xs, "ms_per_step": ms,
                       "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": gbs / peaks["hbm_gbs"], "bytes_per_env_step": step_bytes,
                                    "note": "latency / FP32-issue bound (sequential LP per agent), not HBM bound"}})
        env2.close()

    if rank == 0:
        line = {
            "metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16" if tc else "f32", "data": "synthetic",
            "config": {"workload": workload_name(E, H, a.sim, a.query_env), "envs_per_gpu": E, "humans": H, "actions": 81,
                       "query_env": a.query_env, "precision": a.precision,
                       "weights": "torch.manual_seed(0) default nn.Linear init",
                       "l2": "256 MiB memset between timed steps (outside the event pair)",
                       "wall_s_timed_region": main_res["wall_s"], "phase_ms": main_res["phase_ms"],
                       "preroll_steps": a.preroll,
                       "episodes_finished": st["episodes"], "envs_with_no_finite_value": main_res["bad_envs"]},
            "clocks": main_res["clocks"],
            "e2e": {"value": world * E * ne / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "steps": ne, "shards_per_gpu": a.e2e_shards,
                    "how": "PipelinedHostRollout: pinned host state in and out every step, the copies, host round trip and "
                           "small kernels of one env shard overlap the row kernels of the others; one CUDA-graph launch "
                           "per shard and step",
                    "blocking_single_handle_value": world * E * ne / e2e_blocking_s,
                    "cpu_affinity": ("GPU-local CPUs (%d, NVML)" % numa_cpus) if numa_cpus else "unchanged"},
            "gpu_launches": main_res["launches"],
            "roofline": main_res["roofline"],
            "parity_sample": parity,
        }
        tr = load_dram_bytes(a.precision, E, H)
        line["roofline"]["traffic"] = tr.get("tc_rows_pair_kernel") if tr else None
        line["roofline"]["traffic_lookahead"] = (sum(v for k, v in tr.items() if k.startswith("tc_")) if tr else None)
        line["roofline"]["traffic_source"] = (tr.get("source") if tr else "no ncu capture committed for this configuration")
        line["roofline"]["algorithmic_bytes_per_step"] = E * (48 * (H + 1) + 22)
        if sustained:
            line["sustained"] = sustained
        if extras:
            line["extra_configs"] = extras
        if not a.no_cpu_baseline:
            cores = 1
            n = 16
            rate, steps, el = cpu_port_rate(n, H, a.sim, a.query_env, cores, a.cpu_seconds)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%d steps of %d envs x %d humans, %.1f s, oracle C port, 1 thread" % (
                                        steps, n, H, el)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
