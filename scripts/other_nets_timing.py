"""Lookahead time of the other value networks (CADRL, LSTM-RL, OM-SARL, SARL and OM-SARL without the global state) on the
tensor-core and FP32 paths.

    python scripts/other_nets_timing.py [E] [H]      (GPU box; prints one line per network and precision)
    python scripts/other_nets_timing.py --split      (SARL with / without the global state, alternating in one process:
                                                      lookahead, per-kernel times and the whole rollout step at 8192 x 5,
                                                      8192 x 10 and 4096 x 50, with the card's name and power limit)
"""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import modelcrowdnav_b200 as mcn  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


OM = dict(input_dim=61, with_om=1, cell_num=4, cell_size=1.0, om_channel_size=3)
NOGS = dict(without_global_state=1)


def drop_global_state(w, input_dim):
    """The same weights for [sarl] with_global_state = false: attention.0 keeps its 100 mlp1_out columns (default dims)."""
    off = (input_dim * 150 + 150) + (150 * 100 + 100) + (100 * 100 + 100) + (100 * 50 + 50)     # mlp1.*, mlp2.*
    wa = w[off:off + 100 * 200].reshape(100, 200)[:, :100]
    return np.concatenate([w[:off], wa.ravel(), w[off + 100 * 200:]]).astype(np.float32)


def policy(net, precision):
    if net in ("sarl", "sarl_nogs"):
        return mcn.BatchedSARL(precision=precision, **(NOGS if net == "sarl_nogs" else {}))
    if net in ("om_sarl", "om_sarl_nogs"):
        return mcn.BatchedSARL(precision=precision, **OM, **(NOGS if net == "om_sarl_nogs" else {}))
    if net == "cadrl":
        return mcn.BatchedSARL(precision=precision, network="cadrl", mlp3_dims=[150, 100, 100, 1])
    return mcn.BatchedSARL(precision=precision, network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50,
                           lstm_mlp1_dims=[0, 0, 0, 0])


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip()


def flop_per_env_step(H, gs):
    """Row network + mlp3 of the 81 candidate actions: attention.0 is 200 -> 100 with the global state, 100 -> 100 without."""
    return 81 * ((124100 if gs else 104100) * H + 67000)


def split(rounds=5, n=50):
    trained = np.load(os.path.join(GOLDEN, "sarl_weights_trained.npy"))
    w = {"sarl": trained, "sarl_nogs": drop_global_state(trained, 13)}
    print("card: %s" % card())
    for E, H in ((8192, 5), (8192, 10), (4096, 50)):
        rule = dict(sim_rule=1) if H == 50 else {}
        envs, pols = {}, {}
        for net in ("sarl", "sarl_nogs"):
            envs[net] = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=3, **rule)
            envs[net].reset_device()
            for _ in range(8):
                envs[net].orca()
                envs[net].robot_orca(0.0)
                envs[net].step(update=True, read=False)
            envs[net].orca()
            pols[net] = policy(net, "f16_tc")
            pols[net].load_weights(w[net])
            for _ in range(5):
                pols[net].lookahead(envs[net], 0)
        res = {net: {"look": [], "step": [], "k": []} for net in pols}
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(rounds):
            for net in ("sarl", "sarl_nogs") if r % 2 == 0 else ("sarl_nogs", "sarl"):
                pol, env = pols[net], envs[net]
                torch.cuda.synchronize()
                a.record()
                for _ in range(n):
                    pol.lookahead(env, 0)
                b.record()
                torch.cuda.synchronize()
                res[net]["look"].append(a.elapsed_time(b) / n)
                pol.kernel_timing(True)
                ks = []
                for _ in range(10):
                    pol.lookahead(env, 0)
                    ks.append(pol.kernel_ms())
                pol.kernel_timing(False)
                res[net]["k"].append({k: float(np.median([x[k] for x in ks])) for k in ks[0]})
                torch.cuda.synchronize()
                a.record()
                for _ in range(n):
                    mcn.rollout_step(pol, env)
                b.record()
                torch.cuda.synchronize()
                res[net]["step"].append(a.elapsed_time(b) / n)
        for net in ("sarl", "sarl_nogs"):
            x = res[net]
            look, step = np.median(x["look"]), np.median(x["step"])
            kern = {k: np.median([d[k] for d in x["k"]]) for k in x["k"][0]}
            fl = flop_per_env_step(H, net == "sarl") * E
            print("%-9s E=%d H=%d  lookahead %.4f ms (min %.4f max %.4f)  kernels features %.4f rows %.4f mlp3 %.4f argmax %.4f ms"
                  "  step %.4f ms = %.3e env-steps/s  lookahead %.1f TFLOP/s = %.1f %% of 2250" %
                  (net, E, H, look, min(x["look"]), max(x["look"]), kern["features"], kern["rows"], kern["mlp3"], kern["argmax"],
                   step, E / step * 1e3, fl / look * 1e-9, fl / look * 1e-9 / 2250 * 100))
        for net in pols:
            pols[net].close(); envs[net].close()
    print("card: %s" % card())


def main():
    if "--split" in sys.argv:
        return split()
    E = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
    H = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    nets = np.load(os.path.join(GOLDEN, "units_nets.npz"))
    om = np.load(os.path.join(GOLDEN, "units_om.npz"))
    weights = dict(sarl=np.load(os.path.join(GOLDEN, "sarl_weights_trained.npy")), om_sarl=om["om_sarl_weights"],
                   cadrl=nets["cadrl_weights"], lstm=nets["lstm_weights"])
    weights.update(sarl_nogs=drop_global_state(weights["sarl"], 13), om_sarl_nogs=drop_global_state(weights["om_sarl"], 61))
    env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=3)
    env.reset_device()
    for _ in range(8):
        env.orca()
        env.robot_orca(0.0)
        env.step(update=True, read=False)
    env.orca()
    print("card: %s" % card())
    for net in ("sarl", "om_sarl", "cadrl", "lstm", "sarl_nogs", "om_sarl_nogs"):
        ms = {}
        for precision in ("f16_tc", "f32"):
            pol = policy(net, precision)
            pol.load_weights(weights[net])
            for _ in range(3):
                pol.lookahead(env, 0)
            torch.cuda.synchronize()
            n = 20 if precision == "f16_tc" else 3
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                pol.lookahead(env, 0)
            b.record()
            torch.cuda.synchronize()
            ms[precision] = a.elapsed_time(b) / n
            pol.close()
        print("%-8s E=%d H=%d  lookahead f16_tc %.3f ms  f32 %.3f ms  (x%.1f)" % (net, E, H, ms["f16_tc"], ms["f32"],
                                                                               ms["f32"] / ms["f16_tc"]))


if __name__ == "__main__":
    main()
