#!/usr/bin/env python
"""Bit-for-bit comparison of what library builds compute: for a fixed seeded matrix of networks, precisions and shapes,
20 auto-reset rollout steps (state, reward, done, info, and the number of kernel launches of every step), then one lookahead
(values, action_idx).  Covers the networks bench.py --dump-outputs does not (OM-SARL, CADRL, LSTM-RL) and the pipelined
host rollout.  Each library runs in its own subprocess (ctypes cannot unload).
Usage: python scripts/ab_outputs.py [--envs 1024] lib_a.so lib_b.so ...   (exit status 1 when any output differs)"""
import argparse
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
STEPS = 20
OM = dict(input_dim=61, with_om=1, cell_num=4, cell_size=1.0, om_channel_size=3)
NETS = {"sarl": {}, "om_sarl": OM, "cadrl": dict(network="cadrl", mlp3_dims=[150, 100, 100, 1]),
        "lstm": dict(network="lstm_rl", mlp3_dims=[150, 100, 100, 1], lstm_hidden=50)}


def matrix():
    """(name, network, precision, humans, query_env); the SARL humans pick the row-kernel templates 5, 10 and 0"""
    out = [("sarl_%s_h%d_q%d" % (prec, H, q), "sarl", prec, H, q)
           for prec in ("f32", "f16_tc") for H in (5, 10, 13) for q in (0, 1)]
    out += [("%s_%s_h5" % (net, prec), net, prec, 5, 0) for net in ("om_sarl", "cadrl", "lstm") for prec in ("f32", "f16_tc")]
    return out


def child(lib, E, path):
    sys.path.insert(0, ROOT)
    import numpy as np
    from modelcrowdnav_b200 import _capi
    _capi.LIB_PATH = os.path.abspath(lib)
    import modelcrowdnav_b200 as mcn
    nets = dict(np.load(os.path.join(GOLDEN, "units_nets.npz")))
    weights = {"sarl": np.load(os.path.join(GOLDEN, "sarl_weights_seed0.npy")),
               "om_sarl": dict(np.load(os.path.join(GOLDEN, "units_om.npz")))["om_sarl_weights"],
               "cadrl": nets["cadrl_weights"], "lstm": nets["lstm_weights"]}
    lib_ = _capi.load()
    res = {}
    for seed, (name, net, prec, H, q) in enumerate(matrix()):
        env = mcn.BatchedCrowdSim(E, H, auto_reset=1, seed=seed, sim_rule=seed % 2)
        pol = mcn.BatchedSARL(precision=prec, **NETS[net])
        pol.load_weights(weights[net])
        env.reset_device()
        launches = []
        for _ in range(STEPS):
            n0 = lib_.cn_launch_count()
            mcn.rollout_step(pol, env, q)
            launches.append(lib_.cn_launch_count() - n0)
        res[name + "/state"], res[name + "/time"] = env.get_state()
        res[name + "/reward"], res[name + "/done"], res[name + "/info"], _ = env.read_outputs()
        res[name + "/launches"] = np.array(launches)
        env.orca()
        pol.lookahead(env, q)
        res[name + "/action_idx"], res[name + "/values"] = pol.read(env)
        env.close(); pol.close()
    name = "pipelined_sarl_4_shards"
    pipe = mcn.PipelinedHostRollout(E, 5, weights["sarl"], shards=4, precision="f16_tc", auto_reset=1, seed=99)
    pipe.reset_device()
    launches = []
    for _ in range(STEPS):
        n0 = lib_.cn_launch_count()
        pipe.step()
        launches.append(lib_.cn_launch_count() - n0)
    pipe.sync()
    for k, v in zip(("state", "time", "reward", "action_idx", "done", "info"), pipe.results()):
        res[name + "/" + k] = v
    res[name + "/launches"] = np.array(launches)
    pipe.close()
    np.savez(path, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--child", nargs=2, metavar=("LIB", "NPZ"))
    ap.add_argument("libs", nargs="*")
    a = ap.parse_args()
    if a.child:
        child(a.child[0], a.envs, a.child[1])
        return 0
    import numpy as np
    outs = []
    with tempfile.TemporaryDirectory() as tmp:
        for i, lib in enumerate(a.libs):
            path = os.path.join(tmp, "%d.npz" % i)
            r = subprocess.run([sys.executable, __file__, "--envs", str(a.envs), "--child", lib, path], capture_output=True, text=True)
            if r.returncode:
                print("%s FAILED:\n%s" % (lib, r.stderr[-2000:]))
                return 1
            outs.append(dict(np.load(path)))
    ref, same = outs[0], True
    configs = sorted({k.split("/")[0] for k in ref})
    for lib, got in zip(a.libs[1:], outs[1:]):
        print("%s vs %s" % (a.libs[0], lib))
        for c in configs:
            keys = sorted(k for k in ref if k.startswith(c + "/"))
            bad = [k.split("/")[1] for k in keys
                   if k not in got or ref[k].dtype != got[k].dtype or ref[k].shape != got[k].shape
                   or ref[k].tobytes() != got[k].tobytes()]
            same &= not bad
            print("  %-28s %-22s launches/step %s" % (c, "bit-identical" if not bad else "DIFFERS: " + ",".join(bad),
                                                    " ".join(str(n) for n in got[c + "/launches"][:3]) + " ..."))
    print("all bit-identical" if same else "OUTPUTS DIFFER")
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
