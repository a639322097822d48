#!/usr/bin/env python
"""Per-step time of the fused trainer against the CUDA-graph replay of torch autograd: wall clock vs CUDA events over N
back-to-back steps (cn_trainer_step_indexed / graph replay) on a synthetic replay memory (batch 100 x 5 humans; CADRL: one
human per sample).  Usage: python scripts/trainer_timing.py [network] [steps], network one of sarl (default), om_sarl,
cadrl, lstm_rl, lstm_rl_vn2; lines for a network other than sarl start with its name."""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import modelcrowdnav_b200 as mcn  # noqa: E402
from modelcrowdnav_b200.policy import make_cadrl_network, make_lstm_network, make_value_network  # noqa: E402
from modelcrowdnav_b200.trainer import Trainer, sample_batches  # noqa: E402

NETS = {"sarl": lambda: make_value_network(13, 6, [150, 100], [100, 50], [150, 100, 100, 1], [100, 100, 1]),
        "om_sarl": lambda: make_value_network(61, 6, [150, 100], [100, 50], [150, 100, 100, 1], [100, 100, 1]),
        "cadrl": lambda: make_cadrl_network(13, [150, 100, 100, 1]),
        "lstm_rl": lambda: make_lstm_network(13, 6, None, [150, 100, 100, 1], 50),
        "lstm_rl_vn2": lambda: make_lstm_network(13, 6, [150, 100, 100, 50], [150, 100, 100, 1], 50)}
args = sys.argv[1:]
net = args.pop(0) if args and not args[0].isdigit() else "sarl"
if net not in NETS:
    sys.exit("network must be one of %s" % ", ".join(NETS))
n = int(args[0]) if args else 200
prefix = "" if net == "sarl" else net + " "
dev = torch.device("cuda:0")
torch.manual_seed(0)
model = NETS[net]().to(dev)
memory = mcn.ReplayMemory(100000, device=dev)
shape = (50000, 13) if net == "cadrl" else (50000, 5, 61 if net == "om_sarl" else 13)
memory.push_batch(torch.rand(shape, device=dev), torch.rand((50000,), device=dev))
for mode in ("fused", "graph"):
    tr = Trainer(model, memory, dev, 100, mode=mode)
    tr.set_learning_rate(0.001)
    tr.optimize_batch(20)
    idx = sample_batches(len(memory), 100, n, dev)
    loss = torch.zeros((), device=dev)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(n):
        if mode == "fused":
            tr._fused.step_indexed(memory.states, memory.values, idx[i], loss)
        else:
            loss += tr._step(idx[i])
    e1.record()
    t_launch = time.perf_counter() - t0
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t0
    print("%s%s: %d steps  host enqueue %.1f us/step  wall %.1f us/step  device (events) %.1f us/step" % (
        prefix, mode, n, 1e6 * t_launch / n, 1e6 * t_wall / n, 1e3 * e0.elapsed_time(e1) / n), flush=True)
