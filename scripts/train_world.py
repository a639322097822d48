#!/usr/bin/env python
"""Train a world model (AttentionWorld or MlpWorld) on ORCA transitions, on the device.

Collects the transitions of E circle- or square-crossing episodes with H ORCA humans (the robot follows its own ORCA),
holds out every `--val_every`-th episode for validation, trains with Adam and early stopping, prints the per-epoch losses and
the wall time, and saves the state dict (loadable into the reference's module).
Usage: python scripts/train_world.py --model attention --envs 2048 --humans 5 --output world.pth"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import modelcrowdnav_b200 as mcn  # noqa: E402
from modelcrowdnav_b200.world_model import AttentionWorld, MlpWorld  # noqa: E402
from modelcrowdnav_b200.world_trainer import WorldTrainer, collect_world_transitions  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", choices=("attention", "mlp"), default="attention")
    ap.add_argument("--envs", type=int, default=2048)
    ap.add_argument("--humans", type=int, default=5)
    ap.add_argument("--sim", choices=("circle", "square"), default="circle")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--val_every", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=50)
    ap.add_argument("--batch_size", type=int, default=1000)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--patience", type=int, default=5)
    ap.add_argument("--drop_rate", type=float, default=0.5)
    ap.add_argument("--output", default="world_model.pth")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    t0 = time.perf_counter()
    rule = mcn._capi.CIRCLE_CROSSING if a.sim == "circle" else mcn._capi.SQUARE_CROSSING
    env = mcn.BatchedCrowdSim(a.envs, a.humans, seed=a.seed, sim_rule=rule)
    env.reset_device()
    X, Y, ids = collect_world_transitions(env, robot="orca")
    env.close()
    val = ids % a.val_every == 0
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    print("collected %d pairs (%d train / %d val) from %d episodes in %.2f s" % (
        X.shape[0], int((~val).sum()), int(val.sum()), a.envs, t1 - t0), flush=True)
    torch.manual_seed(a.seed)
    world = AttentionWorld() if a.model == "attention" else MlpWorld(a.humans, drop_rate=a.drop_rate)
    tr = WorldTrainer(world, dev, lr=a.lr, max_batch=a.batch_size, seed=a.seed, max_humans=max(a.humans, 1))
    hist = tr.optimize_epoch(X[~val], Y[~val], a.batch_size, a.epochs, val=(X[val], Y[val]), patience=a.patience,
                             generator=torch.Generator().manual_seed(a.seed))
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    for i, h in enumerate(hist):
        print("epoch %3d  train %.6f  val %.6f" % (i, h["train"], h["val"]))
    print("trained %d epochs in %.2f s (best val %.6f)" % (len(hist), t2 - t1, min(h["val"] for h in hist)))
    torch.save(world.state_dict(), a.output)
    print("saved %s" % a.output)


if __name__ == "__main__":
    main()
