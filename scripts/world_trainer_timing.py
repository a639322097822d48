#!/usr/bin/env python
"""Time per world-model training step: the fused step (cn_world_trainer_step, forward + backward + Adam in two kernels)
against torch eager autograd + torch.optim.Adam on a torch restatement of the same model.  AttentionWorld and MlpWorld(H),
batch sizes 100 / 1,000 / 4,096, H = 5 and 10, drop_rate 0 (the restatement has no dropout).  Each row: 20 warm-up steps,
then `steps` back-to-back steps on fixed random batches of a 50,000-sample set, timed with CUDA events.  Prints the card's
name and power limit, then one line per row; --json writes the rows.
Usage: python scripts/world_trainer_timing.py [--steps 200] [--json out.json]"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as Fn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from modelcrowdnav_b200.world_model import AttentionWorld, MlpWorld  # noqa: E402
from modelcrowdnav_b200.world_trainer import WorldTrainer  # noqa: E402


class TorchAttentionWorld(torch.nn.Module):
    """AttentionWorld's forward (world_model.py:71-106) in torch"""

    def __init__(self):
        super().__init__()
        L = torch.nn.Linear
        self.mlp1 = torch.nn.Sequential(L(4, 150), torch.nn.ReLU(), L(150, 100), torch.nn.ReLU())
        self.mlp2 = torch.nn.Sequential(L(100, 100), torch.nn.ReLU(), L(100, 50))
        self.attention = torch.nn.Sequential(L(200, 100), torch.nn.ReLU(), L(100, 100), torch.nn.ReLU(), L(100, 1))
        self.mlp3 = torch.nn.Sequential(L(54, 150), torch.nn.ReLU(), L(150, 100), torch.nn.ReLU(), L(100, 100), torch.nn.ReLU(),
                                        L(100, 2))

    def forward(self, x):
        e = self.mlp1(x)
        f = self.mlp2(e)
        s = self.attention(torch.cat([e, e.mean(dim=1, keepdim=True).expand_as(e)], dim=-1))[..., 0]
        ex = torch.exp(s) * (s != 0).float()
        w = ex / ex.sum(dim=1, keepdim=True)
        feat = (w.unsqueeze(-1) * f).sum(dim=1)
        return self.mlp3(torch.cat([x, feat.unsqueeze(1).expand(-1, x.shape[1], -1)], dim=-1))


class TorchMlpWorld(torch.nn.Module):
    def __init__(self, H):
        super().__init__()
        L = torch.nn.Linear
        self.mlp = torch.nn.Sequential(L(4 * H, 128), torch.nn.ReLU(), L(128, 64), torch.nn.ReLU(), L(64, 12), torch.nn.ReLU(),
                                       L(12, 2 * H))

    def forward(self, x):
        return torch.tanh(self.mlp(x.reshape(x.shape[0], -1))).reshape(x.shape[0], -1, 2)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def timed(fn, steps):
    for _ in range(20):
        fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    print("card: %s" % card(), flush=True)
    rows = []
    N = 50000
    for kind in ("attention", "mlp"):
        for H in (5, 10):
            g = torch.Generator().manual_seed(H)
            X = (torch.rand((N, H, 4), generator=g) * 2 - 1).to(dev)
            Y = (torch.rand((N, H, 2), generator=g) * 2 - 1).to(dev)
            for B in (100, 1000, 4096):
                idx = [torch.randint(0, N, (B,), generator=g).to(dev) for _ in range(8)]
                torch.manual_seed(0)
                world = AttentionWorld() if kind == "attention" else MlpWorld(H, drop_rate=0.0)
                tr = WorldTrainer(world, dev, lr=1e-3, max_batch=4096)
                loss = torch.zeros((), device=dev)
                fused = timed(lambda i: tr._step(X, Y, idx[i % 8], B, loss), a.steps)
                tr.close()
                model = (TorchAttentionWorld() if kind == "attention" else TorchMlpWorld(H)).to(dev)
                opt = torch.optim.Adam(model.parameters(), lr=1e-3)

                def eager(i):
                    j = idx[i % 8]
                    opt.zero_grad()
                    Fn.mse_loss(model(X[j]), Y[j]).backward()
                    opt.step()
                eager_us = timed(eager, a.steps)
                row = dict(model=kind, H=H, batch=B, fused_us=round(fused, 1), eager_us=round(eager_us, 1),
                           speedup=round(eager_us / fused, 2))
                rows.append(row)
                print("%-9s H=%-2d B=%-4d  fused %8.1f us/step   eager autograd + Adam %8.1f us/step   x%.2f" % (
                    kind, H, B, fused, eager_us, eager_us / fused), flush=True)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(dict(card=card(), steps=a.steps, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
