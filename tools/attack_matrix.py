"""Training outcome of every aggregation rule under every attack, on the fused nvl transport in one process.

Cells are (rule, attack).  The rules are every baseline rule at P = 7 workers with f = 2 liars per step (mean, geometric
median, Krum, multi-Krum, coordinate-wise median, trimmed mean) plus Draco's repetition vote at P = 7, group size 3, f = 1.
The attacks are none, rev_grad (the reference's sign flip x100), alie ("A Little Is Enough", Baruch et al., NeurIPS 2019)
and ipm (inner-product manipulation, Xie et al., UAI 2019).  Each cell trains from the same seeded model and data for
``--steps`` steps (CUDA graphs on) and reports the mean training loss and Prec@1 over the last 20 steps; the ``none`` cell
of a rule is its clean run.

    python tools/attack_matrix.py [--steps 200] [--network LeNet --dataset MNIST] [--rules ...] [--attacks ...]

The last line is one JSON record with every cell, the GPU name and its power limit.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from draco_b200 import JobConfig  # noqa: E402
from draco_b200.parallel.trainer import Trainer  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_rules import gpu_info  # noqa: E402

P = 7
RULES = {
    "mean": dict(approach="baseline", mode="normal", worker_fail=2),
    "geomedian": dict(approach="baseline", mode="geometric_median", worker_fail=2),
    "krum": dict(approach="baseline", mode="krum", worker_fail=2),
    "multi_krum": dict(approach="baseline", mode="multi_krum", worker_fail=2),
    "coord_median": dict(approach="baseline", mode="coord_median", worker_fail=2),
    "trimmed_mean": dict(approach="baseline", mode="trimmed_mean", worker_fail=2),
    "vote": dict(approach="maj_vote", mode="maj_vote", group_size=3, worker_fail=1),
}
ATTACKS = ("none", "rev_grad", "alie", "ipm")
WINDOW = 20


def _finite(x: float):
    return round(x, 4) if math.isfinite(x) else None


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--network", type=str, default="LeNet")
    ap.add_argument("--dataset", type=str, default="MNIST")
    ap.add_argument("--batch-size", type=int, default=64)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--rules", type=str, default=",".join(RULES))
    ap.add_argument("--attacks", type=str, default=",".join(ATTACKS))
    a = ap.parse_args()
    assert a.steps >= WINDOW, f"train at least {WINDOW} steps"
    if not torch.cuda.is_available():
        raise SystemExit("attack_matrix.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(dev)
    print(f"# {info['gpu']}, power limit {info['power_limit']}")
    print(f"# {a.network} / {a.dataset}, P = {P}, batch {a.batch_size} per worker, lr {a.lr}, momentum 0.9, {a.steps} steps per "
          f"cell; loss and Prec@1 are means over the last {WINDOW} steps")
    cells = []
    for rule in a.rules.split(","):
        for attack in a.attacks.split(","):
            cfg = JobConfig(network=a.network, dataset=a.dataset, batch_size=a.batch_size, num_workers=P, transport="nvl",
                            lr=a.lr, momentum=0.9, max_steps=a.steps + 4, eval_freq=10 ** 9, log_interval=10 ** 9,
                            compress_grad="None", err_mode=attack, **RULES[rule])
            t = Trainer(cfg, rank=0, world=1, device=dev, quiet=True)
            hist = [t.train_step() for _ in range(a.steps)]
            t.close()
            loss = float(np.mean([m["loss"] for m in hist[-WINDOW:]]))
            prec1 = float(np.mean([m["prec1"] for m in hist[-WINDOW:]]))
            cells.append(dict(rule=rule, attack=attack, f=cfg.worker_fail, loss=_finite(loss), prec1=_finite(prec1)))
            print(f"{rule:>13} {attack:>9} (f = {cfg.worker_fail}): loss {loss:10.4f}  Prec@1 {prec1:7.2f}", flush=True)
            del t
            torch.cuda.empty_cache()
    print(json.dumps(dict(info, network=a.network, dataset=a.dataset, P=P, steps=a.steps, window=WINDOW, cells=cells)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
