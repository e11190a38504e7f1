"""PS-only microbenchmark of every aggregation rule on the fused path.

For each rule, ``FusedPS.enqueue_step`` (decode + SGD-momentum update, whole arena, no broadcast destinations) is captured in
a CUDA graph and timed with CUDA events over ``--replays`` replays after ``--warmup`` replays.  The arena is ResNet-18's with a
seeded P = 7 gradient slab; at 314 MB (299 MiB) the slab is larger than the B200's 126 MiB L2, so every replay streams it from HBM.
Bytes per step are the least the rule must move, computed from the shapes (fp32):

    slab rows read                              optimizer (params + momentum, read + write)
    mean, coord_median, trimmed_mean: P         + 16 B per element
    vote: P (compare) + G (select-sum)
    krum: P (distances) + 1
    geomedian: P (distances) + P (weighted sum)
    multi_krum: P (distances) + (P - f)

With ``--attack alie|ipm`` every rule's PS runs under that colluding attack: its ``FusedPS`` gets a one-word adversary bitmap
with the same f liar slots at every step (f = the rule's worker_fail; the mean, which has none, gets 2), so each step starts
with the collusion kernel (csrc/cuda/collude.cu).  The step is timed with it, and the kernel alone is timed in a graph of its
own.  The kernel moves 4 * P * D bytes: the P - f honest rows read plus the f liar rows written (its second pass over the
honest rows re-reads the tile from L2).

    python tools/bench_rules.py [--replays 300] [--warmup 20] [--rules mean,coord_median] [--attack none|alie|ipm]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from draco_b200 import JobConfig  # noqa: E402
from draco_b200.models import build_model  # noqa: E402
from draco_b200.parallel.arena import ArenaLayout  # noqa: E402
from draco_b200.parallel.ps import FusedPS, build_codes  # noqa: E402

P = 7
RULES = {       # rule -> job flags (P = 7 workers; f as the benchmark commands use it)
    "mean": dict(approach="baseline", mode="normal", worker_fail=0),
    "vote": dict(approach="maj_vote", mode="maj_vote", group_size=3, worker_fail=1),
    "krum": dict(approach="baseline", mode="krum", worker_fail=2),
    "geomedian": dict(approach="baseline", mode="geometric_median", worker_fail=2),
    "coord_median": dict(approach="baseline", mode="coord_median", worker_fail=3),
    "trimmed_mean": dict(approach="baseline", mode="trimmed_mean", worker_fail=2),
    "multi_krum": dict(approach="baseline", mode="multi_krum", worker_fail=2),
}


def rows_read(rule: str, ps: FusedPS) -> int:
    if rule == "vote":
        return P + ps.group_table.shape[0]
    if rule == "krum":
        return P + 1
    if rule == "geomedian":
        return 2 * P
    if rule == "multi_krum":
        return P + ps.krum_m
    return P


def time_graph(fn, warmup: int, replays: int):
    """Capture ``fn`` after three eager calls on a side stream; returns (µs per replay timed with CUDA events, what the
    captured call returned)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ret = fn()
    for _ in range(warmup):
        graph.replay()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(replays):
        graph.replay()
    t1.record()
    torch.cuda.synchronize()
    del graph
    return t0.elapsed_time(t1) * 1e3 / replays, ret


def gpu_info(dev: torch.device) -> dict:
    info = {"gpu": torch.cuda.get_device_name(dev), "power_limit": "unknown"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(dev.index)],
                           capture_output=True, text=True, timeout=30)
        if q.returncode == 0 and q.stdout.strip():
            pl, clk = (s.strip() for s in q.stdout.strip().split(","))
            info.update(power_limit=pl, max_sm_clock=clk)
    except (OSError, subprocess.SubprocessError):
        pass
    return info


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--replays", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rules", type=str, default=",".join(RULES))
    ap.add_argument("--attack", type=str, default="none", choices=("none", "alie", "ipm"),
                    help="run every rule under this colluding attack (f liar slots at every step)")
    a = ap.parse_args()
    assert a.replays >= 200, "time at least 200 replays"
    if not torch.cuda.is_available():
        raise SystemExit("bench_rules.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    layout = ArenaLayout.from_model(build_model("ResNet18"), bf16=True, channels_last=True)
    D = layout.total
    slab_mib = P * D * 4 / 2 ** 20
    l2_mib = getattr(torch.cuda.get_device_properties(dev), "L2_cache_size", 0) / 2 ** 20
    info = gpu_info(dev)
    print(f"# {info['gpu']}, power limit {info['power_limit']}, max SM clock {info.get('max_sm_clock', 'unknown')}")
    print(f"# ResNet-18 arena: D = {D} fp32 elements, {layout.ntensors} tensors; P = {P} slab = {P * D * 4 / 1e6:.0f} MB = "
          f"{slab_mib:.0f} MiB ({'larger' if slab_mib > l2_mib else 'NOT larger'} than the {l2_mib:.0f} MiB L2"
          f"{': each replay streams it from HBM' if slab_mib > l2_mib else ''})")
    print(f"# FusedPS.enqueue_step per rule, CUDA graph, {a.replays} replays after {a.warmup}; SGD momentum 0.9, no broadcast")
    if a.attack != "none":
        print(f"# under --err-mode {a.attack}: the f highest slots lie at every step; 'collude' = the collusion kernel alone, "
              f"4 * P * D bytes")
    g = torch.Generator(device=dev).manual_seed(1234)
    mask = torch.from_numpy(layout.valid_mask()).to(dev)
    grad_in = torch.randn(P, D, generator=g, device=dev) * 0.01 * mask
    grad_in[2] *= -100.0                                         # one liar row: the robust rules have something to reject
    results = []
    for rule in a.rules.split(","):
        flags = dict(RULES[rule])
        adv = None
        if a.attack != "none":
            flags["worker_fail"] = flags["worker_fail"] or 2
            f = flags["worker_fail"]
            word = np.array([((1 << f) - 1) << (P - f)], dtype=np.uint32)          # slots P-f .. P-1 lie at every step
            adv = torch.from_numpy(word.view(np.int32)).to(dev)
        cfg = JobConfig(network="ResNet18", num_workers=P, transport="nvl", lr=0.01, momentum=0.9, err_mode=a.attack,
                        **flags).resolve(P + 1)
        groups, code = build_codes(cfg)
        params = (torch.randn(D, generator=g, device=dev) * 0.05 * mask).contiguous()
        ps = FusedPS(cfg, layout, dev, params, grad_in, groups, code, adv_bitmap=adv)
        assert ps.rule == rule, (rule, ps.rule)
        assert bool(ps.collusion) == (a.attack != "none")
        step = torch.ones(1, dtype=torch.int64, device=dev)
        us, nk = time_graph(lambda: ps.enqueue_step(step, mc_params=None, dst=[], flags=[]), a.warmup, a.replays)
        nbytes = (4 * rows_read(rule, ps) + 16) * D
        rec = dict(rule=rule, us_per_step=round(us, 1), kernels=nk, rows_read=rows_read(rule, ps), bytes=nbytes,
                   gb_per_s=round(nbytes / us / 1e3, 1), finite=bool(torch.isfinite(params).all()))
        line = f"{rule:>13}: {us:8.1f} us/step  {nk:2d} kernels  {nbytes / 1e6:7.1f} MB  {rec['gb_per_s']:7.1f} GB/s"
        if a.attack != "none":
            cu, _ = time_graph(lambda: ps.collude(step), a.warmup, a.replays)
            cb = 4 * P * D
            rec.update(attack=a.attack, liars=cfg.worker_fail, collude_us=round(cu, 1), collude_bytes=cb,
                       collude_gb_per_s=round(cb / cu / 1e3, 1))
            line += f"  | collude {cu:7.1f} us  {cb / 1e6:6.1f} MB  {rec['collude_gb_per_s']:7.1f} GB/s  (f = {cfg.worker_fail})"
        results.append(rec)
        print(line)
        del ps
    print(json.dumps(dict(info, D=D, P=P, slab_mib=round(slab_mib, 1), l2_mib=round(l2_mib, 1), replays=a.replays,
                     **({"attack": a.attack} if a.attack != "none" else {}), results=results)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
