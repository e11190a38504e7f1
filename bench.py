#!/usr/bin/env python
"""Headline benchmark: ResNet-18/CIFAR-10 steps/sec at r=3 under s adversaries on N B200s (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29500 \
           bench.py --gpus 8 --steps 20 --warmup 5

Job: 1 PS + 7 logical workers (repetition code, groups of 3, majority vote at the PS), per-worker batch 128, 3 sign-flip
adversaries per step, bf16 compute, synthetic CIFAR-shaped data, random-init ResNet-18.  The logical job is the same at
every N (strong scaling): with N < 8 the logical ranks are packed onto the GPUs that exist (parallel/placement.py).

`value`  : steps/s of the whole job, K steps timed on the device with CUDA events (max over ranks), batches gathered
           on the device, no host synchronisation inside the timed region.
`e2e`    : the same metric through the public API (`Trainer.train_step()`): every step copies that step's batches from
           pinned host memory to the device and reads the loss back to the host.
--impl reference : the unmodified reference cannot be installed here (Python 2.7 / torch 0.3 / mpi4py, no setup.py) ->
           prints {"impl": "reference", "unavailable": ...}.
--impl nccl      : our reference-faithful NCCL baseline (per-tensor messages, library-op decode; BASELINE.md section 4).
--impl nccl_flat : the honest library comparator (flat arenas, ONE broadcast + ONE message per worker, vectorised torch vote,
           CUDA graphs, cuDNN / ATen model compute): parallel/flat_engine.py.  `vs_baseline` divides by the FASTER of the two
           library arms recorded in baseline/measured_nccl.json.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

METRIC = "ResNet-18/CIFAR-10 steps/sec at r=3 under s adversaries"
REF_UNAVAILABLE = ("hwang595/Draco is Python-2.7/PyTorch-0.3/mpi4py code with no setup.py or pyproject.toml: "
                   "`pip install --no-index --target baseline/_ref /root/reference` fails with 'Neither setup.py nor "
                   "pyproject.toml found'; mpi4py, blosc, hdmedians and Eigen are not in the offline wheelhouse")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="ours", choices=("ours", "reference", "nccl", "nccl_flat"))
    ap.add_argument("--network", type=str, default="ResNet18")
    ap.add_argument("--dataset", type=str, default="Cifar10", help="Cifar10 (3x32x32) | ImageNet (synthetic 3x224x224, 1000 classes: "
                    "ResNets get the 7x7/s2 stem + max-pool, BASELINE.json config 5) | MNIST")
    ap.add_argument("--synthetic-size", type=int, default=None)
    ap.add_argument("--approach", type=str, default="maj_vote")
    ap.add_argument("--mode", type=str, default="maj_vote")
    ap.add_argument("--batch-size", type=int, default=128)
    ap.add_argument("--num-workers", type=int, default=7)
    ap.add_argument("--group-size", type=int, default=3)
    ap.add_argument("--worker-fail", type=int, default=3)
    ap.add_argument("--err-mode", type=str, default="rev_grad")
    ap.add_argument("--no-cuda-graphs", action="store_true")
    ap.add_argument("--multicast", type=str, default="auto")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--no-overlap-push", action="store_true")
    ap.add_argument("--push-ctas", type=int, default=16)
    ap.add_argument("--no-pipeline-ps", action="store_true")
    ap.add_argument("--sanity-steps", type=int, default=12,
                    help="after the timed runs: train the same job for this many steps with ONE liar (which r=3 provably tolerates) "
                         "and with none, and report that the loss is finite and identical (0 = skip)")
    ap.add_argument("--wgrad-stream", type=str, default="auto", choices=("auto", "on", "off"),
                    help="weight-gradient kernels on a low-priority side stream (auto = on)")
    ap.add_argument("--ps-stream", action="store_true", help="co-located PS on its own stream inside the captured graph")
    ap.add_argument("--timeline", type=str, default=None,
                    help="after the timed runs, record 3 steps under torch.profiler and write <FILE>.rank<R>.txt: every kernel of "
                         "this rank's GPU in start order (start us, duration us, stream, name) -- NOT a timed number")
    ap.add_argument("--timeline-e2e", type=str, default=None,
                    help="like --timeline but for 3 steps of the end-to-end loop (Trainer.train_step_pipelined, pinned H2D + D2H)")
    ap.add_argument("--worker-streams", type=int, default=None,
                    help="concurrent CUDA streams for logical workers sharing a GPU (default: the JobConfig default)")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy: params.npy (the PS's "
                         "fp32 parameter arena, a fixed seeded sample when larger than 48 MB) and metrics.npy (loss, Prec@1, "
                         "Prec@5, fp64)")
    return ap.parse_args()


DUMP_MAX_PARAMS = 12 * 2 ** 20          # fp32 elements (48 MB): params.npy + metrics.npy stay under 64 MB


def _dump_outputs(out_dir, params, metrics):
    """Write the outputs of the last timed step.  Inputs and initial parameters are seeded, so two builds run with the same
    arguments can be compared file for file; an arena above DUMP_MAX_PARAMS is sampled at the same positions every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    p = params.detach().float().cpu().numpy()
    if p.size > DUMP_MAX_PARAMS:
        p = p[np.sort(np.random.default_rng(0).choice(p.size, DUMP_MAX_PARAMS, replace=False))]
    np.save(os.path.join(out_dir, "params.npy"), p)
    np.save(os.path.join(out_dir, "metrics.npy"), np.asarray(metrics, dtype=np.float64))


def _write_timeline(path, trainer, rank, barrier, pipelined=False):
    """Kernel timeline of 3 consecutive steps on this rank's GPU (CUPTI through torch.profiler; graph replays included)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    barrier()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            if pipelined:
                trainer.train_step_pipelined()
            else:
                trainer.train_step_async()
        if pipelined:
            trainer.drain()
        torch.cuda.synchronize()
    barrier()
    raw = f"{path}.rank{rank}.trace.json"
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    prof.export_chrome_trace(raw)
    evs = [e for e in json.load(open(raw)).get("traceEvents", []) if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
    os.remove(raw)
    evs.sort(key=lambda e: e["ts"])
    if not evs:
        return
    t0 = evs[0]["ts"]
    with open(f"{path}.rank{rank}.txt", "w") as fh:
        fh.write("start_us dur_us gap_to_prev_end_us stream name\n")
        last_end = t0
        for e in evs:
            st, en = e["ts"], e["ts"] + e.get("dur", 0)
            fh.write(f"{st - t0:10.1f} {en - st:8.1f} {st - last_end:8.1f} {e.get('args', {}).get('stream', '?'):>4} {e['name'][:110]}\n")
            last_end = max(last_end, en)


def main() -> int:
    a = parse()
    if a.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": REF_UNAVAILABLE}), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    from draco_b200 import JobConfig
    from draco_b200.parallel.trainer import Trainer, init_distributed
    from draco_b200.utils.metrics import ClockSampler

    if not torch.cuda.is_available():
        print(json.dumps({"metric": METRIC, "error": "no CUDA device visible"}), flush=True)
        return 1
    transport = {"ours": "nvl", "nccl": "nccl", "nccl_flat": "nccl_flat"}[a.impl]
    if a.impl == "nccl_flat":
        # the honest library comparator: flat arenas + one broadcast + one message per worker + CUDA graphs, and the LIBRARY
        # compute path (cuDNN / ATen) instead of this repository's kernels (parallel/flat_engine.py)
        os.environ.update(DRACO_CONV="cudnn", DRACO_BN="aten", DRACO_LINEAR="aten", DRACO_FUSED_LOSS="0", DRACO_FUSED_PREP="0")
    rank, world, local = init_distributed(transport)
    if world != a.gpus and rank == 0:
        print(f"[bench] note: --gpus {a.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    total_steps = 2 * (a.warmup + a.steps) + 8
    syn = a.synthetic_size or (8192 if a.dataset != "ImageNet" else max(512, 2 * a.batch_size * a.num_workers))
    cfg = JobConfig(network=a.network, dataset=a.dataset, approach=a.approach, mode=a.mode, batch_size=a.batch_size,
                    num_workers=a.num_workers, group_size=a.group_size, worker_fail=a.worker_fail, err_mode=a.err_mode,
                    lr=0.01, momentum=0.9, max_steps=total_steps + 4, eval_freq=10 ** 9, transport=transport, dtype="bf16",
                    cuda_graphs=not a.no_cuda_graphs and a.impl in ("ours", "nccl_flat"), compress_grad="None", multicast=a.multicast,
                    synthetic_size=syn, log_interval=10 ** 9, overlap_push=not a.no_overlap_push, push_ctas=a.push_ctas,
                    pipeline_ps=not a.no_pipeline_ps, ps_stream=a.ps_stream, wgrad_stream=a.wgrad_stream,
                    **({"worker_streams": a.worker_streams} if a.worker_streams is not None else {}))
    trainer = Trainer(cfg, rank=rank, world=world, device=torch.device("cuda", local), quiet=True)
    eng = trainer.engine
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # clocks / throttle reasons are sampled on the busiest GPU (a worker GPU when the PS has its own) over BOTH timed regions
    busiest = eng.place.worker_procs()[0] if world > 1 else 0
    sampler = ClockSampler(busiest, period_ms=50) if rank == 0 else None
    if sampler:
        sampler.start()

    def mean_loss(m, key="loss"):
        vals = [None] * world
        if world > 1:
            dist.all_gather_object(vals, m.get(key) if m else None)
        else:
            vals = [m.get(key) if m else None]
        vals = [v for v in vals if v is not None]
        return sum(vals) / len(vals) if vals else None

    # ------------------------------------------------------------------ value: device-timed, no host sync in the loop
    # Runs first, from the seeded initial model: what --dump-outputs writes is the state after exactly warmup + steps training
    # steps, whether or not the e2e loop runs.  (The headline's 3 liars out-vote r=3 groups and the model diverges; its
    # parameters overflow fp32 after about 40 steps.)  The engines capture their CUDA graph on the third step, so at least
    # three warm-up steps keep the capture out of the timed window.
    cfg.data_on_device = True
    for _ in range(max(a.warmup, 3)):
        trainer.train_step_async()
    barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(a.steps):
        trainer.train_step_async()
    e.record()
    barrier()
    ms = reduce_max(s.elapsed_time(e))
    launches = reduce_sum(float(getattr(eng, "kernels_per_step", 0) * a.steps))
    # device-side timeline (spin-wait stamps): how long workers wait for parameters / the PS waits for gradients per step
    trace = eng.wait_trace(min(a.steps, 16)) if hasattr(eng, "wait_trace") else {}
    traces = [None] * world
    if world > 1:
        dist.all_gather_object(traces, trace)
    else:
        traces = [trace]
    ww = [t["worker_wait_ms"] for t in traces if t and "worker_wait_ms" in t]
    breakdown = {"ps_wait_for_grads_ms": next((t["ps_wait_ms"] for t in traces if t and "ps_wait_ms" in t), None),
                 "worker_wait_for_params_ms_mean": sum(ww) / len(ww) if ww else None,
                 "worker_wait_for_params_ms_min": min(ww) if ww else None} if traces and any(traces) else None
    m = eng.read_metrics()
    if a.dump_outputs:
        # mean over the ranks hosting workers; the PS's arena (rank 0) is the master copy every worker trains on
        metrics = [mean_loss(m, k) for k in ("loss", "prec1", "prec5")]
        if rank == 0:
            _dump_outputs(a.dump_outputs, eng.master_params(), [float("nan") if v is None else v for v in metrics])
    if a.timeline:
        _write_timeline(a.timeline, trainer, rank, barrier)

    # ------------------------------------------------------------------ e2e: public API, pinned H2D + D2H every step
    e2e = None
    if not a.skip_e2e:
        cfg.data_on_device = False
        for _ in range(a.warmup):
            trainer.train_step_pipelined()
        trainer.drain()
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s.record()
        last = {}
        # public API, pipelined result read: every step copies its inputs pinned-host -> device and its loss / Prec@k
        # device -> host; the host looks at step k's numbers while step k+1 runs (Trainer.train_step_pipelined), and the
        # last one is drained inside the timed region.
        for _ in range(a.steps):
            last = trainer.train_step_pipelined() or last
        last = trainer.drain() or last
        e.record()
        barrier()
        wall = time.perf_counter() - t0
        e2e_ms = reduce_max(max(s.elapsed_time(e), wall * 1e3 if world == 1 else 0.0))
        h2d = reduce_sum(float(eng.worker.h2d_bytes if eng.local_workers else 0))
        # loss/prec1/prec5 + watchdog word + the step's device-side phase stamps (12 x int64)
        d2h = reduce_sum((12.0 if eng.local_workers else 0.0) + (4.0 + 96.0 if a.impl == "ours" else 0.0))
        if a.timeline_e2e:
            _write_timeline(a.timeline_e2e, trainer, rank, barrier, pipelined=True)
        e2e = {"value": a.steps / (e2e_ms / 1e3), "unit": "steps/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / a.steps, "final_loss": mean_loss(last),
               "api": "Trainer.train_step_pipelined() + drain()",
               "result_read": "every step's loss/Prec@k is copied device->host into pinned memory and read by the host one "
                              "step later (while the next step runs); the last one is drained inside the timed region"}
    clocks = sampler.stop() if sampler else None
    trainer.close()

    # ------------------------------------------------------------------ sanity point: the code tolerates what it promises
    # The headline draws 3 liars over 7 workers like the reference, so a group of 3 can be out-voted and the timed model may
    # diverge.  Here: the SAME job with one liar per step (r = 3 tolerates 1) and with none must produce the same finite loss.
    sanity = None
    if a.sanity_steps > 0 and a.impl == "ours" and a.approach == "maj_vote":
        losses = {}
        for fails in (1, 0) if os.environ.get("DRACO_BENCH_SANITY", "1") != "0" else ():
            c2 = JobConfig(network=a.network, dataset=a.dataset, approach=a.approach, mode=a.mode, batch_size=a.batch_size,
                           num_workers=a.num_workers, group_size=a.group_size, worker_fail=fails, err_mode=a.err_mode if fails else "none",
                           lr=0.01, momentum=0.9, max_steps=a.sanity_steps + 4, eval_freq=10 ** 9, transport=transport, dtype="bf16",
                           cuda_graphs=not a.no_cuda_graphs, compress_grad="None", multicast=a.multicast, synthetic_size=syn,
                           log_interval=10 ** 9, data_on_device=True,
                           **({"worker_streams": a.worker_streams} if a.worker_streams is not None else {}))
            t2 = Trainer(c2, rank=rank, world=world, device=dev, quiet=True)
            first = None
            for i in range(a.sanity_steps):
                t2.train_step_async()
                if i == 0:
                    first = mean_loss(t2.engine.read_metrics())
            barrier()
            losses[fails] = (first, mean_loss(t2.engine.read_metrics()))
            t2.close()
    if len(locals().get("losses", {})) == 2:
        l1, l0 = losses[1][1], losses[0][1]
        sanity = {"steps": a.sanity_steps, "one_liar": {"loss_first": losses[1][0], "loss_last": l1},
                  "no_liar": {"loss_first": losses[0][0], "loss_last": l0},
                  "finite": bool(l1 is not None and l1 == l1 and abs(l1) < 1e4),
                  "one_liar_equals_no_liar": bool(l1 is not None and l0 is not None and l1 == l0)}

    if rank == 0:
        value = a.steps / (ms / 1e3)
        base = None
        headline = (a.network == "ResNet18" and a.dataset == "Cifar10" and a.approach == "maj_vote" and a.mode == "maj_vote" and a.group_size == 3
                    and a.worker_fail == 3 and a.num_workers == 7 and a.batch_size == 128)
        try:
            if not headline:
                raise LookupError("no measured baseline for this configuration")
            with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "baseline", "measured_nccl.json")) as fh:
                rec = json.load(fh).get(str(world), {})
                cands = [v for v in (rec.get("steps_per_s"), rec.get("flat_steps_per_s")) if v]
                base = max(cands) if cands else None            # the faster library arm
        except Exception:
            base = None
        out = {
            "metric": METRIC if headline else f"{a.network}/{a.dataset} steps/sec, {a.approach}/{a.mode} r={a.group_size} under "
                                                f"{a.worker_fail} adversaries (not the headline config)",
            "value": value, "unit": "steps/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": (value / base) if base else None, "dtype": "bf16", "data": "synthetic",
            "impl": a.impl,
            "config": {"model": a.network + " (CIFAR variant, 11.17M params)" if a.network == "ResNet18" else a.network,
                       "global_batch": a.batch_size * a.num_workers, "per_worker_batch": a.batch_size,
                       "seq_len": None, "image": {"Cifar10": "3x32x32", "ImageNet": "3x224x224 (synthetic, 1000 classes)", "MNIST": "1x28x28"}.get(a.dataset),
                       "dataset": a.dataset, "parallelism": f"ps1+w{a.num_workers} on {world} gpu",
                       "placement": eng.place.describe(), "code": f"repetition r={a.group_size} majority-vote" if a.approach == "maj_vote" else a.approach,
                       "adversaries_per_step": a.worker_fail, "err_mode": a.err_mode, "transport": transport,
                       "cuda_graphs": bool(cfg.cuda_graphs), "wgrad_stream": a.wgrad_stream, "worker_streams": len(getattr(eng, "worker_streams", None) or getattr(eng, "streams", None) or []) or 1, "nvls_multicast": bool(getattr(eng, "mc_params", None)),
                       "l2": "per-step working set (7x44.7 MB gradient slab + activations) exceeds the 126 MB L2; no explicit flush",
                       "images_per_s": value * a.batch_size * a.num_workers,
                       "note": ("adversaries are drawn over all workers each step like the reference (src/util.py:100-103), so "
                                "with r=3 and 3 liars a group can be out-voted and the loss may diverge; throughput is "
                                "unaffected. Use --worker-fail 1 for a run the code provably tolerates.")},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "breakdown": breakdown, "sanity": sanity,
            "samples_per_s": value * a.batch_size * a.num_workers,
        }
        def clean(o):                      # strict JSON: no NaN / Infinity literals
            if isinstance(o, float) and (o != o or o in (float("inf"), float("-inf"))):
                return None
            if isinstance(o, dict):
                return {k: clean(v) for k, v in o.items()}
            if isinstance(o, list):
                return [clean(v) for v in o]
            return o
        print(json.dumps(clean(out)), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
