"""The product transport (``--transport nvl``): every byte of a training step moves through sm_100a kernels.

Step anatomy (one PS + P logical workers hosted by ``nprocs`` GPU processes; see placement.py):

    worker GPU                                                   PS GPU
    ----------                                                   ------
    wait_flags(params_ready >= t)        [spin on local flag]
    cast_params fp32 -> bf16
    forward / backward  (x R sub-batches under the cyclic code)
    push_encode: encode + adversary + 16 B peer stores  ------>  grad_in[w]   + release flag grad_ready[w] = t
                                                                 wait_flags(grad_ready[*] >= t)
                                                                 vote | project+locate | krum | geomedian   (decode)
    params arena  <------ multimem.st / peer stores  ----------  aggregate_update: SGD-momentum + broadcast
    flag params_ready = t+1  <---------------------------------  (last CTA)

There is no NCCL / MPI call and no host synchronisation anywhere in that loop; ordering between GPUs is carried by
step-stamped, monotonically increasing flag words (acquire/release at system scope).  The whole per-process sequence is
captured once in a CUDA graph and replayed; the step number lives in device memory so replays advance it.  Logical
workers that share a GPU run on concurrent streams inside that graph (``--worker-streams``), their bucket pushes on side
streams overlapped with the rest of the backward pass, and the PS consumes buckets as they complete (pipelined PS).

Reference counterparts: master loops src/master/{baseline,rep,cyclic}_master.py ``start()``; worker loops
src/worker/*_worker.py ``train()``; all mpi4py traffic listed in SURVEY.md section 2.3 "Collective / message call sites".
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist

from ..codes.adversary import ATTACK_OMNISCIENT, COLLUSION_ATTACKS, attack_code, generate_schedule
from ..config import JobConfig
from ..data import BatchPlan, TensorDataset
from ..ops import conv as _conv_ops
from ..ops import kernels as K
from ..utils.metrics import PhaseTimer, limit_host_threads, wait_event
from .arena import ArenaLayout
from .placement import Placement
from .ps import COORDINATE_RULES, FusedPS, build_codes, select_rule
from .symm import SymmContext
from .worker import WorkerCompute, make_model

FLAG_STRIDE = 128            # bytes between flag words (one per 128-B line)
FLAG_BYTES = 65536
MAX_BUCKETS = 8              # per-worker gradient-bucket flags


class FusedEngine:
    def __init__(self, cfg: JobConfig, rank: int, nprocs: int, device: torch.device, dataset: Optional[TensorDataset],
                 group=None):
        assert device.type == "cuda", "the nvl transport needs a GPU"
        limit_host_threads()
        self.cfg, self.rank, self.nprocs, self.device, self.group = cfg, rank, nprocs, device, group
        self.place = Placement(cfg.num_workers, nprocs)
        self.P = cfg.num_workers
        self.is_ps = rank == 0
        self.local_workers = self.place.local_workers(rank)
        self.active = self.is_ps or bool(self.local_workers)
        self.groups, self.code = build_codes(cfg)
        self.cyclic = cfg.approach == "cyclic"
        self.esize = 8 if self.cyclic else 4
        self.step = 1                                   # host mirror of the device step counter
        self.kernels_per_step = 0
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self._use_graph = (cfg.cuda_graphs and cfg.err_mode != "omniscient" and not cfg.profile_phases
                           and not cfg.debug_checksum)
        self.debug_checksum = cfg.debug_checksum
        self._dbg_sums: Dict[int, torch.Tensor] = {}
        self._dbg_ps_sums: Optional[torch.Tensor] = None
        self.checksum_log: List[dict] = []
        self.timer = PhaseTimer(True) if cfg.profile_phases else None
        self._eager_steps = 0
        # --compress-grad compress (reference default, src/compress_gradient.py:7-15): the encoded gradient is packed on the
        # worker GPU and only the packed bytes cross NVLink into a PS staging slot; the PS unpacks into the worker's gradient
        # slot ahead of the decode.  Whole-arena push (no bucket overlap / PS pipelining in this mode).
        self.compress = bool(cfg.compress)
        self.overlap_push = cfg.overlap_push and not self.cyclic and not self.compress
        # PS pipelining: decode + apply + broadcast each gradient bucket as soon as all workers pushed it
        self.pipeline_ps = (self.overlap_push and cfg.pipeline_ps and select_rule(cfg) in ("mean", "vote") + COORDINATE_RULES
                            and cfg.err_mode != "omniscient")
        self.push_stream = torch.cuda.Stream(device=device) if self.overlap_push else None
        ns = min(max(int(cfg.worker_streams), 1), len(self.local_workers))
        # weight gradients on a side stream (auto = on: +5.6 % for a worker that owns its GPU, +2.4 % with seven workers sharing
        # one).  The compute streams then get a higher priority than the side / push streams: the backward chain's CTAs are
        # dispatched ahead of weight-gradient CTAs whenever both are pending
        wgrad_side = (cfg.wgrad_stream in ("on", "auto") and bool(self.local_workers)
                      and not cfg.profile_phases and cfg.zero_copy_grads)
        prio = -1 if wgrad_side else 0
        # (compute stream, push stream) pairs; omniscient liars need the serial order, phase timers one timeline
        self.worker_streams = ([(torch.cuda.Stream(device=device, priority=prio), torch.cuda.Stream(device=device)) for _ in range(ns)]
                               if ns > 1 and cfg.err_mode != "omniscient" and not cfg.profile_phases and not cfg.debug_checksum
                               else [])
        self.push_counters = torch.zeros(cfg.num_workers + 1, dtype=torch.int32, device=device)
        # does ANY process of the job host several workers on concurrent streams?  (decides the BatchNorm variant job-wide)
        self.job_uses_worker_streams = (int(cfg.worker_streams) > 1 and cfg.err_mode != "omniscient" and not cfg.profile_phases
                                        and not cfg.debug_checksum
                                        and max(len(self.place.local_workers(p)) for p in range(nprocs)) > 1)
        self._staged_step = -1
        # one worker on this GPU (the 8-GPU topology): overlap the weight-gradient kernels with the rest of the backward chain
        from ..ops import conv as _conv_ops_mod
        _conv_ops_mod.WGRAD_SIDE_STREAM = wgrad_side                 # stolen (zero-copy) gradients only: see ops/conv.py

        if cfg.deterministic:
            torch.backends.cudnn.deterministic = True
            torch.backends.cudnn.benchmark = False
            os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

        model = make_model(cfg)
        bf16 = cfg.dtype == "bf16"
        self.layout = ArenaLayout.from_model(model, bf16, channels_last=True)
        D = self.layout.total

        # ---------------- symmetric regions -------------------------------------------------------------
        self.symm = SymmContext(device, rank, nprocs, group)
        gran = None
        want_mc = cfg.multicast != "off" and nprocs > 1
        regA = self.symm.alloc("params", D * 4 + FLAG_BYTES, gran)
        self.params_f32 = regA.tensor[: D * 4].view(torch.float32)
        self.flagsA = regA.tensor[D * 4: D * 4 + FLAG_BYTES].view(torch.int64)
        self.params_ready_ptr = regA.ptr + D * 4
        if self.is_ps:
            regB = self.symm.alloc("grad_in", self.P * D * self.esize + FLAG_BYTES)
            self.grad_in = regB.tensor[: self.P * D * self.esize].view(torch.float32)
            self.flagsB = regB.tensor[self.P * D * self.esize: self.P * D * self.esize + FLAG_BYTES].view(torch.int64)
        all_procs = list(range(nprocs))
        mapA = self.symm.share("params", exporters=all_procs, importers=[0])
        mapB = self.symm.share("grad_in", exporters=[0], importers=all_procs)
        self.ps_grad_base = mapB[0].ptr
        self.ps_flag_base = mapB[0].ptr + self.P * D * self.esize
        self.codec = None
        if self.compress:
            from ..utils.codec import DeviceStreamCodec
            self.codec = DeviceStreamCodec(D * self.esize // 4, device)
            cap = self.codec.capacity
            if self.is_ps:
                regS = self.symm.alloc("grad_stage", self.P * cap + 8 * self.P)
                self.stage = regS.tensor[: self.P * cap].view(self.P, cap)
                self.stage_bytes = regS.tensor[self.P * cap: self.P * cap + 8 * self.P].view(torch.int64)
            mapS = self.symm.share("grad_stage", exporters=[0], importers=all_procs)
            self.ps_stage_base = mapS[0].ptr
            # one codec (plan / size scratch) per local worker: workers sharing this GPU pack concurrently on their own streams
            self.codec_w = {w: DeviceStreamCodec(D * self.esize // 4, device) for w in self.local_workers}
            self.enc_local = {w: torch.zeros(D * self.esize // 4, dtype=torch.float32, device=device) for w in self.local_workers}
            self.stream_local = {w: torch.zeros(cap, dtype=torch.uint8, device=device) for w in self.local_workers}
        self.mc_params = None
        if want_mc:
            self.mc_params = self.symm.bind_multicast("params")
            if self.mc_params is None and cfg.multicast == "on":
                raise RuntimeError("--multicast on, but NVLS multicast could not be set up")

        # ---------------- device-side control words -----------------------------------------------------
        self.step_dev = torch.ones(1, dtype=torch.int64, device=device)
        self.error = torch.zeros(1, dtype=torch.int32, device=device)
        self.counters = torch.zeros(16, dtype=torch.int32, device=device)
        self.stamps_worker = torch.zeros(64, 2, dtype=torch.int64, device=device)   # %globaltimer trace of the spin waits
        self.stamps_ps = torch.zeros(64, 2, dtype=torch.int64, device=device)
        # phase stamps [step & 63][col]: 0 worker compute done (push joined) | 1 PS decode done, update + broadcast about to start |
        # 2 PS update + broadcast done.  Together with the wait stamps they give the reference's per-step Comp / Comm / Method /
        # Update times in graph mode, on the device, with no host synchronisation (utils/metrics.py prints them every step).
        self.stamps_phase = torch.zeros(64, 8, dtype=torch.int64, device=device)
        self.default_phases = not cfg.profile_phases
        sched = generate_schedule(self.P, cfg.worker_fail, cfg.max_steps)
        self.schedule = sched
        use_adv = cfg.err_mode != "none" and cfg.worker_fail > 0
        self.adv_bitmap = torch.from_numpy(sched.bitmaps().view(np.int32).copy()).to(device) if use_adv else None
        self.attack = attack_code(cfg.err_mode) if self.adv_bitmap is not None else 0

        # ---------------- roles -------------------------------------------------------------------------
        self.worker: Optional[WorkerCompute] = None
        self.ps: Optional[FusedPS] = None
        if self.local_workers or self.is_ps:
            plan = make_plan(cfg, dataset, self.groups)
            # the PS process also builds the model: its initial parameters are the job's initial parameters
            self.worker = WorkerCompute(cfg, device, self.local_workers, plan, dataset, self.layout, self.params_f32, model)
            self.worker.step_dev = self.step_dev       # dropout masks are keyed by the device step (graph replays advance it)
        if self.is_ps:
            self.ps = FusedPS(cfg, self.layout, device, self.params_f32, self.grad_in, self.groups, self.code,
                              adv_bitmap=self.adv_bitmap)
            self.dst_ptrs = [mapA[p].ptr for p in self.place.worker_procs() if p != 0]
            self.param_flag_ptrs = [mapA[p].ptr + D * 4 for p in self.place.active_procs()]
        self._dbg_buf = (torch.zeros(D * self.esize // 4, dtype=torch.float32, device=device)
                         if self.debug_checksum and self.local_workers else None)
        self._initial_broadcast()

    # ------------------------------------------------------------------ transport self-check (SURVEY 5.2)
    def _dbg_loopback(self, w: int, g32, g16, push_kw) -> None:
        """Re-run the worker's encode + adversary into a LOCAL buffer and keep its 64-bit checksum (sum of the 32-bit
        words): what the PS must find in slot ``w`` if every peer store of the real push landed."""
        K.push_encode(self.layout, g32, g16, self._dbg_buf.data_ptr(), flag=None, **push_kw)
        self._dbg_sums[w] = self._dbg_buf.view(torch.int32).sum(dtype=torch.int64)

    def _dbg_sum_slots(self, tile_range) -> None:
        """PS-side checksums of (one bucket of) every slot, taken before a colluding attack rewrites the liar slots."""
        words = self.grad_in.view(torch.int32).view(self.P, -1)
        if tile_range is not None:
            words = words[:, tile_range[0] * K.N.TILE: tile_range[1] * K.N.TILE]
        self._dbg_ps_sums += words.sum(1, dtype=torch.int64)

    def _verify_checksums(self, step: int) -> None:
        sums = torch.zeros(self.P, dtype=torch.int64, device=self.device)
        have = torch.zeros(self.P, dtype=torch.int64, device=self.device)
        for w, v in self._dbg_sums.items():
            sums[w - 1] = v
            have[w - 1] = 1
        self._dbg_sums = {}
        if self.nprocs > 1:
            dist.all_reduce(sums, group=self.group)
            dist.all_reduce(have, group=self.group)
        if self.is_ps:
            got = self._dbg_ps_sums.cpu()
            exp, hv = sums.cpu(), have.cpu()
            bad = [w + 1 for w in range(self.P) if hv[w] and int(got[w]) != int(exp[w])]
            self.checksum_log.append({"step": step, "checked": int(hv.sum()), "bad": bad})
            if bad:
                raise RuntimeError(f"step {step}: gradient slot checksum mismatch for worker(s) {bad} -- a peer store was "
                                   f"lost or reordered past its flag")

    # ------------------------------------------------------------------ setup helpers
    def _initial_broadcast(self) -> None:
        """PS -> every process: initial parameters, then params_ready = 1 (reference: first Bcast of the loop)."""
        if self.is_ps:
            nbytes = self.layout.total * 4
            lib = K.N.cuda()
            st = torch.cuda.current_stream().cuda_stream
            for d in self.dst_ptrs:
                K.N.check(lib.drc_rt_memcpy_async(d, self.params_f32.data_ptr(), nbytes, st), "initial broadcast")
            torch.cuda.synchronize()
        self._barrier()
        if self.is_ps:
            K.set_flags(self.param_flag_ptrs, self.step_dev, 0)
            torch.cuda.synchronize()
        self._barrier()

    def _barrier(self) -> None:
        if self.nprocs > 1:
            dist.barrier(group=self.group)

    def slot_ptr(self, w: int) -> int:
        return self.ps_grad_base + (w - 1) * self.layout.total * self.esize

    def grad_flag_ptr(self, w: int, b: int = 0) -> int:
        return self.ps_flag_base + ((w - 1) * MAX_BUCKETS + b) * FLAG_STRIDE

    # ------------------------------------------------------------------ the step
    def _enqueue_local_step(self, step_host: Optional[int]) -> int:
        """Enqueue everything this process contributes to one step.  Returns #kernels of ours launched."""
        cfg, L = self.cfg, self.layout
        n = 0
        nvtx = torch.cuda.nvtx
        # PS co-located with workers (N = 1, 2, 4): inside the captured graph the PS part runs on ITS OWN stream, forked here, so it
        # votes / applies / broadcasts every gradient bucket as soon as all P workers (local and remote) pushed it, while the local
        # workers are still back-propagating -- instead of queueing behind them (VERDICT r1, weak 11).  A bucket's parameters are
        # rewritten only after EVERY worker's flag for it arrived, i.e. after every local worker is past those layers.  Eager steps
        # keep the serial order (a first-time kernel load would synchronise with the spinning wait kernel).
        ps_side = (self.is_ps and bool(self.local_workers) and self.pipeline_ps and step_host is None and cfg.ps_stream
                   and torch.cuda.is_current_stream_capturing())
        if ps_side:
            if getattr(self, "_ps_stream", None) is None:
                self._ps_stream = torch.cuda.Stream(device=self.device)
            fork0 = torch.cuda.Event()
            fork0.record(torch.cuda.current_stream())
            self._ps_stream.wait_event(fork0)
            with torch.cuda.stream(self._ps_stream):
                n += self._enqueue_ps_part()
        if self.local_workers:
            wc = self.worker
            nvtx.range_push("draco/worker: fetch params + compute + encode/push")   # reference phases: Comm / Comp / Encode
            with self._phase("t_fetch"):
                K.wait_flags([self.params_ready_ptr], self.step_dev, 0, self.error, cfg.spin_timeout_s, self.stamps_worker); n += 1
                if wc.bf16:
                    K.cast_params(L, wc.binder.params_f32, wc.binder.params_c); n += 1
            comp_phase = self._phase("t_comp_encode_push")         # the push overlaps the backward pass: one phase
            comp_phase.__enter__()
            order = list(self.local_workers)
            if step_host is not None and cfg.err_mode == "omniscient":
                # liars read the honest slots: on a shared stream the honest workers must be enqueued first
                order.sort(key=lambda r: self.schedule.is_adversary(r, step_host))
            if self.worker_streams:
                # Logical workers sharing this GPU are issued round-robin on concurrent streams: the late layers of a
                # CIFAR ResNet launch 16-128 CTAs on 148 SMs, so kernels of different workers fill each other's gaps.
                # Every worker's kernel sequence is unchanged => its gradient stays bit-identical to the serial run.
                from ..ops import norm as _norm
                main = torch.cuda.current_stream()
                fork = torch.cuda.Event()
                fork.record(main)
                try:
                    for i, w in enumerate(order):
                        st, pst = self.worker_streams[i % len(self.worker_streams)]
                        _norm.UPDATE_RUNNING_STATS = (i == 0)
                        if i < len(self.worker_streams):
                            st.wait_event(fork)
                        with torch.cuda.stream(st):
                            n += self._enqueue_worker(w, step_host, pst)
                finally:
                    _norm.UPDATE_RUNNING_STATS = True
                for st, _ in self.worker_streams[: len(order)]:
                    main.wait_stream(st)
            else:
                # (every rank runs the same kernels whatever its stream layout: replicas of a vote group on different GPUs
                # stay bit-identical)
                for w in order:
                    n += self._enqueue_worker(w, step_host, self.push_stream)
        if self.local_workers:
            if self.default_phases:
                K.stamp(self.stamps_phase, self.step_dev, 0); n += 1
            comp_phase.__exit__(None, None, None)
            nvtx.range_pop()
        if ps_side:
            torch.cuda.current_stream().wait_stream(self._ps_stream)
        elif self.is_ps:
            n += self._enqueue_ps_part()
        if self.is_ps and self.debug_checksum and not self.ps.collusion:    # every gradient flag of this step has been waited for
            self._dbg_ps_sums = self.grad_in.view(torch.int32).view(self.P, -1).sum(1, dtype=torch.int64)
        K.step_add(self.step_dev, 1); n += 1
        return n

    def _enqueue_ps_part(self) -> int:
        """Gather (wait for the gradient flags) + decode + optimizer + broadcast on the current stream."""
        cfg = self.cfg
        n = 0
        nvtx = torch.cuda.nvtx
        if True:
            ps_phase = self._phase("t_gather_decode_update_bcast")
            ps_phase.__enter__()
            nvtx.range_push("draco/ps: gather + decode + update + broadcast")            # reference: Method / Update time
            base = self.flagsB.data_ptr()
            before_collude = None
            if self.debug_checksum and self.ps.collusion:
                self._dbg_ps_sums = torch.zeros(self.P, dtype=torch.int64, device=self.device)
                before_collude = self._dbg_sum_slots
            if self.pipeline_ps:
                nb = len(self.worker.buckets)

                def wait_bucket(bi):
                    fl = [base + (i * MAX_BUCKETS + bi) * FLAG_STRIDE for i in range(self.P)]
                    K.wait_flags(fl, self.step_dev, 0, self.error, cfg.spin_timeout_s, self.stamps_ps if bi == nb - 1 else None)
                    return 1

                n += self.ps.enqueue_step(self.step_dev, mc_params=self.mc_params, dst=[] if self.mc_params else self.dst_ptrs,
                                          flags=self.param_flag_ptrs, buckets=self.worker.buckets, wait_bucket=wait_bucket,
                                          before_update=self._stamp_decode_done, before_collude=before_collude)
            else:
                flags = [base + i * MAX_BUCKETS * FLAG_STRIDE for i in range(self.P)]
                K.wait_flags(flags, self.step_dev, 0, self.error, cfg.spin_timeout_s, self.stamps_ps); n += 1
                if self.compress:                               # packed streams -> the workers' gradient slots
                    slots = self.grad_in.view(self.P, -1)
                    for i in range(self.P):
                        self.codec.unpack(self.stage[i], slots[i]); n += 1
                n += self.ps.enqueue_step(self.step_dev, mc_params=self.mc_params,
                                          dst=[] if self.mc_params else self.dst_ptrs, flags=self.param_flag_ptrs,
                                          before_update=self._stamp_decode_done, before_collude=before_collude)
        if self.default_phases:
            K.stamp(self.stamps_phase, self.step_dev, 2); n += 1
        nvtx.range_pop()
        ps_phase.__exit__(None, None, None)
        return n

    def _stamp_decode_done(self) -> int:
        if not self.default_phases:
            return 0
        K.stamp(self.stamps_phase, self.step_dev, 1)
        return 1

    def _phase_row(self, step: int) -> torch.Tensor:
        """[12] int64 on the device: wait stamps (worker begin/end, PS begin/end) + the 8 phase stamps of ``step``."""
        i = step & 63
        return torch.cat([self.stamps_worker[i], self.stamps_ps[i], self.stamps_phase[i]])

    def _phases_from_row(self, row) -> Dict[str, float]:
        """Reference field names (seconds): t_fetch = waiting for parameters ("Comm"), t_comp_encode_push = forward/backward with the
        fused encode + push ("Comp"; "Encode" is inside it), t_gather = PS waiting for the last gradient, t_decode = vote /
        Fourier / Krum / median up to the start of the last update kernel ("Method"), t_update = fused optimizer + broadcast."""
        ww0, ww1, pw0, pw1, comp_end, dec_end, upd_end = [int(v) for v in row[:7]]
        out: Dict[str, float] = {}
        if self.local_workers and ww1 >= ww0 > 0:
            out["t_fetch"] = (ww1 - ww0) * 1e-9
            if comp_end >= ww1:
                out["t_comp_encode_push"] = (comp_end - ww1) * 1e-9
        if self.is_ps and pw1 >= pw0 > 0:
            out["t_gather"] = (pw1 - pw0) * 1e-9
            if dec_end >= pw1:
                out["t_decode"] = (dec_end - pw1) * 1e-9
                if upd_end >= dec_end:
                    out["t_update"] = (upd_end - dec_end) * 1e-9
        return out

    def _enqueue_worker(self, w: int, step_host: Optional[int], push_stream) -> int:
        """Forward/backward + encode/push of logical worker ``w`` on the current stream (bucket pushes on ``push_stream``)."""
        cfg, L, wc = self.cfg, self.layout, self.worker
        n = 0
        g32 = [g[0] for g in wc.grads]
        g16 = [g[1] for g in wc.grads]
        coef = list(self.code.coeffs_of(w - 1)) if self.cyclic else None
        lying_now = (step_host is not None and cfg.err_mode == "omniscient"
                     and self.schedule.is_adversary(w, step_host))
        push_kw = dict(step_ptr=self.step_dev, worker=w - 1, done_counter=self.push_counters[w:w + 1], coef=coef,
                       adv_bitmap=self.adv_bitmap, adv_len=len(self.schedule.ranks),
                       # omniscient / colluding liars push their honest gradient: their lie is made from the honest slots
                       attack=0 if self.attack == ATTACK_OMNISCIENT or self.attack in COLLUSION_ATTACKS else self.attack,
                       magnitude=cfg.attack_magnitude, seed=cfg.seed,
                       src_table=wc.ptr_dev[w] if wc.zero_copy else None)
        if self.overlap_push and not lying_now:
            # bucketed push on a side stream, overlapped with the rest of the backward pass
            state = {"done": 0}
            nb = len(wc.buckets)

            def on_bucket(b, _w=w, _state=state, _g32=g32, _g16=g16, _kw=push_kw):
                t0, t1, idxs = wc.buckets[b]
                _state["done"] += 1
                if wc.zero_copy:                              # pointers of this bucket's gradients -> device table
                    wc.upload_ptrs(_w, wc.R - 1, min(idxs), max(idxs) + 1)
                ev = torch.cuda.Event()
                ev.record()                                   # on the backward stream (autograd thread)
                _conv_ops.join_wgrad_stream(self.device, push_stream)    # ... and the weight gradients of the side stream
                with torch.cuda.stream(push_stream):
                    push_stream.wait_event(ev)
                    # few CTAs: the transfer is NVLink/ingress-bound and must not starve the backward kernels
                    # it overlaps with (a full-GPU grid of store-stalled CTAs would hog every SM's warp slots)
                    if self.pipeline_ps:
                        flag = self.grad_flag_ptr(_w, b)                  # every bucket announces itself
                    else:
                        flag = self.grad_flag_ptr(_w) if _state["done"] == nb else None
                    # remote slot: NVLink-bound, few CTAs; local slot (PS on this GPU): HBM-bound, 2 CTAs per SM
                    grid = self.cfg.push_ctas if self.rank != 0 else 2 * K.sm_count()
                    if _state["done"] == nb and len(self.local_workers) == 1:
                        grid = max(grid, K.sm_count())        # last bucket of the only worker: backward is over, nothing to starve
                    K.push_encode(L, _g32, _g16, self.slot_ptr(_w), tile_range=(t0, t1), grid=min(grid, t1 - t0),
                                  flag=flag, **_kw)

            wc.forward_backward(w, step_host, on_bucket=on_bucket)
            assert state["done"] == nb, "a gradient bucket never became ready"
            torch.cuda.current_stream().wait_stream(push_stream)      # join (also required by capture)
            n += nb
            if self.debug_checksum:
                if wc.zero_copy:
                    wc.upload_ptrs(w, wc.R - 1, 0, L.ntensors)
                self._dbg_loopback(w, g32, g16, push_kw)
            return n
        wc.forward_backward(w, step_host)
        if wc.zero_copy and not lying_now:
            for k in range(wc.R):
                if k < wc.R - 1:
                    # earlier sub-batches: their gradient tensors were detached from the parameters
                    if not torch.cuda.is_current_stream_capturing():
                        host = torch.tensor([g.data_ptr() for g in wc.grad_refs[w][k]], dtype=torch.int64).pin_memory()
                        wc._pinned_keep.append(host)
                        wc.ptr_dev[w][k].copy_(host, non_blocking=True)
                else:
                    wc.upload_ptrs(w, k, 0, L.ntensors)
        if lying_now:
            honest = 0
            for h in range(1, self.P + 1):
                if not self.schedule.is_adversary(h, step_host):
                    honest |= 1 << (h - 1)
            flags = [self.grad_flag_ptr(h) for h in range(1, self.P + 1) if (honest >> (h - 1)) & 1]
            K.wait_flags(flags, self.step_dev, 0, self.error, cfg.spin_timeout_s)
            K.omniscient(self.ps_grad_base, L.total, honest, w - 1, cfg.attack_magnitude, L.total,
                         step_ptr=self.step_dev, done_counter=self.push_counters[w:w + 1], flag=self.grad_flag_ptr(w))
            n += 2
        elif self.compress:
            enc, stream = self.enc_local[w], self.stream_local[w]
            K.push_encode(L, g32, g16, enc.data_ptr(), flag=None, **push_kw)                 # encode + adversary, locally
            nbytes = self.codec_w[w].pack(enc, stream)                                       # DRC2 stream, size on the device
            K.stream_push(stream, self.ps_stage_base + (w - 1) * self.codec.capacity, nbytes,
                          self.ps_stage_base + self.P * self.codec.capacity + 8 * (w - 1), step_ptr=self.step_dev,
                          done_counter=self.push_counters[w:w + 1], flag=self.grad_flag_ptr(w),
                          grid=self.cfg.push_ctas if self.rank != 0 else 2 * K.sm_count())
            n += 4
            if self.debug_checksum:
                self._dbg_loopback(w, g32, g16, push_kw)
        else:
            K.push_encode(L, g32, g16, self.slot_ptr(w), flag=self.grad_flag_ptr(w), **push_kw)
            n += 1
            if self.debug_checksum:
                self._dbg_loopback(w, g32, g16, push_kw)
        return n

    def _phase(self, name: str):
        import contextlib
        return self.timer.phase(name) if self.timer else contextlib.nullcontext()

    def _capture(self) -> None:
        """Capture this process's whole step once; replays then advance the device-side step counter themselves.
        (Called after two eager steps so that lazy cuDNN / cuBLAS initialisation never happens under capture.)"""
        torch.cuda.synchronize()
        self._check_error()
        self.graph = torch.cuda.CUDAGraph()
        # With the weight gradients on a side stream the step is captured on a HIGH-PRIORITY stream: whenever the backward chain
        # (BatchNorm backward -> dgrad -> ...) and a weight-gradient / push kernel both have CTAs pending, the chain's are
        # dispatched first (kernel-node priorities are captured from the stream).  Worker forward+backward 1.61 -> 1.52 ms.
        from ..ops import conv as _conv_ops_mod
        cap = torch.cuda.Stream(device=self.device, priority=-1) if _conv_ops_mod.WGRAD_SIDE_STREAM else None
        with torch.cuda.graph(self.graph, stream=cap):
            self.kernels_per_step = self._enqueue_local_step(None)
        if self.local_workers and self.worker.zero_copy:
            # gradients allocated during capture live at fixed addresses of the graph's pool: publish them once
            for w in self.local_workers:
                self.worker.upload_all_ptrs(w)
            torch.cuda.synchronize()

    def _stage(self, step: int) -> int:
        if self.local_workers and self.worker.dataset is not None:
            return self.worker.stage_batches(step)
        return 0

    def train_step(self, stage: bool = True, prefetch: bool = True) -> None:
        """Enqueue exactly one full step for this process (asynchronous; ``read_metrics``/``synchronize`` wait).
        With CUDA graphs the first two steps run eagerly, the third call captures, and from then on a step is one
        graph replay (plus the input staging copies)."""
        if not self.active:
            if self.debug_checksum and self.nprocs > 1:
                self._verify_checksums(self.step)          # collective: idle processes take part too
            self.step += 1
            return
        if self._use_graph and self.graph is None and self._eager_steps >= 2:
            self._capture()
        if stage and self._staged_step != self.step:
            self._stage(self.step)
        if self.graph is not None:
            self.graph.replay()
        else:
            self.kernels_per_step = self._enqueue_local_step(self.step)
            self._eager_steps += 1
            if self.debug_checksum:
                self._verify_checksums(self.step)
        self.step += 1
        if stage and prefetch:
            self.prefetch_inputs()

    def prefetch_inputs(self) -> None:
        """Gather the next step's batches on the CPU and start their H2D copy (copy stream) while the GPU runs the step that was
        just enqueued; the device-to-device hand-over into the step's input buffers is stream-ordered after that step, so it cannot
        overwrite inputs still in use.  ``train_step(prefetch=False)`` + this call lets a caller enqueue other work (the
        metrics D2H of the step) between the two."""
        if self.active and self._staged_step != self.step:
            self._stage(self.step)
            self._staged_step = self.step

    # ------------------------------------------------------------------ host-visible results
    def _check_error(self) -> None:
        e = int(self.error.item())
        if e:
            raise RuntimeError(f"rank {self.rank}: spin-wait watchdog fired (flag index {e - 1}) -- a peer never arrived")

    def read_metrics(self) -> Dict[str, float]:
        """Device -> host read of the step's loss / Prec@1 / Prec@5 (mean over local workers).  Waits for the step."""
        if self.timer is None:
            return self.resolve_metrics(self.enqueue_metrics_read())
        if not self.local_workers:
            torch.cuda.current_stream().synchronize()
            self._check_error()
            return self.timer.elapsed()
        m = torch.stack([self.worker.metrics[w] for w in self.local_workers]).mean(0)
        vals = m.tolist()
        self._check_error()
        return {"loss": vals[0], "prec1": vals[1], "prec5": vals[2], **self.timer.elapsed()}

    # Pipelined metric reads: the D2H copy of a step's loss / Prec@k (and of the watchdog word) is enqueued behind the
    # step and resolved by the host one step later, so the next step's launch never waits for the previous step to drain.
    def enqueue_metrics_read(self):
        if self.timer is not None:                         # phase timers need the synchronous read
            return self.read_metrics()
        if not hasattr(self, "_mpin"):
            self._mpin = [(torch.zeros(3, dtype=torch.float32).pin_memory(), torch.zeros(1, dtype=torch.int32).pin_memory(),
                           torch.cuda.Event(blocking=True)) for _ in range(4)]
            self._ppin = [torch.zeros(12, dtype=torch.int64).pin_memory() for _ in range(4)]
            self._mslot = 0
        slot = self._mslot
        self._mslot = (slot + 1) % len(self._mpin)
        pin_f, pin_e, ev = self._mpin[slot]
        if self.local_workers:
            m = torch.stack([self.worker.metrics[w] for w in self.local_workers]).mean(0)
            pin_f.copy_(m, non_blocking=True)
        pin_e.copy_(self.error, non_blocking=True)
        if self.default_phases:
            self._ppin[slot].copy_(self._phase_row(self.step - 1), non_blocking=True)      # 96 B: the step's device-side timeline
        ev.record()
        return slot

    def resolve_metrics(self, slot) -> Dict[str, float]:
        if isinstance(slot, dict):
            return slot
        pin_f, pin_e, ev = self._mpin[slot]
        wait_event(ev)
        if int(pin_e[0]):
            raise RuntimeError(f"rank {self.rank}: spin-wait watchdog fired (flag index {int(pin_e[0]) - 1}) -- a peer never arrived")
        phases = self._phases_from_row(self._ppin[slot].tolist()) if self.default_phases else {}
        if not self.local_workers:
            return phases
        v = pin_f.tolist()
        return {"loss": v[0], "prec1": v[1], "prec5": v[2], **phases}

    def synchronize(self) -> None:
        torch.cuda.synchronize()
        self._check_error()

    def wait_trace(self, last: int = 16) -> Dict[str, float]:
        """Device-side timeline of the last ``last`` steps from the %globaltimer stamps of the spin-wait kernels:
        how long this process's workers sat waiting for parameters (= everything that is not their own compute) and how
        long the PS sat waiting for gradients, plus the step period.  Milliseconds, means."""
        torch.cuda.synchronize()
        out: Dict[str, float] = {}
        cur = self.step - 1                                   # last completed step
        idx = [(cur - i) & 63 for i in range(min(last, 60))][::-1]
        for name, st, on in (("worker_wait_ms", self.stamps_worker, bool(self.local_workers)), ("ps_wait_ms", self.stamps_ps, self.is_ps)):
            if not on:
                continue
            t = st.cpu()[idx].double()
            out[name] = float((t[:, 1] - t[:, 0]).mean() / 1e6)
            per = (t[1:, 0] - t[:-1, 0]) / 1e6
            out[name.replace("wait", "period")] = float(per.mean()) if len(per) else float("nan")
        return out

    def master_params(self) -> torch.Tensor:
        """The fp32 parameter arena of this process (the PS's is the master copy)."""
        return self.params_f32

    def close(self) -> None:
        self.symm.close()


def make_plan(cfg: JobConfig, dataset: Optional[TensorDataset], groups) -> BatchPlan:
    n = len(dataset) if dataset is not None else cfg.synthetic_size
    return BatchPlan(cfg.approach, n, cfg.batch_size, cfg.num_workers,
                     group_of=groups.rank_to_group if groups is not None else None,
                     group_seeds=groups.seeds if groups is not None else None,
                     seed=428, redundancy=cfg.redundancy if cfg.approach == "cyclic" else 1)
