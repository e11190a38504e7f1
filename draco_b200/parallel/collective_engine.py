"""Library-collective transports: ``--transport nccl`` (the measured baseline) and ``--transport gloo`` (CPU plumbing).

This engine keeps the *structure* of the reference's step on purpose, so that it can serve as the reference-faithful
baseline BASELINE.md asks for -- the unmodified reference cannot run here (Python 2.7 / torch 0.3 / mpi4py):

* one broadcast per parameter tensor per step        (reference: ``comm.Bcast`` per layer, baseline_master.py:180-186)
* one message per (worker, parameter tensor) upward  (reference: ``isend`` tag 88+layer, baseline_worker.py:258-273)
* decode, optimizer step and broadcast are separate phases built from library ops (TorchPS)
* encode / adversary / (optional) compression are separate passes over the gradient

Only the communication library differs: NCCL (or Gloo) point-to-point and broadcast instead of mpi4py.  Wire dtype is
fp32 (complex64 for the cyclic code); ``--compress-grad compress`` runs the C++ lossless codec on the CPU path.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import torch
import torch.distributed as dist

from ..codes.adversary import generate_schedule
from ..config import COLLUDING_ERR_MODES, JobConfig
from ..data import TensorDataset
from ..utils.codec import compress, decompress
from ..utils.metrics import PhaseTimer, limit_host_threads
from .arena import ArenaLayout
from .fused_engine import make_plan
from .placement import Placement
from .ps import TorchPS, build_codes
from .worker import WorkerCompute, make_model


class CollectiveEngine:
    def __init__(self, cfg: JobConfig, rank: int, nprocs: int, device: torch.device, dataset: Optional[TensorDataset],
                 group=None):
        self.cfg, self.rank, self.nprocs, self.device, self.group = cfg, rank, nprocs, torch.device(device), group
        self.place = Placement(cfg.num_workers, nprocs)
        self.P = cfg.num_workers
        self.is_ps = rank == 0
        self.local_workers = self.place.local_workers(rank)
        self.active = self.is_ps or bool(self.local_workers)
        self.groups, self.code = build_codes(cfg)
        self.cyclic = cfg.approach == "cyclic"
        self.step = 1
        self.kernels_per_step = 0
        if self.device.type == "cuda":
            limit_host_threads()            # same host policy as the fused engine (fair baseline: no OpenMP spin pool)
        if cfg.deterministic and self.device.type == "cuda":
            torch.backends.cudnn.deterministic = True
            torch.backends.cudnn.benchmark = False
            os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
        model = make_model(cfg)
        bf16 = cfg.dtype == "bf16" and self.device.type == "cuda"
        self.layout = ArenaLayout.from_model(model, bf16, channels_last=self.device.type == "cuda")
        plan = make_plan(cfg, dataset, self.groups)
        self.worker = WorkerCompute(cfg, self.device, self.local_workers, plan, dataset, self.layout, None, model)
        self.params_f32 = self.worker.binder.params_f32
        self.schedule = generate_schedule(self.P, cfg.worker_fail, cfg.max_steps)
        self.use_adv = cfg.err_mode != "none" and cfg.worker_fail > 0
        wire = torch.complex64 if self.cyclic else torch.float32
        self.sendbuf = {w: torch.zeros(self.layout.total, dtype=wire, device=self.device) for w in self.local_workers}
        self.ps: Optional[TorchPS] = None
        if self.is_ps:
            self.slots = torch.zeros(self.P, self.layout.total, dtype=wire, device=self.device)
            self.ps = TorchPS(cfg, self.layout, self.device, self.params_f32, self.groups, self.code)
            if self.use_adv and cfg.err_mode in COLLUDING_ERR_MODES:    # the colluded vector keeps the slots' padding zero
                self._valid = torch.from_numpy(self.layout.valid_mask()).to(self.device)
        self.compress = cfg.compress and self.device.type == "cpu"
        self.compress_gpu = cfg.compress and self.device.type == "cuda"
        self.bytes_up = 0
        self.bytes_up_raw = 0
        self.timer = PhaseTimer(self.device.type == "cuda") if cfg.profile_phases else None
        self.last_phases: Dict[str, float] = {}

    # ------------------------------------------------------------------ phases
    def _broadcast_params(self) -> None:
        if self.nprocs > 1 and self.cfg.comm_type == "Async":
            # --comm-type=Async: the PS posts one point-to-point send per (parameter tensor, worker process) instead of a
            # broadcast (reference: async_bcast_layer_weights_async, baseline_master.py:164-178 <-> baseline_worker.py:171-188).
            # Like the reference's, the step stays fully synchronous -- only the fan-out primitive differs.
            ops = []
            peers = [p for p in self.place.worker_procs() if p != 0]
            for i in range(self.layout.ntensors):
                s = self.layout.specs[i]
                view = self.params_f32[s.offset: s.offset + s.numel]
                if self.is_ps:
                    ops += [dist.P2POp(dist.isend, view, p, group=self.group) for p in peers]
                elif self.rank in peers:
                    ops.append(dist.P2POp(dist.irecv, view, 0, group=self.group))
            if ops:
                for r in dist.batch_isend_irecv(ops):
                    r.wait()
        elif self.nprocs > 1:
            for i in range(self.layout.ntensors):
                s = self.layout.specs[i]
                dist.broadcast(self.params_f32[s.offset: s.offset + s.numel], src=0, group=self.group)
        self.worker.binder.refresh_compute_copy()

    def _encode(self, w: int, step: int) -> torch.Tensor:
        wc = self.worker
        buf = self.sendbuf[w]
        if self.cyclic:
            coef = self.code.coeffs_of(w - 1)
            buf.zero_()
            for k in range(wc.R):
                buf.add_(wc.flat_gradient(k).to(torch.complex64), alpha=complex(coef[k]))
        else:
            buf.copy_(wc.flat_gradient(0))
        if self.use_adv and self.schedule.is_adversary(w, step):
            self._corrupt(buf, w, step)
        return buf

    def _corrupt(self, buf: torch.Tensor, w: int, step: int) -> None:
        mag = self.cfg.attack_magnitude
        mode = self.cfg.err_mode
        for s in self.layout.specs:
            v = buf[s.offset: s.offset + s.numel]
            if mode == "rev_grad":
                adv = v * mag
            elif mode == "constant":
                adv = torch.full_like(v, mag)
            elif mode == "random":
                g = torch.Generator(device="cpu").manual_seed((self.cfg.seed * 1000003 + step * 8191 + w) & 0x7FFFFFFF)
                adv = (abs(mag) * torch.randn(s.numel, generator=g)).to(v.device).to(v.dtype)
            elif mode == "omniscient":
                continue            # handled at the PS where the honest gradients are visible (see _omniscient)
            else:
                return
            if self.cyclic:
                v.add_(adv)
            else:
                v.copy_(adv)

    def _omniscient(self, step: int) -> None:
        liars = [w for w in range(1, self.P + 1) if self.schedule.is_adversary(w, step)]
        honest = [w for w in range(1, self.P + 1) if w not in liars]
        if not liars or not honest:
            return
        mean = self.slots[[h - 1 for h in honest]].mean(0)
        for w in liars:
            self.slots[w - 1].copy_(mean * self.cfg.attack_magnitude)

    def _collude(self, step: int) -> None:
        """--err-mode alie / ipm: every liar slot <- mu - z * sigma / -epsilon * mu of the honest slots, per coordinate, in fp64
        (codes/adversary.py::collude), rounded into the fp32 slots.  Padding stays zero."""
        liars = [w - 1 for w in range(1, self.P + 1) if self.schedule.is_adversary(w, step)]
        honest = [r for r in range(self.P) if r not in liars]
        if not liars or not honest:
            return
        X = self.slots[honest].double()
        mu = X.mean(0)
        param = self.cfg.attack_param
        lie = mu - param * X.std(0) if self.cfg.err_mode == "alie" else -param * mu
        self.slots[liars] = torch.where(self._valid, lie, 0.0).to(self.slots.dtype)

    def _exchange_gradients(self, step: int) -> None:
        """Per-tensor point-to-point: every remote worker -> PS."""
        L = self.layout
        ops = []
        recv_tmp = {}
        if self.compress and self.nprocs > 1:
            self._exchange_compressed(step)
            return
        if self.compress_gpu and self.nprocs > 1:
            self._exchange_compressed_gpu(step)
            return
        for w in range(1, self.P + 1):
            src_proc = self.place.proc_of[w]
            if self.is_ps and src_proc == 0:
                self.slots[w - 1].copy_(self.sendbuf[w])
                continue
            for s in L.specs:
                if self.is_ps:
                    ops.append(dist.P2POp(dist.irecv, self.slots[w - 1, s.offset: s.offset + s.numel], src_proc, group=self.group))
                elif src_proc == self.rank:
                    ops.append(dist.P2POp(dist.isend, self.sendbuf[w][s.offset: s.offset + s.numel], 0, group=self.group))
                    self.bytes_up += s.numel * self.sendbuf[w].element_size()
        if ops:
            for r in dist.batch_isend_irecv(ops):
                r.wait()

    def _exchange_compressed_gpu(self, step: int) -> None:
        """NCCL path with the device codec (csrc/cuda/codec.cu): the flat gradient is compressed on the GPU, the byte
        stream travels (length first), and the PS decompresses it straight into the worker's slot."""
        from ..utils.codec import compress_tensor, decompress_tensor
        for w in range(1, self.P + 1):
            src_proc = self.place.proc_of[w]
            if self.is_ps and src_proc == 0:
                self.slots[w - 1].copy_(self.sendbuf[w])
                continue
            if self.is_ps:
                n = torch.zeros(1, dtype=torch.int64, device=self.device)
                dist.recv(n, src=src_proc, group=self.group)
                payload = torch.empty(int(n.item()), dtype=torch.uint8, device=self.device)
                dist.recv(payload, src=src_proc, group=self.group)
                self.slots[w - 1].copy_(decompress_tensor(payload, self.slots.dtype, (self.layout.total,)))
            elif src_proc == self.rank:
                s = compress_tensor(self.sendbuf[w])
                self.bytes_up_raw += self.sendbuf[w].numel() * self.sendbuf[w].element_size()
                self.bytes_up += s.numel()
                dist.send(torch.tensor([s.numel()], dtype=torch.int64, device=self.device), dst=0, group=self.group)
                dist.send(s, dst=0, group=self.group)

    def _exchange_compressed(self, step: int) -> None:
        """Gloo path with the lossless codec: per tensor, length header then payload (reference: blosc + isend)."""
        L = self.layout
        for w in range(1, self.P + 1):
            src_proc = self.place.proc_of[w]
            if self.is_ps and src_proc == 0:
                self.slots[w - 1].copy_(self.sendbuf[w])
                continue
            if self.is_ps:
                lens = torch.zeros(L.ntensors, dtype=torch.int64)
                dist.recv(lens, src=src_proc, group=self.group)
                for i, s in enumerate(L.specs):
                    payload = torch.empty(int(lens[i]), dtype=torch.uint8)
                    dist.recv(payload, src=src_proc, group=self.group)
                    arr = decompress(payload.numpy().tobytes())
                    t = torch.from_numpy(arr)
                    # cyclic codewords travel as [numel, 2] float32 (re, im) pairs
                    t = torch.view_as_complex(t.reshape(-1, 2).contiguous()) if self.cyclic else t.reshape(-1)
                    self.slots[w - 1, s.offset: s.offset + s.numel].copy_(t)
            elif src_proc == self.rank:
                msgs = []
                for s in L.specs:
                    arr = self.sendbuf[w][s.offset: s.offset + s.numel].contiguous()
                    raw = torch.view_as_real(arr).numpy() if arr.is_complex() else arr.numpy()
                    msgs.append(compress(raw))
                    self.bytes_up_raw += raw.nbytes
                    self.bytes_up += len(msgs[-1])
                dist.send(torch.tensor([len(m) for m in msgs], dtype=torch.int64), dst=0, group=self.group)
                for m in msgs:
                    dist.send(torch.frombuffer(bytearray(m), dtype=torch.uint8), dst=0, group=self.group)

    # ------------------------------------------------------------------ the step
    def _phase(self, name: str):
        import contextlib
        return self.timer.phase(name) if self.timer else contextlib.nullcontext()

    def train_step(self, stage: bool = True) -> None:
        step = self.step
        with self._phase("t_fetch"):                      # reference: "Comm" on the worker (weights down)
            self._broadcast_params()
        if self.local_workers:
            if stage and self.worker.dataset is not None:
                self.worker.stage_batches(step)
            for w in self.local_workers:
                with self._phase("t_comp"):
                    self.worker.forward_backward(w, step)
                with self._phase("t_encode"):
                    self._encode(w, step)
        with self._phase("t_comm"):                       # gradients up
            self._exchange_gradients(step)
        if self.is_ps:
            if self.use_adv and self.cfg.err_mode == "omniscient":
                self._omniscient(step)
            elif self.use_adv and self.cfg.err_mode in COLLUDING_ERR_MODES:
                self._collude(step)
            with self._phase("t_decode"):                 # reference: "Method Time Cost"
                grads = self.ps.aggregate(self.slots)
            with self._phase("t_update"):                 # reference: "Update Time Cost"
                self.ps.apply(grads)
        if self.timer:
            self.last_phases = self.timer.elapsed()
        self.step += 1

    def read_metrics(self) -> Dict[str, float]:
        if not self.local_workers:
            return dict(self.last_phases)
        m = torch.stack([self.worker.metrics[w] for w in self.local_workers]).mean(0).tolist()
        return {"loss": m[0], "prec1": m[1], "prec5": m[2], **self.last_phases}

    def enqueue_metrics_read(self):
        """Same protocol as the fused engine's pipelined read; the library-op engine simply reads synchronously."""
        return self.read_metrics()

    def resolve_metrics(self, handle) -> Dict[str, float]:
        return handle

    def synchronize(self) -> None:
        if self.device.type == "cuda":
            torch.cuda.synchronize()

    def master_params(self) -> torch.Tensor:
        return self.params_f32

    def close(self) -> None:
        pass
