"""Parameter-server side: aggregation rules + optimizer.

Two implementations of the same semantics (reference: ``SyncReplicasMaster_NN`` / ``CodedMaster`` / ``CyclicMaster`` in
src/master/*.py):

* ``FusedPS``  -- the product path.  Decode + SGD + parameter broadcast are sm_100a kernels working on the flat
  ``grad_in`` slab that workers filled through peer stores (ops/kernels.py); nothing returns to the host.
* ``TorchPS``  -- reference-faithful structure: per-tensor decode with library ops, a separate optimizer step, used by
  the NCCL baseline transport and the CPU/Gloo transport (where the small dense solves go through the C++ host
  library instead of Eigen/scipy).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from .. import _native as N
from ..codes.adversary import COLLUSION_ATTACKS, attack_code
from ..codes.cyclic import CyclicCode, search_w
from ..codes.repetition import GroupPlan
from ..config import JobConfig
from .arena import ArenaLayout


def select_rule(cfg: JobConfig) -> str:
    """Aggregation rule of a job.  Mirrors the reference's dispatch: cyclic approach -> Fourier decode
    (cyclic_master.py:24); maj_vote approach -> vote only when ``--mode maj_vote``, plain mean for ``--mode normal``
    (rep_master.py:118-129); baseline approach -> mean / geometric median / Krum by ``--mode`` (baseline_master.py:118-129), plus
    the coordinate-wise median and trimmed mean (Yin et al., ICML 2018) and multi-Krum (Blanchard et al., NeurIPS 2017)."""
    if cfg.approach == "cyclic":
        return "cyclic"
    if cfg.approach == "maj_vote":
        return "vote" if cfg.mode == "maj_vote" else "mean"
    return {"normal": "mean", "geometric_median": "geomedian", "krum": "krum", "coord_median": "coord_median",
            "trimmed_mean": "trimmed_mean", "multi_krum": "multi_krum"}.get(cfg.mode, "mean")


COORDINATE_RULES = ("coord_median", "trimmed_mean")


def coordinate_trim(rule: str, P: int, f: int) -> int:
    """Values dropped at each end of every coordinate's sorted column: f for the trimmed mean, all but the middle one
    (odd P) or two (even P) for the median."""
    return (P - 1) // 2 if rule == "coord_median" else f


def hyperparams_tensor(cfg: JobConfig, device) -> torch.Tensor:
    opt = {"sgd": 0, "adam": 2 if getattr(cfg, "amsgrad", False) else 1}[cfg.optimizer]
    hp = N.HyperParams(cfg.lr, cfg.momentum, cfg.weight_decay, cfg.dampening, int(cfg.nesterov), opt,
                       float(cfg.adam_beta1), float(cfg.adam_beta2), float(cfg.adam_eps))
    raw = np.frombuffer(bytes(hp), dtype=np.uint8).copy()
    return torch.from_numpy(raw).to(device)


class FusedPS:
    """Kernel-driven PS state for one job (lives on the PS GPU)."""

    def __init__(self, cfg: JobConfig, layout: ArenaLayout, device: torch.device, params: torch.Tensor,
                 grad_in: torch.Tensor, groups: Optional[GroupPlan], code: Optional[CyclicCode], *,
                 adv_bitmap: Optional[torch.Tensor] = None):
        from ..ops import kernels as K
        self.K = K
        self.cfg, self.layout, self.device = cfg, layout, device
        self.P = cfg.num_workers
        # --err-mode alie / ipm: the liar slots of the step (device bitmap per step, see codes/adversary.py) are overwritten
        # by the collusion kernel after their gradients arrived and before the rule reads them
        self.adv_bitmap = adv_bitmap
        attack = attack_code(cfg.err_mode)
        self.collusion = attack if adv_bitmap is not None and attack in COLLUSION_ATTACKS else 0
        self.collusion_param = cfg.attack_param if self.collusion else 0.0
        self.params = params                       # fp32 [D] master copy (inside the exported region)
        self.grad_in = grad_in                     # fp32 [P, D] or complex64-as-fp32 [P, 2D]
        self.momentum = layout.new_arena(device)             # SGD momentum buffer / Adam first moment
        # Adam / AMSGrad state lives in arenas too (checkpointed with the momentum: utils/checkpoint.py)
        self.exp_avg_sq = layout.new_arena(device) if cfg.optimizer == "adam" else None
        self.max_exp_avg_sq = layout.new_arena(device) if (cfg.optimizer == "adam" and getattr(cfg, "amsgrad", False)) else None
        self.hp = hyperparams_tensor(cfg, device)
        self.counters = torch.zeros(16, dtype=torch.int32, device=device)
        T = layout.ntensors
        self.cyclic = cfg.approach == "cyclic"
        self.slot_stride = layout.total
        self.rule = select_rule(cfg)
        if self.rule == "vote":
            self.group_table = torch.from_numpy(groups.as_table()).to(device)
            G = self.group_table.shape[0]
            self.neq_mask = torch.zeros(G, T, dtype=torch.int32, device=device)
            self.winner_slot = torch.zeros(G, T, dtype=torch.int32, device=device)
            self.winner_member = torch.zeros(G, T, dtype=torch.int32, device=device)
        elif self.rule in ("krum", "multi_krum"):
            self.krum_m = self.P - cfg.worker_fail if self.rule == "multi_krum" else 1
            self.pair_d2 = torch.zeros(T, self.P * (self.P - 1) // 2, dtype=torch.float64, device=device)
            self.select = torch.zeros(self.krum_m, T, dtype=torch.int32, device=device)
        elif self.rule in COORDINATE_RULES:
            self.trim = coordinate_trim(self.rule, self.P, cfg.worker_fail)
        elif self.rule == "geomedian":
            if self.P <= K.GEOMED_FAST_MAXP:      # weight-space Weiszfeld: 2 passes over the slab in total
                self.gm = None
                self.pair_d2 = torch.zeros(T, self.P * (self.P - 1) // 2, dtype=torch.float64, device=device)
                self.gm_weights = torch.zeros(T, self.P, dtype=torch.float32, device=device)
            else:
                self.gm = K.GeoMedianWorkspace(layout, self.P, device)
        elif self.rule == "cyclic":
            self.code = code
            self.E = torch.zeros(T, self.P, 2, dtype=torch.float64, device=device)
            self.recomb = torch.zeros(T, self.P, 2, dtype=torch.float32, device=device)
            self.healthy = torch.zeros(T, dtype=torch.int32, device=device)
            self.flagged = torch.zeros(T, dtype=torch.int32, device=device)
            # per-tensor random projection f ~ N(1,1), fixed at build time (reference: cyclic_master.py:58-61)
            g = torch.Generator().manual_seed(cfg.seed + 4242)
            f = (torch.randn(layout.total, generator=g) + 1.0) * torch.from_numpy(layout.valid_mask()).float()
            self.f = f.to(device)

    @property
    def opt_state(self) -> Dict[str, Optional[torch.Tensor]]:
        """Optimizer arenas beyond ``momentum`` (Adam second moment, AMSGrad maximum) for checkpoints."""
        return {"exp_avg_sq": self.exp_avg_sq, "max_exp_avg_sq": self.max_exp_avg_sq}

    def collude(self, step_ptr: torch.Tensor, tile_range: Optional[tuple] = None, before=None) -> int:
        """Colluding attack of the step on the slab (or one bucket of it): ``before(tile_range)`` runs first, while every
        slot still holds what its worker pushed.  Returns the number of kernels launched (0 without such an attack)."""
        if not self.collusion:
            return 0
        if before is not None:
            before(tile_range)
        self.K.collude(self.layout, self.grad_in, self.slot_stride, self.P, self.adv_bitmap, self.adv_bitmap.numel(),
                       step_ptr, self.collusion, self.collusion_param, tile_range=tile_range)
        return 1

    def enqueue_step(self, step_ptr: torch.Tensor, *, mc_params: Optional[int], dst: Sequence[int], flags: Sequence[int],
                     grad_out: Optional[torch.Tensor] = None, buckets=None, wait_bucket=None, before_update=None,
                     before_collude=None) -> int:
        """Decode + update + broadcast for the step in ``*step_ptr``.  Returns the number of kernels launched.

        With ``buckets`` (the workers' push buckets, in arrival order) and ``wait_bucket(b)`` the PS is pipelined: bucket
        ``b`` is voted on, applied and broadcast as soon as every worker has pushed it, while the workers are still
        back-propagating / pushing the later buckets; only the last bucket is on the critical path.  Under a colluding
        attack each bucket (or the whole slab) first goes through the collusion kernel; ``before_collude(tile_range)`` is
        called right before it."""
        K, L = self.K, self.layout
        before_update = before_update or (lambda: 0)      # called right before the (last) fused update + broadcast kernel
        common = dict(params=self.params, momentum=self.momentum, exp_avg_sq=self.exp_avg_sq, max_exp_avg_sq=self.max_exp_avg_sq,
                      hp=self.hp, step_ptr=step_ptr,
                      done_counter=self.counters[0:1], first_step=1, grad_out=grad_out, mc_params=mc_params, dst=dst)
        n = 0
        if buckets is not None and self.rule in ("mean", "vote") + COORDINATE_RULES:
            for bi, (t0, t1, idxs) in enumerate(buckets):
                n += wait_bucket(bi)
                n += self.collude(step_ptr, (t0, t1), before_collude)
                fl = flags if bi == len(buckets) - 1 else []
                if self.rule == "vote":
                    K.vote(L, self.grad_in, self.slot_stride, self.group_table, self.neq_mask, self.winner_slot,
                           self.winner_member, tile_range=(t0, t1), tensor_range=(min(idxs), max(idxs) + 1)); n += 2
                    G = self.group_table.shape[0]
                    if bi == len(buckets) - 1:
                        n += before_update()
                    K.aggregate_update(L, self.grad_in, self.slot_stride, K=G, scale=1.0 / G, select=self.winner_slot,
                                       tile_range=(t0, t1), flags=fl, **common); n += 1
                elif self.rule in COORDINATE_RULES:
                    if bi == len(buckets) - 1:
                        n += before_update()
                    K.aggregate_update(L, self.grad_in, self.slot_stride, K=self.P, scale=1.0 / (self.P - 2 * self.trim),
                                       trim=self.trim, tile_range=(t0, t1), flags=fl, **common); n += 1
                else:
                    if bi == len(buckets) - 1:
                        n += before_update()
                    K.aggregate_update(L, self.grad_in, self.slot_stride, K=self.P, scale=1.0 / self.P,
                                       tile_range=(t0, t1), flags=fl, **common); n += 1
            return n
        common["flags"] = flags
        n += self.collude(step_ptr, None, before_collude)
        _agg = K.aggregate_update

        def _update(*a, **kw):                             # every rule below ends in exactly one fused update kernel
            nonlocal n
            n += before_update()
            _agg(*a, **kw)
        if self.rule == "mean":
            _update(L, self.grad_in, self.slot_stride, K=self.P, scale=1.0 / self.P, **common); n += 1
        elif self.rule == "vote":
            K.vote(L, self.grad_in, self.slot_stride, self.group_table, self.neq_mask, self.winner_slot, self.winner_member); n += 2
            G = self.group_table.shape[0]
            _update(L, self.grad_in, self.slot_stride, K=G, scale=1.0 / G, select=self.winner_slot, **common); n += 1
        elif self.rule in ("krum", "multi_krum"):
            m = self.krum_m
            K.krum_select(L, self.grad_in, self.slot_stride, self.P, self.cfg.worker_fail, self.pair_d2, self.select, m=m); n += 2
            _update(L, self.grad_in, self.slot_stride, K=m, scale=1.0 / m, select=self.select, **common); n += 1
        elif self.rule in COORDINATE_RULES:
            _update(L, self.grad_in, self.slot_stride, K=self.P, scale=1.0 / (self.P - 2 * self.trim), trim=self.trim,
                    **common); n += 1
        elif self.rule == "geomedian" and self.gm is None:
            K.geometric_median_weights(L, self.grad_in, self.slot_stride, self.P, self.pair_d2, self.gm_weights); n += 2
            _update(L, self.grad_in, self.slot_stride, K=self.P, scale=1.0, weights=self.gm_weights, **common); n += 1
        elif self.rule == "geomedian":
            iters = 48
            K.geometric_median(L, self.grad_in, self.slot_stride, self.P, self.gm, iters=iters); n += 2 * iters + 1
            _update(L, self.gm.median, self.slot_stride, K=1, scale=1.0, **common); n += 1
        elif self.rule == "cyclic":
            K.cyclic_project(L, self.grad_in, self.slot_stride, self.P, self.f, self.E); n += 1
            K.cyclic_locate(self.E, self.P, self.cfg.worker_fail, self.recomb, self.healthy, self.flagged); n += 1
            _update(L, self.grad_in, self.slot_stride, K=self.P, scale=1.0 / self.P, recomb=self.recomb, **common); n += 1
        return n


# =====================================================================================================
# Library-op PS (NCCL baseline + CPU/Gloo)
# =====================================================================================================
class TorchPS:
    """Per-tensor decode with torch / host-C++ ops + a separate optimizer step (reference-faithful structure)."""

    def __init__(self, cfg: JobConfig, layout: ArenaLayout, device: torch.device, params: torch.Tensor,
                 groups: Optional[GroupPlan], code: Optional[CyclicCode]):
        from ..optim import SGDModified, AdamModified
        self.cfg, self.layout, self.device, self.params = cfg, layout, device, params
        self.P = cfg.num_workers
        self.groups, self.code = groups, code
        self.rule = select_rule(cfg)
        # flat per-tensor views in arena element order (the optimizer is element-wise, so order is irrelevant)
        views = [params[s.offset: s.offset + s.numel] for s in layout.specs]
        self._views = views
        if cfg.optimizer == "adam":
            self.optimizer = AdamModified(views, lr=cfg.lr, betas=(cfg.adam_beta1, cfg.adam_beta2), eps=cfg.adam_eps,
                                          weight_decay=cfg.weight_decay, amsgrad=cfg.amsgrad)
        else:
            self.optimizer = SGDModified(views, lr=cfg.lr, momentum=cfg.momentum, weight_decay=cfg.weight_decay,
                                         dampening=cfg.dampening, nesterov=cfg.nesterov)
        if self.rule == "cyclic":
            g = torch.Generator().manual_seed(cfg.seed + 4242)
            f = (torch.randn(layout.total, generator=g) + 1.0) * torch.from_numpy(layout.valid_mask()).float()
            self.f = f.to(device)
        self.last_info: Dict[str, object] = {}

    # --- optimizer state for checkpoints (the reference saves none: src/master/baseline_master.py:237-243) ----------
    @property
    def momentum(self) -> Optional[torch.Tensor]:
        """SGD momentum buffers gathered into a flat arena (a copy), or None when there is nothing to save yet."""
        from ..optim import SGDModified
        if not isinstance(self.optimizer, SGDModified):
            return self._gather("exp_avg")                  # Adam: the first moment plays the momentum's role in checkpoints
        if self.cfg.momentum == 0:
            return None
        arena, found = self.layout.new_arena(self.device), False
        for v, spec in zip(self._views, self.layout.specs):
            buf = self.optimizer.state.get(v, {}).get("momentum_buffer")
            if buf is not None:
                arena[spec.offset: spec.offset + spec.numel].copy_(buf)
                found = True
        return arena if found else None

    def load_momentum(self, arena: torch.Tensor) -> None:
        key = "momentum_buffer" if self.cfg.optimizer != "adam" else "exp_avg"
        for v, spec in zip(self._views, self.layout.specs):
            self.optimizer.state[v][key] = arena[spec.offset: spec.offset + spec.numel].clone()

    def _gather(self, key: str) -> Optional[torch.Tensor]:
        arena, found = self.layout.new_arena(self.device), False
        for v, spec in zip(self._views, self.layout.specs):
            buf = self.optimizer.state.get(v, {}).get(key)
            if buf is not None:
                arena[spec.offset: spec.offset + spec.numel].copy_(buf)
                found = True
        return arena if found else None

    @property
    def opt_state(self) -> Dict[str, Optional[torch.Tensor]]:
        if self.cfg.optimizer != "adam":
            return {}
        return {"exp_avg_sq": self._gather("exp_avg_sq"), "max_exp_avg_sq": self._gather("max_exp_avg_sq")}

    def load_opt_state(self, arenas: Dict[str, torch.Tensor], step: int) -> None:
        """Adam: second moment (+ AMSGrad maximum) and the per-tensor step count (= updates applied so far)."""
        if self.cfg.optimizer != "adam":
            return
        for v, spec in zip(self._views, self.layout.specs):
            st = self.optimizer.state[v]
            st["step"] = int(step)
            st.setdefault("exp_avg", torch.zeros_like(v))
            for key, arena in arenas.items():
                if arena is not None:
                    st[key] = arena[spec.offset: spec.offset + spec.numel].clone()
            st.setdefault("exp_avg_sq", torch.zeros_like(v))

    # --- per-tensor rules -----------------------------------------------------------------------
    def _vote_tensor(self, rows: List[torch.Tensor]) -> int:
        cand, count = 0, 0
        for k, r in enumerate(rows):
            if count == 0:
                cand, count = k, 1
            elif torch.equal(r, rows[cand]):
                count += 1
            else:
                count -= 1
        return cand

    def _geomedian_tensor(self, X: torch.Tensor, iters: int = 100, eps: float = 1e-6) -> torch.Tensor:
        if X.device.type == "cpu":
            out = torch.empty(X.shape[1], dtype=torch.float32)
            Xc = X.contiguous()
            N.host().drc_host_geomedian(Xc.data_ptr(), Xc.shape[0], Xc.shape[1], Xc.stride(0), eps, iters, out.data_ptr())
            return out
        m = X.mean(0)
        for _ in range(iters):
            d = (X - m).norm(dim=1).clamp_min(1e-30)
            w = 1.0 / d
            m_new = (w[:, None] * X).sum(0) / w.sum()
            done = (m_new - m).norm() <= eps * max(1.0, float(m.norm()))
            m = m_new
            if done:
                break
        return m

    def _krum_scores(self, X: torch.Tensor) -> torch.Tensor:
        d2 = torch.cdist(X.double(), X.double()).pow(2)
        P = X.shape[0]
        keep = max(P - self.cfg.worker_fail - 2, 0)
        d2 = d2 + torch.diag(torch.full((P,), float("inf"), dtype=d2.dtype, device=d2.device))
        return d2.sort(dim=1).values[:, :keep].sum(1)

    def _krum_tensor(self, X: torch.Tensor) -> int:
        return int(self._krum_scores(X).argmin())

    def _multi_krum_tensor(self, X: torch.Tensor) -> torch.Tensor:
        """Mean of the P - f lowest-scoring rows (ties to the lower slot), summed in ascending slot order."""
        m = self.P - self.cfg.worker_fail
        rows = sorted(torch.argsort(self._krum_scores(X), stable=True)[:m].tolist())
        acc = X[rows[0]].clone()
        for r in rows[1:]:
            acc += X[r]
        return acc / m

    def _coordinate_tensor(self, X: torch.Tensor) -> torch.Tensor:
        """Coordinate-wise trimmed mean / median: sort every column (NaN last), drop ``trim`` values at each end."""
        b = coordinate_trim(self.rule, self.P, self.cfg.worker_fail)
        return torch.sort(X, dim=0).values[b: self.P - b].sum(0) / (self.P - 2 * b)

    def _cyclic_tensor(self, R: torch.Tensor, f: torch.Tensor) -> torch.Tensor:
        """R: [n, d] complex64 -> Re(v^T R) / n with v from the C++ locator (N1 replacement)."""
        n, s = self.P, self.cfg.worker_fail
        E = (R.to(torch.complex128) @ f.to(torch.complex128))
        Eh = torch.view_as_real(E).contiguous().cpu().double().numpy()
        v = np.zeros((n, 2)); mask = np.zeros(1, dtype=np.uint32); fl = np.zeros(1, dtype=np.int32)
        N.check(N.host().drc_host_locate(Eh.ctypes.data, 1, n, s, 1e-4, v.ctypes.data, mask.ctypes.data, fl.ctypes.data), "locate")
        vt = torch.from_numpy(v[:, 0] + 1j * v[:, 1]).to(R.device).to(torch.complex64)
        self.last_info.setdefault("flagged", []).append(int(fl[0]))
        return (vt @ R).real / n

    # --- step -----------------------------------------------------------------------------------
    def aggregate(self, slots: torch.Tensor) -> List[torch.Tensor]:
        """``slots``: [P, D] fp32 (or [P, D] complex64 for cyclic).  Returns the per-tensor aggregated gradients."""
        L = self.layout
        self.last_info = {}
        out = []
        for i, spec in enumerate(L.specs):
            X = slots[:, spec.offset: spec.offset + spec.numel]
            if self.rule == "mean":
                g = X.sum(0) / self.P
            elif self.rule == "vote":
                acc = torch.zeros(spec.numel, dtype=torch.float32, device=X.device)
                for grp in self.groups.groups:
                    rows = [X[w - 1] for w in grp]
                    acc += rows[self._vote_tensor(rows)]
                g = acc / float(self.groups.num_groups)
            elif self.rule == "krum":
                g = X[self._krum_tensor(X)]
            elif self.rule == "multi_krum":
                g = self._multi_krum_tensor(X)
            elif self.rule in COORDINATE_RULES:
                g = self._coordinate_tensor(X)
            elif self.rule == "geomedian":
                g = self._geomedian_tensor(X)
            elif self.rule == "cyclic":
                g = self._cyclic_tensor(X, self.f[spec.offset: spec.offset + spec.numel])
            else:
                raise ValueError(self.rule)
            out.append(g)
        return out

    def step(self, slots: torch.Tensor) -> None:
        self.apply(self.aggregate(slots))

    def apply(self, grads: List[torch.Tensor]) -> None:
        mode = {"mean": "normal", "vote": "maj_vote", "krum": "krum", "geomedian": "geometric_median", "cyclic": "cyclic",
                "coord_median": "coord_median", "trimmed_mean": "trimmed_mean", "multi_krum": "multi_krum"}[self.rule]
        self.optimizer.step(grads=grads, mode=mode)


def build_codes(cfg: JobConfig):
    """(GroupPlan | None, CyclicCode | None) for a job -- the coding part of the reference's ``prepare``."""
    from ..codes.repetition import group_assign
    groups = group_assign(cfg.num_workers, cfg.group_size) if cfg.approach == "maj_vote" else None
    code = search_w(cfg.num_workers, cfg.worker_fail) if cfg.approach == "cyclic" else None
    return groups, code
