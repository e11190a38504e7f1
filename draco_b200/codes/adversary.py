"""Simulated Byzantine workers: per-step schedule and attack models.

Schedule parity: the reference draws, with numpy's global RNG seeded to 428, ``max_steps+1``
samples of ``worker_fail`` distinct worker ranks out of ``1..P`` (src/util.py:100-103) and a
worker lies at step ``t`` iff ``rank in schedule[t]`` (src/worker/rep_worker.py:162).  We draw the
same stream from a private ``RandomState(428)`` so the *same ranks lie at the same steps*.

Attack parity (src/model_ops/utils.py:3-23), ``mag = -100``:
  rev_grad : replace  g -> mag*g           (cyclic: add, i.e. g + mag*g)
  constant : replace  g -> mag             (cyclic: g + mag)
  random   : reference is a no-op (TODO there).  Here it is a real attack: g -> sigma*N(0,1)
             (cyclic: g + sigma*N(0,1)) from a counter-based generator keyed by (seed, step, worker)
  omniscient (north-star extension): g -> -k * mean(honest gradients); needs a view of the honest
             gradients so it is applied by the engine, not by the per-worker hook.

Colluding attacks, designed to defeat the robust baselines (see ``collude``).  Every liar of the step
sends the same vector, built from the per-coordinate mean ``mu`` and unbiased standard deviation
``sigma`` of the honest slots:
  alie : g -> mu - z * sigma   "A Little Is Enough" (Baruch et al., NeurIPS 2019); z = ``alie_z_max``
  ipm  : g -> -epsilon * mu    inner-product manipulation (Xie et al., UAI 2019)
Both read every honest gradient, so they are applied where all of them meet: at the parameter server,
after the gradients arrived and before the aggregation rule runs (csrc/cuda/collude.cu).

The device implementation of the per-worker hook lives in csrc/cuda/push_encode.cu; the integer codes
below are shared with it and with collude.cu.
"""
from __future__ import annotations

from dataclasses import dataclass
from statistics import NormalDist
from typing import List, Optional, Sequence

import numpy as np

SEED = 428
ADVERSARY_MAG = -100.0     # reference: ADVERSARY_ / CONST_ in src/model_ops/utils.py:3-4

ATTACK_NONE = 0
ATTACK_REV_GRAD = 1
ATTACK_CONSTANT = 2
ATTACK_RANDOM = 3
ATTACK_OMNISCIENT = 4
ATTACK_ALIE = 5
ATTACK_IPM = 6
COLLUSION_ATTACKS = (ATTACK_ALIE, ATTACK_IPM)     # applied by the parameter server, not by the worker's push

_ATTACK_CODES = {
    "none": ATTACK_NONE,
    "rev_grad": ATTACK_REV_GRAD,
    "constant": ATTACK_CONSTANT,
    "random": ATTACK_RANDOM,
    "omniscient": ATTACK_OMNISCIENT,
    "alie": ATTACK_ALIE,
    "ipm": ATTACK_IPM,
}


def attack_code(name: str) -> int:
    try:
        return _ATTACK_CODES[name]
    except KeyError:
        raise ValueError(f"unknown --err-mode {name!r}; choose from {sorted(_ATTACK_CODES)}") from None


@dataclass(frozen=True)
class AdversarySchedule:
    """``ranks[t]`` = sorted worker ranks (1-based) that lie at step ``t`` (t = 0..max_steps)."""

    num_workers: int
    worker_fail: int
    ranks: List[np.ndarray]

    def is_adversary(self, rank: int, step: int) -> bool:
        return bool(np.any(self.ranks[step % len(self.ranks)] == rank))

    def bitmaps(self) -> np.ndarray:
        """uint32 bitmap per step: bit ``w-1`` set iff worker ``w`` lies (consumed on device)."""
        out = np.zeros(len(self.ranks), dtype=np.uint32)
        for t, r in enumerate(self.ranks):
            for w in r:
                out[t] |= np.uint32(1) << np.uint32(int(w) - 1)
        return out


def generate_schedule(num_workers: int, worker_fail: int, max_steps: int, seed: int = SEED) -> AdversarySchedule:
    if worker_fail > num_workers:
        raise ValueError("more adversaries than workers")
    if num_workers > 32:
        raise ValueError("adversary bitmaps are 32-bit: at most 32 workers")
    rng = np.random.RandomState(seed)
    pool = np.arange(1, num_workers + 1)
    ranks = [np.sort(rng.choice(pool, size=worker_fail, replace=False)) for _ in range(max_steps + 1)]
    return AdversarySchedule(num_workers, worker_fail, ranks)


def _philox_like_normal(shape, seed: int, step: int, worker: int) -> np.ndarray:
    rng = np.random.Generator(np.random.Philox(key=[(seed << 32) ^ (step & 0xFFFFFFFF), worker]))
    return rng.standard_normal(shape)


def err_simulation(grad: np.ndarray, mode: str, cyclic: bool = False, *, magnitude: float = ADVERSARY_MAG,
                   seed: int = SEED, step: int = 0, worker: int = 0,
                   honest_mean: Optional[np.ndarray] = None) -> np.ndarray:
    """Host oracle of the adversary hook (same name as the reference's function)."""
    g = np.asarray(grad)
    if mode in ("none", None):
        return g
    if mode == "rev_grad":
        adv = magnitude * g
    elif mode == "constant":
        adv = np.full(g.shape, magnitude, dtype=g.dtype if np.iscomplexobj(g) else np.float64)
    elif mode == "random":
        adv = abs(magnitude) * _philox_like_normal(g.shape, seed, step, worker)
    elif mode == "omniscient":
        if honest_mean is None:
            raise ValueError("omniscient attack needs the honest mean")
        adv = magnitude * np.asarray(honest_mean)
    else:
        raise ValueError(f"unknown err mode {mode!r}")
    if cyclic:
        return g + adv
    return adv if np.iscomplexobj(g) else adv.astype(g.dtype, copy=False)


def alie_z_max(num_workers: int, worker_fail: int) -> float:
    """ALIE's default z (Baruch et al., NeurIPS 2019, section 3): with ``s = floor(P/2 + 1) - f`` honest workers the
    liars must win over, the largest z for which ``s`` of them are still expected to sit farther from the mean than the
    lie, ``z = Phi^{-1}((P - s) / P)``.  Undefined (ValueError) when ``s <= 0``: the liars alone are a majority."""
    P, f = int(num_workers), int(worker_fail)
    s = (P // 2 + 1) - f
    if P < 1 or s <= 0:
        raise ValueError(f"ALIE's default z is undefined for {P} workers with {f} liars (s = floor(P/2 + 1) - f = {s} <= 0); "
                         f"pass --alie-z")
    return NormalDist().inv_cdf((P - s) / P)


def collude(slots: np.ndarray, liars: Sequence[int], mode: str, param: float) -> np.ndarray:
    """Oracle of the colluding attacks.  ``slots``: [P, D] worker gradients; ``liars``: 0-based rows that lie.  Returns an
    fp64 copy of the slab whose liar rows all hold the same vector, computed in fp64 from the honest rows H (every other
    row, ascending): ``mu - param * sigma`` for ``alie`` (``param`` = z), ``-param * mu`` for ``ipm`` (``param`` = epsilon),
    with ``mu`` the mean and ``sigma`` the unbiased (ddof = 1) standard deviation of each coordinate over H.  Honest rows are
    returned unchanged; non-finite honest values propagate per IEEE."""
    out = np.array(slots, dtype=np.float64, copy=True)
    P = out.shape[0]
    lie = sorted({int(r) for r in liars})
    if any(r < 0 or r >= P for r in lie):
        raise ValueError(f"liar rows {lie} outside 0..{P - 1}")
    honest = [r for r in range(P) if r not in lie]
    if not lie or not honest:
        return out
    X = out[honest]
    mu = X.sum(axis=0) / len(honest)
    if mode == "alie":
        sigma = np.sqrt(((X - mu) ** 2).sum(axis=0) / (len(honest) - 1)) if len(honest) > 1 else np.full_like(mu, np.nan)
        v = mu - float(param) * sigma
    elif mode == "ipm":
        v = -float(param) * mu
    else:
        raise ValueError(f"unknown colluding attack {mode!r}")
    out[lie] = v
    return out
