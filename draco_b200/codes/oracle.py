"""fp64 numpy oracles for every PS-side aggregation rule.

They define the semantics the CUDA kernels (csrc/cuda/*.cu) and the C++ host twins
(csrc/host/*.cpp) are tested against, tensor by tensor -- the reference applies every rule
*per parameter tensor*, never on the concatenated model (src/master/rep_master.py:154-168,
src/master/baseline_master.py:271-296).
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np


def boyer_moore_winner(members: Sequence[np.ndarray]) -> int:
    """Index of the Boyer-Moore candidate using whole-tensor equality (``np.array_equal``).

    Mirrors the reference's streaming vote (rep_master.py:157-165) including its behaviour when no
    strict majority exists (the last surviving candidate wins).
    """
    cand, count = 0, 0
    for i, m in enumerate(members):
        if count == 0:
            cand, count = i, 1
        elif np.array_equal(m, members[cand]):
            count += 1
        else:
            count -= 1
    return cand


def majority_vote(slots: np.ndarray, groups: Sequence[Sequence[int]]) -> Tuple[np.ndarray, List[int]]:
    """``slots``: [P, d] one tensor from every worker (row w-1 = worker w).  Returns (mean of group
    winners, winner member index per group)."""
    acc = np.zeros(slots.shape[1], dtype=np.float64)
    winners = []
    for g in groups:
        members = [slots[w - 1] for w in g]
        k = boyer_moore_winner(members)
        winners.append(k)
        acc += members[k]
    return acc / float(len(groups)), winners


def mean(slots: np.ndarray) -> np.ndarray:
    return np.asarray(slots, dtype=np.float64).mean(axis=0)


def geometric_median(slots: np.ndarray, eps: float = 1e-8, max_iter: int = 200) -> np.ndarray:
    """Weiszfeld iteration started at the mean (what hdmedians.geomedian does; baseline_master.py:274)."""
    X = np.asarray(slots, dtype=np.float64)
    m = X.mean(axis=0)
    for _ in range(max_iter):
        d = np.linalg.norm(X - m, axis=1)
        nz = d > 1e-300
        if not nz.any():
            return m
        w = np.zeros_like(d)
        w[nz] = 1.0 / d[nz]
        m_new = (w[:, None] * X).sum(axis=0) / w.sum()
        if np.linalg.norm(m_new - m) <= eps * max(1.0, np.linalg.norm(m)):
            return m_new
        m = m_new
    return m


def geometric_median_weights(slots: np.ndarray, eps: float = 1e-10, max_iter: int = 256) -> np.ndarray:
    """The same Weiszfeld iteration carried out on the convex weights only (host model of ``geomed_weights_kernel``,
    csrc/cuda/robust.cu).  Every iterate is ``m = w @ X`` with ``sum(w) = 1``, for which
    ``||x_i - m||^2 = (D w)_i - w^T D w / 2`` with ``D_ij = ||x_i - x_j||^2`` -- the data is touched once (for D)."""
    X = np.asarray(slots, dtype=np.float64)
    P = X.shape[0]
    D = ((X[:, None, :] - X[None, :, :]) ** 2).sum(axis=2)
    w = np.full(P, 1.0 / P)
    if D.max() <= 0:
        return w
    floor_d = 1e-12 * np.sqrt(D.max()) + 1e-300
    for _ in range(max_iter):
        s = D @ w
        d = np.maximum(np.sqrt(np.maximum(s - 0.5 * (w @ s), 0.0)), floor_d)
        wn = (1.0 / d) / (1.0 / d).sum()
        delta = np.abs(wn - w).max()
        w = wn
        if delta <= eps:
            break
    return w


def krum_index(slots: np.ndarray, s: int) -> int:
    """Krum (arXiv:1703.02757) as the reference implements it (baseline_master.py:278-296):
    score_i = sum of the (P - s - 2) smallest squared distances to the others; argmin wins."""
    X = np.asarray(slots, dtype=np.float64)
    P = X.shape[0]
    keep = max(P - s - 2, 0)
    d2 = ((X[:, None, :] - X[None, :, :]) ** 2).sum(axis=2)
    scores = []
    for i in range(P):
        others = np.sort(np.delete(d2[i], i))
        scores.append(others[:keep].sum())
    return int(np.argmin(scores))


def krum(slots: np.ndarray, s: int) -> np.ndarray:
    return np.asarray(slots, dtype=np.float64)[krum_index(slots, s)]


def multi_krum_indices(slots: np.ndarray, s: int, m: int) -> List[int]:
    """Multi-Krum (Blanchard et al., NeurIPS 2017): the m rows with the lowest Krum scores (ties to the lower slot), in
    ascending slot order.  The aggregate is their mean; m = 1 is Krum.  Defined for finite inputs."""
    X = np.asarray(slots, dtype=np.float64)
    P = X.shape[0]
    keep = max(P - s - 2, 0)
    d2 = ((X[:, None, :] - X[None, :, :]) ** 2).sum(axis=2)
    scores = np.array([np.sort(np.delete(d2[i], i))[:keep].sum() for i in range(P)])
    return sorted(int(i) for i in np.argsort(scores, kind="stable")[:m])


def trimmed_mean(slots: np.ndarray, b: int) -> np.ndarray:
    """Coordinate-wise trimmed mean (Yin et al., ICML 2018): sort every coordinate's P values with ``np.sort`` (NaN of either
    sign after +Inf), drop the b lowest and the b highest, average the rest.  Up to b non-finite values per coordinate are
    trimmed away."""
    X = np.sort(np.asarray(slots, dtype=np.float64), axis=0)
    P = X.shape[0]
    assert 0 <= 2 * b < P
    return X[b: P - b].sum(axis=0) / (P - 2 * b)


def coordinate_median(slots: np.ndarray) -> np.ndarray:
    """Coordinate-wise median: the trimmed mean that keeps the middle value (odd P) or averages the middle two (even P) --
    ``np.median`` on finite inputs."""
    return trimmed_mean(slots, (np.asarray(slots).shape[0] - 1) // 2)


def sgd_momentum_step(p: np.ndarray, buf: np.ndarray, g: np.ndarray, lr: float, momentum: float,
                      weight_decay: float = 0.0, dampening: float = 0.0, nesterov: bool = False,
                      first_step: bool = False) -> Tuple[np.ndarray, np.ndarray]:
    """One SGD step with torch.optim.SGD semantics (reference: src/optim/sgd_modified.py:53-88)."""
    d_p = g + weight_decay * p if weight_decay != 0 else g
    if momentum != 0:
        buf = d_p.copy() if first_step else momentum * buf + (1.0 - dampening) * d_p
        d_p = d_p + momentum * buf if nesterov else buf
    return p - lr * d_p, buf
