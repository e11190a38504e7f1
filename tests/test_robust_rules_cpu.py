"""Coordinate-wise median, trimmed mean and multi-Krum on CPU: the fp64 oracles, configuration checks, the library-op PS
(used by the nccl and gloo transports) against the oracles, training under attack, and multi-process CLI jobs."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from draco_b200 import JobConfig
from draco_b200.codes import oracle
from draco_b200.models import build_model
from draco_b200.parallel.arena import ArenaLayout
from draco_b200.parallel.ps import TorchPS, select_rule
from draco_b200.parallel.trainer import Trainer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_MODES = ("coord_median", "trimmed_mean", "multi_krum")


# ------------------------------------------------------------------------------------------------ oracles
@pytest.mark.parametrize("P", [4, 5, 7, 8, 13, 16])
def test_coordinate_median_is_np_median_on_finite_data(P):
    X = np.random.default_rng(P).standard_normal((P, 257))
    assert np.array_equal(oracle.coordinate_median(X), np.median(X, axis=0))


def test_trimmed_mean_with_no_trim_is_the_mean():
    X = np.random.default_rng(1).standard_normal((7, 300))
    assert np.allclose(oracle.trimmed_mean(X, 0), X.mean(axis=0), rtol=0, atol=1e-14)


@pytest.mark.parametrize("P", [5, 7, 8, 13])
def test_up_to_b_non_finite_rows_are_trimmed(P):
    rng = np.random.default_rng(P)
    b = (P - 1) // 2
    H = rng.standard_normal((P, 64))
    bad = [np.nan, -np.nan, np.inf, -np.inf, 1e300]
    for nb in range(b + 1):
        X = H.copy()
        for r in range(nb):
            X[r] = bad[r % len(bad)]
        honest = H[nb:]
        for trim in range(nb, b + 1):
            got = oracle.trimmed_mean(X, trim)
            assert np.isfinite(got).all(), (nb, trim)
            assert (got >= honest.min(axis=0) - 1e-12).all() and (got <= honest.max(axis=0) + 1e-12).all(), (nb, trim)
        med = oracle.coordinate_median(X)
        assert np.isfinite(med).all() and (med >= honest.min(axis=0)).all() and (med <= honest.max(axis=0)).all()
    # liars that all sort to the top (NaN or +Inf) leave exactly the honest values s_{b+1} .. s_{P-b}
    X = H.copy()
    X[:b] = np.where(np.arange(64) % 2 == 0, np.nan, np.inf)
    hs = np.sort(H[b:], axis=0)
    assert np.allclose(oracle.trimmed_mean(X, b), hs[b: P - b].mean(axis=0), rtol=0, atol=1e-14)


def test_multi_krum_with_one_row_is_krum():
    rng = np.random.default_rng(3)
    for P, s in ((7, 2), (5, 1), (9, 3), (16, 6)):
        X = rng.standard_normal((P, 40))
        X[0] *= -100
        assert oracle.multi_krum_indices(X, s, 1) == [oracle.krum_index(X, s)]
        got = oracle.multi_krum_indices(X, s, P - s)
        assert got == sorted(got) and len(got) == P - s and 0 not in got


def test_multi_krum_ties_go_to_the_lower_slot():
    X = np.zeros((7, 4))                     # every score ties
    assert oracle.multi_krum_indices(X, 2, 5) == [0, 1, 2, 3, 4]


# ------------------------------------------------------------------------------------------------ configuration
def _resolve(mode, P, f, transport="nvl"):
    return JobConfig(approach="baseline", mode=mode, num_workers=P, worker_fail=f, transport=transport).resolve(P + 1)


def test_new_modes_resolve_to_their_own_rules():
    for mode, f in (("coord_median", 3), ("trimmed_mean", 3), ("multi_krum", 2)):
        assert select_rule(JobConfig(approach="baseline", mode=mode, num_workers=7, worker_fail=f).resolve(8)) == mode
    # unknown strings keep the fallback to the mean
    assert select_rule(JobConfig(approach="baseline", mode="no_such_rule", num_workers=7).resolve(8)) == "mean"


@pytest.mark.parametrize("mode,P_ok,P_bad,f", [("coord_median", 7, 6, 3), ("trimmed_mean", 5, 4, 2), ("multi_krum", 7, 6, 2)])
def test_config_enforces_the_worker_bounds(mode, P_ok, P_bad, f):
    _resolve(mode, P_ok, f)
    with pytest.raises(ValueError):
        _resolve(mode, P_bad, f)
    with pytest.raises(ValueError):
        _resolve(mode, P_bad, f, transport="nccl")
    # nvl: at most 16 workers (register budget of the kernels); the library-op transports have no such limit
    _resolve(mode, 16, 1)
    with pytest.raises(ValueError, match="at most 16"):
        _resolve(mode, 17, 1)
    _resolve(mode, 17, 1, transport="nccl")
    _resolve(mode, 17, 1, transport="gloo")


# ------------------------------------------------------------------------------------------------ library-op PS
def _lenet_slots(P, liars, seed):
    L = ArenaLayout.from_model(build_model("LeNet"), bf16=False, channels_last=True)
    g = torch.Generator().manual_seed(seed)
    honest = torch.randn(L.total, generator=g) * 0.1
    slots = honest[None] + 0.01 * torch.randn(P, L.total, generator=g)
    for r, v in liars.items():
        slots[r] = v if not isinstance(v, str) else -100.0 * slots[r]
    return L, slots


@pytest.mark.parametrize("mode,P,f", [("coord_median", 7, 3), ("coord_median", 8, 3), ("trimmed_mean", 7, 2),
                                      ("trimmed_mean", 13, 4), ("multi_krum", 7, 2), ("multi_krum", 9, 3)])
def test_torch_ps_matches_the_oracles(mode, P, f):
    if mode == "multi_krum":
        liars = {1: "flip", P - 1: 30.0, 3: "flip"}
    else:
        liars = {0: float("nan"), 2: float("inf"), 4: float("-inf"), 5: 1e30, 6: -1e30}
    liars = dict(list(liars.items())[:f])
    L, slots = _lenet_slots(P, liars, seed=P + f)
    cfg = JobConfig(approach="baseline", mode=mode, num_workers=P, worker_fail=f, transport="gloo").resolve(P + 1)
    ps = TorchPS(cfg, L, torch.device("cpu"), L.new_arena(torch.device("cpu")), None, None)
    out = ps.aggregate(slots)
    sl = slots.double().numpy()
    for spec, g in zip(L.specs, out):
        X = sl[:, spec.offset: spec.offset + spec.numel]
        if mode == "coord_median":
            want = oracle.coordinate_median(X)
        elif mode == "trimmed_mean":
            want = oracle.trimmed_mean(X, f)
        else:
            want = X[oracle.multi_krum_indices(X, f, P - f)].mean(axis=0)
        assert np.isfinite(g.numpy()).all()
        assert np.allclose(g.double().numpy(), want, rtol=1e-5, atol=1e-7), (spec.name, np.abs(g.numpy() - want).max())


def test_torch_ps_krum_is_unchanged_by_the_shared_score_code():
    P, f = 7, 2
    L, slots = _lenet_slots(P, {2: "flip", 5: 30.0}, seed=11)
    cfg = JobConfig(approach="baseline", mode="krum", num_workers=P, worker_fail=f, transport="gloo").resolve(P + 1)
    ps = TorchPS(cfg, L, torch.device("cpu"), L.new_arena(torch.device("cpu")), None, None)
    sl = slots.double().numpy()
    for spec, g in zip(L.specs, ps.aggregate(slots)):
        X = sl[:, spec.offset: spec.offset + spec.numel]
        assert torch.equal(g, slots[oracle.krum_index(X, f), spec.offset: spec.offset + spec.numel])


# ------------------------------------------------------------------------------------------------ training under attack
@pytest.mark.parametrize("mode,f", [("coord_median", 3), ("trimmed_mean", 3), ("multi_krum", 2)])
def test_new_modes_train_under_attack(mode, f):
    cfg = JobConfig(network="LeNet", dataset="MNIST", batch_size=16, max_steps=8, num_workers=7, transport="gloo", lr=0.05,
                    momentum=0.9, synthetic_size=512, eval_freq=10 ** 6, compress_grad="None", approach="baseline", mode=mode,
                    worker_fail=f, err_mode="rev_grad")
    t = Trainer(cfg, rank=0, world=1, device=torch.device("cpu"), quiet=True)
    assert t.engine.ps.rule == mode
    losses = [t.train_step()["loss"] for _ in range(12)]
    assert losses[-1] < losses[0], losses
    assert torch.isfinite(t.engine.master_params()).all()


# ------------------------------------------------------------------------------------------------ multi-process CLI jobs
@pytest.mark.parametrize("name,flags", [
    ("coord_median", ["--mode", "coord_median", "--worker-fail", "2", "--err-mode", "rev_grad"]),
    ("trimmed_mean", ["--mode", "trimmed_mean", "--worker-fail", "1", "--err-mode", "constant"]),
    ("multi_krum", ["--mode", "multi_krum", "--worker-fail", "1", "--err-mode", "random"]),
])
def test_new_modes_as_multi_process_jobs(tmp_path, name, flags):
    """1 PS + 5 workers packed onto 2 Gloo processes, 3 steps."""
    port = 29760 + list(NEW_MODES).index(name)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), OMP_NUM_THREADS="2")
    r = subprocess.run([sys.executable, "-m", "draco_b200.cli.distributed_nn", "--launch", "2", "--master-port", str(port), "--no-cuda",
                        "--network", "LeNet", "--dataset", "MNIST", "--num-workers", "5", "--batch-size", "8", "--max-steps", "3",
                        "--eval-freq", "1000", "--train-dir", str(tmp_path) + "/", "--synthetic-size", "128", "--log-interval", "1",
                        "--compress-grad", "None", "--approach", "baseline", *flags],
                       capture_output=True, text=True, timeout=420, env=env, cwd=ROOT)
    out = r.stdout + r.stderr
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert out.count("done at step 3") == 2, out[-2500:]
