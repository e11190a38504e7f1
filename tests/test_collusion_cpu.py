"""ALIE and inner-product-manipulation attacks on CPU: ALIE's default z, the fp64 oracle, configuration checks and flags, the
library-op PS (nccl / gloo transports) against the oracle, the vote's immunity, training under attack and a multi-process job."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from draco_b200 import JobConfig
from draco_b200 import _native as N
from draco_b200.codes.adversary import ATTACK_ALIE, ATTACK_IPM, alie_z_max, attack_code, collude
from draco_b200.config import add_fit_args, config_from_args
from draco_b200.parallel.trainer import Trainer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ codes and the oracle
@pytest.mark.parametrize("P,f,z", [(5, 1, 0.2533), (7, 1, 0.1800), (7, 2, 0.5659), (7, 3, 1.0676), (16, 6, 0.8871)])
def test_alie_default_z(P, f, z):
    assert round(alie_z_max(P, f), 4) == z


def test_alie_default_z_is_undefined_when_the_liars_are_a_majority():
    with pytest.raises(ValueError, match="undefined"):
        alie_z_max(7, 4)


def test_attack_codes():
    assert attack_code("alie") == ATTACK_ALIE == 5 and attack_code("ipm") == ATTACK_IPM == 6


@pytest.mark.parametrize("mode,param", [("alie", 0.5659), ("alie", -2.0), ("ipm", 0.1), ("ipm", 4.0)])
@pytest.mark.parametrize("P", [3, 7, 16, 32])
def test_collude_matches_numpy(mode, param, P):
    rng = np.random.default_rng(P)
    X = (rng.standard_normal((P, 300)) + 0.3).astype(np.float32)
    for nl in (1, (P - 1) // 2, P - 2):
        liars = sorted(rng.choice(P, size=max(nl, 1), replace=False).tolist())
        honest = [r for r in range(P) if r not in liars]
        out = collude(X, liars, mode, param)
        assert out.dtype == np.float64 and out.shape == X.shape
        H = X[honest].astype(np.float64)
        want = H.mean(axis=0) - param * H.std(axis=0, ddof=1) if mode == "alie" else -param * H.mean(axis=0)
        assert np.array_equal(out[honest], X[honest].astype(np.float64))
        for r in liars:
            assert np.array_equal(out[r], out[liars[0]])
        assert np.allclose(out[liars[0]], want, rtol=1e-12, atol=1e-14)


def test_collude_without_liars_or_without_honest_rows_changes_nothing():
    X = np.arange(12, dtype=np.float32).reshape(3, 4)
    assert np.array_equal(collude(X, [], "alie", 1.0), X)
    assert np.array_equal(collude(X, [0, 1, 2], "ipm", 1.0), X)


def test_collude_propagates_non_finite_honest_values():
    X = np.ones((5, 4))
    X[1, 0], X[2, 1] = np.nan, np.inf
    out = collude(X, [4], "alie", 1.0)
    assert np.isnan(out[4, 0]) and np.isnan(out[4, 1]) and np.isfinite(out[4, 2:]).all()
    assert np.isinf(collude(X, [4], "ipm", 1.0)[4, 1])


# ------------------------------------------------------------------------------------------------ configuration
def _resolve(err_mode, P=7, f=2, **kw):
    base = dict(approach="baseline", mode="normal", num_workers=P, worker_fail=f, err_mode=err_mode)
    base.update(kw)
    return JobConfig(**base).resolve(P + 1)


@pytest.mark.parametrize("err_mode", ["alie", "ipm"])
def test_resolve_rejects_the_cyclic_code(err_mode):
    with pytest.raises(ValueError, match="cyclic"):
        _resolve(err_mode, approach="cyclic", f=1)
    _resolve(err_mode, approach="maj_vote", mode="maj_vote", group_size=3, f=1)


def test_resolve_bounds_on_honest_workers():
    _resolve("alie", P=3, f=1, alie_z=1.0)
    with pytest.raises(ValueError, match="2 honest"):
        _resolve("alie", P=3, f=2, alie_z=1.0)
    _resolve("ipm", P=3, f=2)
    with pytest.raises(ValueError, match="1 honest"):
        _resolve("ipm", P=3, f=3)


def test_resolve_needs_alie_z_when_the_default_is_undefined():
    assert abs(_resolve("alie", P=7, f=3).attack_param - 1.0676) < 1e-4          # s = 1: the last defined default
    with pytest.raises(ValueError, match="undefined"):
        _resolve("alie", P=7, f=4)
    assert _resolve("alie", P=7, f=4, alie_z=0.5).attack_param == 0.5


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), float("-inf")])
def test_resolve_rejects_non_finite_parameters(bad):
    with pytest.raises(ValueError, match="alie-z"):
        _resolve("alie", alie_z=bad)
    with pytest.raises(ValueError, match="ipm-epsilon"):
        _resolve("ipm", ipm_epsilon=bad)


def test_flags_parse():
    import argparse
    d = config_from_args(add_fit_args(argparse.ArgumentParser()).parse_args([]))
    assert d.alie_z is None and d.ipm_epsilon == 0.1
    a = add_fit_args(argparse.ArgumentParser()).parse_args(["--err-mode", "alie", "--alie-z", "1.5", "--ipm-epsilon", "0.3"])
    cfg = config_from_args(a)
    assert (cfg.err_mode, cfg.alie_z, cfg.ipm_epsilon) == ("alie", 1.5, 0.3)
    assert _resolve("ipm", ipm_epsilon=0.3).attack_param == 0.3


def test_collusion_args_abi_matches_ctypes():
    lib = N.cuda()            # loads without a GPU
    assert lib.drc_sizeof_CollusionArgs() == C.sizeof(N.CollusionArgs)


# ------------------------------------------------------------------------------------------------ library-op engine
def _cfg(**kw):
    base = dict(network="LeNet", dataset="MNIST", batch_size=16, max_steps=12, num_workers=7, worker_fail=2, transport="gloo",
                lr=0.05, momentum=0.9, synthetic_size=512, eval_freq=10 ** 6, compress_grad="None", approach="baseline")
    base.update(kw)
    return JobConfig(**base)


@pytest.mark.parametrize("err_mode", ["alie", "ipm"])
def test_library_op_engine_liar_slots_equal_the_oracle(err_mode):
    t = Trainer(_cfg(mode="coord_median", err_mode=err_mode), rank=0, world=1, device=torch.device("cpu"), quiet=True)
    eng = t.engine
    seen = []
    orig = eng._collude

    def spy(step):
        before = eng.slots.clone()
        orig(step)
        seen.append((step, before, eng.slots.clone()))
    eng._collude = spy
    for _ in range(3):
        t.train_step()
    assert len(seen) == 3
    valid = eng.layout.valid_mask()
    param = eng.cfg.attack_param
    for step, before, after in seen:
        liars = [w - 1 for w in range(1, 8) if eng.schedule.is_adversary(w, step)]
        assert len(liars) == 2
        want = collude(before.numpy(), liars, err_mode, param)
        honest = [r for r in range(7) if r not in liars]
        assert torch.equal(after[honest], before[honest])
        assert all(torch.equal(after[r], after[liars[0]]) for r in liars)
        assert float(after[:, ~valid].abs().sum()) == 0
        assert np.allclose(after[liars[0]].double().numpy()[valid], want[liars[0]][valid], rtol=1e-6, atol=1e-10), step


@pytest.mark.parametrize("err_mode", ["alie", "ipm"])
def test_vote_is_immune_to_collusion(err_mode):
    """Group size 3 on 7 workers, one liar per step: every group's honest replicas still agree, so the parameters are exactly
    those of the clean run."""
    kw = dict(approach="maj_vote", mode="maj_vote", group_size=3, worker_fail=1)
    runs = []
    for em in ("none", err_mode):
        t = Trainer(_cfg(err_mode=em, **kw), rank=0, world=1, device=torch.device("cpu"), quiet=True)
        for _ in range(4):
            t.train_step()
        runs.append(t.engine.master_params().clone())
    assert torch.equal(runs[0], runs[1])


@pytest.mark.parametrize("err_mode", ["alie", "ipm"])
@pytest.mark.parametrize("mode", ["normal", "geometric_median", "krum", "coord_median", "trimmed_mean", "multi_krum"])
def test_baseline_rules_train_under_collusion(mode, err_mode):
    t = Trainer(_cfg(mode=mode, err_mode=err_mode), rank=0, world=1, device=torch.device("cpu"), quiet=True)
    losses = [t.train_step()["loss"] for _ in range(8)]
    assert all(np.isfinite(losses)), losses
    assert torch.isfinite(t.engine.master_params()).all()


def test_alie_as_a_multi_process_job(tmp_path):
    """1 PS + 5 workers packed onto 2 Gloo processes, 3 steps."""
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), OMP_NUM_THREADS="2")
    r = subprocess.run([sys.executable, "-m", "draco_b200.cli.distributed_nn", "--launch", "2", "--master-port", "29770", "--no-cuda",
                        "--network", "LeNet", "--dataset", "MNIST", "--num-workers", "5", "--batch-size", "8", "--max-steps", "3",
                        "--eval-freq", "1000", "--train-dir", str(tmp_path) + "/", "--synthetic-size", "128", "--log-interval", "1",
                        "--compress-grad", "None", "--approach", "baseline", "--mode", "coord_median", "--worker-fail", "2",
                        "--err-mode", "alie"],
                       capture_output=True, text=True, timeout=420, env=env, cwd=ROOT)
    out = r.stdout + r.stderr
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert out.count("done at step 3") == 2, out[-2500:]
