"""Coordinate-wise median / trimmed mean (aggregate_update MODE 3) and multi-Krum on the B200: kernels against the fp64
oracles, the fused engine against the library-op engine, and bit-identity across PS pipelining, graph replay, the wire codec
and process boundaries."""
import hashlib
import json
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
from draco_b200.parallel.ps import hyperparams_tensor
from draco_b200.parallel.trainer import Trainer

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def K():
    from draco_b200.ops import kernels
    return kernels


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


def _layout():
    """LeNet layout: 8 tensors, several of them not a multiple of the tile (padding inside the last tile)."""
    return ArenaLayout.from_model(build_model("LeNet"), bf16=True, channels_last=True)


def _slots(L, P, seed, scale=0.1):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(P, L.total, generator=g) * scale
    x[:, ~torch.from_numpy(L.valid_mask())] = 0
    return x


def _ctrl(dev):
    return torch.ones(1, dtype=torch.int64, device=dev), torch.zeros(4, dtype=torch.int32, device=dev)


NEG_NAN = torch.tensor([-1 << 22], dtype=torch.int32).view(torch.float32).item()     # 0xffc00000: NaN with the sign bit set
LIES = [float("inf"), float("-inf"), float("nan"), 1e30, -1e30, NEG_NAN]


def _with_liars(L, P, b, seed):
    """P slots, b of them (random rows) liars whose every element -- padding included -- is +-Inf, NaN of either sign or +-1e30."""
    x = _slots(L, P, seed)
    rng = np.random.default_rng(seed)
    for j, r in enumerate(rng.choice(P, size=b, replace=False)):
        pick = torch.from_numpy(rng.integers(0, len(LIES), size=L.total))
        x[r] = torch.tensor(LIES)[pick] if j % 2 else LIES[(seed + j) % len(LIES)]
    return x


def _coordinate_update(K, dev, L, slots, trim, tile_ranges=None):
    """MODE 3 + SGD with lr = 1, momentum 0 on zero parameters: returns (grad_out, params) after one step."""
    P = slots.shape[0]
    hp = hyperparams_tensor(JobConfig(lr=1.0, momentum=0.0), dev)
    params = torch.zeros(L.total, device=dev)
    mom = torch.zeros(L.total, device=dev)
    gout = torch.zeros(L.total, device=dev)
    step, cnt = _ctrl(dev)
    for tr in tile_ranges or [None]:
        K.aggregate_update(L, slots, L.total, params=params, momentum=mom, hp=hp, step_ptr=step, done_counter=cnt[0:1], K=P,
                           scale=1.0 / (P - 2 * trim), trim=trim, grad_out=gout, tile_range=tr)
    torch.cuda.synchronize()
    return gout, params


# ------------------------------------------------------------------------------------------------ MODE 3 kernel
@pytest.mark.parametrize("P", [4, 7, 8, 13, 16])
def test_coordinate_kernel_matches_oracles(K, dev, P):
    L = _layout()
    valid = torch.from_numpy(L.valid_mask())
    for b in range((P - 1) // 2 + 1):
        slots = _with_liars(L, P, b, seed=100 * P + b)
        gout, params = _coordinate_update(K, dev, L, slots.to(dev), b)
        gout, params = gout.cpu(), params.cpu()
        sl = slots.double().numpy()
        want = np.zeros(L.total)
        for spec in L.specs:
            X = sl[:, spec.offset: spec.offset + spec.numel]
            want[spec.offset: spec.offset + spec.numel] = oracle.trimmed_mean(X, b)
        assert np.isfinite(want[valid.numpy()]).all()
        if P % 2 == 1 and b == (P - 1) // 2:                         # odd-P median: one kept value, scale 1 -> exact
            assert torch.equal(gout[valid], torch.from_numpy(want).float()[valid]), (P, b)
        else:
            err = np.abs(gout.double().numpy() - want)[valid.numpy()]
            assert np.all(err <= 1e-5 * np.abs(want[valid.numpy()]) + 1e-7), (P, b, err.max())
        assert torch.equal(params, -gout), (P, b)                   # lr = 1, momentum 0: the parameters are -g
        assert float(params[~valid].abs().sum()) == 0 and float(gout[~valid].abs().sum()) == 0, (P, b)


def test_coordinate_kernel_median_is_np_median_for_even_p(K, dev):
    L = _layout()
    slots = _slots(L, 8, seed=5)
    gout, _ = _coordinate_update(K, dev, L, slots.to(dev), 3)
    valid = torch.from_numpy(L.valid_mask())
    want = np.median(slots.double().numpy(), axis=0)
    assert np.allclose(gout.cpu().double().numpy()[valid.numpy()], want[valid.numpy()], rtol=1e-6, atol=1e-8)


def test_coordinate_kernel_buckets_equal_one_launch(K, dev):
    L = _layout()
    slots = _with_liars(L, 7, 2, seed=17).to(dev)
    n = L.ntiles
    whole = _coordinate_update(K, dev, L, slots, 2)
    bucketed = _coordinate_update(K, dev, L, slots, 2, tile_ranges=[(0, n // 3), (n // 3, 2 * n // 3), (2 * n // 3, n)])
    assert torch.equal(whole[0], bucketed[0]) and torch.equal(whole[1], bucketed[1])


def test_coordinate_kernel_rejects_more_than_16_slots(K, dev):
    L = _layout()
    with pytest.raises(RuntimeError, match="aggregate_update"):
        _coordinate_update(K, dev, L, _slots(L, 17, seed=1).to(dev), 8)


# ------------------------------------------------------------------------------------------------ multi-Krum selection
@pytest.mark.parametrize("P,s", [(7, 2), (9, 3), (16, 6)])
def test_multi_krum_selection_matches_oracle(K, dev, P, s):
    L = _layout()
    T = L.ntensors
    slots = _slots(L, 1, seed=6)[0][None] + 0.01 * _slots(L, P, seed=7, scale=1.0)
    slots[1] = -100 * slots[1]
    slots[P - 2] = _slots(L, 1, seed=8, scale=30.0)[0]
    slots = slots.to(dev)
    pair = torch.zeros(T, P * (P - 1) // 2, dtype=torch.float64, device=dev)
    sl = slots.cpu().double().numpy()
    # m = 1 with the [T] table the Krum path has always used: the Krum winner
    sel1 = torch.zeros(T, dtype=torch.int32, device=dev)
    K.krum_select(L, slots, L.total, P, s, pair, sel1)
    torch.cuda.synchronize()
    for t, spec in enumerate(L.specs):
        assert int(sel1[t]) == oracle.krum_index(sl[:, spec.offset:spec.offset + spec.numel], s), t
    m = P - s
    sel = torch.full((m, T), -1, dtype=torch.int32, device=dev)
    K.krum_select(L, slots, L.total, P, s, pair, sel, m=m)
    torch.cuda.synchronize()
    assert float(pair.abs().sum()) == 0
    want = np.zeros(L.total)
    for t, spec in enumerate(L.specs):
        X = sl[:, spec.offset:spec.offset + spec.numel]
        idx = oracle.multi_krum_indices(X, s, m)
        assert sel[:, t].tolist() == idx, (t, sel[:, t].tolist(), idx)
        want[spec.offset:spec.offset + spec.numel] = X[idx].mean(axis=0)
    # the aggregate: MODE 0 select-sum over the m rows, scale 1/m
    hp = hyperparams_tensor(JobConfig(lr=1.0, momentum=0.0), dev)
    params, mom, gout = (torch.zeros(L.total, device=dev) for _ in range(3))
    step, cnt = _ctrl(dev)
    K.aggregate_update(L, slots, L.total, params=params, momentum=mom, hp=hp, step_ptr=step, done_counter=cnt[0:1], K=m,
                       scale=1.0 / m, select=sel, grad_out=gout)
    torch.cuda.synchronize()
    assert np.allclose(gout.cpu().double().numpy(), want, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------ engines
def _cfg(**kw):
    base = dict(network="LeNet", dataset="MNIST", batch_size=16, max_steps=12, num_workers=7, transport="nvl", lr=0.02,
                momentum=0.9, synthetic_size=512, eval_freq=10 ** 6, compress_grad="None", dtype="fp32", cuda_graphs=False,
                approach="baseline")
    base.update(kw)
    return JobConfig(**base)


def _run(cfg, steps):
    t = Trainer(cfg, rank=0, world=1, device=torch.device("cuda", 0), quiet=True)
    losses = [t.train_step()["loss"] for _ in range(steps)]
    t.synchronize()
    return t, losses


_MODES = [dict(mode="coord_median", worker_fail=3, err_mode="rev_grad"),
          dict(mode="trimmed_mean", worker_fail=2, err_mode="constant"),
          dict(mode="multi_krum", worker_fail=2, err_mode="constant")]


@pytest.mark.parametrize("kw", _MODES, ids=[k["mode"] for k in _MODES])
@pytest.mark.parametrize("opt", [dict(), dict(optimizer="adam", lr=1e-3)], ids=["sgd", "adam"])
def test_fused_matches_library_op_engine(kw, opt):
    # Adam: ONE step.  Its update lr * m / sqrt(v) is scale-free, so later steps turn 1-ulp differences of the two transports'
    # trajectories into lr-sized moves wherever an aggregate is tiny -- and a median's aggregate IS one input value, often the
    # one nearest zero.  SGD is compared after 4 steps.
    steps = 1 if opt else 4
    a, _ = _run(_cfg(**kw, **opt), steps)
    b, _ = _run(_cfg(transport="nccl", **kw, **opt), steps)
    assert a.engine.ps.rule == kw["mode"] and b.engine.ps.rule == kw["mode"]
    pa, pb = a.engine.master_params(), b.engine.master_params()
    assert torch.isfinite(pa).all()
    assert torch.allclose(pa, pb, atol=2e-5), (kw, opt, float((pa - pb).abs().max()))


_RESNET = dict(network="ResNet18", dataset="Cifar10", batch_size=8, num_workers=5, worker_fail=2, err_mode="rev_grad",
               dtype="bf16", synthetic_size=256)


@pytest.mark.parametrize("mode", ["coord_median", "trimmed_mean"])
def test_coordinate_rules_are_bit_identical_across_pipelining_graphs_and_codec(mode):
    piped, lp = _run(_cfg(mode=mode, cuda_graphs=True, **_RESNET), 6)
    serial, ls = _run(_cfg(mode=mode, cuda_graphs=True, pipeline_ps=False, **_RESNET), 6)
    eager, le = _run(_cfg(mode=mode, cuda_graphs=False, **_RESNET), 6)
    assert piped.engine.pipeline_ps and not serial.engine.pipeline_ps and piped.engine.graph is not None
    ref = piped.engine.master_params()
    assert torch.isfinite(ref).all()
    assert torch.equal(ref, serial.engine.master_params()) and lp == ls
    assert torch.equal(ref, eager.engine.master_params()) and lp == le
    kw = dict(mode=mode, worker_fail=2, err_mode="rev_grad")
    packed, lc = _run(_cfg(compress_grad="compress", **kw), 4)
    raw, lr = _run(_cfg(compress_grad="None", **kw), 4)
    assert packed.engine.compress and torch.equal(packed.engine.master_params(), raw.engine.master_params()) and lc == lr


def _torchrun(nproc, env_extra, port, timeout=900):
    env = dict(os.environ, PYTHONPATH=ROOT, **env_extra)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mp_equiv.py")],
                         capture_output=True, text=True, timeout=timeout, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


_MEDIAN_JOB = dict(approach="baseline", mode="coord_median", worker_fail=3, err_mode="rev_grad")


@pytest.mark.timeout(900)
def test_coord_median_across_two_processes_on_one_gpu():
    rec = _torchrun(2, {"DRACO_BOOTSTRAP": "gloo", "CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0],
                        "MP_EQUIV_CFG": json.dumps(dict(_MEDIAN_JOB, multicast="off", cuda_graphs=False)), "MP_EQUIV_STEPS": "4"},
                    port=29766)
    assert rec["gpus"] == 1 and rec["world"] == 2
    assert rec["sha"][0] == rec["sha"][1]
    single, _ = _run(_cfg(**_MEDIAN_JOB, network="ResNet18", dataset="Cifar10", batch_size=8, dtype="bf16", synthetic_size=256), 4)
    assert hashlib.sha256(single.engine.master_params().cpu().numpy().tobytes()).hexdigest() == rec["sha"][0]


@pytest.mark.multigpu
@pytest.mark.timeout(1200)
def test_multigpu_coord_median_nvl_equals_nccl(tmp_path):
    """Same seeds through the fused peer-memory transport and through NCCL + the library-op PS.  The median itself is exact on
    both (P = 7: one kept value), but the SGD update is not: the fused kernel applies it with fmaf in registers, the library PS
    with separate torch ops, so after the first step the parameters -- and with them the next steps' gradients -- differ in the
    last bits.  Hence fp32 round-off agreement, like test_fused_engine_gpu.py's nvl-vs-nccl case, not bit equality."""
    nproc = min(8, torch.cuda.device_count())
    outs = []
    for j, tr in enumerate(("nvl", "nccl")):
        f = str(tmp_path / f"p_{tr}.pt")
        _torchrun(nproc, {"MP_EQUIV_CFG": json.dumps(dict(_MEDIAN_JOB, transport=tr, cuda_graphs=(tr == "nvl"))), "MP_EQUIV_OUT": f,
                          "MP_EQUIV_STEPS": "4"}, port=29767 + j)
        outs.append(torch.load(f)["params"])
    assert torch.allclose(outs[0], outs[1], atol=5e-5), float((outs[0] - outs[1]).abs().max())
