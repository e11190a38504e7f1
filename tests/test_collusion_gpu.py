"""ALIE and inner-product manipulation on the B200: the collusion kernel against the fp64 oracle (buckets, graph replay), the fused
engine against the library-op engine, bit-identity across PS pipelining, graph replay, the wire codec and process boundaries,
the vote's immunity and the transport self-check."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from draco_b200 import JobConfig
from draco_b200.codes.adversary import ATTACK_ALIE, ATTACK_IPM, collude
from draco_b200.models import build_model
from draco_b200.parallel.arena import ArenaLayout
from draco_b200.parallel.trainer import Trainer

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = {"alie": (ATTACK_ALIE, 0.8), "ipm": (ATTACK_IPM, 0.1)}


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


def _slots(L, P, seed):
    g = torch.Generator().manual_seed(seed)
    x = 0.05 + 0.1 * torch.randn(P, L.total, generator=g)
    x[:, ~torch.from_numpy(L.valid_mask())] = 0
    return x


def _bitmaps(P, n, seed, min_honest):
    """n random liar masks over P slots, each with at least one liar and ``min_honest`` honest slots."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        k = int(rng.integers(1, P - min_honest + 1))
        out.append(sum(1 << int(r) for r in rng.choice(P, size=k, replace=False)))
    return torch.tensor(np.array(out, dtype=np.uint32).view(np.int32))


def _check(L, before, after, mask, mode, param):
    P = before.shape[0]
    valid = L.valid_mask()
    liars = [r for r in range(P) if (mask >> r) & 1]
    honest = [r for r in range(P) if r not in liars]
    assert torch.equal(after[honest], before[honest])                               # honest rows bitwise unchanged
    assert float(after[:, ~valid].abs().sum()) == 0                                 # padding stays zero
    want = collude(before.double().numpy(), liars, mode, param)[liars[0]][valid]
    H = before[honest].double().numpy()[:, valid]
    mu, sigma = H.mean(axis=0), H.std(axis=0, ddof=1)
    for r in liars:
        got = after[r].double().numpy()[valid]
        err = np.abs(got - want)
        assert np.all(err <= 1e-5 * (np.abs(mu) + abs(param) * sigma) + 1e-7), (mode, P, r, err.max())


def _launch(K, L, x, bm, step, mode, tile_ranges=None):
    code, param = MODES[mode]
    for tr in tile_ranges or [None]:
        K.collude(L, x, L.total, x.shape[0], bm, bm.numel(), step, code, param, tile_range=tr)


# ------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("mode", ["alie", "ipm"])
@pytest.mark.parametrize("P", [4, 7, 13, 16, 32])
def test_kernel_matches_oracle(K, dev, P, mode):
    L = _layout()
    bm = _bitmaps(P, 6, seed=P, min_honest=2).to(dev)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    valid = torch.from_numpy(L.valid_mask())
    for t in range(bm.numel()):
        mask = int(bm[t].item()) & 0xFFFFFFFF
        before = _slots(L, P, seed=100 * P + t)
        for r in range(P):
            if (mask >> r) & 1:
                before[r, valid] = 1e4                           # what a liar pushed must not matter
        x = before.to(dev)
        step.fill_(t + bm.numel())                               # step % adv_len picks the word
        _launch(K, L, x, bm, step, mode)
        torch.cuda.synchronize()
        _check(L, before, x.cpu(), mask, mode, MODES[mode][1])


def test_kernel_buckets_equal_one_launch(K, dev):
    L = _layout()
    n = L.ntiles
    bm = _bitmaps(7, 1, seed=3, min_honest=2).to(dev)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    for mode in MODES:
        a = _slots(L, 7, seed=9).to(dev)
        b = a.clone()
        _launch(K, L, a, bm, step, mode)
        _launch(K, L, b, bm, step, mode, tile_ranges=[(0, n // 3), (n // 3, 2 * n // 3), (2 * n // 3, n)])
        torch.cuda.synchronize()
        assert torch.equal(a, b), mode
        c = _slots(L, 7, seed=9).to(dev)
        _launch(K, L, c, bm, step, mode, tile_ranges=[(n // 2, n // 2)])      # an empty bucket touches nothing
        torch.cuda.synchronize()
        assert torch.equal(c, _slots(L, 7, seed=9).to(dev)), mode


def test_kernel_graph_replay_follows_the_device_step(K, dev):
    """Captured once; each replay reads that step's liar set from the bitmap."""
    L = _layout()
    P = 7
    bm = _bitmaps(P, 5, seed=11, min_honest=2).to(dev)
    orig = _slots(L, P, seed=12).to(dev)
    x = torch.empty_like(orig)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    for mode in MODES:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                       # warm-up outside the capture
            x.copy_(orig)
            _launch(K, L, x, bm, step, mode)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            x.copy_(orig)
            _launch(K, L, x, bm, step, mode)
        for t in range(7):
            step.fill_(t)
            g.replay()
            torch.cuda.synchronize()
            _check(L, orig.cpu(), x.cpu(), int(bm[t % bm.numel()].item()) & 0xFFFFFFFF, mode, MODES[mode][1])
        del g


def test_kernel_rejects_more_than_32_slots(K, dev):
    L = _layout()
    bm = torch.ones(1, dtype=torch.int32, device=dev)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    x = torch.zeros(33, L.total, device=dev)
    with pytest.raises(RuntimeError, match="collude"):
        K.collude(L, x, L.total, 33, bm, 1, step, ATTACK_ALIE, 1.0)


# ------------------------------------------------------------------------------------------------ engines
def _cfg(**kw):
    base = dict(network="LeNet", dataset="MNIST", batch_size=16, max_steps=12, num_workers=7, worker_fail=2, transport="nvl",
                lr=0.02, momentum=0.9, synthetic_size=512, eval_freq=10 ** 6, compress_grad="None", dtype="fp32",
                cuda_graphs=False, approach="baseline")
    base.update(kw)
    return JobConfig(**base)


def _run(cfg, steps):
    t = Trainer(cfg, rank=0, world=1, device=torch.device("cuda", 0), quiet=True)
    losses = [t.train_step()["loss"] for _ in range(steps)]
    t.synchronize()
    return t, losses


_RULES = ["normal", "coord_median", "trimmed_mean", "krum", "multi_krum", "geometric_median"]


@pytest.mark.parametrize("err_mode", ["alie", "ipm"])
@pytest.mark.parametrize("mode", _RULES)
def test_fused_matches_library_op_engine(mode, err_mode):
    a, _ = _run(_cfg(mode=mode, err_mode=err_mode), 3)
    b, _ = _run(_cfg(transport="nccl", mode=mode, err_mode=err_mode), 3)
    assert a.engine.ps.collusion and a.engine.ps.rule == b.engine.ps.rule
    pa, pb = a.engine.master_params(), b.engine.master_params()
    assert torch.isfinite(pa).all()
    assert torch.allclose(pa, pb, atol=2e-5), (mode, err_mode, float((pa - pb).abs().max()))


_RESNET = dict(network="ResNet18", dataset="Cifar10", batch_size=8, num_workers=5, worker_fail=2, err_mode="alie",
               dtype="bf16", synthetic_size=256)


def test_coord_median_under_alie_is_bit_identical_across_pipelining_graphs_and_codec():
    piped, lp = _run(_cfg(mode="coord_median", cuda_graphs=True, **_RESNET), 6)
    serial, ls = _run(_cfg(mode="coord_median", cuda_graphs=True, pipeline_ps=False, **_RESNET), 6)
    eager, le = _run(_cfg(mode="coord_median", cuda_graphs=False, **_RESNET), 6)
    assert piped.engine.pipeline_ps and not serial.engine.pipeline_ps and piped.engine.graph is not None
    assert piped.engine.ps.collusion == ATTACK_ALIE
    ref = piped.engine.master_params()
    assert torch.isfinite(ref).all()
    assert torch.equal(ref, serial.engine.master_params()) and lp == ls
    assert torch.equal(ref, eager.engine.master_params()) and lp == le
    packed, lc = _run(_cfg(mode="coord_median", compress_grad="compress", err_mode="alie"), 4)
    raw, lr = _run(_cfg(mode="coord_median", compress_grad="None", err_mode="alie"), 4)
    assert packed.engine.compress and torch.equal(packed.engine.master_params(), raw.engine.master_params()) and lc == lr


@pytest.mark.parametrize("err_mode", ["alie", "ipm"])
def test_vote_under_collusion_equals_the_clean_run(err_mode):
    kw = dict(network="ResNet18", dataset="Cifar10", batch_size=8, dtype="bf16", synthetic_size=256, approach="maj_vote",
              mode="maj_vote", group_size=3, worker_fail=1, cuda_graphs=True)
    clean, lc = _run(_cfg(err_mode="none", **kw), 5)
    lied, ll = _run(_cfg(err_mode=err_mode, **kw), 5)
    assert lied.engine.graph is not None and lied.engine.ps.collusion
    assert torch.equal(clean.engine.master_params(), lied.engine.master_params()) and lc == ll


@pytest.mark.parametrize("compress", ["None", "compress"])
def test_debug_checksum_under_alie(compress):
    t, _ = _run(_cfg(mode="coord_median", err_mode="alie", debug_checksum=True, compress_grad=compress), 3)
    log = t.engine.checksum_log
    assert len(log) == 3 and all(r["bad"] == [] and r["checked"] == 7 for r in log), log


def _torchrun(nproc, env_extra, port, timeout=900):
    env = dict(os.environ, PYTHONPATH=ROOT, **env_extra)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mp_equiv.py")],
                         capture_output=True, text=True, timeout=timeout, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


@pytest.mark.timeout(900)
def test_alie_across_two_processes_on_one_gpu():
    job = dict(approach="baseline", mode="coord_median", worker_fail=3, err_mode="alie")
    rec = _torchrun(2, {"DRACO_BOOTSTRAP": "gloo", "CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0],
                        "MP_EQUIV_CFG": json.dumps(dict(job, multicast="off", cuda_graphs=False)), "MP_EQUIV_STEPS": "4"},
                    port=29776)
    assert rec["gpus"] == 1 and rec["world"] == 2
    assert rec["sha"][0] == rec["sha"][1]
    single, _ = _run(_cfg(**job, network="ResNet18", dataset="Cifar10", batch_size=8, dtype="bf16", synthetic_size=256), 4)
    assert hashlib.sha256(single.engine.master_params().cpu().numpy().tobytes()).hexdigest() == rec["sha"][0]
