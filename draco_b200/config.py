"""Job configuration: the reference's flag surface (src/distributed_nn.py:23-77) as a dataclass + parser.

Every reference flag keeps its name and default.  Flags the reference parses but ignores are honoured here where that
is meaningful (``--seed`` seeds model init, ``--adversarial`` scales the attack magnitude, ``--log-interval`` throttles
logging, ``--no-cuda`` forces the CPU/Gloo path) -- see DESIGN.md "flag semantics".  New flags are additive.
"""
from __future__ import annotations

import argparse
import math
from dataclasses import asdict, dataclass
from typing import Optional

APPROACHES = ("baseline", "maj_vote", "cyclic")
MODES = ("normal", "geometric_median", "krum", "maj_vote", "coord_median", "trimmed_mean", "multi_krum")
ROBUST_NVL_MAXP = 16            # P limit of coord_median / trimmed_mean / multi_krum on nvl (register budget of their kernels)
ERR_MODES = ("rev_grad", "constant", "random", "omniscient", "alie", "ipm", "none")
COLLUDING_ERR_MODES = ("alie", "ipm")   # every liar sends one vector built from the honest gradients, applied at the PS
TRANSPORTS = ("nvl", "nccl", "nccl_flat", "gloo")


@dataclass
class JobConfig:
    # ---- reference flags ------------------------------------------------------------------
    batch_size: int = 128
    test_batch_size: int = 100
    max_steps: int = 10000
    epochs: int = 100
    lr: float = 0.01
    momentum: float = 0.5
    no_cuda: bool = False
    seed: int = 1
    log_interval: int = 10
    network: str = "LeNet"
    mode: str = "normal"
    dataset: str = "MNIST"
    comm_type: str = "Bcast"
    err_mode: str = "rev_grad"
    approach: str = "maj_vote"
    num_aggregate: int = 5
    eval_freq: int = 50
    train_dir: str = "output/models/"
    adversarial: int = 1
    worker_fail: int = 2
    group_size: int = 5
    compress_grad: str = "compress"  # lossless DRC2 codec on the wire (reference default: blosc on every gradient message)
    checkpoint_step: int = 0
    # ---- additions --------------------------------------------------------------------------
    num_workers: int = 0            # logical workers P (0: world_size - 1, like `mpirun -n P+1`)
    transport: str = "nvl"          # nvl: fused sm_100a kernels over peer memory | nccl: baseline | gloo: CPU
    dtype: str = "bf16"             # compute dtype on workers (bf16 | fp32)
    cuda_graphs: bool = True
    weight_decay: float = 0.0
    nesterov: bool = False
    dampening: float = 0.0
    optimizer: str = "sgd"          # sgd | adam (reference: src/optim/{sgd,adam}_modified.py); every transport
    amsgrad: bool = False
    adam_beta1: float = 0.9
    adam_beta2: float = 0.999
    adam_eps: float = 1e-8
    data_root: str = "./data"
    synthetic_size: int = 8192
    augment: bool = False
    data_on_device: bool = False    # keep the dataset in HBM and gather batches on the device
    metrics_file: Optional[str] = None
    debug_checksum: bool = False    # verify every pushed gradient: loopback re-encode vs what landed in the PS slot (eager mode)
    profile_phases: bool = False    # CUDA-event timers per phase (fetch/comp/encode/comm/decode/update); disables CUDA graphs
    multicast: str = "auto"         # auto | on | off  (NVLS multimem.st broadcast)
    wgrad_stream: str = "auto"      # weight-gradient kernels on a low-priority side stream: auto (= on with zero-copy gradients) | on | off
    spin_timeout_s: float = 60.0
    ps_stream: bool = False         # PS co-located with workers consumes gradient buckets on its own stream (captured graph only).
                                    # Off by default: its spin-wait kernels then depend on kernels of OTHER graph branches making
                                    # progress, which holds only while every branch gets its own hardware queue
                                    # (CUDA_DEVICE_MAX_CONNECTIONS >= number of concurrent streams)
    num_classes: int = 10
    deterministic: bool = True
    overlap_push: bool = True       # ship gradient buckets while the remaining layers are still back-propagating
    pipeline_ps: bool = True        # PS votes / applies / broadcasts a bucket as soon as every worker pushed it
    push_ctas: int = 16             # CTAs of an overlapped bucket push (NVLink-bound: a handful of SMs saturates the link)
    worker_streams: int = 4         # >1: logical workers sharing a GPU run on (up to) this many concurrent CUDA streams
    zero_copy_grads: bool = True    # push reads gradients where autograd left them (pointer table), no flat gather
    alie_z: Optional[float] = None  # --err-mode alie: the lie is mu - z * sigma; None = Baruch et al.'s z_max(P, worker_fail)
    ipm_epsilon: float = 0.1        # --err-mode ipm: the lie is -epsilon * mu

    # ---- derived --------------------------------------------------------------------------
    def resolve(self, world_size: int) -> "JobConfig":
        if self.num_workers <= 0:
            self.num_workers = max(world_size - 1, 1)
        if self.approach not in APPROACHES:
            raise ValueError(f"--approach must be one of {APPROACHES}")
        if self.err_mode not in ERR_MODES:
            raise ValueError(f"--err-mode must be one of {ERR_MODES}")
        if self.compress_grad not in ("compress", "None", "none"):
            # the reference deadlocks on anything but the two magic strings (baseline_master.py:92-96)
            raise ValueError("--compress-grad must be 'compress' or 'None'")
        if self.approach == "cyclic" and self.num_workers < 2 * self.worker_fail + 1:
            raise ValueError("cyclic code needs num_workers >= 2*worker_fail + 1")
        if self.approach == "cyclic" and 2 * self.worker_fail + 1 > 8:
            raise ValueError("cyclic code: redundancy 2*worker_fail + 1 is limited to 8 (DRC_MAX_R)")
        if self.approach == "maj_vote" and self.num_workers >= self.group_size > 0:
            # all remainder workers join the last group (codes/repetition.py): it can hold up to 2r-1 members, the vote kernel 8
            largest = self.group_size + self.num_workers % self.group_size
            if largest > 8:
                raise ValueError(f"repetition code: the last group would have {largest} members (num_workers % group_size "
                                 f"remainder joins it); the vote kernel handles at most 8 (DRC_MAX_R) -- pick a group size that "
                                 f"divides num_workers more evenly")
        if self.no_cuda:
            self.transport = "gloo"
        if self.approach == "baseline" and self.mode in ("coord_median", "trimmed_mean", "multi_krum"):
            P, f = self.num_workers, self.worker_fail
            if f < 0:
                raise ValueError(f"--mode {self.mode} needs --worker-fail >= 0")
            if self.mode in ("coord_median", "trimmed_mean") and P < 2 * f + 1:
                raise ValueError(f"--mode {self.mode} needs num_workers >= 2*worker_fail + 1 (got {P} workers, "
                                 f"worker_fail {f}): a majority of every coordinate's values must be honest")
            if self.mode == "multi_krum" and P < 2 * f + 3:
                raise ValueError(f"--mode multi_krum needs num_workers >= 2*worker_fail + 3 (got {P} workers, worker_fail {f})")
            if self.transport == "nvl" and P > ROBUST_NVL_MAXP:
                raise ValueError(f"--mode {self.mode} on --transport nvl handles at most {ROBUST_NVL_MAXP} workers (got {P}); "
                                 f"use --transport nccl for more")
        if self.err_mode in COLLUDING_ERR_MODES:
            self._check_collusion()
        if self.compress and self.transport == "nvl" and self.err_mode == "omniscient":
            raise ValueError("--err-mode omniscient reads the honest slots in PS memory while they arrive; with --compress-grad "
                             "compress they only exist after the PS unpacked them -- pass --compress-grad None")
        if self.compress and self.transport == "nccl_flat":
            raise ValueError("--transport nccl_flat is the uncompressed library comparator: pass --compress-grad None")
        if self.transport == "gloo":
            self.dtype = "fp32"
            self.cuda_graphs = False
        return self

    def _check_collusion(self) -> None:
        P, f = self.num_workers, self.worker_fail
        if self.approach == "cyclic":
            raise ValueError(f"--err-mode {self.err_mode} is defined over real gradients; the cyclic code's adversary adds an "
                             f"error to a complex codeword -- use another --approach")
        for name, v in (("--alie-z", self.alie_z), ("--ipm-epsilon", self.ipm_epsilon)):
            if v is not None and not math.isfinite(float(v)):
                raise ValueError(f"{name} must be finite (got {v})")
        if self.err_mode == "alie" and P - f < 2:
            raise ValueError(f"--err-mode alie needs at least 2 honest workers for the standard deviation (got {P} workers, "
                             f"worker_fail {f})")
        if self.err_mode == "ipm" and P - f < 1:
            raise ValueError(f"--err-mode ipm needs at least 1 honest worker (got {P} workers, worker_fail {f})")
        if self.err_mode == "alie" and self.alie_z is None:
            from .codes.adversary import alie_z_max
            alie_z_max(P, f)                    # raises when the default z is undefined (the liars alone are a majority)

    @property
    def attack_param(self) -> float:
        """z of ``--err-mode alie`` (``--alie-z``, else Baruch et al.'s default for P workers and worker_fail liars) or
        epsilon of ``--err-mode ipm``."""
        if self.err_mode == "ipm":
            return float(self.ipm_epsilon)
        if self.alie_z is not None:
            return float(self.alie_z)
        from .codes.adversary import alie_z_max
        return alie_z_max(self.num_workers, self.worker_fail)

    @property
    def compress(self) -> bool:
        return self.compress_grad == "compress"

    @property
    def redundancy(self) -> int:
        if self.approach == "cyclic":
            return 2 * self.worker_fail + 1
        if self.approach == "maj_vote":
            return self.group_size
        return 1

    @property
    def attack_magnitude(self) -> float:
        return -100.0 * float(self.adversarial)

    def to_dict(self) -> dict:
        return asdict(self)


def add_fit_args(parser: argparse.ArgumentParser) -> argparse.ArgumentParser:
    """Same flag names/defaults as the reference's ``add_fit_args`` plus the additive ones."""
    d = JobConfig()
    a = parser.add_argument
    a("--batch-size", type=int, default=d.batch_size, help="per-worker batch size")
    a("--test-batch-size", type=int, default=d.test_batch_size)
    a("--max-steps", type=int, default=d.max_steps)
    a("--epochs", type=int, default=d.epochs)
    a("--lr", type=float, default=d.lr)
    a("--momentum", type=float, default=d.momentum)
    a("--no-cuda", action="store_true", default=False, help="run on CPU over the Gloo transport")
    a("--seed", type=int, default=d.seed)
    a("--log-interval", type=int, default=d.log_interval)
    a("--worker-streams", type=int, default=d.worker_streams,
      help="logical workers that share one GPU are issued round-robin on this many CUDA streams (small layers of "
           "different workers overlap); 1 = serial")
    a("--debug-checksum", action="store_true", default=d.debug_checksum,
      help="transport self-check: each worker re-encodes its gradient into a local buffer and the PS compares 64-bit "
           "checksums with what arrived in its slots, every step (eager mode, nvl transport)")
    a("--profile-phases", action="store_true", default=d.profile_phases,
      help="time the reference's phases (Comm / Comp / Encode / Method / Update) with CUDA events each step; eager mode")
    a("--network", type=str, default=d.network)
    a("--mode", type=str, default=d.mode,
      help="normal | geometric_median | krum | coord_median | trimmed_mean | multi_krum (baseline); normal | maj_vote (maj_vote)")
    a("--dataset", type=str, default=d.dataset)
    a("--comm-type", type=str, default=d.comm_type)
    a("--err-mode", type=str, default=d.err_mode,
      help="rev_grad | constant | random | omniscient | alie | ipm | none.  alie (Baruch et al., 2019) and ipm (Xie et al., "
           "2019) collude: every liar sends mu - z * sigma / -epsilon * mu of the honest gradients (not with --approach cyclic)")
    a("--alie-z", type=float, default=d.alie_z,
      help="z of --err-mode alie (default: Phi^-1((P - s) / P) with s = floor(P/2 + 1) - worker_fail)")
    a("--ipm-epsilon", type=float, default=d.ipm_epsilon, help="epsilon of --err-mode ipm")
    a("--approach", type=str, default=d.approach, help="baseline | maj_vote | cyclic")
    a("--num-aggregate", type=int, default=d.num_aggregate)
    a("--eval-freq", type=int, default=d.eval_freq)
    a("--train-dir", type=str, default=d.train_dir)
    a("--adversarial", type=int, default=d.adversarial, help="attack magnitude multiplier (x -100)")
    a("--worker-fail", type=int, default=d.worker_fail)
    a("--group-size", type=int, default=d.group_size)
    a("--compress-grad", type=str, default=d.compress_grad)
    a("--checkpoint-step", type=int, default=d.checkpoint_step)
    a("--num-workers", type=int, default=0, help="logical workers P (default world_size-1)")
    a("--transport", type=str, default=d.transport, choices=TRANSPORTS)
    a("--dtype", type=str, default=d.dtype, choices=("bf16", "fp32"))
    a("--no-cuda-graphs", dest="cuda_graphs", action="store_false", default=True)
    a("--weight-decay", type=float, default=0.0)
    a("--nesterov", action="store_true", default=False)
    a("--dampening", type=float, default=0.0)
    a("--optimizer", type=str, default="sgd", choices=("sgd", "adam"))
    a("--amsgrad", action="store_true", default=False, help="AMSGrad variant of --optimizer adam (reference: adam_modified.py:16)")
    a("--data-root", type=str, default=d.data_root)
    a("--synthetic-size", type=int, default=d.synthetic_size)
    a("--augment", action="store_true", default=False)
    a("--data-on-device", action="store_true", default=False)
    a("--metrics-file", type=str, default=None)
    a("--multicast", type=str, default="auto", choices=("auto", "on", "off"))
    a("--wgrad-stream", type=str, default=d.wgrad_stream, choices=("auto", "on", "off"))
    a("--spin-timeout-s", type=float, default=d.spin_timeout_s)
    a("--ps-stream", action="store_true", default=d.ps_stream,
      help="co-located PS on its own stream inside the captured graph (set CUDA_DEVICE_MAX_CONNECTIONS=32)")
    a("--num-classes", type=int, default=10)
    a("--no-overlap-push", dest="overlap_push", action="store_false", default=True)
    return parser


def config_from_args(args: argparse.Namespace) -> JobConfig:
    fields = JobConfig.__dataclass_fields__
    return JobConfig(**{k: v for k, v in vars(args).items() if k in fields})
