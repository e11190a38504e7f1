"""``distributed_nn`` entry point -- same flags as the reference's ``src/distributed_nn.py``.

Reference launch: ``mpirun -n P+1 --hostfile hosts_address python distributed_nn.py <flags>`` (src/run_pytorch.sh:1-19),
rank 0 = PS, ranks 1..P = workers (src/distributed_nn.py:87-133).

Here:
  * one process per GPU under torchrun:
        python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 -m draco_b200.cli.distributed_nn <flags>
    (8 processes = 1 PS + 7 workers, like ``mpirun -n 8``; with fewer GPUs pass ``--num-workers 7`` and the logical
    workers are packed onto the GPUs that exist)
  * or let this script spawn the processes:  ``python -m draco_b200.cli.distributed_nn --launch 8 <flags>``
  * or a single process hosting every role:  ``python -m draco_b200.cli.distributed_nn --num-workers 7 <flags>``
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

from ..config import add_fit_args, config_from_args


RULES = """aggregation rules (per parameter tensor, P workers, f = --worker-fail):
  --approach maj_vote --mode maj_vote       repetition-code majority vote (Draco)
  --approach cyclic                         cyclic-code decode (Draco)
  --approach baseline --mode normal         mean
  --approach baseline --mode geometric_median
  --approach baseline --mode krum           Krum
  --approach baseline --mode multi_krum     mean of the P - f best Krum rows       (P >= 2f + 3)
  --approach baseline --mode coord_median   coordinate-wise median                 (P >= 2f + 1)
  --approach baseline --mode trimmed_mean   coordinate-wise mean without the f lowest and f highest values  (P >= 2f + 1)
"""


def main(argv=None) -> int:
    ap = add_fit_args(argparse.ArgumentParser(description="Draco on B200 (draco_b200)", epilog=RULES,
                                              formatter_class=argparse.RawDescriptionHelpFormatter))
    ap.add_argument("--launch", type=int, default=0, help="spawn this many local processes with torchrun semantics")
    ap.add_argument("--master-port", type=int, default=29511)
    args = ap.parse_args(argv)
    if args.launch and "RANK" not in os.environ:
        argv_child = [a for a in (argv if argv is not None else sys.argv[1:])]
        # strip --launch N
        out, skip = [], False
        for a in argv_child:
            if skip:
                skip = False
                continue
            if a == "--launch":
                skip = True
                continue
            if a.startswith("--launch="):
                continue
            out.append(a)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.launch}",
               "--master-addr", "127.0.0.1", "--master-port", str(args.master_port), "-m", "draco_b200.cli.distributed_nn", *out]
        return subprocess.call(cmd)

    from ..parallel.trainer import Trainer
    cfg = config_from_args(args)
    trainer = Trainer(cfg)
    role = "master" if trainer.rank == 0 else "worker"
    print(f"I am {role}: rank {trainer.rank} of {trainer.world} processes; job = 1 PS + {cfg.num_workers} workers; "
          f"placement: {trainer.engine.place.describe()}; transport={cfg.transport}", flush=True)
    try:
        last = trainer.fit()
        if last:
            print(f"rank {trainer.rank} done at step {trainer.step - 1}: loss {last.get('loss', float('nan')):.4f}", flush=True)
    finally:
        trainer.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
