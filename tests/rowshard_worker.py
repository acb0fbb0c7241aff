"""torchrun worker (one rank per GPU): the library's row-sharded step loop, with either exchange, equals the
single-process emulation."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import isingmodel_jl_b200 as pkg  # noqa: E402,F401
from isingmodel_jl_b200 import rowshard, synth  # noqa: E402


def main():
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, R, seed, nsteps = 1024, 600, 17, 4
    S0 = synth.spins(3, R, n)
    T = np.array([1.0, 0.8, 0.6, 0.4])
    ok, modes = True, []
    # the step loop inside the library (isb_shard_run_*): NCCL through the library's own communicator, and the
    # copy-engine exchange over CUDA IPC; bf16 terms and int8 digit planes
    for prec in (pkg._lib.PREC_BF16X3, pkg._lib.PREC_I8X3):
        emu = rowshard.RowShardedSCA(n, R, seed=seed, q=1.0, prec=prec, emulate_blocks=dist.get_world_size(), device=local)
        emu.set_spins(S0)
        emu.run(nsteps, T, seed=7)
        for exchange in ("nccl", "copy"):
            abi = rowshard.ShardRunSCA(n, R, seed=seed, q=1.0, prec=prec, device=local, exchange=exchange)
            for rep in range(2):      # a second run on the same object exercises the re-initialisation path
                abi.set_spins(S0)
                abi.run(nsteps, T, seed=7)
                same = np.array_equal(abi.get_spins(), emu.get_spins()) and np.array_equal(abi.get_hidden(), emu.get_hidden())
                ok = ok and same
            modes.append(f"{abi.exchange}/{'i8' if prec == pkg._lib.PREC_I8X3 else 'bf16'}:{'ok' if same else 'MISMATCH'}")
            del abi
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if dist.get_rank() == 0:
        print("ROWSHARD-OK" if int(flag.item()) == 1 else "ROWSHARD-MISMATCH", modes, flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
