"""Multi-GPU check of the single lattice in a field schedule, launched with torchrun (one process per GPU,
NCCL):

  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tests/multi_gpu_strip_field_check.py

SingleLattice2D split in row strips over the ranks - the library's own NCCL loop (exchange_every = k > 0)
and the per-phase exchange overlapped with the interior (k = 0) - runs a field schedule that changes sign
and passes through 0; the gathered rows equal one strip on one GPU and the field strip mirror, and the
global energy and magnetization equal the single strip's.  Rank 0 prints MULTI_GPU_STRIP_FIELD_OK."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def main():
    import torch
    import torch.distributed as dist

    import pyisingmontecarlo_b200 as pkg
    from strip_field_check import mirror_single_field

    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    Lx, Ly = 256, 16 * world
    betas = [0.3, 0.44, 0.8, 0.44, 0.5, 0.2, 0.6]
    fields = [0.3, -0.3, 0.0, -0.0, 2.0, -7.0, 0.1]
    ref, _, _ = mirror_single_field(Lx, Ly, -1.0, 9, betas, fields)
    for k in (0, 1, 3):
        lat = pkg.SingleLattice2D(Lx, Ly, j=-1.0, seed=9, device=local, exchange_every=k)
        lat.sweeps(betas, fields)
        e, m = lat.energy(), lat.magnetization()
        rows = torch.from_numpy(lat.local_rows().astype(np.uint8)).cuda(local)
        parts = [torch.empty_like(rows) for _ in range(world)]
        dist.all_gather(parts, rows)
        if rank == 0:
            got = torch.cat(parts).cpu().numpy().astype(bool)
            assert (got == ref).all(), (k, int((got != ref).sum()))
            one = pkg.SingleLattice2D(Lx, Ly, j=-1.0, seed=9, device=local, process_group=dist.new_group([0]),
                                      exchange_every=k)
            one.sweeps(betas, fields)
            assert (one.local_rows() == ref).all(), k
            assert (e, m) == (one.energy(), one.magnetization()), (k, e, m)
        else:
            dist.new_group([0])                       # new_group is collective
        dist.barrier()
    if rank == 0:
        print("MULTI_GPU_STRIP_FIELD_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
