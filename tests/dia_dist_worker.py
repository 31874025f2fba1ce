"""Worker for test_gpu_spmv_dia.py::test_multi_gpu_operator_stays_csr, launched through torchrun (one process per
GPU, NCCL): a row slab of a multi-GPU operator addresses its halo through the local extended index, so its col - row
offsets are not those of the global matrix and it must not get an offset-diagonal copy."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    N = 32
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import iterativesolvers_jl_b200 as isb
    ctx = isb.Context.distributed(local)
    offs = np.array([N * r // world * N * N for r in range(world + 1)], dtype=np.int64)
    lo, m = int(offs[rank]), int(offs[rank + 1] - offs[rank])
    plan = isb.HaloPlan(rank, world, offs).scan_laplacian(N, 3).exchange()
    A = isb.B200CSR.laplacian(N, 3, np.float64, lo, m, plan, ctx)
    rp, ci, va = isb.laplace_csr_slab(np.float64, N, 3, lo, m)
    plan2 = isb.HaloPlan(rank, world, offs).scan_csr(rp, ci).exchange()
    A2 = isb.B200CSR.from_csr_slab(rp, ci, va, N ** 3, lo, 0, plan2, ctx)
    assert A.format == "csr" and A.dia_offsets == [], (A.format, A.dia_offsets)
    assert A2.format == "csr" and A2.dia_offsets == [], (A2.format, A2.dia_offsets)
    dist.barrier()
    if rank == 0:
        print("DIA_DIST_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
