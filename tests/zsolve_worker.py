"""Worker of tests/test_gpu_complex_solve.py (one process per GPU, launched by torch.distributed.run): the doublecomplex
factorization and solve on a 1 x 1 x Pz grid through the C-ABI (slu_b200_z_factor, slu_b200_z_solve).  Every rank
passes the same b and must receive the full x."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from superlu_dist_b200 import capi  # noqa: E402
from test_gpu_complex_solve import complex_csr, crandn, permuted_matvec  # noqa: E402
from util import complex_problem  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 14
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    kw = dict(N=N, leaf=16, relax=16, maxsup=64)
    rp, ci, val = complex_csr(**kw)
    prob = complex_problem(**kw, npdep=world, layers=[rank])
    xtrue = crandn(np.random.default_rng(5), 2, prob.n)
    b = permuted_matvec(prob.perm, rp, ci, val, xtrue)
    box = [capi.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    h = capi.Handle(prob, rank, device=local, world_size=world, world_rank=rank, nccl_id=box[0])
    h.upload()
    assert h.factor() == 0
    errs = []
    for rhs, ref in ((b, xtrue), (b[1], xtrue[1])):
        x = h.solve(rhs)
        errs.append(float(np.abs(x - ref).max() / np.abs(ref).max()))
    h.close()
    assert max(errs) < 1e-10, errs
    print(f"rank {rank}/{world}: complex solve err {max(errs):.2e}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
