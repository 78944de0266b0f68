"""
Two-rank parity of SimulationBoxPairCount, run under torchrun (one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29543 tests/mgpu_paircount_check.py
Every rank holds half of the rows of a seeded clumpy catalogue and of a uniform one; npairs gathered over the GPUs must
equal a one-GPU count on rank 0 exactly, the sums to 1e-12 (every mode, periodic and not, auto and cross).
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    rank = int(os.environ["RANK"]); local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from nbodykit_b200 import CurrentMPIComm
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.lab import ArrayCatalog, SimulationBoxPairCount
    from test_gpu_fof import clumpy
    comm = CurrentMPIComm.get()
    P = comm.size
    pos = clumpy(seed=7)[0]
    rng = np.random.RandomState(5)
    w = rng.uniform(size=len(pos))
    pos2, w2 = rng.uniform(0, 100., (20000, 3)), rng.uniform(size=20000)
    failures = []
    self_comm = SelfComm()
    for mode, kw in (('1d', {}), ('2d', {'Nmu': 8}), ('projected', {'pimax': 8.})):
        for periodic in (True, False):
            for cross in (False, True):
                edges = np.geomspace(0.5, 10., 7)

                def count(comm, sl1, sl2):
                    a = ArrayCatalog({'Position': pos[sl1], 'Weight': w[sl1]}, comm=comm, BoxSize=100.)
                    b = ArrayCatalog({'Position': pos2[sl2], 'Weight': w2[sl2]}, comm=comm, BoxSize=100.) \
                        if cross else None
                    return SimulationBoxPairCount(mode, a, edges, second=b, periodic=periodic, **kw).pairs
                n1, n2 = len(pos), len(pos2)
                many = count(comm, slice(rank * n1 // P, (rank + 1) * n1 // P), slice(rank * n2 // P, (rank + 1) * n2 // P))
                if rank == 0:
                    one = count(self_comm, slice(None), slice(None))
                    ok = np.array_equal(many['npairs'], one['npairs']) and \
                        np.allclose(many['wnpairs'], one['wnpairs'], rtol=1e-12, atol=0) and \
                        np.allclose(many[one.dims[0]], one[one.dims[0]], rtol=1e-12, atol=0)
                    tag = "%s periodic=%s cross=%s" % (mode, periodic, cross)
                    print("%s: %s (%d pairs)" % (tag, "ok" if ok else "MISMATCH", int(one['npairs'].sum())))
                    if not ok:
                        failures.append(tag)
    failures = comm.bcast(failures)
    dist.destroy_process_group()
    if failures:
        print("FAILED:", failures)
        sys.exit(1)
    if rank == 0:
        print("mgpu paircount check: %d GPUs agree with 1 GPU" % P)


if __name__ == "__main__":
    main()
