"""
Two-rank parity of FOF, run under torchrun (one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 tests/mgpu_fof_check.py
Every rank holds half of the rows of a seeded clumpy catalogue; the gathered labels must equal those of a one-GPU run
on rank 0 exactly, and the gathered find_features columns must match to 1e-6 (periodic and non-periodic).
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
    from nbodykit_b200.lab import ArrayCatalog, FOF
    from test_gpu_fof import clumpy
    comm = CurrentMPIComm.get()
    P = comm.size
    failures = []
    pos, vel = clumpy(seed=7)
    peak = np.random.RandomState(2).uniform(size=len(pos))
    n = len(pos)
    sl = slice(rank * n // P, (rank + 1) * n // P)
    cols = ('CMPosition', 'CMVelocity', 'Length', 'PeakPosition', 'PeakVelocity')
    for periodic in (True, False):
        attrs = {'BoxSize': 100.} if periodic else {}
        cat = ArrayCatalog({'Position': pos[sl], 'Velocity': vel[sl], 'Peak': peak[sl]}, comm=comm, **attrs)
        f = FOF(cat, 0.25, 20, absolute=True, periodic=periodic)
        h = f.find_features(peakcolumn='Peak')
        labels = np.concatenate(comm.allgather(f.labels.cpu().numpy()))
        feats = {k: np.concatenate(comm.allgather(np.asarray(h[k]))) for k in cols}
        if rank == 0:
            one = FOF(ArrayCatalog({'Position': pos, 'Velocity': vel, 'Peak': peak}, comm=SelfComm(), **attrs), 0.25, 20,
                      absolute=True, periodic=periodic)
            h1 = one.find_features(peakcolumn='Peak')
            if not np.array_equal(labels, one.labels.cpu().numpy()):
                failures.append("labels differ (periodic=%s)" % periodic)
            for k in cols:
                try:
                    np.testing.assert_allclose(feats[k], np.asarray(h1[k]), rtol=1e-6, atol=1e-4)
                except AssertionError as e:
                    failures.append("%s (periodic=%s): %s" % (k, periodic, str(e)[:300]))
            print("periodic=%s: %d groups, %d merge iterations" % (periodic, one.max_label[0], f.merge_iterations))
    failures = comm.bcast(failures)
    dist.destroy_process_group()
    if failures:
        print("FAILED:\n" + "\n".join(failures))
        sys.exit(1)
    print("mgpu_fof_check ok")


if __name__ == "__main__":
    main()
