"""
Two-rank parity of the mixed-radix FFT (mesh sides 2^a 3^b 5^c 7^d), run under torchrun (one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 tests/mgpu_mixed_check.py
The distributed transform (z and y passes on x slabs, pack + NCCL all-to-all + unpack, x pass) must reproduce the
single-GPU one computed on rank 0: an r2c / c2r round trip of a random field, and FFTPower at Nmesh = 96 and
[96, 60, 40] with the tolerances of tests/mgpu_check.py (mode counts bit-exact, P(k) to 2e-8 in f8, 2e-5 in f4).
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from nbodykit_b200 import CurrentMPIComm
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.lab import ArrayCatalog, FFTPower
    from nbodykit_b200.pmesh.pm import ParticleMesh, RealField
    comm = CurrentMPIComm.get()
    failures = []

    # ---- r2c / c2r of a random field on x slabs
    for N, dtype in (([96, 60, 40], "f8"), ([48, 48, 30], "f4")):
        full = np.random.RandomState(3).standard_normal(N).astype(dtype)
        pm = ParticleMesh(BoxSize=1.0, Nmesh=N, dtype=dtype, comm=comm)
        assert pm.mixed_fft
        f = RealField(pm)
        f[...] = full[pm.x_start:pm.x_start + pm.x_n]
        c = f.r2c()                                   # [y_n][Nx][Nzc] on each rank
        back = c.c2r().numpy()
        cparts = comm.allgather(c.numpy())
        bparts = comm.allgather(back)
        if rank == 0:
            want = np.fft.rfftn(full.astype("f8")) / full.size
            got = np.concatenate(cparts, axis=0).transpose(1, 0, 2)
            tol = 1e-13 if dtype == "f8" else 2e-6
            rms = np.sqrt((np.abs(want) ** 2).mean())
            ok = np.abs(got - want).max() <= tol * rms * np.log2(full.size)
            ok &= np.abs(np.concatenate(bparts, axis=0) - full).max() <= tol * 10 * np.log2(full.size)
            print("case r2c/c2r %s %s: %s" % (N, dtype, "OK" if ok else "MISMATCH"), flush=True)
            if not ok:
                failures.append("r2c %s" % N)

    # ---- FFTPower on mixed meshes
    L = 1000.
    rng = np.random.RandomState(1234)
    pos_all = rng.uniform(-50, 1050, size=(400000, 3)).astype("f4")
    w_all = rng.uniform(0.5, 1.5, size=len(pos_all))
    mine = slice(rank * len(pos_all) // world, (rank + 1) * len(pos_all) // world)
    cases = [dict(Nmesh=96, resampler="cic", interlaced=False, dtype="f8", mode="1d", kw={}),
             dict(Nmesh=[96, 60, 40], resampler="tsc", interlaced=True, dtype="f4", mode="2d", kw=dict(Nmu=4, poles=[0, 2])),
             dict(Nmesh=[96, 60, 40], resampler="cic", interlaced=False, dtype="f8", mode="1d", kw={})]
    for c in cases:
        cat = ArrayCatalog({"Position": torch.from_numpy(pos_all[mine]).cuda(), "Weight": torch.from_numpy(w_all[mine]).cuda()},
                           comm=comm, BoxSize=L)
        mesh = cat.to_mesh(Nmesh=c["Nmesh"], resampler=c["resampler"], interlaced=c["interlaced"], compensated=True,
                           dtype=c["dtype"])
        r = FFTPower(mesh, mode=c["mode"], **c["kw"])
        if rank == 0:
            cat1 = ArrayCatalog({"Position": torch.from_numpy(pos_all).cuda(), "Weight": torch.from_numpy(w_all).cuda()},
                                comm=SelfComm(), BoxSize=L)
            mesh1 = cat1.to_mesh(Nmesh=c["Nmesh"], resampler=c["resampler"], interlaced=c["interlaced"], compensated=True,
                                 dtype=c["dtype"])
            r1 = FFTPower(mesh1, mode=c["mode"], **c["kw"])
            tol = 2e-8 if c["dtype"] == "f8" else 2e-5
            ok = np.array_equal(r.power["modes"], r1.power["modes"])
            ok &= np.allclose(np.nan_to_num(r.power["power"].real), np.nan_to_num(r1.power["power"].real), rtol=tol,
                              atol=tol * np.nanmax(np.abs(r1.power["power"])))
            ok &= np.allclose(np.nan_to_num(r.power["k"]), np.nan_to_num(r1.power["k"]), rtol=1e-12)
            ok &= r.attrs["N1"] == r1.attrs["N1"]
            if "poles" in c["kw"]:
                ok &= np.allclose(np.nan_to_num(r.poles["power_2"].real), np.nan_to_num(r1.poles["power_2"].real),
                                  rtol=tol, atol=tol * np.nanmax(np.abs(r1.poles["power_0"])))
            print("case FFTPower %s: %s" % (c, "OK" if ok else "MISMATCH"), flush=True)
            if not ok:
                failures.append(c)
    flag = torch.tensor([len(failures)], device="cuda")
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(1 if int(flag.item()) else 0)


if __name__ == "__main__":
    main()
