"""
FOF timing on the B200 (writes one JSON line per workload to --out, default profiles/r04_fof_bench.jsonl):

  lognormal  LogNormalCatalog 1e8 particles (f4), L = 1024, bias 2, b = 0.2 of the mean separation, nmin = 20 (the C2
             catalogue of bench.py)
  clumpy     the worst case for the link pass: 1e7 particles, a fifth of them in 100 Plummer spheres (a = 2) whose cores
             hold hundreds of particles per cell -- the pair loop is quadratic in the cell occupancy there
  parity     LogNormal 1e7: labels against oracle/fof_oracle.py (cKDTree.query_pairs + connected components), with the
             oracle's host time for context

Per workload: FOF + find_features wall time (CUDA events, best and median of --repeat after one warm-up run), the
per-stage device times (bucket, link, compress, labels, features; events recorded by _lib.stage), particles/s, the
group count, the card name and power limit (nvidia-smi, read in the same run).  Under torchrun (2 GPUs) each rank keeps
its share of the rows and the merge iteration count is reported as well.

    python tools/fof_bench.py [--workloads lognormal,clumpy,parity] [--repeat 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAGES = ("fof_bucket", "fof_link", "fof_compress", "fof_labels", "fof_features")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def lognormal(npart, box, comm, seed=42):
    from nbodykit_b200.cosmology import NoWiggleEHPower
    from nbodykit_b200.source.catalog.lognormal import LogNormalCatalog
    return LogNormalCatalog(Plin=NoWiggleEHPower(), nbar=npart / box ** 3, BoxSize=box, Nmesh=256, bias=2.0, seed=seed,
                            comm=comm)


def clumpy(n, box, comm, seed=3):
    import torch
    from nbodykit_b200.lab import ArrayCatalog
    rng = np.random.RandomState(seed)
    nclump, per = 100, n // 500
    parts = []
    for c in rng.uniform(0, box, (nclump, 3)):
        r = 2.0 / np.sqrt(rng.uniform(1e-3, 1, per) ** (-2. / 3) - 1)
        v = rng.standard_normal((per, 3))
        parts.append(c + v / np.linalg.norm(v, axis=1)[:, None] * np.minimum(r, 20.)[:, None])
    parts.append(rng.uniform(0, box, (n - nclump * per, 3)))
    pos = (np.concatenate(parts) % box).astype('f4')
    pos = pos[rng.permutation(len(pos))]
    vel = rng.standard_normal(pos.shape).astype('f4')
    sl = slice(comm.rank * n // comm.size, (comm.rank + 1) * n // comm.size)
    return ArrayCatalog({'Position': torch.as_tensor(pos[sl]).cuda(), 'Velocity': torch.as_tensor(vel[sl]).cuda()},
                        comm=comm, BoxSize=box)


def time_fof(cat, b, nmin, repeat):
    import torch
    from nbodykit_b200 import _lib
    from nbodykit_b200.lab import FOF
    FOF(cat, b, nmin).find_features()                  # warm-up
    torch.cuda.synchronize()
    totals, stages = [], {s: [] for s in STAGES}
    for _ in range(repeat):
        _lib.profiler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f = FOF(cat, b, nmin)
        h = f.find_features()
        e1.record()
        rec = _lib.profiler.stop()
        totals.append(e0.elapsed_time(e1))
        for s in STAGES:
            stages[s].append(sum(rec.get(s, [0.0])))
    return f, h, totals, stages


def run(name, cat, b, nmin, repeat, comm, out):
    f, h, totals, stages = time_fof(cat, b, nmin, repeat)
    n = int(cat.csize)
    best = min(totals)
    rec = {"workload": name, "particles": n, "linking_length_rel": b, "nmin": nmin, "ranks": comm.size,
           "groups": int(max(f.max_label)), "merge_iterations": int(getattr(f, "merge_iterations", 0)),
           "total_ms_best": round(best, 3), "total_ms_median": round(float(np.median(totals)), 3),
           "particles_per_s": n / (best * 1e-3),
           "stage_ms_median": {s: round(float(np.median(v)), 3) for s, v in stages.items()},
           "card": card()}
    if comm.rank == 0:
        print(json.dumps(rec))
        out.write(json.dumps(rec) + "\n")
        out.flush()


def parity(comm, out):
    import torch
    from nbodykit_b200.lab import FOF
    from oracle import fof_oracle as fo
    cat = lognormal(1e7, 1024., comm)
    f = FOF(cat, 0.2, 20)
    torch.cuda.synchronize()
    labels = np.concatenate(comm.allgather(f.labels.cpu().numpy()))
    pos = np.concatenate(comm.allgather(cat['Position'].compute().cpu().numpy()))
    if comm.rank != 0:
        return
    ll = f._linking_length
    t0 = time.perf_counter()
    want = fo.labels(pos, ll, 20, 1024.)
    t_oracle = time.perf_counter() - t0
    ties = len(fo.near_ties(pos, ll, 1024.))
    rec = {"workload": "parity_lognormal_1e7", "particles": len(pos), "ranks": comm.size,
           "labels_equal": bool(np.array_equal(labels, want)), "groups": int(want.max()), "near_ties": ties,
           "oracle_host_s": round(t_oracle, 2), "host_cores": os.cpu_count(), "card": card()}
    print(json.dumps(rec))
    out.write(json.dumps(rec) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="lognormal,clumpy,parity")
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_fof_bench.jsonl"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fof_bench needs a CUDA device")
    from nbodykit_b200 import CurrentMPIComm
    comm = CurrentMPIComm.get()
    with open(a.out, "a") as out:
        for w in a.workloads.split(","):
            if w == "lognormal":
                run("lognormal_1e8", lognormal(1e8, 1024., comm), 0.2, 20, a.repeat, comm, out)
            elif w == "clumpy":
                run("clumpy_1e7", clumpy(10 ** 7, 1024., comm), 0.2, 20, a.repeat, comm, out)
            elif w == "parity":
                parity(comm, out)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
