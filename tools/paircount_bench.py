"""
Pair-count timing on the B200 (writes one JSON line per workload to --out, default profiles/r05_paircount_bench.jsonl):

  a_uniform_1d     UniformCatalog 1e6 in L = 1000, '1d', 20 log bins over 0.1 - 150 (a halo-catalogue xi(r)); the
                   CPU oracle's time (cKDTree.count_neighbors over all host cores) is reported beside it
  b_lognormal_2d   LogNormalCatalog 1e7 in L = 1024 (bias 2), '2d', 50 r bins up to 50, Nmu = 20
  c_lognormal_proj the same catalogue, 'projected', 25 log r_p bins over 0.5 - 30, pimax = 40
  d_fof_groups_1d  FOF groups (b = 0.2, nmin = 20) of the C2 catalogue (LogNormal 1e8, L = 1024) ->
                   SimulationBox2PCF('1d'), 20 log bins over 1 - 100

Per workload: the time per call (CUDA events, median and best of --repeat after one warm-up call), the per-stage
device times (bucket, count, reduce; events recorded by _lib.stage), the distance evaluations the stencil implies
(sum over cells of primaries x secondaries in the stencil cells, from the cell occupancies), the pairs in range,
evaluations per second, and the card name and power limit (nvidia-smi, read in the same run).

    python tools/paircount_bench.py [--workloads a,b,c,d] [--repeat 3] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAGES = ("pc_bucket", "pc_count", "pc_reduce")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def lognormal(npart, box, seed=42, Nmesh=256):
    from nbodykit_b200.cosmology import NoWiggleEHPower
    from nbodykit_b200.source.catalog.lognormal import LogNormalCatalog
    return LogNormalCatalog(Plin=NoWiggleEHPower(), nbar=npart / box ** 3, BoxSize=box, Nmesh=Nmesh, bias=2.0, seed=seed)


def _pos(cat, col='Position'):
    c = cat[col]
    return c.compute() if hasattr(c, 'compute') else c


def stencil_evaluations(pos, box, rmax):
    """distance evaluations of an auto count: sum over cells of n_c * (secondaries in the stencil cells of c)"""
    import torch
    from nbodykit_b200._lib import darr, lib
    n = int(pos.shape[0])
    nc = (ctypes.c_int64 * 3)()
    bc = darr([box] * 3)
    lib().nbk_pc_workspace(n, n, rmax, bc, None, None, nc)
    st = (ctypes.c_int32 * 125)()
    k = lib().nbk_pc_stencil(n, rmax, bc, None, None, st)
    ncell = [int(v) for v in nc]
    p = torch.as_tensor(pos).double()
    idx = torch.stack([torch.clamp((torch.remainder(p[:, d], box) * (ncell[d] / box)).long(), 0, ncell[d] - 1)
                       for d in range(3)], 1)
    occ = torch.zeros(ncell, dtype=torch.float64, device=p.device)
    occ.index_put_((idx[:, 0], idx[:, 1], idx[:, 2]), torch.ones(n, dtype=torch.float64, device=p.device),
                   accumulate=True)
    nb = torch.zeros_like(occ)
    for o in st[:k]:
        nb += torch.roll(occ, shifts=(-(o // 25 - 2), -((o // 5) % 5 - 2), -(o % 5 - 2)), dims=(0, 1, 2))
    return float((occ * nb).sum())


def time_calls(fn, repeat):
    import torch
    from nbodykit_b200 import _lib
    fn()                                               # warm-up
    torch.cuda.synchronize()
    totals, stages = [], {s: [] for s in STAGES}
    res = None
    for _ in range(repeat):
        _lib.profiler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        rec = _lib.profiler.stop()
        totals.append(e0.elapsed_time(e1))
        for s in STAGES:
            stages[s].append(sum(rec.get(s, [0.0])))
    return res, totals, stages


def record(name, n, totals, stages, evals, pairs, extra, out):
    med = float(np.median(totals))
    rec = {"workload": name, "objects": n, "ms_median": round(med, 3), "ms_best": round(min(totals), 3),
           "stage_ms_median": {s: round(float(np.median(v)), 3) for s, v in stages.items()},
           "stencil_distance_evaluations": evals, "pairs_in_range": pairs,
           "evaluations_per_s": evals / (med * 1e-3), "card": card()}
    rec.update(extra)
    print(json.dumps(rec))
    out.write(json.dumps(rec) + "\n")
    out.flush()


def _oracle_chunk(args):
    from scipy.spatial import cKDTree
    pos, lo, hi, edges, box = args
    tree = cKDTree(pos, boxsize=box)
    sub = cKDTree(pos[lo:hi], boxsize=box)
    return sub.count_neighbors(tree, edges)


def oracle_time(pos, edges, box):
    """host time of the cumulative pair counts at the edges, primaries split over every host core"""
    from concurrent.futures import ProcessPoolExecutor
    ncore = os.cpu_count() or 1
    stops = np.linspace(0, len(pos), ncore + 1).astype(int)
    t0 = time.perf_counter()
    with ProcessPoolExecutor(ncore) as ex:
        cum = sum(ex.map(_oracle_chunk, [(pos, stops[i], stops[i + 1], edges, box) for i in range(ncore)]))
    return time.perf_counter() - t0, ncore, np.diff(cum)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="a,b,c,d")
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_paircount_bench.jsonl"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("paircount_bench needs a CUDA device")
    from nbodykit_b200.lab import FOF, SimulationBox2PCF, SimulationBoxPairCount, UniformCatalog
    todo = a.workloads.split(",")
    with open(a.out, "a") as out:
        if "a" in todo:
            cat = UniformCatalog(nbar=1e6 / 1000. ** 3, BoxSize=1000., seed=42)
            edges = np.geomspace(0.1, 150., 21)
            r, totals, stages = time_calls(lambda: SimulationBoxPairCount('1d', cat, edges), a.repeat)
            pos = _pos(cat)
            evals = stencil_evaluations(pos, 1000., 150.)
            t_cpu, ncore, cpu_counts = oracle_time(pos.cpu().numpy().astype('f8'), edges, 1000.)
            record("a_uniform_1d", int(cat.csize), totals, stages, evals, int(r.pairs['npairs'].sum()),
                   {"oracle_host_s": round(t_cpu, 2), "host_cores": ncore,
                    "oracle_npairs_rel_diff": float(np.abs(cpu_counts - r.pairs['npairs']).sum()
                                                    / max(1, r.pairs['npairs'].sum()))}, out)
            del cat, r
        if "b" in todo or "c" in todo:
            cat = lognormal(1e7, 1024.)
            pos = _pos(cat)
            if "b" in todo:
                edges = np.linspace(1., 50., 51)
                r, totals, stages = time_calls(lambda: SimulationBoxPairCount('2d', cat, edges, Nmu=20), a.repeat)
                record("b_lognormal_2d", int(cat.csize), totals, stages, stencil_evaluations(pos, 1024., 50.),
                       int(r.pairs['npairs'].sum()), {"bins": [50, 20]}, out)
            if "c" in todo:
                edges = np.geomspace(0.5, 30., 26)
                r, totals, stages = time_calls(lambda: SimulationBoxPairCount('projected', cat, edges, pimax=40.),
                                               a.repeat)
                record("c_lognormal_projected", int(cat.csize), totals, stages,
                       stencil_evaluations(pos, 1024., float(np.hypot(30., 40.))), int(r.pairs['npairs'].sum()),
                       {"bins": [25, 40]}, out)
            del cat, pos
            torch.cuda.empty_cache()
        if "d" in todo:
            cat = lognormal(1e8, 1024.)
            groups = FOF(cat, 0.2, 20).find_features()
            groups['Position'] = groups['CMPosition']
            del cat
            torch.cuda.empty_cache()
            edges = np.geomspace(1., 100., 21)
            r, totals, stages = time_calls(lambda: SimulationBox2PCF('1d', groups, edges), a.repeat)
            record("d_fof_groups_1d", int(groups.csize), totals, stages,
                   stencil_evaluations(_pos(groups), 1024., 100.), int(r.D1D2['npairs'].sum()), {}, out)


if __name__ == "__main__":
    main()
