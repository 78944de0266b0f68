#!/usr/bin/env python
"""
bench.py -- the FFTPower hot path on synthetic log-normal particles.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--order sorted|random]
                  [--dump-outputs DIR]

One "step" = one full FFTPower(...) / ConvolvedFFTPower(...) call on already-materialised particle columns:
paint -> r2c -> compensate -> |delta(k)|^2 V -> binning -> BinnedStatistic on the host.

Configurations (BASELINE.json / SURVEY.md 8d):
  headline (default)  LogNormal 1e9 f4 particles, L = 2048 -> 1024^3 f8 mesh, CIC, FFTPower 1d   -- the metric's config
  c2                  LogNormal 1e8, L = 1024 -> 512^3 f8, CIC, 1d                                  (configs[1])
  c3                  LogNormal 1e9 -> 1024^3 f4, TSC interlaced, 1d                                (configs[2])
  c4                  LogNormal 1e9 -> 1024^3 f8, CIC, mode='2d' Nmu=5                              (configs[3])
  c5                  FKP 1e8 data + 1e8 randoms -> 1024^3 f8, ConvolvedFFTPower poles 0,2,4        (configs[4])
`--gpus N` runs the SAME global problem on N x-slabs (strong scaling): rank r holds the r-th contiguous 1/N of the
generator's cell-ordered output (what the reference's generators leave on rank r), or of a random permutation
(`--order random`); decompose / exchange / ghosts run inside every step.

Prints ONE JSON line (rank 0).  `value` = particles/s through the whole step with columns resident in HBM; `e2e` = the
same call fed from pinned HOST arrays (H2D inside the timed region); `parity` = the result of the timed configuration
checked against an independent evaluation (N > 1: the single-GPU result on the gathered catalogue; N = 1: the same
catalogue in randomly permuted order, i.e. through the other bucketing configuration).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: particles, BoxSize, Nmesh, generator Nmesh, mesh dtype, resampler, interlaced, mode, Nmu, poles
    "headline": dict(npart=1.0e9, box=2048.0, nmesh=1024, gen=512, dtype="f8", resampler="cic", interlaced=False, mode="1d"),
    "c2": dict(npart=1.0e8, box=1024.0, nmesh=512, gen=256, dtype="f8", resampler="cic", interlaced=False, mode="1d"),
    "c3": dict(npart=1.0e9, box=2048.0, nmesh=1024, gen=512, dtype="f4", resampler="tsc", interlaced=True, mode="1d"),
    "c4": dict(npart=1.0e9, box=2048.0, nmesh=1024, gen=512, dtype="f8", resampler="cic", interlaced=False, mode="2d", Nmu=5),
    "c5": dict(npart=1.0e8, box=2048.0, nmesh=1024, gen=256, dtype="f8", resampler="cic", interlaced=False, mode="fkp",
               poles=[0, 2, 4]),
}
DESCR = {
    "headline": "LogNormal %.3g particles (f4) -> %d^3 mesh CIC f8 compensated, FFTPower mode=1d (BASELINE metric: 1024^3)",
    "c2": "LogNormal %.3g particles (f4) -> %d^3 mesh CIC f8 compensated, FFTPower mode=1d (BASELINE configs[1])",
    "c3": "LogNormal %.3g particles (f4) -> %d^3 mesh TSC interlaced f4 compensated, FFTPower mode=1d (BASELINE configs[2])",
    "c4": "LogNormal %.3g particles (f4) -> %d^3 mesh CIC f8, FFTPower mode=2d Nmu=5 (BASELINE configs[3])",
    "c5": "FKP %.3g data (log-normal) + as many uniform randoms -> %d^3 mesh f8, ConvolvedFFTPower poles 0,2,4 (BASELINE configs[4])",
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(config):
    """DRAM bytes per paint call from the committed ncu summary (profiles/r02_paint_traffic.json), or (None, None)"""
    p = os.path.join(ROOT, "profiles", "r02_paint_traffic.json")
    try:
        d = json.load(open(p))
        e = d[config]
        return float(e["dram_bytes"]), "profiles/r02_paint_traffic.json <- " + e["source"]
    except Exception:
        return None, None


class ClockSampler(object):
    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = [float(r[1]) for r in rows]
        pw = [float(r[3]) for r in rows if r[3].strip().replace(".", "").isdigit()]
        if pw:      # samples under load: upper half of the power draw
            thr = 0.5 * (max(pw) + min(pw))
            load = [s for s, r in zip(sm, rows) if float(r[3]) >= thr] or sm
        else:
            load = sm
        out["sm_mhz"] = float(np.median(load))
        out["sm_max_mhz"] = float(rows[0][2])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for j, n in enumerate(names):
            if any("Active" == r[5 + j].strip() for r in rows):
                out["reasons"].append(n)
        out["samples"] = len(rows)
        return out


def bind_to_gpu_numa(local):
    """pin this process (and so the pinned host buffers it first-touches) to the CPU cores next to its GPU: with one
    rank per GPU the H2D copies of the e2e leg then never cross the socket interconnect"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1 and 64 * i + b < ncpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


def generate(cfg, seed=42):
    """the config's particles on the current GPU (device float32 positions in the generator's cell order)"""
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.cosmology import NoWiggleEHPower
    from nbodykit_b200.source.catalog.lognormal import LogNormalCatalog
    import torch
    nbar = cfg["npart"] / cfg["box"] ** 3
    cat = LogNormalCatalog(Plin=NoWiggleEHPower(), nbar=nbar, BoxSize=cfg["box"], Nmesh=cfg["gen"], bias=2.0, seed=seed,
                           comm=SelfComm())
    pos = cat['Position'].compute()
    del cat
    torch.cuda.empty_cache()
    return pos


def fkp_columns(pos, cfg, device=True):
    """C5: data = the log-normal particles seen by an off-origin observer, randoms = as many uniform points"""
    import torch
    n = int(pos.shape[0])
    g = torch.Generator(device=pos.device)
    g.manual_seed(4242)
    ran = torch.rand((n, 3), device=pos.device, dtype=torch.float32, generator=g) * float(cfg["box"])
    off = torch.tensor([500.0, 300.0, 1500.0], device=pos.device)      # observer at the origin, box centre off-axis
    nbar = n / cfg["box"] ** 3
    return pos + off, ran + off, nbar, (off.cpu().numpy() + 0.5 * cfg["box"])


def make_step(cfg, comm, cols):
    """the timed call for a config on the given columns (device tensors or pinned host tensors)"""
    from nbodykit_b200.lab import ArrayCatalog, FFTPower
    Nmesh, Box = cfg["nmesh"], cfg["box"]
    if cfg["mode"] == "fkp":
        from nbodykit_b200.lab import ConvolvedFFTPower, FKPCatalog
        dpos, rpos, nbar, center = cols

        def step():
            d = ArrayCatalog({'Position': dpos}, comm=comm)
            r = ArrayCatalog({'Position': rpos}, comm=comm)
            for c in (d, r):
                c['NZ'] = nbar
                c['FKPWeight'] = 1.0 / (1.0 + 1e4 * nbar)
            fkp = FKPCatalog(d, r)
            mesh = fkp.to_mesh(Nmesh=Nmesh, BoxSize=Box, BoxCenter=center, dtype=cfg["dtype"], resampler=cfg["resampler"])
            return ConvolvedFFTPower(mesh, poles=cfg["poles"], dk=2 * np.pi / Box, kmin=0.)
        return step
    pos = cols

    def step():
        c = ArrayCatalog({'Position': pos}, comm=comm, BoxSize=Box)
        if cfg["interlaced"] or cfg["resampler"] != "cic" or cfg["dtype"] != "f8":
            src = c.to_mesh(Nmesh=Nmesh, resampler=cfg["resampler"], interlaced=cfg["interlaced"], compensated=True,
                            dtype=cfg["dtype"])
            return FFTPower(src, mode=cfg["mode"], Nmu=cfg.get("Nmu", 5))
        return FFTPower(c, mode=cfg["mode"], Nmesh=Nmesh, Nmu=cfg.get("Nmu", 5))
    return step


def result_arrays(r, cfg):
    if cfg["mode"] == "fkp":
        p = r.poles
        return np.asarray(p['modes']), np.stack([np.asarray(p['power_%d' % l]) for l in cfg["poles"]])
    return np.asarray(r.power['modes']), np.asarray(r.power['power'])


def dump_outputs(r, directory):
    """what a caller of the timed path receives, as DIR/<name>.npy: every column and the bin edges of the result's
    BinnedStatistics (power, poles) and its non-empty numeric attrs.  Complex columns are split into <name>.real / <name>.imag;
    float32 stays float32, everything else (integer mode counts included, exact below 2**53) becomes float64."""
    os.makedirs(directory, exist_ok=True)
    out = {}
    for which in ("power", "poles"):
        stat = getattr(r, which, None)
        if stat is None:
            continue
        for v in stat.variables:
            a = np.asarray(stat[v])
            if np.iscomplexobj(a):
                out["%s.%s.real" % (which, v)], out["%s.%s.imag" % (which, v)] = a.real, a.imag
            else:
                out["%s.%s" % (which, v)] = a
        for d in stat.dims:
            out["%s.edges.%s" % (which, d)] = stat.edges[d]
    for k, v in r.attrs.items():
        a = np.asarray(v)
        if a.dtype.kind in "iuf" and a.size:        # numbers only; an empty setting (poles=[]) is no output
            out["attrs.%s" % k] = a
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def compare(a, b, tol):
    ma, pa = a
    mb, pb = b
    ok_modes = bool(np.array_equal(ma, mb))
    with np.errstate(invalid="ignore", divide="ignore"):
        ref = np.nanmax(np.abs(pb))
        err = float(np.nanmax(np.abs(pa - pb)) / ref) if ref > 0 else 0.0
    return {"ok": bool(ok_modes and err <= tol), "modes_equal": ok_modes, "max_rel_dP": err, "tol": tol}


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        bind_to_gpu_numa(local)
    # keep stdout clean for the ONE JSON line: libraries (e.g. the NCCL version banner) write to fd 1 directly
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from nbodykit_b200 import CurrentMPIComm, _lib
    from nbodykit_b200.comm import SelfComm
    comm = CurrentMPIComm.get()
    assert comm.size == world
    cfg = dict(CONFIGS[args.config])
    if args.npart:
        cfg["npart"] = float(args.npart)
    Nmesh, Box = cfg["nmesh"], cfg["box"]

    # every rank generates the same catalogue (same seed, same device type) and keeps its contiguous 1/N of it
    full = generate(cfg, seed=42)
    n_total = int(full.shape[0])
    if args.order == "random":
        g = torch.Generator(device=full.device)
        g.manual_seed(45)
        full = full[torch.randperm(n_total, device=full.device, generator=g)].contiguous()
    lo, hi = (n_total * rank) // world, (n_total * (rank + 1)) // world
    keep_full = (world > 1 and rank == 0 and not args.no_parity)
    if cfg["mode"] == "fkp":
        fc = fkp_columns(full, cfg)             # data + randoms of the whole problem, then this rank's share of both
        cols = (fc[0][lo:hi].contiguous(), fc[1][lo:hi].contiguous(), fc[2], fc[3]) if world > 1 else fc
        full_cols = fc if keep_full else None
        pos = cols[0]
        del fc
    else:
        pos = full[lo:hi].contiguous() if world > 1 else full
        cols = pos
        full_cols = full if keep_full else None
    del full
    n_local = int(pos.shape[0])
    step = make_step(cfg, comm, cols)
    n_count = n_total * (2 if cfg["mode"] == "fkp" else 1)       # particles painted per step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the clock sampler needs ~1 s to come up: start it before the warm-up
    sampler = ClockSampler(local) if rank == 0 else None
    t_w = time.time()
    nw = 0
    while nw < args.warmup or (time.time() - t_w < 1.5 and nw < 50):
        r = step()
        nw += 1
    barrier()

    l0 = _lib.launch_count()
    _lib.profiler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        r = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    stages = _lib.profiler.stop()
    if _lib.profiler.host and rank == 0:
        for k, (t, c) in sorted(_lib.profiler.wall.items()):
            sys.stderr.write("TRACE %-20s %8.3f ms/step (%d calls)\n" % (k, 1e3 * t / max(1, nw + args.steps), c))
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_step = float(tms.item()) / args.steps
    res_timed = result_arrays(r, cfg)
    if args.dump_outputs and rank == 0:
        dump_outputs(r, args.dump_outputs)

    # ---- e2e: same call, columns start in pinned host memory
    def pinned(t):
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        return h
    if cfg["mode"] == "fkp":
        hcols = (pinned(cols[0]), pinned(cols[1]), cols[2], cols[3])
        h2d = 2 * n_local * 12
    else:
        hcols = pinned(pos)
        h2d = n_local * 12
    step_host = make_step(cfg, comm, hcols)
    del cols, step
    if world > 1:
        del pos
    torch.cuda.empty_cache()
    step_host()
    barrier()
    e0.record()
    for _ in range(args.steps):
        rh = step_host()
    e1.record()
    barrier()
    tms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_e2e = float(tms.item()) / args.steps
    nb = len(np.ravel(res_timed[0]))
    d2h = int(np.asarray(res_timed[1]).nbytes + np.asarray(res_timed[0]).nbytes) + 8 * 3 * (nb + 2) * 3
    parity = {"e2e_equals_resident": compare(result_arrays(rh, cfg), res_timed, 1e-12)}
    del step_host, rh
    torch.cuda.empty_cache()

    # ---- parity of the timed configuration against an independent evaluation
    if not args.no_parity:
        if world > 1:
            if rank == 0:
                ref = result_arrays(make_step(cfg, SelfComm(), full_cols)(), cfg)
                parity["vs"] = "single-GPU evaluation of the gathered catalogue on rank 0"
                parity.update(compare(res_timed, ref, 2e-8))
                del full_cols
        else:
            if cfg["mode"] != "fkp":
                g = torch.Generator(device=pos.device)
                g.manual_seed(46)
                perm = torch.randperm(n_local, device=pos.device, generator=g)
                other = pos[perm].contiguous()
                del perm
                ref = result_arrays(make_step(cfg, comm, other)(), cfg)
                parity["vs"] = "the same catalogue in randomly permuted order (other bucketing configuration)"
                parity.update(compare(res_timed, ref, 2e-8))
                del other, pos
            else:
                parity["vs"] = "e2e only"
                parity.update(parity["e2e_equals_resident"])
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    hbm, which = peaks()
    per_step = {k: float(np.sum(v)) / args.steps for k, v in stages.items()}       # SUM of the records of a step
    paint_ms = per_step.get("paint", float('nan'))
    sf = 4 if cfg["dtype"] == "f4" else 8
    nmeshes = 2 if cfg["interlaced"] else 1
    mesh_cells = float(Nmesh) ** 3 / world
    npaint_local = n_local * (2 if cfg["mode"] == "fkp" else 1)
    alg_bytes = npaint_local * 12.0 + nmeshes * mesh_cells * sf    # particles read once + mesh(es) written once (DESIGN.md)
    if cfg["mode"] == "fkp":
        alg_bytes += mesh_cells * sf                               # data and randoms are two paints of one mesh each
    achieved = alg_bytes / (paint_ms * 1e-3) / 1e9
    traffic, traffic_src = committed_traffic(args.config if args.order == "sorted" else args.config + "_random") if world == 1 else (None, None)
    other = {}
    field_bytes = mesh_cells * sf
    cplx_bytes = mesh_cells / Nmesh * (Nmesh // 2 + 1) * 2 * sf
    if world == 1 and "r2c" in per_step and not cfg["interlaced"] and cfg["mode"] != "fkp":
        a = 4.0 * field_bytes / (per_step["r2c"] * 1e-3) / 1e9
        other["r2c"] = {"algorithmic_bytes": 4.0 * field_bytes, "kernel_ms": per_step["r2c"], "achieved": a, "frac": a / hbm}
    if world > 1 and "fft_y_scatter" in per_step:
        out_bytes = cplx_bytes * (world - 1) / world
        nv = out_bytes / (per_step["fft_y_scatter"] * 1e-3) / 1e9
        other["fft_y_scatter"] = {"nvlink_bytes_out": out_bytes, "kernel_ms": per_step["fft_y_scatter"], "achieved_GBps": nv,
                                  "peak_GBps": 770.0, "frac": nv / 770.0,
                                  "note": "fused y pass + peer-store transpose; peak = measured peer copy (B200_PROFILING.md)"}
    if "power_bin" in per_step and cfg["mode"] in ("1d", "2d"):
        a = cplx_bytes / (per_step["power_bin"] * 1e-3) / 1e9
        other["power_bin"] = {"algorithmic_bytes": cplx_bytes, "kernel_ms": per_step["power_bin"], "achieved": a, "frac": a / hbm}
    out = {
        "metric": "particles/sec painted + P(k) end-to-end, 1024^3 mesh" if Nmesh == 1024 else
                  "particles/sec painted + P(k) end-to-end",
        "value": n_count / (ms_step * 1e-3),
        "unit": "particles/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step,
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f64" if cfg["dtype"] == "f8" else "f32",
        "data": "synthetic",
        "config": {"workload": DESCR[args.config] % (n_total, Nmesh), "name": args.config,
                   "particles": n_count, "Nmesh": [Nmesh] * 3, "BoxSize": [Box] * 3, "resampler": cfg["resampler"],
                   "interlaced": cfg["interlaced"], "mesh_dtype": cfg["dtype"], "mode": cfg["mode"],
                   "particle_order": "generator (cell-ordered, Zel'dovich-displaced)" if args.order == "sorted" else "random permutation",
                   "l2": "inputs (%.1f GB particles, %.1f GB mesh per GPU) exceed the 126 MB L2; no flush needed"
                         % (n_local * 12 / 1e9, mesh_cells * sf / 1e9),
                   "parallelism": "x-slab x%d" % world,
                   "placement": "rank r holds the r-th contiguous 1/N of the particle array; decompose + exchange + ghosts run "
                                "inside every step"},
        "paint_particles_per_sec": n_count / (paint_ms * 1e-3),
        "pk_seconds": ms_step * 1e-3,
        "stage_ms": per_step,
        "e2e": {"value": n_count / (ms_e2e * 1e-3), "unit": "particles/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "parity": parity,
        "roofline": {"kernel": "paint = nbk_paint_tiled (k_bucket_probe, k_bucket_count, k_tile_scan*, k_bucket_scatter, "
                               "k_tile_paint, k_apply_deferred), all paint launches of a step summed" + ("; rank 0's slab" if world > 1 else ""),
                     "bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s",
                     "frac": achieved / hbm, "peak_source": which, "algorithmic_bytes": alg_bytes,
                     "kernel_ms": paint_ms, "traffic": traffic, "traffic_source": traffic_src,
                     "other_stages": other},
    }
    if world == 1 and not args.no_cpu:
        try:
            if cfg["mode"] in ("1d", "2d") and not cfg["interlaced"]:
                base = cpu_step(hcols.numpy(), cfg)
                o = base.pop("_result")
                base["sample"] = "ONE full step of this workload (every particle, full mesh): " + base["sample"]
                out["cpu_baseline"] = base
                # the oracle's result on the very same particles: parity of the timed GPU result at full size
                out["parity"]["vs_cpu_oracle"] = compare(res_timed, (np.squeeze(o["modes"]), np.squeeze(o["power"])), 1e-5)
                if not out["parity"]["vs_cpu_oracle"]["ok"]:
                    out["parity"]["ok"] = False
        except Exception as e:      # the baseline leg must never cost the bench line
            out["cpu_baseline"] = {"error": repr(e)}
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not parity.get("ok", True):
        sys.exit(3)


def cpu_step(pos, cfg, nproc=None, single=True):
    """one full step of the reference's CPU algorithm (oracle port) on all host cores: C/OpenMP restatement of the
    pmesh scatter over EVERY particle, scipy (pocketfft) r2c with all workers, and the mesh stages (compensation,
    |delta_k|^2 V, project_to_basis -- the reference's own per-slab NumPy code) spread over one process per core the
    way the reference spreads them over MPI ranks."""
    from oracle import build_c, parallel as opar, pmesh_oracle as po
    cores = os.cpu_count() or 1
    # mesh-stage workers are fork()ed from this process, which holds the catalogue, pinned buffers and a CUDA context: every
    # fork costs ~40-110 ms of page-table copying (measured on the 128-core GPU host: 128 workers were no faster than ONE
    # process, 4.88 s vs 4.85 s at 512^3).  24 workers balance that cost against the per-slab NumPy work.
    nproc = nproc or min(cores, int(os.environ.get("NBK_REF_PROCS", "24")))
    Nm = [cfg["nmesh"]] * 3
    Bx = [cfg["box"]] * 3
    n = len(pos)
    t0 = time.time()
    mesh = build_c.paint(pos, None, Nm, Bx, cfg["resampler"])
    t1 = time.time()
    mesh /= (n / float(np.prod(Nm)))
    c = po.r2c(mesh)
    del mesh
    t2 = time.time()
    comp = po.COMPENSATION[(cfg["interlaced"], cfg["resampler"])]
    res = opar.power_from_complex(c, None, Nm, Bx, mode=cfg["mode"], Nmu=cfg.get("Nmu", 5), compensation=comp, nproc=nproc)
    t3 = time.time()
    total = t3 - t0
    single = single_core_sample(pos, c, cfg, comp) if single else None
    return {"value": n / total, "unit": "particles/s", "cores": cores, "kind": "port", "seconds": total,
            "single_core": single,
            "paint_seconds": t1 - t0, "r2c_seconds": t2 - t1, "mesh_stage_seconds": t3 - t2,
            "paint_particles_per_sec": n / (t1 - t0), "omp_threads": os.environ.get("OMP_NUM_THREADS"),
            "processes_mesh_stages": nproc,
            "sample": "paint %d particles (C/OpenMP, %s threads) + normalise + r2c (scipy pocketfft, %d workers) + "
                      "compensate / power / project_to_basis (NumPy, %d processes over x-slabs) at %d^3"
                      % (n, os.environ.get("OMP_NUM_THREADS"), cores, nproc, cfg["nmesh"]),
            "_result": res}


def single_core_sample(pos, c, cfg, comp):
    """BASELINE.md 3: the single-core numbers next to the all-cores ones, on BOUNDED samples of the same workload (never
    part of `value`): the C scatter of the first 2e7 particles on one OpenMP thread, and the reference's per-slab NumPy
    mesh stages (compensation, |delta_k|^2 V, project_to_basis) of 4 x-planes in this process, scaled to the mesh."""
    out = {}
    try:
        import ctypes
        from oracle import build_c, parallel as opar
        Nm = [cfg["nmesh"]] * 3
        Bx = [cfg["box"]] * 3
        ns = int(min(len(pos), 2e7))
        gomp = None
        try:
            gomp = ctypes.CDLL("libgomp.so.1")
            gomp.omp_set_num_threads(1)
        except Exception:
            gomp = None
        t0 = time.time()
        build_c.paint(pos[:ns], None, Nm, Bx, cfg["resampler"])
        dt = time.time() - t0
        if gomp is not None:
            gomp.omp_set_num_threads(os.cpu_count() or 1)
        out["paint_particles_per_sec"] = ns / dt
        out["paint_threads"] = 1 if gomp is not None else None
        planes = min(4, c.shape[0])
        t0 = time.time()
        opar._G.update(c=c, c2=None, N=(np.asarray(Nm, dtype="i8")), L=np.asarray(Bx, dtype="f8"), comp=comp, coord_dtype="f4",
                       edges=[np.arange(0., np.pi * cfg["nmesh"] / cfg["box"] + np.pi / cfg["box"], 2 * np.pi / cfg["box"]),
                              np.linspace(-1, 1, (1 if cfg["mode"] == "1d" else cfg.get("Nmu", 5)) + 1)],
                       los=(0, 0, 1), poles=[])
        try:
            opar._worker((0, planes))
        finally:
            opar._G.clear()
        dt = time.time() - t0
        out["mesh_stage_seconds_projected"] = dt * c.shape[0] / planes
        out["sample"] = ("scatter of the first %d particles on 1 thread; mesh stages of %d of %d x-planes in one process, "
                         "scaled by the plane count" % (ns, planes, c.shape[0]))
    except Exception as e:      # a diagnostic, never worth the bench line
        out["error"] = repr(e)
    return out


def run_reference(args):
    """the reference's CPU algorithm for this path (oracle port: /root/reference needs pmesh + mpi4py, absent here),
    all host cores, on the FULL workload of the chosen config; the number of steps actually run is bounded by a time
    budget (steps are dropped, never work) and reported in `steps`."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch
    cfg = dict(CONFIGS[args.config])
    if args.npart:
        cfg["npart"] = float(args.npart)
    if cfg["mode"] == "fkp" or cfg["interlaced"]:
        print(json.dumps({"impl": "reference", "unavailable": "the CPU arm covers the FFTPower configs (headline, c2, c4)"}))
        return
    cache = os.path.join(tempfile.gettempdir(), "nbk_bench_%s_%d.npy" % (args.config, int(cfg["npart"])))
    if os.path.exists(cache):
        pos = np.load(cache, mmap_mode=None)
    elif torch.cuda.is_available():
        torch.cuda.set_device(0)
        pos = generate(cfg, seed=42).cpu().numpy()
        try:
            np.save(cache, pos)
        except Exception:
            pass
        torch.cuda.empty_cache()
    else:
        n = int(cfg["npart"])
        pos = (np.random.RandomState(42).uniform(size=(n, 3)) * cfg["box"]).astype("f4")
    budget = float(os.environ.get("NBK_REF_BUDGET_S", "200"))
    t_start = time.time()
    runs = []
    want = args.warmup + args.steps
    done_w = 0
    last = None
    for i in range(want):
        t0 = time.time()
        step_i = cpu_step(pos, cfg, single=(i == 0))
        if last is not None and step_i.get("single_core") is None:
            step_i["single_core"] = last.get("single_core")
        last = step_i
        dt = time.time() - t0
        if done_w < min(args.warmup, 1) and want > 1 and (time.time() - t_start) + 2 * dt < budget:
            done_w += 1                     # at most one warm-up pass (page faults, thread pools), only if affordable
            continue
        runs.append(dt)
        if (time.time() - t_start) + dt > budget:
            break
    n = len(pos)
    sec = float(np.mean(runs))
    last.pop("_result", None)
    last["value"] = n / sec
    last["steps_run"] = len(runs)
    last["sample"] = "FULL workload every step; %d of the %d requested steps fit the %.0f s budget: %s" % (
        len(runs), args.steps, budget, last["sample"])
    out = {"impl": "reference", "metric": "particles/sec painted + P(k) end-to-end, 1024^3 mesh" if cfg["nmesh"] == 1024
           else "particles/sec painted + P(k) end-to-end",
           "value": n / sec, "unit": "particles/s", "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": len(runs),
           "warmup": done_w, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": DESCR[args.config] % (n, cfg["nmesh"]), "name": args.config, "particles": n,
                      "Nmesh": [cfg["nmesh"]] * 3, "BoxSize": [cfg["box"]] * 3, "resampler": cfg["resampler"],
                      "interlaced": cfg["interlaced"], "mesh_dtype": cfg["dtype"], "mode": cfg["mode"]},
           "cpu_baseline": last,
           "e2e": {"value": n / sec, "unit": "particles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS))
    ap.add_argument("--order", default="sorted", choices=["sorted", "random"])
    ap.add_argument("--npart", type=float, default=None, help="override the particle count (scratch runs)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity self-check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/<name>.npy (inputs are seeded: two builds "
                         "run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        # all host threads, also under torchrun (which exports OMP_NUM_THREADS=1); must precede the first OpenMP load
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1) if int(os.environ.get("WORLD_SIZE", 1)) == 1 else os.environ.get("OMP_NUM_THREADS", "1")
        run_ours(args)


if __name__ == "__main__":
    main()
