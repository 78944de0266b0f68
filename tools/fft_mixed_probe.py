"""
Per-pass timing of the 3-D r2c on the B200: z, y and x passes and the whole transform, through whichever
implementation the mesh size selects (power of two: fft.cu; otherwise the mixed-radix fft_mixed.cu); power-of-two sizes
are also timed through the mixed-radix entry points for context.  CUDA events, 2 warm-up calls, best of 5; every field
is larger than the 126 MB L2.  Each result is reported against the 4 x field-bytes roofline (one read + one write of
the real field and of the complex field, ~4 x N^3 x sizeof(real)) at the measured 6.58 TB/s copy bandwidth.
Optionally (--fftpower) times FFTPower(cat, Nmesh=...) end to end on the C2 catalogue (1e8 log-normal particles).

    python tools/fft_mixed_probe.py [--out DIR] [--fftpower]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nbodykit_b200._lib import lib, check, iarr, F4, F8      # noqa: E402

COPY_BW = 6.58e12           # bytes/s, the project's measured device-to-device copy rate (profiles/r02_fft.md)
CASES = [(384, "f8", "auto"), (768, "f8", "auto"), (1536, "f8", "auto"), (768, "f4", "auto"),
         (512, "f8", "auto"), (512, "f8", "mixed"), (1024, "f8", "auto"), (1024, "f8", "mixed")]


def _best(fn, n=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def probe(N, dtype, impl):
    code = F8 if dtype == "f8" else F4
    rt, ct = (torch.float64, torch.complex128) if dtype == "f8" else (torch.float32, torch.complex64)
    Nzc = N // 2 + 1
    real = torch.randn((N, N, N), dtype=rt, device="cuda")
    cplx = torch.empty((N, N, Nzc), dtype=ct, device="cuda")
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    pow2 = (N & (N - 1)) == 0
    mixed = impl == "mixed" or not pow2
    L = lib()
    if mixed:
        z = lambda: check(L.nbk_fft_mr_z(p(real), p(cplx), code, N * N, N, 0, 1.0, s), "z")
        y = lambda: check(L.nbk_fft_mr_lines(p(cplx), p(cplx), code, N, Nzc, Nzc, N, N * Nzc, 0, 1.0, s), "y")
        x = lambda: check(L.nbk_fft_mr_lines(p(cplx), p(cplx), code, N, N * Nzc, N * Nzc, 1, 0, 0, 1.0, s), "x")
        whole = lambda: check(L.nbk_r2c_mr(p(real), p(cplx), code, iarr([N] * 3), 1.0, s), "r2c_mr")
    else:
        z = lambda: check(L.nbk_fft_z_forward(p(real), p(cplx), code, N * N, N, s), "z")
        y = lambda: check(L.nbk_fft_lines(p(cplx), code, N, Nzc, Nzc, N, N * Nzc, 0, 1.0, s), "y")
        x = lambda: check(L.nbk_fft_lines(p(cplx), code, N, N * Nzc, N * Nzc, 1, 0, 0, 1.0, s), "x")
        whole = lambda: check(L.nbk_r2c(p(real), p(cplx), code, iarr([N] * 3), 1.0, s), "r2c")
    t = dict(z=_best(z), y=_best(y), x=_best(x), r2c=_best(whole))
    field = real.numel() * real.element_size()
    bound_ms = 4 * field / COPY_BW * 1e3
    out = dict(mesh="%d^3" % N, dtype=dtype, impl="mixed-radix" if mixed else "power-of-two", field_GB=field / 1e9,
               bound_4x_ms=bound_ms, ms={k: round(v, 3) for k, v in t.items()},
               share_of_4x_bound=round(bound_ms / t["r2c"], 3),
               pass_share_of_2x_bound={k: round(0.5 * bound_ms / t[k], 3) for k in ("z", "y", "x")})
    del real, cplx
    torch.cuda.empty_cache()
    return out


def fftpower_c2(nmeshes, steps=3):
    import bench
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.lab import ArrayCatalog, FFTPower
    cfg = bench.CONFIGS["c2"]
    pos = bench.generate(cfg)
    res = []
    for n in nmeshes:
        def step():
            FFTPower(ArrayCatalog({'Position': pos}, comm=SelfComm(), BoxSize=cfg["box"]), mode="1d", Nmesh=n)
        ms = _best(step, steps)
        res.append(dict(workload="FFTPower C2 (%.3g log-normal particles, L=%g, CIC f8, 1d)" % (pos.shape[0], cfg["box"]),
                        Nmesh=n, ms=round(ms, 2)))
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--fftpower", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("fft_mixed_probe needs a CUDA device")
    rows = [dict(card=card(), copy_bw_TBps=COPY_BW / 1e12)]
    print(json.dumps(rows[0]), flush=True)
    for N, dt, impl in CASES:
        rows.append(probe(N, dt, impl))
        print(json.dumps(rows[-1]), flush=True)
    if args.fftpower:
        for r in fftpower_c2([512, 768, 1024]):
            rows.append(r)
            print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "fft_mixed_probe.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
