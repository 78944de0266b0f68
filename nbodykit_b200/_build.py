"""
Build libnbk_b200.so (sm_100a only) in-tree with nvcc.  `python -m nbodykit_b200._build`
or `__graft_entry__.build()`.  The built .so is git-ignored but travels with gpurun.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJDIR = os.path.join(CSRC, "build")
LIB = os.path.join(CSRC, "libnbk_b200.so")

# (source, extra flags).  paint/binning carry bit-exact index arithmetic, and paircount bins float64 separations that
# must equal the CPU oracle's: no FMA contraction there.
SOURCES = [
    ("core.cu", []),
    ("paint.cu", ["--fmad=false"]),
    ("fft.cu", []),
    ("fft_mixed.cu", []),
    ("binning.cu", ["--fmad=false"]),
    ("ylm.cu", []),
    ("route.cu", ["--fmad=false"]),
    ("fof.cu", []),
    ("paircount.cu", ["--fmad=false"]),
]
COMMON = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
          "-Xcompiler", "-fPIC", "-Xcompiler", "-O3"]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found; cannot build libnbk_b200.so")


def _stamp(path, flags):
    h = hashlib.sha1()
    for dep in [path, os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "fft_common.cuh"),
                os.path.join(CSRC, "cellscan.cuh"),
                os.path.join(CSRC, "ylm_table.inc"),
                os.path.join(HERE, "..", "include", "nbk_b200.h")]:
        with open(dep, "rb") as f:
            h.update(f.read())
    h.update(" ".join(flags).encode())
    return h.hexdigest()


def build(verbose=False, force=False):
    nvcc = _nvcc()
    os.makedirs(OBJDIR, exist_ok=True)
    objs = []
    jobs = []
    for src, extra in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        stampf = obj + ".stamp"
        flags = COMMON + extra
        stamp = _stamp(path, flags)
        old = open(stampf).read() if os.path.exists(stampf) else ""
        if force or not os.path.exists(obj) or old != stamp:
            cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            jobs.append((cmd, stampf, stamp))
        objs.append(obj)
    rebuilt = bool(jobs)
    if jobs:
        # the translation units are independent: compile them side by side (paint.cu alone takes ~90 s)
        from concurrent.futures import ThreadPoolExecutor

        def run(job):
            cmd, stampf, stamp = job
            if verbose:
                print(" ".join(cmd))
            subprocess.check_call(cmd)
            with open(stampf, "w") as f:
                f.write(stamp)
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            list(ex.map(run, jobs))
    if rebuilt or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
