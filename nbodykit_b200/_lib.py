"""
ctypes binding of libnbk_b200.so (the C ABI in include/nbk_b200.h).

There is NO fallback: if the library is missing or a call fails, this raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libnbk_b200.so")

F4, F8 = 4, 8
WINDOW = {"nnb": 1, "nearest": 1, "cic": 2, "tsc": 3, "pcs": 4}
COMP = {"CompensateCIC": 1, "CompensateTSC": 2, "CompensatePCS": 3,
        "CompensateCICShotnoise": 4, "CompensateTSCShotnoise": 5, "CompensatePCSShotnoise": 6}


class NbkError(RuntimeError):
    pass


_lib = None

_vp, _i, _i64, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
_pd = ctypes.POINTER(ctypes.c_double)
_pi64 = ctypes.POINTER(ctypes.c_int64)
_pi = ctypes.POINTER(ctypes.c_int)

# name -> argtypes; must list every symbol include/nbk_b200.h declares (checked by tests/test_abi.py)
SIGNATURES = {
    "nbk_version": ([], _i),
    "nbk_last_error": ([], ctypes.c_char_p),
    "nbk_launch_count": ([], _i64),
    "nbk_paint": ([_vp, _i, _i64, _vp, _i, _i, _d, _pd, _pi64, _i64, _i64, _vp, _i, _vp], _i),
    "nbk_paint_interlaced": ([_vp, _i, _i64, _vp, _i, _i, _pd, _pi64, _i64, _i64, _vp, _vp, _i, _vp], _i),
    "nbk_paint_tiled_supported": ([_pi64, _i64, _i], _i),
    "nbk_paint_tiled_workspace": ([_i64, _i, _i, _pi64, _i64], _i64),
    "nbk_paint_tiled": ([_vp, _i, _i64, _vp, _i, _i, _d, _pd, _pi64, _i64, _i64, _vp, _vp, _i, _vp, _i64, _i, _vp], _i),
    "nbk_route_count": ([_vp, _i, _i64, _d, _pd, _pi64, _i, _i, _vp, _vp, _vp], _i),
    "nbk_route_scatter": ([_vp, _i, _vp, _i, _vp, _i64, _i, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "nbk_cell_index": ([_vp, _i, _i64, _i, _d, _pd, _pi64, _vp, _vp], _i),
    "nbk_readout": ([_vp, _i, _vp, _i, _i64, _i, _d, _pd, _pi64, _i64, _i64, _vp, _i, _i, _vp], _i),
    "nbk_recon_displacement": ([_vp, _vp, _i, _pi64, _pd, _i, _i64, _i64, _i, _d, _d, _d, _pd, _vp], _i),
    "nbk_sum_w_w2": ([_vp, _i, _i64, _vp, _vp], _i),
    "nbk_r2c": ([_vp, _vp, _i, _pi64, _d, _vp], _i),
    "nbk_c2r": ([_vp, _vp, _i, _pi64, _vp, _vp], _i),
    "nbk_fft_zy_forward": ([_vp, _vp, _i, _i64, _i64, _i64, _vp], _i),
    "nbk_fft_zy_backward": ([_vp, _vp, _i, _i64, _i64, _i64, _vp], _i),
    "nbk_fft_lines": ([_vp, _i, _i64, _i64, _i64, _i64, _i64, _i, _d, _vp], _i),
    "nbk_fft_lines_oop": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _i64, _i, _d, _vp], _i),
    "nbk_fft_z_forward": ([_vp, _vp, _i, _i64, _i64, _vp], _i),
    "nbk_fft_mr_lines": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _i64, _i, _d, _vp], _i),
    "nbk_fft_mr_z": ([_vp, _vp, _i, _i64, _i64, _i, _d, _vp], _i),
    "nbk_r2c_mr": ([_vp, _vp, _i, _pi64, _d, _vp], _i),
    "nbk_c2r_mr": ([_vp, _vp, _i, _pi64, _vp, _vp], _i),
    "nbk_fft_lines_scatter": ([_vp, ctypes.POINTER(ctypes.c_void_p), _i, _i64, _i64, _i64, _i64, _i, _i, _d, _vp], _i),
    "nbk_transpose_pack": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _vp], _i),
    "nbk_transpose_unpack": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _vp], _i),
    "nbk_transpose_pack_back": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _vp], _i),
    "nbk_transpose_unpack_back": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _vp], _i),
    "nbk_compensate": ([_vp, _i, _i, _pi64, _i, _i64, _i64, _vp], _i),
    "nbk_interlace_combine": ([_vp, _vp, _i, _pi64, _pd, _i, _i64, _i64, _vp], _i),
    "nbk_power_bin": ([_vp, _vp, _i, _i, _d, _i, _pi64, _pd, _i, _i64, _i64, _i, _pd, _i, _pd, _i, _pd, _pi,
                       _i, _i, _i, _i, _i, _pd, _vp, _vp, _vp, _vp, _vp], _i),
    "nbk_power_bin2": ([_vp, _vp, _vp, _i, _i, _d, _i, _pi64, _pd, _i, _i64, _i64, _i, _pd, _i, _pd, _i, _pd, _pi,
                        _i, _i, _i, _i, _i, _pd, _vp, _vp, _vp, _vp, _vp], _i),
    "nbk_ylm_mul_complex_acc2": ([_vp, _vp, _vp, _i, _i, _i, _pi64, _pd, _i, _i64, _i64, _vp], _i),
    "nbk_hermitian_expand": ([_vp, _vp, _i, _pi64, _vp], _i),
    "nbk_hermitian_compress": ([_vp, _vp, _i, _i64, _i64, _vp], _i),
    "nbk_resample_complex": ([_vp, _vp, _i, _pi64, _pi64, _vp], _i),
    "nbk_fft_lines_pack": ([_vp, _vp, _i, _i64, _i64, _i64, _i, _i, _d, _vp], _i),
    "nbk_slab_push": ([_vp, ctypes.POINTER(ctypes.c_void_p), _i, _i64, _i64, _i64, _i64, _i, _i, _vp], _i),
    "nbk_fft_lines_pack_range": ([_vp, _vp, _i, _i64, _i64, _i64, _i64, _i64, _i, _i, _d, _vp], _i),
    "nbk_slab_push_range": ([_vp, ctypes.POINTER(ctypes.c_void_p), _i, _i64, _i64, _i64, _i64, _i64, _i64, _i, _i, _vp], _i),
    "nbk_ylm_mul_real": ([_vp, _vp, _i, _i, _i, _pi64, _pd, _pd, _i64, _i64, _vp], _i),
    "nbk_ylm_mul_complex_acc": ([_vp, _vp, _i, _i, _i, _pi64, _pd, _i, _i64, _i64, _vp], _i),
    "nbk_cross_power": ([_vp, _vp, _vp, _i, _i64, _d, _i, _vp], _i),
    "nbk_fof_workspace": ([_i64, _d, _pd, _pd, _pd, _pi64], _i64),
    "nbk_fof_bucket": ([_vp, _i, _i64, _d, _pd, _pd, _pd, _vp, _i64, _vp, _vp, _vp], _i),
    "nbk_fof_link": ([_vp, _i, _i64, _d, _pd, _pd, _pd, _vp, _i64, _vp, _vp], _i),
    "nbk_fof_compress": ([_vp, _i64, _vp, _vp, _vp], _i),
    "nbk_fof_minid": ([_vp, _i64, _vp, _i64, _vp, _vp, _vp], _i),
    "nbk_fof_reduce": ([_i, _vp, _i64, _vp, _i64, _vp, _i, _i, _vp, _pd, _vp, _vp, _i64, _vp, _vp, _vp, _vp], _i),
    "nbk_pc_workspace": ([_i64, _i64, _d, _pd, _pd, _pd, _pi64], _i64),
    "nbk_pc_stencil": ([_i64, _d, _pd, _pd, _pd, _vp], _i),
    "nbk_pc_bucket": ([_vp, _i, _vp, _i, _i64, _i64, _d, _pd, _pd, _pd, _vp, _i64, _vp, _vp, _vp, _vp, _vp], _i),
    "nbk_pc_count": ([_i, _pd, _i, _i, _d, _i, _d, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _pd, _pd, _pd,
                      _vp, _vp, _vp, _vp], _i),
    "nbk_fill": ([_vp, _i, _i64, _d, _vp], _i),
    "nbk_scale": ([_vp, _i, _i64, _d, _vp], _i),
    "nbk_axpy": ([_vp, _vp, _i, _i64, _d, _vp], _i),
    "nbk_sum": ([_vp, _i, _i64, _vp, _vp], _i),
}


def lib():
    """the loaded library; raises NbkError if it has not been built"""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NbkError("libnbk_b200.so not found at %s -- run `python -m nbodykit_b200._build` "
                           "(there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (args, res) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = res
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().nbk_last_error().decode("utf-8", "replace")
        raise NbkError("%s failed (%d): %s" % (what or "nbk call", rc, msg))


def darr(x):
    """3-vector of doubles as a ctypes array"""
    return (ctypes.c_double * len(x))(*[float(v) for v in x])


def iarr(x):
    return (ctypes.c_int64 * len(x))(*[int(v) for v in x])


def i32arr(x):
    return (ctypes.c_int * len(x))(*[int(v) for v in x])


def launch_count():
    return int(lib().nbk_launch_count())


# ---------------------------------------------------------------------------------------------
# optional per-stage device timing (CUDA events on the launching stream); used by bench.py to
# attribute time inside the timed region to individual kernels.  Off by default: zero overhead.
# ---------------------------------------------------------------------------------------------
class _Profiler(object):
    def __init__(self):
        self.enabled = False
        self.records = []
        # NBK_TRACE=1: additionally bracket every stage with a device synchronize and accumulate host wall time
        # (diagnosis only -- it serialises the pipeline)
        self.host = bool(os.environ.get("NBK_TRACE"))
        self.wall = {}

    def start(self):
        self.enabled = True
        self.records = []

    def stop(self):
        """synchronise and return {name: [ms, ...]}"""
        import torch
        self.enabled = False
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.records:
            out.setdefault(name, []).append(a.elapsed_time(b))
        self.records = []
        return out


profiler = _Profiler()


class stage(object):
    """with stage('paint'): ...  -- records a CUDA event pair when profiling is on"""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if profiler.host:
            import time
            import torch
            torch.cuda.synchronize()
            self.t0 = time.perf_counter()
        if profiler.enabled:
            import torch
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if profiler.enabled:
            self.b.record()
            profiler.records.append((self.name, self.a, self.b))
        if profiler.host:
            import time
            import torch
            torch.cuda.synchronize()
            w = profiler.wall.setdefault(self.name, [0.0, 0])
            w[0] += time.perf_counter() - self.t0
            w[1] += 1
        return False
