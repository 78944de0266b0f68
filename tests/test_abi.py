"""The C-ABI library loads and exports every symbol include/nbk_b200.h declares (no GPU needed)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "nbk_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nbk_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from nbodykit_b200 import _build, _lib
    if not os.path.exists(_lib.LIB_PATH):
        _build.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), "libnbk_b200.so does not export %s" % n


def test_python_binding_covers_the_header():
    from nbodykit_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()


def test_version_and_error_calls_work_without_gpu():
    from nbodykit_b200 import _lib
    L = _lib.lib()
    assert L.nbk_version() >= 100
    assert L.nbk_launch_count() >= 0
    # argument validation happens before any CUDA call: a bad dtype is rejected with a message
    rc = L.nbk_fill(None, 3, 10, 0.0, None)
    assert rc == -1 and b"dtype" in L.nbk_last_error()
    rc = L.nbk_r2c(None, None, 8, _lib.iarr([12, 12, 12]), 1.0, None)
    assert rc == -1 and b"power of two" in L.nbk_last_error()


def test_missing_library_fails_loudly(monkeypatch):
    from nbodykit_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libnbk_b200.so")
    import pytest
    with pytest.raises(_lib.NbkError):
        _lib.lib()


def test_no_cpu_fallback_for_fields(monkeypatch):
    """creating a field without CUDA raises instead of silently computing on the host (a present device is hidden)"""
    import pytest
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    from nbodykit_b200 import _lib
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.pmesh.pm import ParticleMesh, RealField
    pm = ParticleMesh(BoxSize=1.0, Nmesh=8, dtype='f4', comm=SelfComm())
    with pytest.raises(_lib.NbkError):
        RealField(pm)


def test_product_never_imports_oracle():
    import subprocess
    out = subprocess.run(["grep", "-rlE", r"^\s*(from|import)\s+oracle|from oracle", os.path.join(ROOT, "nbodykit_b200")],
                         capture_output=True, text=True).stdout.strip()
    assert out == "", "product code imports the oracle: %s" % out


def test_binding_argument_counts_match_the_header():
    """every ctypes signature lists as many arguments as the prototype in include/nbk_b200.h (ABI drift guard)"""
    from nbodykit_b200 import _lib
    text = open(os.path.join(ROOT, "include", "nbk_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = dict(re.findall(r"\b(nbk_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S))
    assert sorted(protos) == sorted(_lib.SIGNATURES)
    for name, args in protos.items():
        args = args.strip()
        n = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
        assert n == len(_lib.SIGNATURES[name][0]), "%s: header has %d parameters, the binding %d" % (
            name, n, len(_lib.SIGNATURES[name][0]))


def test_range_exchange_entry_points_validate_before_cuda():
    """nbk_fft_lines_pack_range / nbk_slab_push_range reject bad sub-ranges, peers and dtypes without touching the GPU"""
    from nbodykit_b200 import _lib
    L = _lib.lib()
    ptrs = (ctypes.c_void_p * 2)(None, None)
    assert L.nbk_fft_lines_pack_range(None, None, 3, 64, 9, 8, 0, 8, 2, 0, 1.0, None) == -1 and b"dtype" in L.nbk_last_error()
    assert L.nbk_fft_lines_pack_range(None, None, 8, 48, 9, 8, 0, 8, 2, 0, 1.0, None) == -1 and b"line length" in L.nbk_last_error()
    assert L.nbk_fft_lines_pack_range(None, None, 8, 64, 9, 8, 6, 4, 2, 0, 1.0, None) == -1 and b"sub-range" in L.nbk_last_error()
    assert L.nbk_fft_lines_pack_range(None, None, 8, 64, 9, 8, 0, 8, 3, 0, 1.0, None) == -1 and b"peer count" in L.nbk_last_error()
    assert L.nbk_fft_lines_pack_range(None, None, 8, 64, 9, 8, 4, 0, 2, 0, 1.0, None) == 0          # empty part: nothing to do
    assert L.nbk_slab_push_range(None, ptrs, 8, 32, 8, 9, 0, 6, 4, 2, 0, None) == -1 and b"sub-range" in L.nbk_last_error()
    assert L.nbk_slab_push_range(None, ptrs, 8, 32, 8, 9, 0, 0, 8, 2, 5, None) == -1 and b"rank" in L.nbk_last_error()
    assert L.nbk_slab_push_range(None, ptrs, 8, 32, 8, 9, 0, 4, 0, 2, 0, None) == 0
