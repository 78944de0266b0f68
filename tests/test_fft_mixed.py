"""Mixed-radix FFT (sides 2^a 3^b 5^c 7^d): argument validation of the new entry points and the transform selection of
ParticleMesh, without a GPU."""

import pytest

F4, F8 = 4, 8


@pytest.fixture(scope="module")
def L():
    from nbodykit_b200 import _build, _lib
    import os
    if not os.path.exists(_lib.LIB_PATH):
        _build.build()
    return _lib.lib()


def _err(L):
    return L.nbk_last_error()


@pytest.mark.parametrize("n", [11, 13, 22, 26, 9216, 16384, 1, 0])
def test_lines_reject_unsupported_lengths(L, n):
    assert L.nbk_fft_mr_lines(None, None, F8, n, 1, 4, 1, 0, 0, 1.0, None) == -1
    assert b"line length" in _err(L) and "7^d".encode() in _err(L)


def test_lines_reject_bad_dtype(L):
    assert L.nbk_fft_mr_lines(None, None, 3, 48, 1, 4, 1, 0, 0, 1.0, None) == -1 and b"dtype" in _err(L)


@pytest.mark.parametrize("n", [2, 3, 5, 7, 15, 45, 343, 768, 2187, 6000, 8000, 8192])
def test_lines_accept_smooth_lengths(L, n):
    """odd lengths included (a line pass is complex-to-complex); nothing to transform -> success without CUDA"""
    assert L.nbk_fft_mr_lines(None, None, F8, n, 1, 0, 1, 0, 0, 1.0, None) == 0
    assert L.nbk_fft_mr_lines(None, None, F4, n, 1, 4, 0, 0, 1, 1.0, None) == 0
    # with work to do, the size check passes and the call stops at the buffers
    assert L.nbk_fft_mr_lines(None, None, F8, n, 1, 4, 1, 0, 0, 1.0, None) == -1 and b"null buffer" in _err(L)


@pytest.mark.parametrize("nz", [15, 45, 7, 22, 26, 18432, 0])
def test_z_rejects_odd_or_unsupported(L, nz):
    assert L.nbk_fft_mr_z(None, None, F8, 4, nz, 0, 1.0, None) == -1
    assert b"Nz" in _err(L) and b"even" in _err(L)


def test_z_rejects_bad_dtype(L):
    assert L.nbk_fft_mr_z(None, None, 2, 4, 48, 0, 1.0, None) == -1 and b"dtype" in _err(L)


@pytest.mark.parametrize("nz", [2, 6, 30, 90, 768, 1000, 3000, 16384])
def test_z_accepts_even_smooth(L, nz):
    assert L.nbk_fft_mr_z(None, None, F8, 0, nz, 0, 1.0, None) == 0
    assert L.nbk_fft_mr_z(None, None, F4, 4, nz, 1, 1.0, None) == -1 and b"distinct buffers" in _err(L)


@pytest.mark.parametrize("fn", ["nbk_r2c_mr", "nbk_c2r_mr"])
@pytest.mark.parametrize("nmesh", [[12, 12, 15], [15, 12, 12], [12, 22, 12], [12, 12, 26], [9216, 12, 12],
                                   [12, 12, 18432], [0, 12, 12]])
def test_whole_mesh_rejects(L, fn, nmesh):
    from nbodykit_b200._lib import iarr
    f = getattr(L, fn)
    last = 1.0 if fn == "nbk_r2c_mr" else None
    assert f(None, None, F8, iarr(nmesh), last, None) == -1
    msg = _err(L)
    assert b"unsupported" in msg and "2^a·3^b·5^c·7^d".encode() in msg and b"every side even" in msg


@pytest.mark.parametrize("fn", ["nbk_r2c_mr", "nbk_c2r_mr"])
def test_whole_mesh_rejects_bad_dtype(L, fn):
    from nbodykit_b200._lib import iarr
    last = 1.0 if fn == "nbk_r2c_mr" else None
    assert getattr(L, fn)(None, None, 16, iarr([12, 12, 12]), last, None) == -1 and b"dtype" in _err(L)


@pytest.mark.parametrize("nmesh", [[12, 12, 12], [768, 768, 768], [8192, 8192, 16384], [2, 6, 1536], [64, 64, 64]])
def test_whole_mesh_accepts_valid_sizes_up_to_the_cuda_call(L, nmesh):
    """the size check passes; the first pass then refuses the null buffers before launching anything"""
    from nbodykit_b200._lib import iarr
    assert L.nbk_r2c_mr(None, None, F8, iarr(nmesh), 1.0, None) == -1 and b"distinct buffers" in _err(L)
    assert L.nbk_c2r_mr(None, None, F4, iarr(nmesh), None, None) == -1 and b"null buffer" in _err(L)


def test_power_of_two_entry_points_keep_their_domain(L):
    from nbodykit_b200._lib import iarr
    assert L.nbk_r2c(None, None, F8, iarr([12, 12, 12]), 1.0, None) == -1 and b"power of two" in _err(L)
    assert L.nbk_fft_lines(None, F8, 48, 1, 4, 1, 0, 0, 1.0, None) == -1 and b"power of two" in _err(L)


def test_hermitian_expand_takes_mixed_sides(L):
    from nbodykit_b200._lib import iarr
    assert L.nbk_hermitian_expand(None, None, F8, iarr([12, 12, 15]), None) == -1 and b"every side even" in _err(L)
    # a valid mixed size gets past the size check to the buffer check
    assert L.nbk_hermitian_expand(None, None, F8, iarr([12, 48, 30]), None) == -1 and b"distinct buffers" in _err(L)
    assert L.nbk_hermitian_expand(None, None, F8, iarr([1, 64, 64]), None) == -1 and b"distinct buffers" in _err(L)


@pytest.mark.parametrize("nmesh,mixed", [(64, False), ([1, 64, 64], False), ([16, 32, 4096], False), (48, True),
                                         ([64, 64, 96], True), ([768, 512, 512], True), (15, True)])
def test_transform_selection_by_mesh_size(nmesh, mixed):
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.pmesh.pm import ParticleMesh
    assert ParticleMesh(BoxSize=1.0, Nmesh=nmesh, comm=SelfComm()).mixed_fft is mixed
