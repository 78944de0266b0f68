"""
Mixed-radix FFT (mesh sides 2^a 3^b 5^c 7^d) on the GPU: the line pass and the 3-D r2c / c2r against NumPy / SciPy in
f8 on the host, the transform selection of RealField / ComplexField, and the algorithms end to end on non-power-of-two
meshes against the CPU oracle.  Tolerances of the FFT checks follow test_gpu_kernels.test_r2c_c2r:
max |error| <= tol * rms(spectrum) * log2(size), tol = 1e-13 (f8) / 2e-6 (f4).
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import pmesh_oracle as po, convpower_oracle as co

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"f8": 1e-13, "f4": 2e-6}
RTOL = 1e-5


def _pm(N, L, dtype):
    from nbodykit_b200.pmesh.pm import ParticleMesh
    from nbodykit_b200.comm import SelfComm
    return ParticleMesh(BoxSize=L, Nmesh=N, dtype=dtype, comm=SelfComm())


def _within(got, want, tol, size):
    rms = np.sqrt((np.abs(want) ** 2).mean())
    err = np.abs(got - want).max()
    assert err <= tol * rms * np.log2(max(size, 2)), "max error %.3e, bound %.3e" % (err, tol * rms * np.log2(max(size, 2)))


# ---- 1. the strided line pass ----------------------------------------------------------------------------------------
LINE_SIZES = [2, 3, 5, 7, 6, 12, 45, 49, 60, 96, 105, 125, 343, 360, 384, 625, 768, 1000, 1536, 2187, 2401, 4096, 6000,
              8000]


@pytest.mark.parametrize("N", LINE_SIZES)
@pytest.mark.parametrize("dtype", ["f8", "f4"])
@pytest.mark.parametrize("inverse", [0, 1])
@pytest.mark.parametrize("inplace", [True, False])
def test_line_pass(cuda, N, dtype, inverse, inplace):
    """lines along the middle axis of [n_outer][N][stride], n_inner = 13 of `stride` columns: a ragged last tile for
    every tile width, n_outer = 2, padding columns that must stay untouched"""
    import torch
    from nbodykit_b200._lib import lib, check, F4, F8
    n_outer, n_inner, stride = 2, 13, 16
    rng = np.random.RandomState(N)
    x = (rng.standard_normal((n_outer, N, stride)) + 1j * rng.standard_normal((n_outer, N, stride)))
    ct = torch.complex128 if dtype == "f8" else torch.complex64
    src = torch.from_numpy(x).to(ct).to(cuda)
    x = src.cpu().numpy().astype("c16")                 # what the device holds
    dst = src if inplace else torch.full_like(src, 7.0)
    scale = 0.5
    check(lib().nbk_fft_mr_lines(ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(dst.data_ptr()), F8 if dtype == "f8" else F4,
                                 N, stride, n_inner, n_outer, N * stride, inverse, scale,
                                 ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "nbk_fft_mr_lines")
    got = dst.cpu().numpy()
    sub = x[:, :, :n_inner]
    want = scale * (np.fft.ifft(sub, axis=1) * N if inverse else np.fft.fft(sub, axis=1))
    _within(got[:, :, :n_inner], want, TOL[dtype], N)
    pad = x[:, :, n_inner:] if inplace else np.full_like(x[:, :, n_inner:], 7.0)
    np.testing.assert_array_equal(got[:, :, n_inner:], pad)
    if not inplace:
        np.testing.assert_array_equal(src.cpu().numpy(), x.astype(got.dtype))


# ---- 2. 3-D transforms through RealField / ComplexField ---------------------------------------------------------------
SHAPES = [[12, 12, 12], [48, 48, 48], [96, 60, 40], [6, 10, 14], [384, 8, 6], [8, 384, 10], [6, 8, 768], [8, 8, 3000],
          [2, 6, 1536]]


@pytest.mark.parametrize("N", SHAPES)
@pytest.mark.parametrize("dtype", ["f8", "f4"])
def test_r2c_c2r_mixed(cuda, N, dtype):
    from nbodykit_b200.pmesh.pm import RealField
    rng = np.random.RandomState(3)
    real = rng.standard_normal(N).astype(dtype)
    pm = _pm(N, 1.0, dtype)
    assert pm.mixed_fft
    f = RealField(pm)
    f[...] = real
    c = f.r2c()
    want = np.fft.rfftn(real.astype("f8")) / real.size
    got = c.numpy()
    assert got.shape == want.shape
    _within(got, want, TOL[dtype], real.size)
    back = c.c2r().numpy()
    assert np.abs(back - real).max() <= TOL[dtype] * 10 * np.log2(real.size)
    np.testing.assert_array_equal(c.numpy(), got)       # c2r preserves its input


@pytest.mark.parametrize("N", SHAPES[:4])
def test_complex_dtype_mesh_mixed(cuda, N):
    """dtype='c16': full spectrum (Hermitian completion) and back"""
    from nbodykit_b200.pmesh.pm import RealField
    real = np.random.RandomState(4).standard_normal(N)
    pm = _pm(N, 1.0, "c16")
    f = RealField(pm)
    f[...] = real
    c = f.r2c()
    want = np.fft.fftn(real) / real.size
    _within(c.numpy(), want, TOL["f8"], real.size)
    assert np.abs(c.c2r().numpy() - real).max() <= TOL["f8"] * 10 * np.log2(real.size)


def test_768_cubed_matches_scipy(cuda):
    import scipy.fft
    import torch
    from nbodykit_b200.pmesh.pm import RealField
    N = [768, 768, 768]
    pm = _pm(N, 1.0, "f8")
    f = RealField(pm)
    g = torch.Generator(device=cuda)
    g.manual_seed(11)
    f.value.normal_(generator=g)
    real = f.numpy()
    got = f.r2c().numpy()
    want = scipy.fft.rfftn(real, workers=os.cpu_count())
    want /= real.size
    del real
    rms = np.sqrt(np.mean(np.abs(want) ** 2))
    err = max(float(np.abs(got[i:i + 64] - want[i:i + 64]).max()) for i in range(0, N[0], 64))
    assert err <= TOL["f8"] * rms * np.log2(768 ** 3)


@pytest.mark.parametrize("N", [[64, 64, 64], [16, 32, 64], [256, 256, 256]])
@pytest.mark.parametrize("dtype", ["f8", "f4"])
def test_mixed_entry_points_agree_with_power_of_two_transform(cuda, N, dtype):
    import torch
    from nbodykit_b200._lib import lib, check, iarr, F4, F8
    code = F8 if dtype == "f8" else F4
    rt, ct = (torch.float64, torch.complex128) if dtype == "f8" else (torch.float32, torch.complex64)
    g = torch.Generator(device=cuda)
    g.manual_seed(2)
    real = torch.randn(N, generator=g, dtype=rt, device=cuda)
    shape_c = (N[0], N[1], N[2] // 2 + 1)
    a, b = torch.empty(shape_c, dtype=ct, device=cuda), torch.empty(shape_c, dtype=ct, device=cuda)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    check(lib().nbk_r2c(p(real), p(a), code, iarr(N), 1.0, s), "nbk_r2c")
    check(lib().nbk_r2c_mr(p(real), p(b), code, iarr(N), 1.0, s), "nbk_r2c_mr")
    want = a.cpu().numpy().astype("c16")
    _within(b.cpu().numpy(), want, TOL[dtype], real.numel())
    r1, r2, w = torch.empty_like(real), torch.empty_like(real), torch.empty_like(a)
    check(lib().nbk_c2r(p(a), p(r1), code, iarr(N), p(w), s), "nbk_c2r")
    check(lib().nbk_c2r_mr(p(a), p(r2), code, iarr(N), p(w), s), "nbk_c2r_mr")
    assert float((r1 - r2).abs().max()) <= TOL[dtype] * 10 * np.log2(real.numel()) * float(real.abs().max())


# ---- 3. transform selection -----------------------------------------------------------------------------------------
class _Recorder(object):
    def __init__(self, L):
        self._L, self.calls = L, []

    def __getattr__(self, name):
        fn = getattr(self._L, name)
        if name.startswith("nbk_"):
            self.calls.append(name)
        return fn


@pytest.mark.parametrize("N,mixed", [([32, 32, 32], False), ([16, 8, 64], False), ([48, 48, 48], True),
                                     ([32, 32, 48], True), ([24, 32, 32], True)])
def test_path_selection(cuda, monkeypatch, N, mixed):
    from nbodykit_b200 import _lib
    from nbodykit_b200.pmesh import pm as pmmod
    rec = _Recorder(_lib.lib())
    monkeypatch.setattr(pmmod, "lib", lambda: rec)
    monkeypatch.setattr(_lib, "lib", lambda: rec)
    f = pmmod.RealField(_pm(N, 1.0, "f8"))
    f[...] = 1.0
    f.r2c().c2r()
    mr = [c for c in rec.calls if "_mr" in c]
    if mixed:
        assert "nbk_r2c_mr" in rec.calls and "nbk_c2r_mr" in rec.calls
        assert "nbk_r2c" not in rec.calls and "nbk_c2r" not in rec.calls
    else:
        assert "nbk_r2c" in rec.calls and "nbk_c2r" in rec.calls and mr == []


# ---- 4. algorithms end to end against the CPU oracle -------------------------------------------------------------------
def _compare_power(r, o, dtype, poles, interlaced):
    assert np.array_equal(r.power['modes'], np.squeeze(o['modes']))
    np.testing.assert_allclose(r.power['k'], np.squeeze(o['k']), rtol=RTOL, equal_nan=True)
    scale = np.nanmax(np.abs(o['poles_power'][0])) if poles else np.nanmax(np.abs(o['power']))
    # wedges / ell > 0 are sums with cancellations: errors are measured against the monopole.  The oracle forms the
    # compensation factors from float32 coordinates (the reference's dtype flow), the kernel in f8; for the steep
    # CompensateTSC of an interlaced mesh that alone moves the oracle's P by up to 7e-7 of the monopole (f8 fields)
    atol = {(False, "f8"): 1e-7, (True, "f8"): 1e-6, (False, "f4"): 1e-5, (True, "f4"): 3e-5}[interlaced, dtype] * scale
    np.testing.assert_allclose(np.nan_to_num(r.power['power'].real), np.nan_to_num(np.squeeze(o['power']).real),
                               rtol=RTOL, atol=atol)
    if 'mu' in r.power and np.ndim(o['mu']) == 2:
        np.testing.assert_allclose(r.power['mu'], o['mu'], rtol=RTOL, atol=1e-7, equal_nan=True)
    if poles:
        assert np.array_equal(r.poles['modes'], o['poles_modes'])
        for i, ell in enumerate(poles):
            np.testing.assert_allclose(np.nan_to_num(r.poles['power_%d' % ell].real), np.nan_to_num(o['poles_power'][i].real),
                                       rtol=RTOL, atol=atol)


@pytest.mark.parametrize("Nmesh", [48, [48, 60, 40]])
@pytest.mark.parametrize("resampler,interlaced", [("cic", False), ("tsc", True)])
@pytest.mark.parametrize("dtype", ["f4", "f8"])
@pytest.mark.parametrize("mode", ["1d", "2d"])
def test_fftpower_mixed_vs_oracle(cuda, Nmesh, resampler, interlaced, dtype, mode):
    from nbodykit_b200.lab import UniformCatalog, FFTPower
    # non-cubic boxes with cells of 8 x 10 x 6 length units
    L = [384., 480., 288.] if np.isscalar(Nmesh) else [384., 600., 240.]
    cat = UniformCatalog(nbar=3e-4, BoxSize=L, seed=42)
    mesh = cat.to_mesh(Nmesh=Nmesh, resampler=resampler, interlaced=interlaced, compensated=True, dtype=dtype)
    kw = dict(Nmu=5, poles=[0, 2, 4]) if mode == "2d" else {}
    r = FFTPower(mesh, mode=mode, **kw)
    pos, _ = po.uniform_catalog(3e-4, L, 42)
    o = po.fftpower(pos, Nmesh, L, mode=mode, resampler=resampler, interlaced=interlaced, compensated=True, dtype=dtype,
                    **kw)
    assert r.attrs['N1'] == len(pos) and r.attrs['N2'] == len(pos)
    _compare_power(r, o, dtype, kw.get("poles", []), interlaced)


def test_fftcorr_mixed_vs_oracle(cuda):
    from nbodykit_b200.lab import UniformCatalog, FFTCorr
    N, L = 48, 256.
    cat = UniformCatalog(nbar=1e-3, BoxSize=L, seed=11)
    mesh = cat.to_mesh(Nmesh=N, dtype='f8', resampler='cic', compensated=True)
    r = FFTCorr(mesh, mode='2d', Nmu=4, poles=[0, 2])
    pos, _ = po.uniform_catalog(1e-3, L, 11)
    real, _ = po.paint_field(pos, N, L, 'cic', dtype='f8')
    c = po.compensate('CompensateCICShotnoise', po.k_coords(N, L, 'f4', kind='circular'), po.r2c(real))
    p3d = c * np.conj(c)
    p3d[0, 0, 0] = 0
    xi = po.c2r(p3d * L ** 3, N) / L ** 3
    dr = L / N
    res, pres = po.project_to_basis(xi, co.x_coords(N, L, 'f4'), [np.arange(0., 0.5 * L + dr / 2, dr), np.linspace(0, 1, 5)],
                                    poles=[0, 2], hermitian_symmetric=False)
    assert np.array_equal(r.corr['modes'], res[3])
    scale = np.nanmax(np.abs(res[2]))
    np.testing.assert_allclose(np.nan_to_num(r.corr['corr'].real), np.nan_to_num(res[2].real), rtol=1e-6, atol=1e-7 * scale)
    np.testing.assert_allclose(np.nan_to_num(r.poles['corr_2'].real), np.nan_to_num(pres[1][1].real), rtol=1e-6,
                               atol=1e-7 * scale)


NBAR = 3e-4


def _fkp():
    from nbodykit_b200.lab import UniformCatalog, FKPCatalog
    d = UniformCatalog(nbar=NBAR, BoxSize=512., seed=42)
    r = UniformCatalog(nbar=10 * NBAR, BoxSize=512., seed=84)
    for c in (d, r):
        c['Position'] = c['Position'] + np.array((1000., -300., 700.))
        c['NZ'] = NBAR
    d['Weight'] = np.random.RandomState(5).uniform(0.8, 1.2, size=d.size)
    return FKPCatalog(d, r, P0=1e4), d, r


@pytest.mark.parametrize("dtype", ["f8", "c16"])
def test_convolved_power_mixed_vs_oracle(cuda, dtype):
    from nbodykit_b200.lab import ConvolvedFFTPower
    fkp, d, r = _fkp()
    mesh = fkp.to_mesh(Nmesh=48, dtype=dtype)
    ells = [0, 1, 2, 3, 4]
    res = ConvolvedFFTPower(mesh, poles=ells, dk=0.02)
    C, L = mesh.attrs['BoxCenter'], mesh.attrs['BoxSize']
    wfd = 1. / (1 + 1e4 * NBAR)
    args = (np.asarray(d['Position']), np.asarray(r['Position']),
            (np.asarray(d['Weight']), wfd * np.ones(d.size)), (np.ones(r.size), wfd * np.ones(r.size)),
            NBAR * np.ones(d.size), NBAR * np.ones(r.size), 48, L, C, ells)
    full = co.convpower_full(*args, dk=0.02)
    # an 'f8' mesh keeps the reference's Hermitian fold for the odd multipoles (convpower); even ones are the same
    herm = co.convpower(*args, dk=0.02) if dtype == "f8" else full
    assert np.array_equal(res.poles['modes'], full['modes'])
    np.testing.assert_allclose(res.poles['k'], full['k'], rtol=1e-6, equal_nan=True)
    scale = np.nanmax(np.abs(full['power_0']))
    for ell in ells:
        want = (herm if ell % 2 else full)['power_%d' % ell]
        got = res.poles['power_%d' % ell]
        for part in ('real', 'imag'):
            np.testing.assert_allclose(np.nan_to_num(getattr(got, part)), np.nan_to_num(getattr(want, part)), rtol=1e-5,
                                       atol=2e-6 * scale)


@pytest.mark.parametrize("N,M", [(64, 96), (96, 64)])
def test_resample_between_power_of_two_and_mixed(cuda, N, M):
    from nbodykit_b200.lab import ArrayMesh
    L = 64.

    def f(X, Y, Z):
        q = 2 * np.pi / L
        return 1.5 + np.cos(2 * q * X) * np.sin(3 * q * Y + 0.3) + 0.25 * np.cos(q * (X - 2 * Y + 4 * Z))
    x = np.arange(N) * (L / N)
    mesh = ArrayMesh(f(*np.meshgrid(x, x, x, indexing='ij')), BoxSize=L)
    xm = np.arange(M) * (L / M)
    got = mesh.compute(mode='real', Nmesh=M)
    assert got.value.shape == (M, M, M)
    np.testing.assert_allclose(got.numpy(), f(*np.meshgrid(xm, xm, xm, indexing='ij')), rtol=0, atol=1e-12)


def test_lognormal_catalog_on_a_mixed_mesh(cuda):
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.cosmology import NoWiggleEHPower
    from nbodykit_b200.lab import FFTPower
    from nbodykit_b200.source.catalog.lognormal import LogNormalCatalog
    Plin = NoWiggleEHPower()
    cat = LogNormalCatalog(Plin=Plin, nbar=2e-3, BoxSize=1024., Nmesh=96, bias=2.0, seed=7, growth_rate=0.5, comm=SelfComm())
    r = FFTPower(cat, mode='1d', Nmesh=96, dk=0.01, kmin=0.01)
    k, P = r.power['k'], r.power['power'].real - r.attrs['shotnoise']
    sel = (k > 0.02) & (k < 0.06)
    ratio = P[sel] / (4.0 * np.asarray(Plin(k[sel])))
    assert 0.8 < np.average(ratio, weights=r.power['modes'][sel]) < 1.25


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
def test_shot_noise_chi2_on_a_mixed_mesh(cuda, resampler):
    """a compensated uniform catalogue has a flat shot-noise spectrum: reduced chi^2 of P(k) - 1/nbar below 1
    (the reference's aliasing test, algorithms/tests/test_fftpower.py, at Nmesh = 48)"""
    from nbodykit_b200.lab import UniformCatalog, FFTPower
    mesh = UniformCatalog(nbar=3e-4, BoxSize=512., seed=42).to_mesh(resampler=resampler, Nmesh=48, compensated=True)
    r = FFTPower(mesh, mode='1d', kmin=0.02)
    Pk = r.power['power'].real
    err = np.sqrt(2 * Pk ** 2 / r.power['modes'])
    assert (((Pk - r.attrs['shotnoise']) / err) ** 2).sum() / len(Pk) < 1.0


# ---- 5. x slabs on several ranks --------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,dtype", [([96, 60, 40], "f8"), ([48, 48, 30], "f4")])
def test_slab_decomposed_transform_on_emulated_ranks(cuda, N, dtype):
    """the P > 1 route (z, y passes on the x slab, pack + all-to-all + unpack, x pass, and back) with two ranks
    emulated by two threads on one GPU: the transposed [y_n][Nx][Nzc] shares assemble to the one-GPU spectrum"""
    import threading
    import torch
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.pmesh.pm import ParticleMesh, RealField
    P = 2
    shared = dict(buf=[None] * P, bar=threading.Barrier(P))

    class ThreadComm(SelfComm):
        def __init__(self, rank):
            SelfComm.__init__(self)
            self._r = rank
        rank = property(lambda self: self._r)
        size = property(lambda self: P)

        def all_to_all_single(self, out, inp, out_splits=None, in_splits=None):
            torch.cuda.synchronize()
            shared["buf"][self._r] = inp
            shared["bar"].wait()
            n = inp.numel() // P
            out.copy_(torch.cat([shared["buf"][q].reshape(-1)[self._r * n:(self._r + 1) * n] for q in range(P)]))
            torch.cuda.synchronize()
            shared["bar"].wait()

    full = np.random.RandomState(9).standard_normal(N).astype(dtype)
    res, errs = [None] * P, []

    def rank_main(r):
        try:
            torch.cuda.set_device(cuda)
            pm = ParticleMesh(BoxSize=1.0, Nmesh=N, dtype=dtype, comm=ThreadComm(r))
            assert pm.mixed_fft and pm.transposed
            f = RealField(pm)
            f[...] = full[pm.x_start:pm.x_start + pm.x_n]
            c = f.r2c()
            res[r] = (c.numpy(), c.c2r().numpy())
        except Exception as e:      # noqa: BLE001
            errs.append(e)
            shared["bar"].abort()
    th = [threading.Thread(target=rank_main, args=(r,)) for r in range(P)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]
    got = np.concatenate([x[0] for x in res], axis=0).transpose(1, 0, 2)
    _within(got, np.fft.rfftn(full.astype("f8")) / full.size, TOL[dtype], full.size)
    back = np.concatenate([x[1] for x in res], axis=0)
    assert np.abs(back - full).max() <= TOL[dtype] * 10 * np.log2(full.size)


# ---- 6. two GPUs ------------------------------------------------------------------------------------------------------
def test_two_gpu_mixed_sizes_match_one_gpu():
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "mgpu_mixed_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(out.stdout[-3000:])
    sys.stderr.write(out.stderr[-3000:])
    assert out.returncode == 0
