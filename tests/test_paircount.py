"""Pair counting without a GPU: the argument errors of SimulationBoxPairCount / SimulationBox2PCF, attrs, total_wnpairs,
config validation, the nbk_pc_* rejections (no CUDA call is reached), the stencil, the CPU oracle against a brute-force
double loop, the estimators, wp, to_poles and a save/load round trip of a result built on the host."""
import ctypes

import numpy as np
import pytest

from oracle import paircount_oracle as po

F4, F8 = 4, 8


@pytest.fixture(scope="module")
def L():
    from nbodykit_b200 import _build, _lib
    import os
    if not os.path.exists(_lib.LIB_PATH):
        _build.build()
    return _lib.lib()


def _cat(n=100, box=100., seed=1, **cols):
    from nbodykit_b200 import CurrentMPIComm
    from nbodykit_b200.lab import ArrayCatalog
    rng = np.random.RandomState(seed)
    data = {'Position': rng.uniform(0, 100., size=(n, 3))}
    data.update(cols)
    return ArrayCatalog(data, comm=CurrentMPIComm.get(), **({'BoxSize': box} if box is not None else {}))


@pytest.fixture
def norun(monkeypatch):
    """pair counters without the GPU count"""
    from nbodykit_b200.algorithms import paircount
    monkeypatch.setattr(paircount.SimulationBoxPairCount, 'run', lambda self: None)
    return paircount.SimulationBoxPairCount


E = np.linspace(1., 20., 5)


def test_exported():
    from nbodykit_b200 import lab
    from nbodykit_b200.algorithms import SimulationBox2PCF, SimulationBoxPairCount
    assert lab.SimulationBoxPairCount is SimulationBoxPairCount and lab.SimulationBox2PCF is SimulationBox2PCF


@pytest.mark.parametrize("kw, match", [
    (dict(mode='bad'), "allowed 'mode' values"),
    (dict(edges=np.linspace(0, 10, 5)), "greater than zero"),
    (dict(mode='2d'), "'Nmu' keyword is required"),
    (dict(Nmu=5), "mode should be '2d'"),
    (dict(mode='projected'), "'pimax' keyword is required"),
    (dict(pimax=10.), "mode should be 'projected'"),
    (dict(mode='projected', pimax=0.5), "at least 1.0"),
    (dict(los='a'), "one of 'x', 'y', 'z'"),
    (dict(los=3), r"\[0,1,2\]"),
    (dict(los=[0, 0, 1]), r"\[0,1,2\]"),
    (dict(weight='BAD'), "the column 'BAD' is missing"),
    (dict(position='BAD'), "the column 'BAD' is missing"),
    (dict(edges=np.linspace(1, 60, 5)), "Rmax > BoxSize/2"),
    (dict(mode='projected', pimax=60.), "Rmax > BoxSize/2"),
    (dict(BoxSize=300.), "mismatch between sources and the pair count"),
    (dict(nthread=4), "unknown pair-count keyword"),
])
def test_argument_errors(norun, kw, match):
    args = dict(mode='1d', first=_cat(), edges=E)
    args.update(kw)
    with pytest.raises(ValueError, match=match):
        norun(**args)


def test_box_errors(norun):
    with pytest.raises(ValueError, match="BoxSize must be supplied"):
        norun('1d', _cat(box=None), E)
    with pytest.raises(ValueError, match="mismatch between pair count cross-correlation"):
        norun('1d', _cat(), E, second=_cat(box=50.))
    with pytest.raises(NotImplementedError, match="non-cubic"):
        norun('1d', _cat(box=[100., 100., 50.]), E)
    # non-periodic: a large separation and a non-cubic box are fine
    norun('1d', _cat(box=[100., 100., 50.]), np.linspace(1, 80, 4), periodic=False)
    norun('1d', _cat(box=None), E, periodic=False, BoxSize=100.)


def test_angular_not_implemented(norun):
    from nbodykit_b200.lab import SimulationBox2PCF
    for cls in (norun, SimulationBox2PCF):
        with pytest.raises(NotImplementedError, match="angular and survey pair counters are not implemented"):
            cls('angular', _cat(), E)


def test_los_forms(norun):
    assert norun('1d', _cat(), E, los='x').attrs['los'] == 0
    assert norun('1d', _cat(), E, los=-1).attrs['los'] == 2
    assert norun('1d', _cat(), E, los=np.int64(1)).attrs['los'] == 1


def test_attrs_and_totals(norun):
    rng = np.random.RandomState(2)
    w1, w2 = rng.uniform(size=100), rng.uniform(size=70)
    a = _cat(Weight=w1)
    b = _cat(n=70, seed=3, Weight=w2.astype('f4'))
    auto = norun('2d', a, E, Nmu=4, nthreads=8, isa='avx')
    assert set(auto.attrs) == {'mode', 'edges', 'Nmu', 'pimax', 'show_progress', 'N1', 'N2', 'total_wnpairs',
                               'is_cross', 'BoxSize', 'periodic', 'weight', 'position', 'config', 'los'}
    assert auto.attrs['config'] == {'nthreads': 8, 'isa': 'avx'}
    assert auto.attrs['is_cross'] is False and auto.attrs['N1'] == 100 and auto.attrs['N2'] is None
    np.testing.assert_allclose(auto.attrs['total_wnpairs'], po.total_wnpairs(w1), rtol=1e-12)
    same = norun('1d', a, E, second=a)
    assert same.attrs['is_cross'] is False and same.attrs['N2'] == 100
    np.testing.assert_allclose(same.attrs['total_wnpairs'], po.total_wnpairs(w1), rtol=1e-12)
    cross = norun('1d', a, E, second=b)
    assert cross.attrs['is_cross'] is True and cross.attrs['N2'] == 70
    np.testing.assert_allclose(cross.attrs['total_wnpairs'], po.total_wnpairs(w1, w2.astype('f4')), rtol=1e-6)
    np.testing.assert_array_equal(cross.attrs['BoxSize'], [100.] * 3)


def test_2pcf_errors():
    from nbodykit_b200.lab import SimulationBox2PCF
    with pytest.raises(ValueError, match="unknown pair-count keyword"):
        SimulationBox2PCF('1d', _cat(), E, bogus=1)
    with pytest.raises(ValueError, match="randoms must be specified"):
        SimulationBox2PCF('1d', _cat(), E, periodic=False)


# ---- the C ABI -----------------------------------------------------------------------------------------------------
def test_abi_rejections(L):
    box = (ctypes.c_double * 3)(100., 100., 100.)
    nc = (ctypes.c_int64 * 3)()
    assert L.nbk_pc_workspace(-1, 10, 5., box, None, None, nc) < 0
    assert b"row count" in L.nbk_last_error()
    assert L.nbk_pc_workspace(10, 10, 0., box, None, None, nc) < 0
    assert b"largest separation must be > 0" in L.nbk_last_error()
    assert L.nbk_pc_workspace(10, 10, 5., None, None, None, nc) < 0
    assert b"needs the data bounds" in L.nbk_last_error()
    assert L.nbk_pc_bucket(None, 2, None, F8, 0, 0, 5., box, None, None, None, 0, None, None, None, None, None) < 0
    assert b"position dtype 2 not accepted (4 = f4 or 8 = f8)" in L.nbk_last_error()
    assert L.nbk_pc_bucket(None, F8, None, 3, 0, 0, 5., box, None, None, None, 0, None, None, None, None, None) < 0
    assert b"weight dtype 3" in L.nbk_last_error()
    assert L.nbk_pc_bucket(None, F8, None, F8, 10, 10, 5., box, None, None, None, 0, None, None, None, None, None) < 0
    assert b"workspace of 0 bytes is too small" in L.nbk_last_error()
    e = (ctypes.c_double * 3)(1., 2., 3.)

    def count(mode=0, edges=e, nedges=3, nmu=0, pimax=0., los=2, rmax=3.):
        return L.nbk_pc_count(mode, edges, nedges, nmu, pimax, los, rmax, None, None, None, None, 0, None, None, None,
                              0, box, None, None, None, None, None, None)
    assert count(mode=3) < 0 and b"mode 3 not accepted (0 = 1d, 1 = 2d, 2 = projected)" in L.nbk_last_error()
    assert count(nedges=1) < 0 and b"separation edges not accepted" in L.nbk_last_error()
    assert count(edges=(ctypes.c_double * 3)(0., 2., 3.)) < 0 and b"lowest edge must be > 0" in L.nbk_last_error()
    assert count(edges=(ctypes.c_double * 3)(1., 3., 2.)) < 0 and b"increase strictly" in L.nbk_last_error()
    assert count(los=3) < 0 and b"line of sight 3" in L.nbk_last_error()
    assert count(mode=1, nmu=0) < 0 and b"2d mode needs 1 <= nmu" in L.nbk_last_error()
    assert count(mode=2, pimax=0.5) < 0 and b"projected mode needs 1 <= pimax" in L.nbk_last_error()
    assert count(rmax=2.) < 0 and b"below the largest separation" in L.nbk_last_error()
    assert count() < 0 and b"null output" in L.nbk_last_error()


def _stencil(L, n2, rmax, box):
    out = (ctypes.c_int32 * 125)()
    n = L.nbk_pc_stencil(n2, rmax, (ctypes.c_double * 3)(*box), None, None, out)
    assert n > 0
    return {(o // 25 - 2, (o // 5) % 5 - 2, o % 5 - 2) for o in out[:n]}


def _expected_stencil(L, n2, rmax, box):
    """the rule: offsets in [-2, 2]^3 whose cells come closer than r_max, on the grid nbk_pc_workspace plans"""
    ncell = (ctypes.c_int64 * 3)()
    L.nbk_pc_workspace(0, n2, rmax, (ctypes.c_double * 3)(*box), None, None, ncell)
    side = np.asarray(box, 'f8') / np.asarray(list(ncell))
    out = set()
    for o in np.ndindex(5, 5, 5):
        o = np.asarray(o) - 2
        gap = np.maximum(np.abs(o) - 1, 0) * side
        if (gap ** 2).sum() < rmax ** 2:
            out.add(tuple(int(v) for v in o))
    return out, list(ncell)


def test_stencil(L):
    # cells just wider than r_max / 2: the whole 5^3 block (the corners come within sqrt(3) r_max / 2)
    st = _stencil(L, 10 ** 6, 10., [100.] * 3)
    want, nc = _expected_stencil(L, 10 ** 6, 10., [100.] * 3)
    assert nc == [19, 19, 19] and st == want and len(st) == 125
    # cells of 100/17: the eight (+-2, +-2, +-2) corners are r_max or more away
    st = _stencil(L, 2457, 10., [100.] * 3)
    want, nc = _expected_stencil(L, 2457, 10., [100.] * 3)
    assert nc == [17, 17, 17] and st == want and len(st) == 117
    # a periodic axis of 2 cells: offsets wrap onto the same cells, each cell visited once
    st = _stencil(L, 10 ** 6, 10., [100., 100., 12.])
    assert len({(a, b, c % 2) for a, b, c in st}) == len(st) and len({c % 2 for _, _, c in st}) == 2
    assert len(st) == 50
    # the cell cap binds for few secondaries: cells of 20 > r_max, only the 27 nearest cells
    st = _stencil(L, 10, 10., [100.] * 3)
    assert st == {(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)}


# ---- the oracle against a double loop ------------------------------------------------------------------------------
def _brute(mode, pos1, pos2, w1, w2, edges, box, Nmu=None, pimax=None, los=2):
    nb = po.nbins_of(mode, edges, Nmu, pimax)
    n, wn, s = np.zeros(nb, 'u8'), np.zeros(nb), np.zeros(nb)
    u1, u2 = po.wrap(pos1, box), po.wrap(pos2, box)
    for a in range(len(pos1)):
        d = u2 - u1[a]
        if box is not None:
            d = d - box * np.rint(d * (1.0 / box))
        keep, b, sep = po.bin_pairs(mode, d[:, 0], d[:, 1], d[:, 2], edges, Nmu, pimax, los)
        for j in np.nonzero(keep)[0]:
            n[b[j]] += 1
            wn[b[j]] += w1[a] * w2[j]
            s[b[j]] += sep[j]
    return n, wn, s


@pytest.mark.parametrize("mode, kw", [('1d', {}), ('2d', {'Nmu': 4}), ('projected', {'pimax': 6.5})])
@pytest.mark.parametrize("periodic", [True, False])
@pytest.mark.parametrize("los", [0, 2])
def test_oracle_matches_double_loop(mode, kw, periodic, los):
    rng = np.random.RandomState(4)
    L = 20.
    p1 = rng.uniform(-2, L + 2, (150, 3))           # some rows outside the box: they are wrapped
    p2 = rng.uniform(0, L, (120, 3)).astype('f4')
    w1, w2 = rng.uniform(size=150), rng.uniform(size=120)
    edges = np.array([0.5, 1.5, 3., 6.])
    box = L if periodic else None
    got = po.paircount(mode, p1, edges, box=box, pos2=p2, w1=w1, w2=w2, los=los, **kw)
    n, wn, s = _brute(mode, p1, p2.astype('f8'), w1, w2, edges, box, los=los, **kw)
    np.testing.assert_array_equal(got['npairs'].ravel(), n)
    np.testing.assert_allclose(got['wnpairs'].ravel(), wn, rtol=1e-12)
    nz = n > 0
    np.testing.assert_allclose(got['sep'].ravel()[nz], s[nz] / n[nz], rtol=1e-12)
    assert (got['sep'].ravel()[~nz] == 0).all() and n.sum() > 100


def test_oracle_boundaries():
    # a pair at exactly an edge counts in the upper bin; along the line of sight mu = 1 is dropped; pi = pimax dropped
    p = np.array([[0., 0., 0.], [0., 0., 2.], [3., 0., 0.]])
    r = po.paircount('1d', p, [1., 2., 3., 4.])
    np.testing.assert_array_equal(r['npairs'], [0, 2, 4])
    r = po.paircount('2d', p, [1., 2.5, 4.], Nmu=2)
    # (0,0,2) - (0,0,0) has mu = 1: gone; the other two pairs have mu = 0 and 2 / sqrt(13)
    np.testing.assert_array_equal(r['npairs'], [[0, 0], [2, 2]])
    r = po.paircount('projected', p, [1., 4.], pimax=2.)
    np.testing.assert_array_equal(r['npairs'], [[2, 0]])
    assert len(po.near_ties('1d', p, [1., 2., 3., 4.])[0]) == 4


# ---- estimators on hand-made counts --------------------------------------------------------------------------------
def _pairs(mode, npairs, wnpairs, edges, Nmu=None, pimax=None):
    from nbodykit_b200.algorithms.paircount import _make_pairs
    n = np.asarray(npairs, 'i8').ravel()
    return _make_pairs(mode, edges, Nmu, pimax, n, np.asarray(wnpairs, 'f8').ravel(), n * 1.5)


def test_natural_estimator():
    from nbodykit_b200.algorithms.paircount import natural_estimator
    edges = np.array([1., 2., 4.])
    DD = _pairs('1d', [10, 90], [12., 80.], edges)
    for attrs, N2 in ((dict(N1=1000, N2=None, is_cross=False, total_wnpairs=4.5e5), None),
                      (dict(N1=1000, N2=500, is_cross=True, total_wnpairs=2.6e5), 500)):
        attrs.update(mode='1d', BoxSize=np.array([50.] * 3))
        R1R2, corr = natural_estimator(DD, attrs)
        RR, tRR = po.analytic_rr('1d', edges, 50., 1000, N2)
        np.testing.assert_allclose(R1R2['npairs'], RR, rtol=1e-12)
        np.testing.assert_allclose(corr['corr'], po.natural(np.array([12., 80.]), attrs['total_wnpairs'], RR, tRR),
                                   rtol=1e-12)
        np.testing.assert_allclose(corr['r'], 1.5)
    for mode, kw in (('2d', dict(Nmu=3)), ('projected', dict(pimax=4.))):
        shape = po.shape_of(mode, edges, **kw)
        DD = _pairs(mode, np.full(shape, 7), np.full(shape, 7.), edges, **kw)
        R1R2, corr = natural_estimator(DD, dict(N1=100, N2=None, is_cross=False, total_wnpairs=4950., mode=mode,
                                                BoxSize=np.array([20.] * 3)))
        np.testing.assert_allclose(R1R2['npairs'], po.analytic_rr(mode, edges, 20., 100, **kw)[0], rtol=1e-12)


def test_landy_szalay_wp_poles():
    from nbodykit_b200.algorithms.paircount import compute_wp, landy_szalay
    edges = np.array([1., 2., 4.])
    rng = np.random.RandomState(5)
    shape = (2, 3)
    DD, DR, RD, RR = [_pairs('projected', rng.randint(1, 100, shape), rng.uniform(1, 100, shape), edges, pimax=3.)
                      for _ in range(4)]
    RR.data['npairs'][0, 1] = 0
    with pytest.warns(UserWarning, match="contains separation bins with no bins"):
        corr = landy_szalay(DD, DR, RD, RR, (10., 20., 30., 40.))
    want = po.landy_szalay(DD['wnpairs'], DR['wnpairs'], RD['wnpairs'], RR['npairs'] * 1.0, 10., 20., 30., 40.)
    want[RR['npairs'] > 0] = po.landy_szalay(DD['wnpairs'], DR['wnpairs'], RD['wnpairs'], RR['wnpairs'], 10., 20.,
                                             30., 40.)[RR['npairs'] > 0]
    np.testing.assert_allclose(corr['corr'], want, rtol=1e-12)
    assert np.isnan(corr['corr'][0, 1])
    corr.data['corr'][0, 1] = 0.5
    wp = compute_wp(corr)
    assert wp.dims == ['rp']
    np.testing.assert_allclose(wp['corr'], po.wp(corr['corr'], 3.), rtol=1e-12)
    # to_poles of 2d wedges
    from nbodykit_b200.algorithms.paircount import _corr_result
    D = _pairs('2d', np.ones((2, 5)), np.ones((2, 5)), edges, Nmu=5)
    xi = rng.uniform(-1, 1, (2, 5))
    poles = _corr_result(D, xi).to_poles([0, 2, 4])
    want = po.to_poles(xi, 5, [0, 2, 4])
    for ell in (0, 2, 4):
        np.testing.assert_allclose(poles['corr_%d' % ell], want[ell], rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(poles['r'], 1.5)


def test_save_load_round_trip(tmp_path):
    from nbodykit_b200.algorithms.paircount import SimulationBox2PCF, SimulationBoxPairCount, natural_estimator
    from nbodykit_b200.comm import SelfComm
    edges = np.array([1., 2., 4.])
    pc = object.__new__(SimulationBoxPairCount)
    pc.comm = SelfComm()
    pc.attrs = dict(mode='2d', edges=edges, Nmu=3, pimax=None, show_progress=False, N1=10, N2=None,
                    total_wnpairs=45., is_cross=False, BoxSize=np.array([10.] * 3), periodic=True, weight='Weight',
                    position='Position', config={'nthreads': 2}, los=2)
    pc.pairs = _pairs('2d', np.arange(6).reshape(2, 3), np.arange(6.).reshape(2, 3) * 0.5, edges, Nmu=3)
    pc.save(str(tmp_path / "pc.json"))
    back = SimulationBoxPairCount.load(str(tmp_path / "pc.json"), comm=SelfComm())
    np.testing.assert_array_equal(back.pairs.data, pc.pairs.data)
    assert back.pairs.dims == ['r', 'mu'] and back.attrs['config'] == {'nthreads': 2}
    np.testing.assert_array_equal(back.pairs.edges['mu'], np.linspace(0, 1, 4))

    tp = object.__new__(SimulationBox2PCF)
    tp.comm = SelfComm()
    tp.attrs = dict(pc.attrs)
    tp.R1R2, tp.corr = natural_estimator(pc.pairs, pc.attrs)
    tp.D1D2, tp.D1R2, tp.D2R1 = pc.pairs, None, None
    tp.save(str(tmp_path / "tp.json"))
    back = SimulationBox2PCF.load(str(tmp_path / "tp.json"), comm=SelfComm())
    np.testing.assert_array_equal(back.corr['corr'], tp.corr['corr'])
    np.testing.assert_array_equal(back.R1R2['npairs'], tp.R1R2['npairs'])
    assert back.D1R2 is None and back.wp is None
    assert hasattr(back.corr, 'to_poles')
