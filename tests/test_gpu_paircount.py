"""
Pair counts on the GPU: the reference's simulation-box cases (pair_counters/tests/test_{1d,2d,projected}.py and
paircount_tpcf/tests/test_*.py, with the CPU oracle oracle/paircount_oracle.py in place of kdcount and halotools),
exact parity with the oracle on uniform, log-normal and clumpy inputs in every mode, boundary cases on an integer
lattice, the estimators, FOF groups -> SimulationBox2PCF, and several ranks emulated by threads on one GPU.  Inputs are
checked to have no pair within a relative 1e-9 of a bin boundary, so npairs must agree exactly.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import paircount_oracle as po
from test_gpu_fof import _run_ranks, _split, clumpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KW = {'1d': {}, '2d': {'Nmu': 7}, 'projected': {'pimax': 9.5}}
# xi is a difference of O(1) ratios of float64 sums whose order depends on the GPU's atomic schedule (two runs of the
# same count differ in the last bits), so bins where xi is near 0 are compared absolutely
XI_ATOL = 1e-12


def _cat(cols, box=None, comm=None):
    from nbodykit_b200 import CurrentMPIComm
    from nbodykit_b200.lab import ArrayCatalog
    return ArrayCatalog(cols, comm=comm or CurrentMPIComm.get(), **({'BoxSize': box} if box is not None else {}))


def _assert_matches(pairs, want, exact=True):
    dim = pairs.dims[0]
    if exact:
        np.testing.assert_array_equal(pairs['npairs'], want['npairs'])
    else:
        np.testing.assert_allclose(pairs['npairs'].astype('f8'), want['npairs'], rtol=1e-12)
    np.testing.assert_allclose(pairs['wnpairs'], want['wnpairs'], rtol=1e-10, atol=1e-300)
    np.testing.assert_allclose(pairs[dim], want['sep'], rtol=1e-10, atol=1e-300)


def _parity(mode, pos1, edges, box, pos2=None, w1=None, w2=None, los=2, **kw):
    """SimulationBoxPairCount against the oracle, after checking that no pair sits on a boundary"""
    from nbodykit_b200.lab import SimulationBoxPairCount
    kw = dict(KW[mode], **kw)
    assert len(po.near_ties(mode, pos1, edges, box=box, pos2=pos2, los=los, **kw)[0]) == 0, "a pair is on a boundary"
    L = box if box is not None else 1.0
    first = _cat({'Position': pos1, 'Weight': w1 if w1 is not None else np.ones(len(pos1))}, box=L)
    second = None
    if pos2 is not None:
        second = _cat({'Position': pos2, 'Weight': w2 if w2 is not None else np.ones(len(pos2))}, box=L)
    r = SimulationBoxPairCount(mode, first, edges, periodic=box is not None, second=second, los=los, **kw)
    want = po.paircount(mode, pos1, edges, box=box, pos2=pos2, w1=w1, w2=w2, los=los, **kw)
    _assert_matches(r.pairs, want)
    return r, want


# ---- the reference's cases ---------------------------------------------------------------------------------------
def _uniform(nbar, seed, dtype='f8', weights=False):
    from nbodykit_b200.lab import UniformCatalog
    cat = UniformCatalog(nbar=nbar, BoxSize=512., seed=seed, dtype=dtype)
    if weights:
        cat['Weight'] = cat.rng.uniform()
    return cat


def _np(cat, col):
    c = cat[col]
    c = c.compute() if hasattr(c, 'compute') else c
    return c.cpu().numpy() if hasattr(c, 'cpu') else np.asarray(c)


@pytest.mark.parametrize("mode", ["1d", "2d", "projected"])
@pytest.mark.parametrize("periodic", [True, False])
def test_reference_auto(cuda, mode, periodic):
    from nbodykit_b200.lab import SimulationBoxPairCount
    src = _uniform(3e-6, 42, weights=True)
    edges = np.linspace(10, 150, 10)
    kw = {'2d': {'Nmu': 10}, 'projected': {'pimax': 50}, '1d': {}}[mode]
    r = SimulationBoxPairCount(mode, src, edges, periodic=periodic, weight='Weight', **kw)
    pos, w = _np(src, 'Position'), _np(src, 'Weight')
    want = po.paircount(mode, pos, edges, box=512. if periodic else None, w1=w, **kw)
    _assert_matches(r.pairs, want)
    assert r.pairs.attrs['total_wnpairs'] == r.attrs['total_wnpairs']
    with pytest.raises(ValueError):
        SimulationBoxPairCount(mode, src, np.linspace(0, 10.0, 10), **kw)


@pytest.mark.parametrize("mode", ["1d", "2d", "projected"])
def test_reference_cross_f4_f8(cuda, mode):
    from nbodykit_b200.lab import SimulationBoxPairCount
    first, second = _uniform(3e-6, 42, 'f4'), _uniform(3e-6, 84, 'f8')
    edges = np.linspace(10, 150, 10)
    kw = {'2d': {'Nmu': 10}, 'projected': {'pimax': 50}, '1d': {}}[mode]
    r = SimulationBoxPairCount(mode, first, edges, second=second, periodic=True, **kw)
    want = po.paircount(mode, _np(first, 'Position'), edges, box=512., pos2=_np(second, 'Position'), **kw)
    _assert_matches(r.pairs, want)


def test_natural_estimator_reference_catalogue(cuda):
    from nbodykit_b200.lab import SimulationBox2PCF
    src = _uniform(3e-4, 42)
    edges = np.linspace(0.01, 20, 10)
    r = SimulationBox2PCF('1d', src, edges)
    pos = _np(src, 'Position')
    dd = po.paircount('1d', pos, edges, box=512.)
    RR, tRR = po.analytic_rr('1d', edges, 512., len(pos))
    want = po.natural(dd['wnpairs'], po.total_wnpairs(np.ones(len(pos))), RR, tRR)
    np.testing.assert_allclose(r.corr['corr'], want, rtol=1e-10, atol=XI_ATOL)
    np.testing.assert_array_equal(r.D1D2['npairs'], dd['npairs'])
    assert r.D1R2 is None and r.D2R1 is None


def test_landy_szalay_matches_corrfunc_numbers(cuda):
    # the reference's test_sim_nonperiodic_auto: the values Corrfunc gave for these catalogues
    from nbodykit_b200.lab import SimulationBox2PCF
    source, randoms = _uniform(3e-4, 42), _uniform(3e-4, 84)
    r = SimulationBox2PCF('1d', source, np.linspace(0.01, 20, 10), periodic=False, randoms1=randoms)
    cf = [0.1158045, -0.03074509, -0.0227549, 0.01194295, -0.01553021, -0.001123882, -0.005164478, -0.002296215,
          0.003764593]
    np.testing.assert_allclose(cf, r.corr['corr'], rtol=1e-5, atol=1e-5)
    with pytest.raises(ValueError):
        SimulationBox2PCF('1d', source, np.linspace(0.01, 20, 10), periodic=False)


def test_low_nbar_randoms_warn(cuda):
    from nbodykit_b200.lab import SimulationBox2PCF, UniformCatalog
    source = _uniform(3e-4, 42)
    randoms = UniformCatalog(nbar=3e-6, BoxSize=512., seed=84)
    with pytest.warns(UserWarning, match="no bins"):
        r = SimulationBox2PCF('1d', source, np.linspace(0.01, 5.0, 2), periodic=False, randoms1=randoms)
    assert np.isnan(r.corr['corr']).all()


# ---- exact parity with the oracle ------------------------------------------------------------------------------------
def _lognormal():
    from nbodykit_b200.cosmology import NoWiggleEHPower
    from nbodykit_b200.lab import LogNormalCatalog
    cat = LogNormalCatalog(Plin=NoWiggleEHPower(), nbar=3e-3, BoxSize=200., Nmesh=64, bias=2.0, seed=42)
    return _np(cat, 'Position'), 200.


def _input(kind, dtype):
    rng = np.random.RandomState(11)
    if kind == 'uniform':
        return rng.uniform(0, 100., (20000, 3)).astype(dtype), 100.
    if kind == 'clumpy':
        return clumpy(seed=5, dtype=dtype)[0][::3], 100.
    pos, L = _lognormal()
    return pos.astype(dtype), L


@pytest.mark.parametrize("kind", ["uniform", "clumpy", "lognormal"])
@pytest.mark.parametrize("mode", ["1d", "2d", "projected"])
@pytest.mark.parametrize("periodic", [True, False])
def test_parity(cuda, kind, mode, periodic):
    pos, L = _input(kind, 'f4' if periodic else 'f8')
    rng = np.random.RandomState(3)
    w = rng.uniform(0.5, 1.5, len(pos))
    edges = np.geomspace(0.3, 12., 9)
    los = {'uniform': 0, 'clumpy': 1, 'lognormal': 2}[kind]
    box = L if periodic else None
    _parity(mode, pos, edges, box, w1=w, los=los)
    # cross with the other precision and a second weight column
    pos2 = (rng.uniform(0, L, (5000, 3))).astype('f8' if periodic else 'f4')
    _parity(mode, pos, edges, box, pos2=pos2, w1=w, w2=rng.uniform(size=5000).astype('f4'), los=los)


# ---- boundaries on an integer lattice (exact arithmetic) -------------------------------------------------------------
def _lattice(n=8):
    return np.indices((n, n, n)).reshape(3, -1).T.astype('f8')


def test_lattice_edges_and_coincident_points(cuda):
    from nbodykit_b200.lab import SimulationBoxPairCount
    pos = _lattice()
    N = len(pos)
    edges = np.array([1., 2., 3.])
    r = SimulationBoxPairCount('1d', _cat({'Position': pos, 'Weight': np.ones(N)}, box=8.), edges)
    # d = 1, sqrt2, sqrt3 land in [1, 2): 6 + 12 + 8 neighbours; d = 2 (exactly the edge) goes to [2, 3)
    np.testing.assert_array_equal(r.pairs['npairs'], [26 * N, (6 + 24 + 24 + 12) * N])
    _assert_matches(r.pairs, po.paircount('1d', pos, edges, box=8.))
    # every point twice: coincident copies never pair, every other pair four times
    two = np.concatenate([pos, pos])
    r2 = SimulationBoxPairCount('1d', _cat({'Position': two, 'Weight': np.ones(2 * N)}, box=8.), edges)
    np.testing.assert_array_equal(r2.pairs['npairs'], 4 * r.pairs['npairs'])
    # an empty bin: separation 0 and wnpairs 0
    r3 = SimulationBoxPairCount('1d', _cat({'Position': pos, 'Weight': np.ones(N)}, box=8.), [0.2, 0.5, 1.2])
    assert r3.pairs['npairs'][0] == 0 and r3.pairs['r'][0] == 0 and r3.pairs['wnpairs'][0] == 0
    assert r3.pairs['r'][1] == 1.0


def test_lattice_los_and_pimax(cuda):
    from nbodykit_b200.lab import SimulationBoxPairCount
    pos = _lattice()
    N = len(pos)
    cat = _cat({'Position': pos, 'Weight': np.ones(N)}, box=8.)
    for los in (0, 1, 2):
        r = SimulationBoxPairCount('2d', cat, [0.5, 1.2], Nmu=2, los=los)
        # of the 6 nearest neighbours the two along the line of sight have mu = 1 and are dropped
        np.testing.assert_array_equal(r.pairs['npairs'], [[4 * N, 0]])
        _assert_matches(r.pairs, po.paircount('2d', pos, [0.5, 1.2], box=8., Nmu=2, los=los))
    r = SimulationBoxPairCount('projected', cat, [0.5, 1.2], pimax=2.)
    # r_p = 1 (4 neighbours in the plane) at |pi| = 0 and 1; |pi| = 2 = pimax is dropped
    np.testing.assert_array_equal(r.pairs['npairs'], [[4 * N, 8 * N]])
    _assert_matches(r.pairs, po.paircount('projected', pos, [0.5, 1.2], box=8., pimax=2.))


def test_tiny_catalogues(cuda):
    from nbodykit_b200.lab import SimulationBoxPairCount
    edges = np.array([1., 2.])
    for n in (0, 1):
        cat = _cat({'Position': np.full((n, 3), 3.), 'Weight': np.ones(n)}, box=10.)
        for periodic in (True, False):
            r = SimulationBoxPairCount('1d', cat, edges, periodic=periodic)
            assert r.pairs['npairs'].sum() == 0 and r.pairs['wnpairs'].sum() == 0
    one = _cat({'Position': np.full((1, 3), 3.), 'Weight': np.ones(1)}, box=10.)
    other = _cat({'Position': np.array([[4.5, 3., 3.]]), 'Weight': np.full(1, 2.)}, box=10.)
    r = SimulationBoxPairCount('1d', one, edges, second=other)
    assert list(r.pairs['npairs']) == [1] and list(r.pairs['wnpairs']) == [2.] and list(r.pairs['r']) == [1.5]


def test_one_cell_and_global_histogram(cuda):
    rng = np.random.RandomState(9)
    pos = 50. + rng.uniform(0, 0.4, (3000, 3))          # every particle in one cell
    for box in (100., None):
        _parity('1d', pos, np.array([0.01, 0.1, 0.3]), box)
    # 100 r_p bins x 40 pi bins x 3 fields do not fit in shared memory: the global-atomics path
    pos = rng.uniform(0, 100., (20000, 3))
    edges = np.linspace(0.2, 10., 101)
    _parity('projected', pos, edges, 100., pimax=40.)


def test_show_progress_chunks(cuda, caplog):
    import logging
    from nbodykit_b200.lab import SimulationBoxPairCount
    rng = np.random.RandomState(1)
    cat = _cat({'Position': rng.uniform(0, 50., (5000, 3)), 'Weight': rng.uniform(size=5000)}, box=50.)
    a = SimulationBoxPairCount('2d', cat, np.linspace(1, 10, 5), Nmu=3)
    with caplog.at_level(logging.INFO, logger='SimulationBoxPairCount'):
        b = SimulationBoxPairCount('2d', cat, np.linspace(1, 10, 5), Nmu=3, show_progress=True)
    assert sum("% done" in m for m in caplog.messages) == 10
    np.testing.assert_array_equal(a.pairs['npairs'], b.pairs['npairs'])
    np.testing.assert_allclose(a.pairs['wnpairs'], b.pairs['wnpairs'], rtol=1e-12)


# ---- estimators ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["1d", "2d", "projected"])
def test_2pcf_natural_auto_cross_wp_poles(cuda, mode, tmp_path):
    from nbodykit_b200.lab import SimulationBox2PCF
    rng = np.random.RandomState(2)
    p1, p2 = rng.uniform(0, 100., (20000, 3)), rng.uniform(0, 100., (15000, 3))
    d1, d2 = _cat({'Position': p1}, box=100.), _cat({'Position': p2}, box=100.)
    edges = np.linspace(1., 10., 6)
    kw = {'1d': {}, '2d': {'Nmu': 5}, 'projected': {'pimax': 10.}}[mode]
    for data2, pos2 in ((None, None), (d2, p2)):
        r = SimulationBox2PCF(mode, d1, edges, data2=data2, **kw)
        dd = po.paircount(mode, p1, edges, box=100., pos2=pos2, **kw)
        N2 = None if pos2 is None else len(pos2)
        RR, tRR = po.analytic_rr(mode, edges, 100., len(p1), N2, **kw)
        tDD = po.total_wnpairs(np.ones(len(p1)), None if pos2 is None else np.ones(len(pos2)))
        np.testing.assert_allclose(r.corr['corr'], po.natural(dd['wnpairs'], tDD, RR, tRR), rtol=1e-10,
                                   atol=XI_ATOL)
    if mode == 'projected':
        np.testing.assert_allclose(r.wp['corr'], po.wp(r.corr['corr'], 10.), rtol=1e-12, atol=XI_ATOL)
    if mode == '2d':
        poles = r.corr.to_poles([0, 2])
        want = po.to_poles(r.corr['corr'], 5, [0, 2])
        np.testing.assert_allclose(poles['corr_2'], want[2], rtol=1e-12, atol=1e-14)
    r.save(str(tmp_path / "x.json"))
    back = SimulationBox2PCF.load(str(tmp_path / "x.json"))
    np.testing.assert_array_equal(back.corr['corr'], r.corr['corr'])


def test_2pcf_landy_szalay_reuses_r1r2(cuda, monkeypatch):
    from nbodykit_b200.algorithms import paircount
    from nbodykit_b200.lab import SimulationBox2PCF, SimulationBoxPairCount
    rng = np.random.RandomState(4)
    D1, D2 = [_cat({'Position': rng.uniform(0, 100., (8000, 3)), 'Weight': rng.uniform(size=8000)}, box=100.)
              for _ in range(2)]
    R1, R2 = [_cat({'Position': rng.uniform(0, 100., (12000, 3)), 'Weight': np.ones(12000)}, box=100.)
              for _ in range(2)]
    edges = np.linspace(2., 10., 5)
    r = SimulationBox2PCF('projected', D1, edges, pimax=8., data2=D2, randoms1=R1, randoms2=R2, periodic=False)
    RR = SimulationBoxPairCount('projected', R1, edges, pimax=8., second=R2, periodic=False)
    calls = []
    orig = paircount.SimulationBoxPairCount.run
    monkeypatch.setattr(paircount.SimulationBoxPairCount, 'run', lambda self: calls.append(1) or orig(self))
    r2 = SimulationBox2PCF('projected', D1, edges, pimax=8., data2=D2, randoms1=R1, randoms2=R2, periodic=False,
                           R1R2=RR)
    assert len(calls) == 3                        # DD, DR, RD: R1R2 reused
    assert r2.R1R2 is RR.pairs
    np.testing.assert_allclose(r2.corr['corr'], r.corr['corr'], rtol=1e-10, atol=XI_ATOL)
    col = lambda c, k: _np(c, k)
    cnt = lambda a, b: po.paircount('projected', col(a, 'Position'), edges, pos2=col(b, 'Position'),
                                    w1=col(a, 'Weight'), w2=col(b, 'Weight'), pimax=8.)['wnpairs']
    tot = lambda a, b: po.total_wnpairs(col(a, 'Weight'), col(b, 'Weight'))
    want = po.landy_szalay(cnt(D1, D2), cnt(D1, R2), cnt(D2, R1), cnt(R1, R2), tot(D1, D2), tot(D1, R2), tot(D2, R1),
                           tot(R1, R2))
    np.testing.assert_allclose(r.corr['corr'], want, rtol=1e-10, atol=XI_ATOL)
    np.testing.assert_allclose(r.wp['corr'], po.wp(want, 8.), rtol=1e-10, atol=XI_ATOL)


def test_fof_groups_workflow(cuda):
    from nbodykit_b200.lab import FOF, SimulationBox2PCF
    pos, vel = clumpy()
    halos = FOF(_cat({'Position': pos, 'Velocity': vel}, box=100.), 0.25, 5, absolute=True).find_features()
    halos['Position'] = halos['CMPosition']
    halos['Weight'] = np.ones(halos.size)
    r = SimulationBox2PCF('1d', halos, np.linspace(0.5, 20., 8))
    hp = _np(halos, 'CMPosition')
    dd = po.paircount('1d', hp, np.linspace(0.5, 20., 8), box=100.)
    np.testing.assert_array_equal(r.D1D2['npairs'], dd['npairs'])
    assert np.isfinite(r.corr['corr']).all() and r.D1D2['npairs'].sum() > 0


def test_launches_the_paircount_kernels(cuda, monkeypatch):
    from nbodykit_b200 import _lib
    from nbodykit_b200.lab import SimulationBoxPairCount
    L = _lib.lib()
    called = []
    for name in ("nbk_pc_bucket", "nbk_pc_count"):
        orig = getattr(L, name)
        monkeypatch.setattr(L, name, (lambda o, nm: lambda *a: called.append(nm) or o(*a))(orig, name))
    rng = np.random.RandomState(0)
    cat = _cat({'Position': rng.uniform(0, 50., (2000, 3)), 'Weight': np.ones(2000)}, box=50.)
    n0 = _lib.launch_count()
    SimulationBoxPairCount('1d', cat, np.linspace(1, 5, 4))
    assert _lib.launch_count() - n0 >= 9
    assert called == ["nbk_pc_bucket", "nbk_pc_bucket", "nbk_pc_count"]


# ---- several ranks emulated by threads on one GPU ------------------------------------------------------------------
def _multi_rank(P, mode, pos, w, edges, box, pos2=None, w2=None, **kw):
    from nbodykit_b200.lab import SimulationBoxPairCount

    def fn(comm):
        c1 = _cat({'Position': _split(pos, P, comm.rank), 'Weight': _split(w, P, comm.rank)}, box=box or 1., comm=comm)
        c2 = None
        if pos2 is not None:
            c2 = _cat({'Position': _split(pos2, P, comm.rank), 'Weight': _split(w2, P, comm.rank)}, box=box or 1.,
                      comm=comm)
        r = SimulationBoxPairCount(mode, c1, edges, second=c2, periodic=box is not None, **kw)
        return r.pairs
    res = _run_ranks(P, fn)
    for other in res[1:]:
        np.testing.assert_array_equal(other.data, res[0].data)
    return res[0]


@pytest.mark.parametrize("P", [2, 3])
@pytest.mark.parametrize("periodic", [True, False])
@pytest.mark.parametrize("mode", ["1d", "projected"])
def test_emulated_ranks_match_one_rank(cuda, P, periodic, mode):
    from nbodykit_b200.lab import SimulationBoxPairCount
    pos = clumpy(seed=7)[0][::2]
    rng = np.random.RandomState(5)
    w = rng.uniform(size=len(pos))
    pos2, w2 = rng.uniform(0, 100., (6000, 3)), rng.uniform(size=6000)
    box = 100. if periodic else None
    edges = np.geomspace(0.5, 8., 6)
    kw = {'1d': {}, 'projected': {'pimax': 6.}}[mode]
    for p2, ww2 in ((None, None), (pos2, w2)):
        c2 = _cat({'Position': p2, 'Weight': ww2}, box=box or 1.) if p2 is not None else None
        one = SimulationBoxPairCount(mode, _cat({'Position': pos, 'Weight': w}, box=box or 1.), edges, second=c2,
                                     periodic=periodic, **kw).pairs
        many = _multi_rank(P, mode, pos, w, edges, box, pos2=p2, w2=ww2, **kw)
        np.testing.assert_array_equal(many['npairs'], one['npairs'])
        np.testing.assert_allclose(many['wnpairs'], one['wnpairs'], rtol=1e-12)
        np.testing.assert_allclose(many[one.dims[0]], one[one.dims[0]], rtol=1e-12)


def test_emulated_ranks_all_gather_fallback(cuda):
    # 3 slabs of 33.3 are not wider than 2 r_max = 40: every rank gathers the secondaries
    from nbodykit_b200.lab import SimulationBoxPairCount
    rng = np.random.RandomState(6)
    pos, w = rng.uniform(0, 100., (6000, 3)), rng.uniform(size=6000)
    edges = np.linspace(5., 20., 4)
    one = SimulationBoxPairCount('2d', _cat({'Position': pos, 'Weight': w}, box=100.), edges, Nmu=4).pairs
    many = _multi_rank(3, '2d', pos, w, edges, 100., Nmu=4)
    np.testing.assert_array_equal(many['npairs'], one['npairs'])
    np.testing.assert_allclose(many['wnpairs'], one['wnpairs'], rtol=1e-12)


# ---- two GPUs --------------------------------------------------------------------------------------------------------
def test_two_gpu_paircount_matches_one_gpu():
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tests", "mgpu_paircount_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(out.stdout[-3000:])
    sys.stderr.write(out.stderr[-3000:])
    assert out.returncode == 0
