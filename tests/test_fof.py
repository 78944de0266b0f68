"""FOF without a GPU: argument checks, the linking length, attrs, to_halos, argument validation of the nbk_fof_* entry
points (no CUDA call is reached), and the CPU oracle on cases with a known answer."""
import ctypes

import numpy as np
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


def _cat(n=1000, box=True, **cols):
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.lab import ArrayCatalog
    rng = np.random.RandomState(1)
    data = {'Position': rng.uniform(0, 100., size=(n, 3))}
    data.update(cols)
    return ArrayCatalog(data, comm=SelfComm(), **({'BoxSize': 100.} if box else {}))


@pytest.fixture
def norun(monkeypatch):
    """FOF objects without the GPU run"""
    from nbodykit_b200.algorithms import fof
    monkeypatch.setattr(fof.FOF, 'run', lambda self: None)
    return fof.FOF


def test_exported():
    from nbodykit_b200 import lab
    from nbodykit_b200.algorithms import FOF
    assert lab.FOF is FOF


def test_needs_position(norun):
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.lab import ArrayCatalog
    cat = ArrayCatalog({'Velocity': np.zeros((10, 3))}, comm=SelfComm(), BoxSize=1.)
    with pytest.raises(ValueError, match="Position"):
        norun(cat, 0.2, 20)


def test_periodic_needs_boxsize(norun):
    with pytest.raises(ValueError, match="BoxSize"):
        norun(_cat(box=False), 0.2, 20, absolute=True)
    norun(_cat(box=False), 0.2, 20, absolute=True, periodic=False)


def test_relative_linking_length(norun):
    f = norun(_cat(1000), 0.2, 20)
    assert f._linking_length == pytest.approx(0.2 * (100. ** 3 / 1000) ** (1 / 3.))
    f = norun(_cat(1000), 0.7, 20, absolute=True)
    assert f._linking_length == 0.7


def test_attrs_hold_the_arguments(norun):
    f = norun(_cat(), 0.2, 5, absolute=False, periodic=True, domain_factor=3)
    assert f.attrs == {'linking_length': 0.2, 'nmin': 5, 'absolute': False, 'periodic': True, 'domain_factor': 3}


def test_to_halos_is_out_of_scope(norun):
    f = norun(_cat(), 0.2, 5)
    with pytest.raises(NotImplementedError, match="cosmology"):
        f.to_halos(1e12, None, 0.)


def test_find_features_needs_velocity(norun):
    f = norun(_cat(), 0.2, 5)
    with pytest.raises(ValueError, match="Velocity"):
        f.find_features()


def test_scatter_share_splits_like_scatterarray():
    from nbodykit_b200.algorithms.fof import _scatter_share

    class C(object):
        def __init__(self, r, p):
            self.rank, self.size = r, p
    for ntot, P in [(10, 3), (2, 3), (7, 1), (9, 3)]:
        shares = [_scatter_share(ntot, C(r, P)) for r in range(P)]
        sizes = [b - a for a, b in shares]
        assert shares[0][0] == 0 and shares[-1][1] == ntot
        assert all(shares[i][1] == shares[i + 1][0] for i in range(P - 1))
        assert sizes == [ntot // P + (1 if r < ntot % P else 0) for r in range(P)]


# ---- C ABI validation (before any CUDA call) ------------------------------------------------------------------------
def _box(v=1.0):
    from nbodykit_b200._lib import darr
    return darr([v, v, v])


def test_workspace_validates(L):
    from nbodykit_b200._lib import darr
    nc = (ctypes.c_int64 * 3)()
    assert L.nbk_fof_workspace(-1, 0.1, _box(), None, None, nc) == -1 and b"0 <= n <= 2^31-1" in _err(L)
    assert L.nbk_fof_workspace(2 ** 31, 0.1, _box(), None, None, nc) == -1 and b"2^31-1" in _err(L)
    assert L.nbk_fof_workspace(10, 0.0, _box(), None, None, nc) == -1 and b"> 0" in _err(L)
    assert L.nbk_fof_workspace(10, 0.1, darr([1, 0, 1]), None, None, nc) == -1 and b"box sides must be > 0" in _err(L)
    assert L.nbk_fof_workspace(10, 0.1, None, None, None, nc) == -1 and b"lo and hi" in _err(L)
    assert L.nbk_fof_workspace(10, 0.1, None, darr([1, 0, 0]), darr([0, 1, 1]), nc) == -1 and b"lo <= hi" in _err(L)


def test_grid_side_at_least_ll_and_cells_capped(L):
    from nbodykit_b200._lib import darr
    nc = (ctypes.c_int64 * 3)()
    assert L.nbk_fof_workspace(10 ** 6, 0.01, _box(), None, None, nc) > 0
    assert list(nc) == [99, 99, 99]                       # side 1/99 >= 0.01
    assert L.nbk_fof_workspace(1000, 1e-6, _box(), None, None, nc) > 0
    assert np.prod(list(nc)) <= 2000                      # capped at 2n cells
    assert L.nbk_fof_workspace(64, 0.5, _box(), None, None, nc) > 0 and list(nc) == [1, 1, 1]
    assert L.nbk_fof_workspace(10, 0.3, None, darr([0, 0, 0]), darr([1, 0, 2]), nc) > 0 and list(nc) == [3, 1, 6]


def test_bucket_and_link_validate(L):
    from nbodykit_b200._lib import darr
    assert L.nbk_fof_bucket(None, 3, 10, 0.1, _box(), None, None, None, 0, None, None, None) == -1
    assert b"4 = f4 or 8 = f8" in _err(L)
    wb = L.nbk_fof_workspace(10, 0.1, _box(), None, None, None)
    assert L.nbk_fof_bucket(None, F8, 10, 0.1, _box(), None, None, None, wb - 1, None, None, None) == -1
    assert b"workspace" in _err(L) and b"too small" in _err(L)
    assert L.nbk_fof_link(None, F4, 10, -2., _box(), None, None, None, wb, None, None) == -1 and b"> 0" in _err(L)
    assert L.nbk_fof_link(None, 16, 10, 0.1, _box(), None, None, None, wb, None, None) == -1 and b"dtype" in _err(L)
    assert L.nbk_fof_link(None, F4, 10, 0.1, darr([1, 1, -1]), None, None, None, wb, None, None) == -1
    assert b"box sides" in _err(L)
    assert L.nbk_fof_bucket(None, F8, 10, 0.1, _box(), None, None, None, wb, None, None, None) == -1
    assert b"null buffer" in _err(L)
    # nothing to do -> success without CUDA
    assert L.nbk_fof_bucket(None, F8, 0, 0.1, _box(), None, None, None, L.nbk_fof_workspace(0, 0.1, _box(), None, None, None),
                            None, None, None) == 0


def test_compress_minid_reduce_validate(L):
    from nbodykit_b200._lib import darr
    assert L.nbk_fof_compress(None, -5, None, None, None) == -1 and b"2^31-1" in _err(L)
    assert L.nbk_fof_minid(None, 2 ** 31, None, 0, None, None, None) == -1 and b"2^31-1" in _err(L)
    assert L.nbk_fof_minid(None, 10, None, -1, None, None, None) == -1 and b"offset" in _err(L)
    r = L.nbk_fof_reduce
    assert r(3, None, 10, None, 10, None, F8, 3, None, None, None, None, 4, None, None, None, None) == -1
    assert b"0 = sum, 1 = min, 2 = max" in _err(L)
    assert r(0, None, 10, None, 10, ctypes.c_void_p(8), 2, 3, None, None, None, None, 4, None, None, None, None) == -1
    assert b"4 = f4 or 8 = f8" in _err(L)
    assert r(0, None, 10, None, 10, ctypes.c_void_p(8), F8, 4, None, None, None, None, 4, None, None, None, None) == -1
    assert b"dim" in _err(L)
    assert r(0, None, 10, None, 10, None, F8, 3, None, None, None, None, 0, None, None, None, None) == -1
    assert b"ngroups" in _err(L)
    assert r(0, None, 10, None, 9, None, F8, 3, None, None, None, None, 4, None, None, None, ctypes.c_void_p(8)) == -1
    assert b"n_visit" in _err(L)
    assert r(0, None, 10, None, 10, ctypes.c_void_p(8), F8, 3, None, _box(), None, None, 4, ctypes.c_void_p(8), None,
             None, None) == -1 and b"anchors" in _err(L)
    assert r(1, None, 10, None, 10, ctypes.c_void_p(8), F8, 3, None, None, None, None, 4, None, None, None, None) == -1
    assert b"okey" in _err(L)


# ---- the oracle -----------------------------------------------------------------------------------------------------
def test_oracle_grid_links():
    from oracle import fof_oracle as fo
    g = np.indices((4, 4, 4)).reshape(3, -1).T.astype('f8')
    # spacing 1: ll 0.9 links nothing, ll 1.0 links all (separation <= ll), periodic or not
    assert len(np.unique(fo.components(g, 0.9, 4.))) == 64
    assert len(np.unique(fo.components(g, 1.0, 4.))) == 1
    assert len(np.unique(fo.components(g, 1.0))) == 1
    assert len(fo.near_ties(g, 1.0, 4.)) == 3 * 64 and len(fo.near_ties(g, 0.9, 4.)) == 0


def test_oracle_periodic_pairs_and_labels():
    from oracle import fof_oracle as fo
    pos = np.array([[0.1, 5, 5], [9.9, 5, 5], [5, 5, 5], [5.5, 5, 5], [5.9, 5, 5], [2, 2, 2]])
    assert list(fo.components(pos, 0.55, 10.)) == [0, 0, 2, 2, 2, 5]
    assert list(fo.components(pos, 0.55)) == [0, 1, 2, 2, 2, 5]
    # sizes 2, 3, 1 -> the triple is label 1, the pair 2, the single is below nmin = 1
    assert list(fo.labels(pos, 0.55, 1, 10.)) == [2, 2, 1, 1, 1, 0]
    # ties by smallest row
    assert list(fo.assign_labels(np.array([4, 4, 0, 0, 7]), 0)) == [2, 2, 1, 1, 3]
    # label 0 excludes groups of exactly nmin
    assert list(fo.assign_labels(np.array([4, 4, 0, 0, 0]), 2)) == [0, 0, 1, 1, 1]


def test_oracle_periodic_center_of_mass():
    from oracle import fof_oracle as fo
    pos = np.array([[9.8, 1, 1], [0.2, 1, 1], [5, 5, 5]])
    vel = np.array([[1., 0, 0], [3, 0, 0], [0, 0, 0]])
    f = fo.find_features(np.array([1, 1, 0]), pos, vel, boxsize=10., peak=np.array([1., 2., 0.]))
    np.testing.assert_allclose(f['CMPosition'][1], [0.0, 1, 1], atol=1e-12)
    np.testing.assert_allclose(f['CMVelocity'][1], [2., 0, 0])
    np.testing.assert_allclose(f['PeakPosition'][1], [0.2, 1, 1])
    assert list(f['Length']) == [0, 2]
    f = fo.find_features(np.array([1, 1, 1]), pos, vel, boxsize=10.)
    assert np.isnan(f['CMPosition'][0]).all()
