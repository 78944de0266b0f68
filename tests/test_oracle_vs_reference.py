"""Pin the oracle restatement against the reference's own code: the reference's outputs for these cases are stored in
tests/golden/oracle_vs_reference.npz (tests/golden/make_golden.py runs the reference to write them)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import pmesh_oracle as po

GOLD = os.path.join(os.path.dirname(__file__), "golden", "oracle_vs_reference.npz")
# project_to_basis cases, in the order of the stored reference outputs
CASES = [
    ([16, 16, 16], [64.] * 3, "c16", "f4", 5, [0, 2, 4], [0, 0, 1]),
    ([12, 8, 10], [100., 50., 70.], "c8", "f4", 3, [1, 2], [0, 1, 0]),
    ([16, 16, 16], [100.] * 3, "c16", "f8", 4, [3], [0.6, 0.0, 0.8]),
    ([8, 8, 8], [1.] * 3, "c16", "f4", 1, [], [0, 0, 1]),
]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _assert_stream_equal(got, gold, key):
    """`got` equals, bit for bit, the reference stream stored as a SHA-256 digest plus 257 evenly spaced rows"""
    got = np.ascontiguousarray(got)
    np.testing.assert_array_equal(got[np.linspace(0, len(got) - 1, 257).astype("i8")], gold[key + "_rows"])
    h = hashlib.sha256(("%s%s" % (got.dtype.str, got.shape)).encode())
    h.update(got.tobytes())
    assert h.hexdigest() == str(gold[key + "_sha256"]), "%s differs from the reference stream" % key


@pytest.mark.parametrize("N,L,cd,coord,Nmu,poles,los", CASES)
def test_project_to_basis(gold, N, L, cd, coord, Nmu, poles, los):
    case = CASES.index((N, L, cd, coord, Nmu, poles, los))
    rng = np.random.RandomState(3)
    shape = (N[0], N[1], N[2] // 2 + 1)
    y = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(cd)
    x = po.k_coords(N, L, coord)
    dk = 2 * np.pi / min(L)
    kedges = np.arange(0., np.pi * min(N) / max(L) + dk / 2, dk)
    muedges = np.linspace(-1, 1, Nmu + 1)
    ref = [gold["project%d_res%d" % (case, j)] for j in range(4)]
    got, pgot = po.project_to_basis(y, x, [kedges, muedges], los=los, poles=poles)
    assert np.array_equal(ref[3], got[3])
    tol = 1e-12 if cd == "c16" else 1e-6
    for a, b in zip(ref[:3], got[:3]):
        np.testing.assert_allclose(b, a, rtol=tol, atol=tol, equal_nan=True)
    if poles:
        pref = [gold["project%d_pole%d" % (case, j)] for j in range(3)]
        assert np.array_equal(pref[2], pgot[2])
        np.testing.assert_allclose(pgot[1], pref[1], rtol=tol, atol=tol, equal_nan=True)


def test_compensation_functions(gold):
    N, L = [8, 16, 12], [10., 20., 30.]
    rng = np.random.RandomState(4)
    v = rng.standard_normal((8, 16, 7)) + 0j
    for coord in ["f4", "f8"]:
        w = po.k_coords(N, L, coord, kind="circular")
        for interlaced in (True, False):
            for res in ("cic", "tsc", "pcs"):
                key = "comp_%s_%d_%s" % (coord, interlaced, res)
                name = str(gold[key + "_name"])
                assert name == po.COMPENSATION[(interlaced, res)]
                np.testing.assert_array_equal(po.compensate(name, w, v.copy()), gold[key])


def test_mpirng(gold):
    mine = po.SerialMPIRandomState(7, 123456)
    _assert_stream_equal(mine.uniform(itemshape=(3,)), gold, "mpirng_uniform")
    _assert_stream_equal(mine.normal(), gold, "mpirng_normal")


def test_product_mpirng_matches_reference(gold):
    from nbodykit_b200.mpirng import MPIRandomState
    from nbodykit_b200.comm import SelfComm
    mine = MPIRandomState(SelfComm(), seed=9, size=250001)
    _assert_stream_equal(mine.uniform(itemshape=(3,)), gold, "product_uniform")
    lam = np.linspace(0.5, 3, 250001)
    _assert_stream_equal(mine.poisson(lam=lam), gold, "product_poisson")
    _assert_stream_equal(mine.normal(loc=1., scale=3.), gold, "product_normal")
