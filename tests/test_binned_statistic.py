"""BinnedStatistic against states recorded from the reference implementation (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest

from nbodykit_b200.binned_statistic import BinnedStatistic

GOLD = os.path.join(os.path.dirname(__file__), "golden", "binned_statistic_state.json")


@pytest.fixture(scope="module")
def gold():
    return json.load(open(GOLD))


@pytest.fixture()
def ds(gold):
    i = gold["input"]
    dt = np.dtype([("k", "f8"), ("mu", "f8"), ("power", "c16"), ("modes", "i8")])
    data = np.empty((10, 5), dtype=dt)
    data["k"] = i["k"]; data["mu"] = i["mu"]; data["modes"] = i["modes"]
    re, im = np.array(i["power_re"]), np.array(i["power_im"])
    re[re == -999.] = np.nan; im[im == -999.] = np.nan
    data["power"] = re + 1j * im
    return BinnedStatistic(["k", "mu"], [np.array(i["kedges"]), np.array(i["muedges"])], data,
                           fields_to_sum=["modes"], N1=10, shotnoise=1.5)


def _check(o, g):
    assert o.dims == g["dims"]
    for d, e, c in zip(o.dims, g["edges"], g["coords"]):
        np.testing.assert_allclose(o.edges[d], e, rtol=1e-14)
        np.testing.assert_allclose(o.coords[d], c, rtol=1e-14)
    assert o.mask.tolist() == g["mask"]
    assert o["modes"].tolist() == g["modes"]
    np.testing.assert_allclose(np.nan_to_num(o["power"].real, nan=-999.), g["power_re"], rtol=1e-13)
    np.testing.assert_allclose(np.nan_to_num(o["k"], nan=-999.), g["k"], rtol=1e-13)


def test_matches_reference_states(ds, gold):
    _check(ds, gold["full"])
    _check(ds[2:7], gold["slice_k"])
    _check(ds[:, 1], gold["slice_int"])
    _check(ds.sel(mu=slice(-0.6, 0.6), method="nearest"), gold["sel_mu"])
    _check(ds.sel(k=0.35, method="nearest"), gold["sel_k_scalar"])
    _check(ds.take(k=[1, 3, 5]), gold["take"])
    _check(ds.average("mu"), gold["average_mu"])
    _check(ds.reindex("k", 0.2), gold["reindex_k"])
    _check(ds.reindex("k", 0.2, weights="modes"), gold["reindex_k_weighted"])
    _check(ds[:, [2]].squeeze(), gold["squeeze"])


def test_protocol(ds):
    assert ds.shape == (10, 5) and ds.variables == ["k", "mu", "power", "modes"]
    assert "power" in ds and list(ds) == ds.variables
    assert ds.attrs["N1"] == 10
    sub = ds[["k", "power"]]
    assert sub.variables == ["k", "power"]
    with pytest.raises(KeyError):
        ds["nope"]
    with pytest.raises(KeyError):
        ds[["k", "nope"]]
    with pytest.raises(IndexError):
        ds[0, 0]
    with pytest.raises(IndexError):
        ds.sel(k=0.123)
    ds["extra"] = np.ones((10, 5))
    assert "extra" in ds.variables
    with pytest.raises(ValueError):
        ds["bad"] = np.ones(3)
    ds.rename_variable("extra", "renamed")
    assert "renamed" in ds and "extra" not in ds
    c = ds.copy()
    c["k"][:] = 0
    assert not np.all(ds["k"] == 0)
    with pytest.raises(ValueError):
        ds.squeeze()
    with pytest.raises(TypeError):
        BinnedStatistic(["k"], [np.arange(3)], np.zeros(2))
    with pytest.raises(ValueError):
        BinnedStatistic(["k"], [np.arange(4)], np.zeros(2, dtype=[("a", "f8")]))


def test_json_roundtrip(ds, tmp_path):
    fn = str(tmp_path / "ds.json")
    ds.to_json(fn)
    back = BinnedStatistic.from_json(fn)
    assert back.dims == ds.dims and back.attrs["shotnoise"] == 1.5
    for name in ds.variables:
        np.testing.assert_array_equal(np.nan_to_num(back[name]), np.nan_to_num(ds[name]))
    assert back.mask.tolist() == ds.mask.tolist()


def test_reads_reference_fixture_json():
    """a result file written by the reference (its nbodykit/tests/data/dataset_2d.json, copied verbatim) loads unchanged"""
    ds = BinnedStatistic.from_json(os.path.join(os.path.dirname(GOLD), "dataset_2d.json"))
    assert ds.dims == ["k", "mu"] and ds.shape == (64, 5)
    assert ds.attrs["N1"] == 4033
    assert int(np.nansum(ds["modes"])) == 1097911
