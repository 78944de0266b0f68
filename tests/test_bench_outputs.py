"""bench.py --dump-outputs: what the timed call returned, as float32 / float64 .npy files (no GPU needed)."""
import os
import types

import numpy as np

from nbodykit_b200.binned_statistic import BinnedStatistic


def test_dump_outputs_writes_every_column_as_real_floats(tmp_path):
    import bench
    kedges, muedges = np.linspace(0, 1, 5), np.linspace(-1, 1, 3)
    data = np.zeros((4, 2), dtype=[("k", "f8"), ("mu", "f4"), ("power", "c16"), ("modes", "i8")])
    data["k"] = np.arange(8.).reshape(4, 2)
    data["mu"] = 0.5
    data["power"] = np.arange(8).reshape(4, 2) * (1 - 2j)
    data["modes"] = 2 ** 40 + 3
    attrs = {"shotnoise": 1.5, "N1": 10, "Nmesh": np.array([8, 8, 8]), "mode": "2d", "kmax": None, "poles": []}
    power = BinnedStatistic(["k", "mu"], [kedges, muedges], data, **attrs)
    poles = BinnedStatistic(["k"], [kedges], np.zeros(4, dtype=[("k", "f8"), ("power_0", "c8")]), **attrs)
    bench.dump_outputs(types.SimpleNamespace(power=power, poles=poles, attrs=attrs), str(tmp_path / "out"))

    got = {f[:-4]: np.load(str(tmp_path / "out" / f)) for f in os.listdir(str(tmp_path / "out"))}
    assert sorted(got) == sorted([
        "power.k", "power.mu", "power.power.real", "power.power.imag", "power.modes", "power.edges.k", "power.edges.mu",
        "poles.k", "poles.power_0.real", "poles.power_0.imag", "poles.edges.k",
        "attrs.shotnoise", "attrs.N1", "attrs.Nmesh"])
    assert all(a.dtype in (np.float32, np.float64) and a.size for a in got.values())
    assert got["power.mu"].dtype == np.float32 and got["poles.power_0.real"].dtype == np.float32
    np.testing.assert_array_equal(got["power.power.imag"], -2 * data["k"])
    assert (got["power.modes"] == 2 ** 40 + 3).all()
    np.testing.assert_array_equal(got["power.edges.mu"], muedges)
    np.testing.assert_array_equal(got["attrs.Nmesh"], [8., 8., 8.])
