"""
Generates the golden vectors under tests/golden/ by running the REFERENCE's own code
(/root/reference, loaded verbatim by oracle/refload.py) in the build container.  The GPU box has no
/root/reference, so the outputs are committed.  Re-run: `python tests/golden/make_golden.py`.

  project_to_basis_*.npz : inputs (seeded complex field, edges, los, poles) + outputs of the reference's
                           nbodykit.algorithms.fftpower.project_to_basis on float32 / float64 coordinates
  compensate.npz         : the six Compensate* transfer functions of source/mesh/catalog.py evaluated by
                           the reference on float32 circular coordinates
  mpirng.npz             : MPIRandomState streams (uniform / normal / poisson) + UniformCatalog N
  dataset_2d_modes.json  : sum over mu of `modes` in nbodykit/tests/data/dataset_2d.json
  binned_statistic_state.json : BinnedStatistic.__getstate__ of reference objects after slicing/reindexing
  dataset_2d.json        : nbodykit/tests/data/dataset_2d.json, copied verbatim (a result file the reference wrote)
  oracle_vs_reference.npz : the reference's outputs for the cases of tests/test_oracle_vs_reference.py; the long
                           random streams are stored as a SHA-256 digest of their bytes plus 257 evenly spaced rows
"""
import hashlib
import json
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import refload, pmesh_oracle as po  # noqa: E402

ns = refload.load()


def field(N, seed, cdtype):
    rng = np.random.RandomState(seed)
    shape = (N[0], N[1], N[2] // 2 + 1)
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(cdtype)


def golden_project():
    cases = [
        dict(name="a", N=[16, 16, 16], L=[64.] * 3, cd="c16", coord="f4", Nmu=1, poles=[], los=[0, 0, 1]),
        dict(name="b", N=[16, 16, 16], L=[64.] * 3, cd="c16", coord="f4", Nmu=5, poles=[0, 2, 4], los=[0, 0, 1]),
        dict(name="c", N=[8, 16, 32], L=[10., 20., 30.], cd="c8", coord="f4", Nmu=4, poles=[1, 2], los=[0, 1, 0]),
        dict(name="d", N=[16, 16, 16], L=[100.] * 3, cd="c16", coord="f8", Nmu=3, poles=[2], los=[0.6, 0, 0.8]),
        dict(name="e", N=[32, 32, 32], L=[1024.] * 3, cd="c8", coord="f4", Nmu=1, poles=[], los=[1, 0, 0]),
    ]
    for c in cases:
        y = field(c["N"], 11, c["cd"])
        x = po.k_coords(c["N"], c["L"], c["coord"])
        dk = 2 * np.pi / min(c["L"])
        kedges = np.arange(0., np.pi * min(c["N"]) / max(c["L"]) + dk / 2, dk)
        muedges = np.linspace(-1, 1, c["Nmu"] + 1)
        f = refload.RefComplexField(y, x)
        res, pres = ns.project_to_basis(f, [kedges, muedges], los=c["los"], poles=c["poles"])
        out = dict(N=np.array(c["N"]), L=np.array(c["L"]), seed=11, cdtype=c["cd"], coord=c["coord"], kedges=kedges,
                   muedges=muedges, los=np.array(c["los"], dtype="f8"), poles=np.array(c["poles"], dtype="i8"),
                   xmean=res[0], mumean=res[1], y2d=res[2], N2d=res[3])
        if pres is not None:
            out.update(pole_k=pres[0], pole_y=pres[1], pole_N=pres[2])
        np.savez_compressed(os.path.join(HERE, "project_to_basis_%s.npz" % c["name"]), **out)


def golden_compensate():
    N, L = [16, 8, 32], [10., 20., 30.]
    w = po.k_coords(N, L, "f4", kind="circular")
    v = field(N, 2, "c16")
    out = dict(N=np.array(N), L=np.array(L), seed=2)
    for interlaced in (True, False):
        for res in ("cic", "tsc", "pcs"):
            mode, func, kind = ns.get_compensation(interlaced, res)[0]
            assert (mode, kind) == ("complex", "circular")
            out[func.__name__] = func(w, v.copy())
    np.savez_compressed(os.path.join(HERE, "compensate.npz"), **out)


def golden_mpirng():
    comm = ns.FakeComm()
    out = {}
    rng = ns.MPIRandomState(comm, seed=42, size=250000)
    u1 = rng.uniform(itemshape=(3,))
    u2 = rng.uniform(itemshape=(3,))
    out["uniform_first"] = u1[:5]
    out["uniform_rows"] = u1[[0, 99999, 100000, 199999, 200000, 249999]]
    out["uniform_sum"] = np.array([u1.sum(), u2.sum()])
    out["normal_rows"] = rng.normal(loc=1.0, scale=2.0)[[0, 100000, 249999]]
    lam = np.linspace(0.1, 5.0, 250000)
    p = rng.poisson(lam=lam)
    out["poisson_rows"] = p[[0, 100000, 249999]]
    out["poisson_sum"] = np.array([p.sum()])
    out["N_uniformcatalog"] = np.array([np.random.RandomState(42).poisson(1e5), np.random.RandomState(42).poisson(100)])
    np.savez_compressed(os.path.join(HERE, "mpirng.npz"), **out)


def golden_dataset2d():
    src = os.path.join(refload.REF, "nbodykit/tests/data/dataset_2d.json")
    shutil.copyfile(src, os.path.join(HERE, "dataset_2d.json"))
    d = json.load(open(src))
    dt = [tuple(x) for x in d["data"]["__dtype__"]]
    names = [x[0] for x in dt]
    modes = np.array([[rec[names.index("modes")] for rec in row] for row in d["data"]["__data__"]])
    json.dump({"Nmesh": 128, "BoxSize": 512.0,
               "source": "nbodykit/tests/data/dataset_2d.json (sum over mu of modes)",
               "modes_k": [int(v) for v in modes.sum(axis=1)]},
              open(os.path.join(HERE, "dataset_2d_modes.json"), "w"))


def golden_binned_statistic():
    """exercise the reference BinnedStatistic and record the resulting states"""
    from nbodykit.utils import FrontPadArray  # noqa: F401  (stub)
    BS = ns.BinnedStatistic
    rng = np.random.RandomState(5)
    kedges = np.linspace(0, 1.0, 11)
    muedges = np.linspace(-1, 1, 6)
    dt = np.dtype([("k", "f8"), ("mu", "f8"), ("power", "c16"), ("modes", "i8")])
    data = np.empty((10, 5), dtype=dt)
    data["k"] = rng.uniform(size=(10, 5)); data["mu"] = rng.uniform(size=(10, 5))
    data["power"] = rng.standard_normal((10, 5)) + 1j * rng.standard_normal((10, 5))
    data["modes"] = rng.randint(1, 100, size=(10, 5))
    data["power"][0, 0] = np.nan
    ds = BS(["k", "mu"], [kedges, muedges], data, fields_to_sum=["modes"], N1=10, shotnoise=1.5)

    def state(o):
        s = o.__getstate__()
        return dict(dims=s["dims"], edges=[np.asarray(e).tolist() for e in s["edges"]],
                    coords=[np.asarray(c).tolist() for c in s["coords"]],
                    mask=o.mask.tolist(), modes=o["modes"].tolist(),
                    power_re=np.nan_to_num(o["power"].real, nan=-999.).tolist(),
                    k=np.nan_to_num(o["k"], nan=-999.).tolist())

    out = dict(
        input=dict(kedges=kedges.tolist(), muedges=muedges.tolist(),
                   k=data["k"].tolist(), mu=data["mu"].tolist(), power_re=np.nan_to_num(data["power"].real, nan=-999.).tolist(),
                   power_im=np.nan_to_num(data["power"].imag, nan=-999.).tolist(), modes=data["modes"].tolist()),
        full=state(ds),
        slice_k=state(ds[2:7]),
        slice_int=state(ds[:, 1]),
        sel_mu=state(ds.sel(mu=slice(-0.6, 0.6), method="nearest")),
        sel_k_scalar=state(ds.sel(k=0.35, method="nearest")),
        take=state(ds.take(k=[1, 3, 5])),
        average_mu=state(ds.average("mu")),
        reindex_k=state(ds.reindex("k", 0.2)),
        reindex_k_weighted=state(ds.reindex("k", 0.2, weights="modes")),
        squeeze=state(ds[:, [2]].squeeze()),
    )
    json.dump(out, open(os.path.join(HERE, "binned_statistic_state.json"), "w"))


# the cases of tests/test_oracle_vs_reference.py (same order as its parametrisation)
PROJECT_CASES = [
    ([16, 16, 16], [64.] * 3, "c16", "f4", 5, [0, 2, 4], [0, 0, 1]),
    ([12, 8, 10], [100., 50., 70.], "c8", "f4", 3, [1, 2], [0, 1, 0]),
    ([16, 16, 16], [100.] * 3, "c16", "f8", 4, [3], [0.6, 0.0, 0.8]),
    ([8, 8, 8], [1.] * 3, "c16", "f4", 1, [], [0, 0, 1]),
]


def stream_digest(a):
    """(sha256 of dtype, shape and bytes, 257 evenly spaced rows): an exact fingerprint of an array too large to store"""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest(), a[np.linspace(0, len(a) - 1, 257).astype("i8")]


def golden_oracle_vs_reference():
    out = {}
    for i, (N, L, cd, coord, Nmu, poles, los) in enumerate(PROJECT_CASES):
        rng = np.random.RandomState(3)
        shape = (N[0], N[1], N[2] // 2 + 1)
        y = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(cd)
        x = po.k_coords(N, L, coord)
        dk = 2 * np.pi / min(L)
        kedges = np.arange(0., np.pi * min(N) / max(L) + dk / 2, dk)
        muedges = np.linspace(-1, 1, Nmu + 1)
        res, pres = ns.project_to_basis(refload.RefComplexField(y, x), [kedges, muedges], los=los, poles=poles)
        for j in range(4):
            out["project%d_res%d" % (i, j)] = res[j]
        if poles:
            for j in range(3):
                out["project%d_pole%d" % (i, j)] = pres[j]

    N, L = [8, 16, 12], [10., 20., 30.]
    rng = np.random.RandomState(4)
    v = rng.standard_normal((8, 16, 7)) + 0j
    for coord in ["f4", "f8"]:
        w = po.k_coords(N, L, coord, kind="circular")
        for interlaced in (True, False):
            for res in ("cic", "tsc", "pcs"):
                func = ns.get_compensation(interlaced, res)[0][1]
                key = "comp_%s_%d_%s" % (coord, interlaced, res)
                out[key + "_name"] = np.array(func.__name__)
                out[key] = func(w, v.copy())

    def stream(key, a):
        digest, rows = stream_digest(a)
        out[key + "_sha256"] = np.array(digest)
        out[key + "_rows"] = rows

    ref = ns.MPIRandomState(ns.FakeComm(), seed=7, size=123456)
    stream("mpirng_uniform", ref.uniform(itemshape=(3,)))
    stream("mpirng_normal", ref.normal())
    ref = ns.MPIRandomState(ns.FakeComm(), seed=9, size=250001)
    stream("product_uniform", ref.uniform(itemshape=(3,)))
    stream("product_poisson", ref.poisson(lam=np.linspace(0.5, 3, 250001)))
    stream("product_normal", ref.normal(loc=1., scale=3.))
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **out)


if __name__ == "__main__":
    golden_project()
    golden_compensate()
    golden_mpirng()
    golden_dataset2d()
    golden_binned_statistic()
    golden_oracle_vs_reference()
    print("golden vectors written to", HERE)


def golden_ylm():
    """values of the REFERENCE's get_real_Ylm (algorithms/convpower/fkp.py:12-73, executed from its source with
    sympy.lambdify's 'numexpr' backend swapped for 'numpy') on seeded unit vectors and at the origin"""
    import ast
    import sympy
    src = open(os.path.join(refload.REF, "nbodykit/algorithms/convpower/fkp.py")).read()
    tree = ast.parse(src)
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "get_real_Ylm"][0]
    code = compile(ast.Module(body=[fn], type_ignores=[]), "fkp.py:get_real_Ylm", "exec")
    ns_ = {"numpy": np}
    exec(code, ns_)
    orig = sympy.lambdify
    sympy.lambdify = lambda args, expr, modules=None, **kw: orig(args, expr, "numpy", **kw)
    try:
        rng = np.random.RandomState(3)
        v = rng.standard_normal((64, 3))
        v /= np.sqrt((v ** 2).sum(axis=1))[:, None]
        out = {"vec": v}
        for l in range(0, 5):
            for m in range(-l, l + 1):
                f = ns_["get_real_Ylm"](l, m)
                val = np.broadcast_to(np.asarray(f(v[:, 0], v[:, 1], v[:, 2]), dtype="f8"), (64,))
                out["Y_%d_%d" % (l, m)] = val.copy()
                out["Y0_%d_%d" % (l, m)] = np.array(float(f(0.0, 0.0, 0.0)))
    finally:
        sympy.lambdify = orig
    np.savez_compressed(os.path.join(HERE, "ylm_reference.npz"), **out)


if __name__ == "__main__":
    golden_ylm()
    print("ylm golden written")
