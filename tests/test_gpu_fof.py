"""
FOF on the GPU: the reference's own cases (algorithms/tests/test_fof.py), exact label parity with the CPU oracle
(oracle/fof_oracle.py: cKDTree pairs + connected components) on uniform, log-normal and clumpy inputs in f4 and f8,
periodic and not, several ranks emulated by threads on one GPU, and FFTPower of the groups found.  Inputs are checked
to have no pair within a relative 1e-9 of the linking length, so partitions must agree exactly.
"""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fof_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cat(cols, box=None, comm=None, **attrs):
    from nbodykit_b200.comm import SelfComm
    from nbodykit_b200.lab import ArrayCatalog
    if box is not None:
        attrs['BoxSize'] = box
    return ArrayCatalog(cols, comm=comm or SelfComm(), **attrs)


def _grid(n, shift=0.5):
    return (np.indices((n, n, n)).reshape(3, -1).T + shift).astype('f8')


def _plummer(rng, n, center, a):
    r = a / np.sqrt(rng.uniform(1e-3, 1, n) ** (-2. / 3) - 1)
    r = np.minimum(r, 10 * a)
    v = rng.standard_normal((n, 3))
    return center + v / np.linalg.norm(v, axis=1)[:, None] * r[:, None]


def clumpy(seed=5, L=100., n_bg=3000, dtype='f8'):
    """seeded Plummer spheres (one centred on a box corner, straddling every periodic face) on a uniform background"""
    rng = np.random.RandomState(seed)
    parts = [_plummer(rng, 4000, np.zeros(3), 1.5)]
    for k in range(8):
        parts.append(_plummer(rng, int(rng.randint(200, 2000)), rng.uniform(10, 90, 3), rng.uniform(0.5, 2.0)))
    parts.append(rng.uniform(0, L, (n_bg, 3)))
    pos = np.concatenate(parts) % L
    pos = pos[rng.permutation(len(pos))]
    vel = rng.standard_normal(pos.shape) * 3.0
    return pos.astype(dtype), vel.astype(dtype)


def _features_match(got, want, L=None):
    """Length exact; centres of mass to 1e-6 of the box (periodic) or of the column's scale"""
    np.testing.assert_array_equal(np.asarray(got['Length']), want['Length'])
    for name, w in want.items():
        if name == 'Length':
            continue
        g = np.asarray(got[name]).astype('f8')
        assert g.shape == w.shape, name
        nan = np.isnan(w)
        assert np.array_equal(np.isnan(g), nan), name
        d = np.where(nan, 0, g - w)
        if L is not None and name in ('CMPosition', 'PeakPosition', 'InitialPosition'):
            d = (d + 0.5 * L) % L - 0.5 * L
            scale = L
        else:
            scale = np.nanmax(np.abs(w)) if np.isfinite(w).any() else 1.0
        assert np.abs(d).max() <= 1e-6 * scale, "%s: max deviation %.3g, scale %.3g" % (name, np.abs(d).max(), scale)


def _parity(pos, vel, ll, nmin, L, periodic, extra=None, peak=None):
    from nbodykit_b200.lab import FOF
    box = L if periodic else None
    assert len(fo.near_ties(pos, ll, box)) == 0, "input has a pair at the linking length"
    cols = {'Position': pos, 'Velocity': vel}
    cols.update(extra or {})
    if peak is not None:
        cols['Peak'] = peak
    cat = _cat(cols, box=L if periodic else None)
    f = FOF(cat, ll, nmin, absolute=True, periodic=periodic)
    want = fo.labels(pos, ll, nmin, box)
    got = f.labels.cpu().numpy()
    assert f.labels.dtype.__str__() == 'torch.int32'
    np.testing.assert_array_equal(got, want)
    assert f.max_label == [int(want.max())]
    h = f.find_features(peakcolumn='Peak' if peak is not None else None)
    wf = fo.find_features(want, pos, vel, boxsize=box, peak=peak,
                          initpos=(extra or {}).get('InitialPosition'))
    _features_match(h, wf, L if periodic else None)
    return f, h


# ---- the reference's cases ---------------------------------------------------------------------------------------
def test_unit_grid_every_particle_alone(cuda):
    from nbodykit_b200.lab import FOF
    cat = _cat({'Position': _grid(8)}, box=8., Nmesh=np.array([8, 8, 8]))
    f = FOF(cat, linking_length=0.9, nmin=0)
    # one particle per group; equal Lengths are ordered by row
    np.testing.assert_array_equal(f.labels.cpu().numpy(), np.arange(1, 513))
    assert f.max_label == [512]


def test_four_offset_grids_merge_in_fours(cuda):
    from nbodykit_b200.lab import FOF
    Q = _grid(8, shift=0)
    pos = np.concatenate([Q, Q + 0.01, Q - 0.01, Q + 0.02])
    f = FOF(_cat({'Position': pos}, box=8.), linking_length=0.011 * 3 ** 0.5, nmin=0, absolute=True)
    lab = f.labels.cpu().numpy()
    assert lab.max() == 512 and lab.min() == 1
    assert (np.bincount(lab)[1:] == 4).all()
    np.testing.assert_array_equal(lab, fo.labels(pos, 0.011 * 3 ** 0.5, 0, 8.))


def test_fully_connected_two_cells_per_axis(cuda):
    from nbodykit_b200.lab import FOF
    f = FOF(_cat({'Position': _grid(4, shift=0)}, box=4.), linking_length=2, nmin=63, absolute=True)
    np.testing.assert_array_equal(f.labels.cpu().numpy(), 1)


def test_nonperiodic_translation_invariance(cuda):
    from nbodykit_b200.lab import FOF
    pos, vel = clumpy(seed=11)
    dens = np.random.RandomState(3).uniform(size=len(pos))
    assert len(fo.near_ties(pos, 0.3)) == 0
    peaks = []
    for shift in (-100.0, 100.0):
        cat = _cat({'Position': pos + shift, 'Velocity': vel, 'Density': dens})
        f = FOF(cat, linking_length=0.3, nmin=20, periodic=False, absolute=True)
        peaks.append(f.find_features(peakcolumn='Density'))
    p1, p2 = peaks
    assert np.asarray(p1['Length'])[1:].min() > 20
    np.testing.assert_allclose(np.asarray(p1['CMPosition']) + 200.0, np.asarray(p2['CMPosition']), rtol=1e-6)
    np.testing.assert_allclose(np.asarray(p1['CMVelocity']), np.asarray(p2['CMVelocity']), rtol=1e-6)
    np.testing.assert_allclose(np.asarray(p1['PeakPosition']) + 200.0, np.asarray(p2['PeakPosition']), rtol=1e-6)
    np.testing.assert_allclose(np.asarray(p1['PeakVelocity']), np.asarray(p2['PeakVelocity']), rtol=1e-6)


# ---- parity with the oracle --------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f4", "f8"])
@pytest.mark.parametrize("periodic", [True, False])
def test_uniform_parity(cuda, dtype, periodic):
    from nbodykit_b200.lab import UniformCatalog
    cat = UniformCatalog(nbar=2e-1, BoxSize=64., seed=21, dtype=dtype)
    pos, vel = np.asarray(cat['Position']), np.asarray(cat['Velocity'])
    ll = 0.2 * (64. ** 3 / len(pos)) ** (1 / 3.)
    _parity(pos, vel, ll, 2, 64., periodic)


@pytest.mark.parametrize("dtype", ["f4", "f8"])
@pytest.mark.parametrize("periodic", [True, False])
def test_clumpy_parity(cuda, dtype, periodic):
    pos, vel = clumpy(dtype=dtype)
    rng = np.random.RandomState(8)
    init = (pos + rng.uniform(-2, 2, pos.shape)).astype(dtype) % 100.
    peak = rng.uniform(size=len(pos))
    f, h = _parity(pos, vel, 0.25, 20, 100., periodic, extra={'InitialPosition': init}, peak=peak)
    if periodic:
        assert np.asarray(h['Length'])[1] >= 1000      # the corner sphere is found whole across the faces


def test_lognormal_parity(cuda):
    import torch
    from nbodykit_b200.cosmology import NoWiggleEHPower
    from nbodykit_b200.lab import LogNormalCatalog
    L = 256.
    cat = LogNormalCatalog(Plin=NoWiggleEHPower(), nbar=6e-2, BoxSize=L, Nmesh=64, bias=2.0, seed=42)
    pos = cat['Position'].compute()
    vel = cat['Velocity'].compute()
    assert isinstance(pos, torch.Tensor) and pos.is_cuda and 8e5 < len(pos) < 1.3e6
    pos, vel = pos.cpu().numpy(), vel.cpu().numpy()
    ll = 0.2 * (L ** 3 / len(pos)) ** (1 / 3.)
    f, h = _parity(pos, vel, ll, 20, L, True)
    assert f._ngroups > 50


# ---- the GPU path ------------------------------------------------------------------------------------------------
def test_launches_the_fof_kernels(cuda, monkeypatch):
    from nbodykit_b200 import _lib
    from nbodykit_b200.lab import FOF
    L = _lib.lib()
    called = []
    for name in ("nbk_fof_bucket", "nbk_fof_link", "nbk_fof_compress", "nbk_fof_minid", "nbk_fof_reduce"):
        orig = getattr(L, name)
        monkeypatch.setattr(L, name, (lambda o, nm: lambda *a: called.append(nm) or o(*a))(orig, name))
    pos, vel = clumpy()
    n0 = _lib.launch_count()
    f = FOF(_cat({'Position': pos, 'Velocity': vel}, box=100.), 0.25, 20, absolute=True)
    f.find_features()
    assert _lib.launch_count() - n0 >= 10
    assert set(called) == {"nbk_fof_bucket", "nbk_fof_link", "nbk_fof_compress", "nbk_fof_minid", "nbk_fof_reduce"}


def test_fftpower_of_the_haloes(cuda):
    from nbodykit_b200.lab import ArrayCatalog, FFTPower, FOF
    pos, vel = clumpy()
    halos = FOF(_cat({'Position': pos, 'Velocity': vel}, box=100.), 0.25, 5, absolute=True).find_features()
    assert np.isfinite(np.asarray(halos['CMPosition'])).all()
    r = FFTPower(ArrayCatalog({'Position': halos['CMPosition']}, BoxSize=100.), mode='1d', Nmesh=64)
    assert np.isfinite(r.power['power'].real).all() and r.attrs['N1'] == halos.csize


# ---- several ranks emulated by threads on one GPU ------------------------------------------------------------------
def _thread_comm_class():
    import torch
    from nbodykit_b200.comm import SelfComm

    class ThreadComm(SelfComm):
        """one rank per thread on one GPU: collectives through a shared list and a barrier"""

        def __init__(self, rank, P, shared):
            self._r, self._P, self._sh = rank, P, shared
        rank = property(lambda self: self._r)
        size = property(lambda self: self._P)

        def allgather(self, x):
            sh = self._sh
            sh['bar'].wait()
            sh['buf'][self._r] = x
            sh['bar'].wait()
            out = list(sh['buf'])
            sh['bar'].wait()
            return out

        def barrier(self):
            self._sh['bar'].wait()

        def bcast(self, x, root=0):
            return self.allgather(x)[root]

        def alltoall(self, xs):
            g = self.allgather(list(xs))
            return [g[src][self._r] for src in range(self._P)]

        def alltoall_ints(self, xs):
            return [int(v) for v in self.alltoall(xs)]

        def allreduce(self, x, op="sum"):
            if isinstance(x, torch.Tensor):
                return self.allreduce_tensor(x.clone(), op)
            vals = np.asarray(self.allgather(x))
            r = {"sum": np.sum, "min": np.min, "max": np.max}[op](vals, axis=0)
            return r.item() if np.ndim(r) == 0 else r

        def allreduce_floats(self, xs):
            return [float(v) for v in np.sum(self.allgather([float(x) for x in xs]), axis=0)]

        def allreduce_tensor(self, t, op="sum"):
            torch.cuda.synchronize()
            s = torch.stack(self.allgather(t.clone()))
            r = {"sum": lambda a: a.sum(0), "min": lambda a: a.amin(0), "max": lambda a: a.amax(0)}[op](s)
            t.copy_(r.to(t.dtype))
            torch.cuda.synchronize()
            self.barrier()
            return t

        def all_to_all_single(self, out, inp, out_splits=None, in_splits=None):
            torch.cuda.synchronize()
            P = self._P
            ins = in_splits if in_splits is not None else [inp.shape[0] // P] * P
            g = self.allgather((inp, list(ins)))
            pieces = []
            for src in range(P):
                t, sp = g[src]
                o = int(sum(sp[:self._r]))
                pieces.append(t[o:o + int(sp[self._r])])
            if out.shape[0]:
                out.copy_(torch.cat(pieces))
            torch.cuda.synchronize()
            self.barrier()
            return out

    return ThreadComm


def _run_ranks(P, fn):
    import torch
    ThreadComm = _thread_comm_class()
    shared = dict(buf=[None] * P, bar=threading.Barrier(P, timeout=300))
    res, errs = [None] * P, []

    def main(r):
        try:
            torch.cuda.set_device(0)
            res[r] = fn(ThreadComm(r, P, shared))
        except Exception as e:      # noqa: BLE001
            errs.append(e)
            shared['bar'].abort()
    th = [threading.Thread(target=main, args=(r,)) for r in range(P)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]
    return res


def _split(a, P, r):
    n = len(a)
    return a[r * n // P:(r + 1) * n // P]


def _multi_rank(P, pos, vel, ll, nmin, L, periodic, peak=None):
    """labels and features on P emulated ranks, gathered; and the merge iteration count"""
    from nbodykit_b200.lab import FOF

    def fn(comm):
        cols = {'Position': _split(pos, P, comm.rank), 'Velocity': _split(vel, P, comm.rank)}
        if peak is not None:
            cols['Peak'] = _split(peak, P, comm.rank)
        f = FOF(_cat(cols, box=L if periodic else None, comm=comm), ll, nmin, absolute=True, periodic=periodic)
        h = f.find_features(peakcolumn='Peak' if peak is not None else None)
        return f.labels.cpu().numpy(), {k: np.asarray(h[k]) for k in h.columns if k in
                                        ('CMPosition', 'CMVelocity', 'Length', 'PeakPosition', 'PeakVelocity')}, \
            f.merge_iterations, f.max_label
    res = _run_ranks(P, fn)
    labels = np.concatenate([r[0] for r in res])
    feats = {k: np.concatenate([r[1][k] for r in res]) for k in res[0][1]}
    return labels, feats, res[0][2], res[0][3]


@pytest.mark.parametrize("P", [2, 3])
@pytest.mark.parametrize("periodic", [True, False])
def test_emulated_ranks_match_one_rank(cuda, P, periodic):
    from nbodykit_b200.lab import FOF
    pos, vel = clumpy(seed=7)
    peak = np.random.RandomState(2).uniform(size=len(pos))
    box = 100. if periodic else None
    one = FOF(_cat({'Position': pos, 'Velocity': vel, 'Peak': peak}, box=box), 0.25, 20, absolute=True,
              periodic=periodic)
    h1 = one.find_features(peakcolumn='Peak')
    labels, feats, iters, max_label = _multi_rank(P, pos, vel, 0.25, 20, 100., periodic, peak=peak)
    np.testing.assert_array_equal(labels, one.labels.cpu().numpy())
    assert len(max_label) == P and max(max_label) == one.max_label[0]
    for k, v in feats.items():
        np.testing.assert_allclose(v, np.asarray(h1[k]), rtol=1e-6, atol=1e-6 * 100, err_msg=k)


def _winding_chain(L=100., ll=1.0, passes=6, seed=4):
    """one chain of friends (spacing ll/2) running along x from wall to wall and back `passes` times, so it crosses
    every slab boundary again and again; rows shuffled over the ranks; plus isolated points"""
    pts = []
    for k in range(passes):
        y = 10. + 6. * k
        xs = np.arange(2., L - 2. + 1e-9, 0.5 * ll)
        xs = xs if k % 2 == 0 else xs[::-1]
        pts.append(np.stack([xs, np.full_like(xs, y), np.full_like(xs, 50.)], 1))
        if k + 1 < passes:                    # the turn at the wall
            ys = np.arange(y + 0.5 * ll, y + 6., 0.5 * ll)
            pts.append(np.stack([np.full_like(ys, xs[-1]), ys, np.full_like(ys, 50.)], 1))
    rng = np.random.RandomState(seed)
    iso = np.stack([np.arange(5., 95., 3.), np.full(30, 90.), np.full(30, 20.)], 1)
    pos = np.concatenate(pts + [iso])
    pos = pos[rng.permutation(len(pos))] + rng.uniform(-0.05, 0.05, pos.shape)
    return pos, np.zeros_like(pos)


@pytest.mark.parametrize("P", [2, 3])
def test_winding_chain_needs_several_merges(cuda, P):
    pos, vel = _winding_chain()
    ll = 0.75
    assert len(fo.near_ties(pos, ll, 100.)) == 0
    want = fo.labels(pos, ll, 1, 100.)
    assert want.max() == 1 and (want == 1).sum() > 1000
    labels, feats, iters, _ = _multi_rank(P, pos, vel, ll, 1, 100., True)
    np.testing.assert_array_equal(labels, want)
    assert iters >= 2


def test_thin_slab_raises(cuda):
    from nbodykit_b200.lab import FOF
    pos, vel = clumpy()

    def fn(comm):
        FOF(_cat({'Position': _split(pos, 3, comm.rank)}, box=100., comm=comm), 20., 5, absolute=True)
    with pytest.raises(ValueError, match="thinner than the routing reach"):
        _run_ranks(3, fn)


# ---- two GPUs --------------------------------------------------------------------------------------------------------
def test_two_gpu_fof_matches_one_gpu():
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "mgpu_fof_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(out.stdout[-3000:])
    sys.stderr.write(out.stderr[-3000:])
    assert out.returncode == 0
