"""
FOF -- friends-of-friends groups on the GPU (API of nbodykit/algorithms/fof.py: `FOF` :10-195, `_assign_labels`
:197-287, `_fof_merge` :311-337, `fof_catalog` :427-533, `centerofmass` :647-700).

The local step is csrc/fof.cu: a counting sort of the rows into cells of side >= ll, a lock-free union-find over each
cell and its 13 forward neighbours (link: squared separation <= ll^2 in float64, minimum image when periodic), path
compression, and a per-group atomicMin of the global row index (`minid`).  With several ranks the rows near every x slab
are copied there (`ParticleMesh.decompose` with a reach of ll, the route `readout` uses) and the minid of every copy is
merged back to its source row until no rank changes.  Group sizes, labels and the sort by size are small torch steps on
at most n / (nmin + 1) groups.

Deviations from the reference, on purpose:
  * equal-Length groups are labelled in the order of their smallest global row index (the reference's order for ties
    comes from an unstable argsort);
  * with several ranks, an x slab (BoxSize[0] / P, or the data extent + ll when not periodic) must be wider than 2 ll.
"""
import ctypes
import logging

import numpy
import torch

from .._lib import F4, F8, check, darr, lib, stage
from ..pmesh.pm import _ptr, _stream, as_device_tensor
from ..source.catalog.array import ArrayCatalog

_I64_MAX = 0x7fffffffffffffff
_SUM, _MIN, _MAX = 0, 1, 2


class FOF(object):
    """
    Friends-of-friends groups of a catalogue: every particle gets the label of its group, groups ordered by size.

    Parameters
    ----------
    source : CatalogSource
        must have a 'Position' column (and attrs['BoxSize'] when `periodic`)
    linking_length : float
        absolute, or in units of the mean separation (prod(BoxSize) / csize) ** (1 / ndim) unless `absolute`
    nmin : int
        groups of nmin particles or fewer get label 0
    absolute : bool
        whether `linking_length` is in absolute units
    periodic : bool
        minimum-image separations in the box attrs['BoxSize']
    domain_factor : int
        accepted for compatibility; the load-balancing knob of the reference's domain grid has no role here

    Results: `labels` (device int32 tensor, int64 beyond 2^31 - 1 groups, one entry per local row; 0 = not in a
    group of more than nmin particles, then 1, 2, ... from the largest group down) and `max_label` (the largest label
    of every rank).
    """
    logger = logging.getLogger('FOF')

    def __init__(self, source, linking_length, nmin, absolute=False, periodic=True, domain_factor=1):
        self.comm = source.comm
        self._source = source
        if 'Position' not in source:
            raise ValueError("cannot compute FOF without 'Position' column")
        self.attrs = {'linking_length': linking_length, 'nmin': nmin, 'absolute': absolute, 'periodic': periodic,
                      'domain_factor': domain_factor}
        if periodic and 'BoxSize' not in source.attrs:
            raise ValueError("Periodic FOF requires BoxSize in .attrs['BoxSize']")
        if not absolute:
            if 'BoxSize' not in source.attrs:
                raise ValueError("a linking length relative to the mean separation needs BoxSize in .attrs['BoxSize']")
            if 'Nmesh' in source.attrs:
                ndim = len(source.attrs['Nmesh'])
            else:
                ndim = source['Position'].shape[1]
            # a scalar BoxSize stands for a cubic box
            box = numpy.broadcast_to(numpy.asarray(source.attrs['BoxSize'], dtype='f8'), (ndim,))
            mean_separation = pow(numpy.prod(box) / source.csize, 1.0 / ndim)
            linking_length = linking_length * mean_separation
        self._linking_length = float(linking_length)
        self.run()

    def run(self):
        """find the groups: sets `labels` and `max_label` (and what find_features needs)"""
        pos = _device_column(self._source['Position'])
        if pos.ndim != 2 or pos.shape[1] != 3:
            raise ValueError("FOF needs 3-D positions, got a Position column of shape %s" % (tuple(pos.shape),))
        box = None
        if self.attrs['periodic']:
            box = numpy.empty(3, dtype='f8')
            box[:] = self._source.attrs['BoxSize']
        self._box = box
        if self.comm.size == 1:
            local = _local_fof(pos, self._linking_length, box)
            minid, self.merge_iterations = local.minid, 0
        else:
            minid, local, self.merge_iterations = _fof_slabs(pos, self._linking_length, box, self.comm)
        self._order, self._nvisit = local.order, int(local.order.shape[0])
        with stage("fof_labels"):
            self.labels, self._ngroups = _assign_labels(minid, self.comm, self.attrs['nmin'])
        self.max_label = self.comm.allgather(int(self.labels.max()) if self.labels.numel() else 0)

    def find_features(self, peakcolumn=None):
        """
        ArrayCatalog of the groups, K + 1 rows split over the ranks as the reference's ScatterArray does: row 0 collects
        the particles of label 0 (its Length is set to 0), row k the group of label k.  Columns CMPosition, CMVelocity
        (f4, 3) and Length (i4); InitialPosition (f4, 3) when the source has it; PeakPosition and PeakVelocity when
        `peakcolumn` is given (centre of mass of the particles at the group's maximum of that column; as in the
        reference, the other particles of a group count for row 0 there).  Periodic centres of mass are taken from the
        per-axis minimum of the group with differences wrapped into [-L/2, L/2), accumulated in float64.
        """
        src = self._source
        for col in ('Position', 'Velocity'):
            if col not in src:
                raise ValueError("the column '%s' is missing from parent source; cannot compute halos" % col)
        if self.attrs['periodic'] and 'BoxSize' not in src.attrs:
            raise ValueError("cannot compute halo catalog from source without 'BoxSize' in ``attrs`` dict")
        if peakcolumn is not None and peakcolumn not in src:
            raise ValueError("the peak column '%s' is missing from parent source" % peakcolumn)
        with stage("fof_features"):
            red = _GroupReducer(self.labels, self._order, self._nvisit, self._ngroups + 1, self.comm)
            pos = _device_column(src['Position'])
            vel = _device_column(src['Velocity'])
            cmpos, count = red.center_of_mass(pos, self._box)
            cmvel, _ = red.center_of_mass(vel, None)
            length = count.clone()
            length[0] = 0
            cols = {'CMPosition': cmpos, 'CMVelocity': cmvel, 'Length': length}
            if 'InitialPosition' in src:
                cols['InitialPosition'] = red.center_of_mass(_device_column(src['InitialPosition']), self._box)[0]
            if peakcolumn is not None:
                peak = _device_column(src[peakcolumn]).reshape(-1).to(torch.float64).contiguous()
                red.set_peak(peak)
                cols['PeakPosition'] = red.center_of_mass(pos, self._box)[0]
                cols['PeakVelocity'] = red.center_of_mass(vel, None)[0]
            start, stop = _scatter_share(self._ngroups + 1, self.comm)
            out = {k: (v[start:stop].to(torch.int32) if k == 'Length' else v[start:stop].to(torch.float32)).contiguous()
                   for k, v in cols.items()}
        attrs = src.attrs.copy()
        attrs.update(self.attrs)
        return ArrayCatalog(out, comm=self.comm, **attrs)

    def to_halos(self, particle_mass, cosmo, redshift, mdef='vir', posdef='cm', peakcolumn='Density'):
        raise NotImplementedError(
            "FOF.to_halos needs the cosmology and halo-model layer (HaloCatalog with halotools mass definitions, "
            "concentration and radius), which nbodykit_b200 does not implement; use find_features() for the group "
            "catalogue")


def _device_column(col):
    """a catalogue column as a contiguous device tensor, f4 / f8 kept, any other type as f8"""
    data = col.compute() if hasattr(col, 'compute') else col
    t = as_device_tensor(data)
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    return t.contiguous()


def _code(t):
    return F4 if t.dtype == torch.float32 else F8


class _Local(object):
    """what the local FOF leaves: cell order of the rows, component root of every row, minid"""

    def __init__(self, order, root, rootmin, minid):
        self.order, self.root, self.rootmin, self.minid = order, root, rootmin, minid


def _local_fof(pos, ll, box, gidx=None, row_offset=0):
    """FOF over the rows of one rank; minid = smallest of gidx (default row_offset + row) over each group"""
    n = int(pos.shape[0])
    dev = pos.device
    if box is not None:
        box_c, lo_c, hi_c = darr(box), None, None
    else:
        box_c = None
        if n:
            lo_c, hi_c = darr(pos.min(dim=0).values.double().tolist()), darr(pos.max(dim=0).values.double().tolist())
        else:
            lo_c, hi_c = darr([0.0] * 3), darr([0.0] * 3)
    ncell = (ctypes.c_int64 * 3)()
    wb = int(lib().nbk_fof_workspace(n, ll, box_c, lo_c, hi_c, ncell))
    check(min(wb, 0), "nbk_fof_workspace")
    work = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    order = torch.empty(n, dtype=torch.int32, device=dev)
    spos = torch.empty(3 * n, dtype=pos.dtype, device=dev)
    parent = torch.empty(n, dtype=torch.int32, device=dev)
    root = torch.empty(n, dtype=torch.int32, device=dev)
    rootmin = torch.empty(n, dtype=torch.int64, device=dev)
    minid = torch.empty(n, dtype=torch.int64, device=dev)
    s = _stream()
    with stage("fof_bucket"):
        check(lib().nbk_fof_bucket(_ptr(pos), _code(pos), n, ll, box_c, lo_c, hi_c, _ptr(work), wb, _ptr(order),
                                   _ptr(spos), s), "nbk_fof_bucket")
    with stage("fof_link"):
        check(lib().nbk_fof_link(_ptr(spos), _code(pos), n, ll, box_c, lo_c, hi_c, _ptr(work), wb, _ptr(parent), s),
              "nbk_fof_link")
    with stage("fof_compress"):
        check(lib().nbk_fof_compress(_ptr(parent), n, _ptr(order), _ptr(root), s), "nbk_fof_compress")
        check(lib().nbk_fof_minid(_ptr(root), n, _ptr(gidx), int(row_offset), _ptr(rootmin), _ptr(minid), s),
              "nbk_fof_minid")
    return _Local(order, root, rootmin, minid)


def _routing_mesh(ll, box, comm):
    """a ParticleMesh whose x slabs are the ranks' slabs, with `smoothing` = ll in cells; raises when a slab is not
    wider than the 2 ll a routed particle reaches across"""
    from ..pmesh.pm import ParticleMesh
    P = comm.size
    s0 = ll * P / float(box[0])           # smoothing per plane of slab width
    m = int(numpy.ceil(1.0 / (1.0 - 2.0 * s0))) if s0 < 0.5 else 0
    if m < 1 or s0 * m >= 64:
        raise ValueError("FOF on %d ranks: the x slab (%g wide) is thinner than the routing reach 2 * ll = %g; use "
                         "fewer ranks or a smaller linking length" % (P, float(box[0]) / P, 2 * ll))
    pm = ParticleMesh(BoxSize=box, Nmesh=[P * m, P, 2], comm=comm)
    return pm, ll * P * m / float(box[0])


def _send_rows(layout, values, sidx):
    """the rows `route` sent (send order `sidx`) of a per-row column, as received by the destinations"""
    out = torch.empty((int(sum(layout.recvcounts)),) + tuple(values.shape[1:]), dtype=values.dtype, device=values.device)
    layout.comm.all_to_all_single(out, values.index_select(0, sidx).contiguous(), list(layout.recvcounts),
                                  list(layout.sendcounts))
    return out


def _fof_slabs(pos, ll, box, comm):
    """FOF over several ranks (reference `_fof_local` + `_fof_merge`): (minid of the local rows, local FOF of local +
    received rows, number of merge iterations)"""
    from ..utils import get_data_bounds
    n = int(pos.shape[0])
    dev = pos.device
    offset = int(sum(comm.allgather(n)[:comm.rank]))
    if box is not None:
        rbox, rpos = box, pos
    else:
        # route as if periodic in a box one linking length wider than the data; the local FOF is not periodic, so the
        # copies that wrap around cannot link
        lo, hi = get_data_bounds(pos, comm)
        rbox = (hi - lo) + ll
        rpos = pos.to(torch.float64) - torch.as_tensor(lo, dtype=torch.float64, device=dev)
    pm, smoothing = _routing_mesh(ll, rbox, comm)
    layout = pm.decompose(rpos, smoothing)
    recv_pos, _, sidx = layout.route(rpos, want_index=True)
    gid = torch.arange(offset, offset + n, dtype=torch.int64, device=dev)
    allpos = torch.cat([rpos, recv_pos]).contiguous()
    allgid = torch.cat([gid, _send_rows(layout, gid, sidx)])
    local = _local_fof(allpos, ll, box, gidx=allgid)
    minid = local.minid
    ntot = int(allpos.shape[0])
    iterations = 0
    while True:
        own = minid[:n].clone()
        layout.gather_back(minid[n:], sidx, own, mode='min')
        new = torch.cat([own, _send_rows(layout, own, sidx)])
        if int(comm.allreduce(int((new != minid).sum()))) == 0:
            break
        iterations += 1
        check(lib().nbk_fof_minid(_ptr(local.root), ntot, _ptr(new), 0, _ptr(local.rootmin), _ptr(minid), _stream()),
              "nbk_fof_minid")
    return minid[:n], local, iterations


def _assign_labels(minid, comm, nmin):
    """(labels, K): groups of more than nmin rows get 1..K by decreasing size, ties by increasing minid; others 0"""
    dev = minid.device
    P = comm.size
    u, c = torch.unique(minid, return_counts=True)
    if P > 1:
        # (minid, count) pairs travel to the rank that owns row minid, which adds them up
        ends = torch.tensor(numpy.cumsum(comm.allgather(int(minid.shape[0]))), dtype=torch.int64, device=dev)
        owner = torch.searchsorted(ends, u, right=True)
        sendcounts = [int(v) for v in torch.bincount(owner, minlength=P).tolist()]
        recvcounts = comm.alltoall_ints(sendcounts)
        ru = torch.empty(sum(recvcounts), dtype=torch.int64, device=dev)
        rc = torch.empty_like(ru)
        comm.all_to_all_single(ru, u.contiguous(), recvcounts, sendcounts)
        comm.all_to_all_single(rc, c.to(torch.int64).contiguous(), recvcounts, sendcounts)
        u, inv = torch.unique(ru, return_inverse=True)
        c = torch.zeros(u.shape[0], dtype=torch.int64, device=dev).index_add_(0, inv, rc)
    keep = c > nmin
    su, sc = u[keep], c[keep].to(torch.int64)
    if P > 1:
        # every rank gets all survivors, in owner order: minid ascending overall
        parts = comm.allgather((su.cpu().numpy(), sc.cpu().numpy()))
        su = torch.as_tensor(numpy.concatenate([p[0] for p in parts]), device=dev)
        sc = torch.as_tensor(numpy.concatenate([p[1] for p in parts]), device=dev)
    K = int(su.shape[0])
    dtype = torch.int64 if K + 1 > 2 ** 31 else torch.int32
    if K == 0:
        return torch.zeros(minid.shape[0], dtype=dtype, device=dev), 0
    perm = torch.argsort(-sc, stable=True)              # su is ascending: ties keep increasing minid
    label_of = torch.empty(K, dtype=torch.int64, device=dev)
    label_of[perm] = torch.arange(1, K + 1, dtype=torch.int64, device=dev)
    at = torch.searchsorted(su, minid).clamp_(max=K - 1)
    labels = torch.where(su[at] == minid, label_of[at], torch.zeros((), dtype=torch.int64, device=dev))
    return labels.to(dtype), K


def _scatter_share(ntot, comm):
    """rows [start, stop) of rank r when ntot rows are split as ScatterArray does (the first ntot % P get one more)"""
    P, r = comm.size, comm.rank
    q, extra = divmod(ntot, P)
    start = r * q + min(r, extra)
    return start, start + q + (1 if r < extra else 0)


def _decode(keys):
    """order-preserving int64 keys of nbk_fof_reduce -> float64"""
    return torch.where(keys >= 0, keys, keys ^ _I64_MAX).view(torch.float64)


class _GroupReducer(object):
    """dense per-group reductions over all ranks (the reference's equiv_class + Allreduce)"""

    def __init__(self, labels, order, nvisit, ngroups, comm):
        self.label = labels.to(torch.int64).contiguous()
        self.order, self.nvisit, self.ngroups, self.comm = order, nvisit, ngroups, comm
        self.peak = self.peakmax = None
        self.dev = labels.device

    def _reduce(self, op, val, dim, anchor=None, box=None, osum=None, okey=None, ocount=None):
        check(lib().nbk_fof_reduce(op, _ptr(self.label), int(self.label.shape[0]), _ptr(self.order), self.nvisit,
                                   _ptr(val), _code(val) if val is not None else F8, dim, _ptr(anchor),
                                   darr(box) if box is not None else None, _ptr(self.peak), _ptr(self.peakmax),
                                   self.ngroups, _ptr(osum), _ptr(okey), _ptr(ocount), _stream()), "nbk_fof_reduce")

    def set_peak(self, peak):
        """from now on only the rows at their group's maximum of `peak` count for the group (the others for group 0)"""
        self.peak = None
        self.peakmax = None
        pmax = torch.full((self.ngroups,), _key(-numpy.inf), dtype=torch.int64, device=self.dev)
        self._reduce(_MAX, peak, 1, okey=pmax)
        self.peakmax = self.comm.allreduce_tensor(pmax, "max")
        self.peak = peak

    def center_of_mass(self, val, box):
        """(per-group mean of val [n][3], float64 [ngroups][3]; per-group count) -- periodic when box is given"""
        dim = int(val.shape[1]) if val.ndim == 2 else 1
        anchor = None
        if box is not None:
            anchor = torch.full((self.ngroups, dim), _I64_MAX, dtype=torch.int64, device=self.dev)
            self._reduce(_MIN, val, dim, okey=anchor)
            anchor = self.comm.allreduce_tensor(anchor, "min")
        sums = torch.zeros((self.ngroups, dim), dtype=torch.float64, device=self.dev)
        count = torch.zeros(self.ngroups, dtype=torch.int64, device=self.dev)
        self._reduce(_SUM, val, dim, anchor=anchor, box=box, osum=sums, ocount=count)
        sums = self.comm.allreduce_tensor(sums, "sum")
        count = self.comm.allreduce_tensor(count, "sum")
        mean = sums / count[:, None].to(torch.float64)
        if box is not None:
            L = torch.as_tensor(numpy.asarray(box, dtype='f8')[:dim], device=self.dev)
            mean = torch.remainder(_decode(anchor) + mean, L)
        return mean, count


def _key(x):
    b = int(numpy.array(x, dtype='f8').view('i8'))
    return b if b >= 0 else b ^ _I64_MAX
