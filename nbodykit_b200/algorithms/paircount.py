"""
Pair counts and pair-count correlation functions in a simulation box on the GPU (API of nbodykit
algorithms/pair_counters/{base,simbox}.py and paircount_tpcf/{tpcf,estimators}.py: `SimulationBoxPairCount`,
`SimulationBox2PCF`).

The reference hands the catalogues to Corrfunc (theory DD / DDsmu / DDrppi with autocorr=0 and the catalogue passed
twice), so every ORDERED pair (i in first, j in second) is counted: an auto-correlation counts each unordered pair
twice.  Here the counting is csrc/paircount.cu: both catalogues are bucketed on one cell grid (side >= r_max / 2),
and every primary visits the cells of a host-computed stencil, secondaries staged through shared memory.

What counts as a pair, pinned from Corrfunc's documented behaviour (there is no binary to compare with):
  * separations are float64 from the stored positions (f4 or f8), wrapped into [0, L) when periodic (the reference's
    `pos %= BoxSize`), minimum image per axis;
  * a pair is in separation bin k when edges[k]^2 <= d^2 < edges[k+1]^2 (squared edges in float64), so self-pairs and
    coincident points never count (edges[0] > 0);
  * '2d': mu = |d_los| / d, bin floor(mu * Nmu); pairs with mu >= 1 are dropped (Corrfunc's 0 <= mu < mu_max);
  * 'projected': r_p over the two axes other than the line of sight, pi = |d_los|; a pair counts when pi < pimax, in
    pi bin floor(pi * npi / pimax) clamped to npi - 1, npi = int(pimax);
  * the first-dimension field is the UNWEIGHTED mean of r (r_p) over the pairs of the bin, 0 for an empty bin;
    `wnpairs` is the sum of w1 * w2, weights of any type taken as float64.
Deviation from the reference, on purpose: Corrfunc evaluates separations in the input precision; here they are always
float64 (as FOF does), so f4 catalogues may differ from Corrfunc for pairs within float32 rounding of an edge.

With several ranks the rows of the x slab of a rank are its primaries, and every secondary within r_max of a slab is
copied there (`ParticleMesh.decompose` / `SlabLayout.route`, as FOF routes); the histograms are then all-reduced.
"""
import ctypes
import logging
import math
import warnings

import numpy
import torch

from .._lib import F4, F8, check, darr, lib, stage
from ..binned_statistic import BinnedStatistic
from .. import CurrentMPIComm
from ..pmesh.pm import _ptr, _stream, as_device_tensor

_MODES = {'1d': 0, '2d': 1, 'projected': 2}
_VALID_MODES = ['1d', '2d', 'projected', 'angular']

# keywords the reference forwards to Corrfunc; they only tune its CPU execution, so here they are recorded in
# attrs['config'] and otherwise ignored
CONFIG_KEYS = ('nthreads', 'verbose', 'isa', 'c_api_timer', 'xbin_refine_factor', 'ybin_refine_factor',
               'zbin_refine_factor', 'max_cells_per_dim', 'copy_particles', 'enable_min_sep_opt',
               'fast_divide_and_NR_steps', 'bin_type')


def _check_config(config):
    bad = sorted(k for k in config if k not in CONFIG_KEYS)
    if bad:
        raise ValueError("unknown pair-count keyword(s) %s; the accepted Corrfunc tuning keywords are %s (they are "
                         "recorded in attrs['config'] and have no effect on the GPU)" % (bad, list(CONFIG_KEYS)))


def _parse_los(los):
    if isinstance(los, str):
        if los not in ('x', 'y', 'z'):
            raise ValueError("``los`` should be one of 'x', 'y', 'z'")
        los = 'xyz'.index(los)
    if isinstance(los, (int, numpy.integer)) and not isinstance(los, bool):
        los = int(los)
        if los < 0:
            los += 3
    if not isinstance(los, int) or los not in (0, 1, 2):
        raise ValueError("``los`` should be either ['x', 'y', 'z'] or [0,1,2]")
    return los


def _verify_input_sources(first, second, BoxSize, required_columns):
    """required columns present; the box of the sources and of the keyword agree (base.py verify_input_sources)"""
    if second is None:
        second = first
    assert second.comm is first.comm, "communicator mismatch between input sources"
    for source in (first, second):
        for col in required_columns:
            if col not in source:
                raise ValueError("the column '%s' is missing from input source; cannot do pair count" % col)
    box = numpy.zeros(3)
    box1 = first.attrs.get('BoxSize', None)
    if box1 is not None:
        box[:] = box1
    if BoxSize is not None:
        box[:] = BoxSize
    if (box == 0.).all():
        raise ValueError("BoxSize must be supplied in the source ``attrs`` or via the ``BoxSize`` keyword")
    box2 = second.attrs.get('BoxSize', None)
    if box1 is not None and box2 is not None:
        if not numpy.all(numpy.asarray(box1) == numpy.asarray(box2)):
            raise ValueError("BoxSize mismatch between pair count cross-correlation sources")
        if not numpy.all(numpy.asarray(box1) == box):
            raise ValueError("BoxSize mismatch between sources and the pair count algorithm")
    return box


def _column(source, name, what):
    """a catalogue column as a contiguous device tensor; positions keep f4 / f8, anything else becomes f8"""
    col = source[name]
    t = as_device_tensor(col.compute() if hasattr(col, 'compute') else col)
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    if what == 'weight':
        return t.reshape(-1).contiguous()
    if t.ndim != 2 or t.shape[1] != 3:
        raise ValueError("pair counts need 3-D positions, got a column of shape %s" % (tuple(t.shape),))
    return t.contiguous()


def _weight_sum(source, name, power):
    """local sum of w ** power in float64, where the column lives (device tensor or host array)"""
    col = source[name]
    w = col.compute() if hasattr(col, 'compute') else col
    if isinstance(w, torch.Tensor):
        w = w.to(torch.float64)
        return float((w if power == 1 else w * w).sum())
    w = numpy.asarray(w, dtype='f8')
    return float((w if power == 1 else w * w).sum())


def _code(t):
    return F4 if t.dtype == torch.float32 else F8


def _pair_edges(mode, edges, Nmu, pimax):
    """(dims, edges per dim) of the result grid"""
    if mode == '1d':
        return ['r'], [edges]
    if mode == '2d':
        return ['r', 'mu'], [edges, numpy.linspace(0, 1., Nmu + 1)]
    return ['rp', 'pi'], [edges, numpy.linspace(0, pimax, int(pimax + 1))]


def _reach(mode, edges, pimax):
    """largest separation a counted pair can have: the grid and the routing reach"""
    emax = float(edges[-1])
    return math.sqrt(emax * emax + float(pimax) * float(pimax)) if mode == 'projected' else emax


class SimulationBoxPairCount(object):
    r"""
    Count (weighted) pairs of objects in a simulation box as a function of :math:`r`, :math:`(r,\mu)` or
    :math:`(r_p, \pi)`, on the GPU.

    Parameters
    ----------
    mode : '1d', '2d', 'projected'
        the coordinates of the result ('angular' is not implemented)
    first : CatalogSource
        the first source, with the `position` and `weight` columns
    edges : array_like
        separation bin edges along r (or r_p); edges[0] > 0
    BoxSize : float or 3-vector, optional
        the box; taken from first.attrs['BoxSize'] when not given
    periodic : bool
        minimum-image separations in a cubic box
    second : CatalogSource, optional
        the second source of a cross-correlation (`second is first` is an auto-correlation)
    los : 'x', 'y', 'z' or 0, 1, 2 (negative wraps)
        the line-of-sight axis for '2d' and 'projected'
    Nmu : int
        number of mu bins in [0, 1]; required for '2d'
    pimax : float
        largest pi for 'projected', >= 1; int(pimax) pi bins of equal width
    weight, position : str
        column names
    show_progress : bool
        count the primaries in 10 chunks and log after each
    **config :
        Corrfunc tuning keywords (see `CONFIG_KEYS`): recorded in attrs['config'], no effect here

    The result `pairs` is a BinnedStatistic with dims ['r'], ['r', 'mu'] or ['rp', 'pi'] and the fields r (or rp, the
    mean separation of the counted pairs, 0 for an empty bin), npairs (u8) and wnpairs (f8, sum of w1 * w2).
    """
    logger = logging.getLogger('SimulationBoxPairCount')

    def __init__(self, mode, first, edges, BoxSize=None, periodic=True, second=None, los='z', Nmu=None, pimax=None,
                 weight='Weight', position='Position', show_progress=False, **config):
        if mode == 'angular':
            raise NotImplementedError("mode='angular': the angular and survey pair counters are not implemented "
                                      "(they, like SurveyDataPairCount and SurveyData2PCF, need the sky transforms "
                                      "and the cosmology layer, which nbodykit_b200 does not have)")
        los = _parse_los(los)
        _check_config(config)
        BoxSize = _verify_input_sources(first, second, BoxSize, [position, weight])

        if mode not in _VALID_MODES:
            raise ValueError("allowed 'mode' values are: %s" % _VALID_MODES)
        if numpy.min(edges) <= 0.:
            raise ValueError("the lower edge of the 1st separation bin must greater than zero (no self-pairs)")
        if mode == '2d' and Nmu is None:
            raise ValueError("'Nmu' keyword is required when 'mode' is '2d'")
        if Nmu is not None and mode != '2d':
            raise ValueError("mode should be '2d' if 'Nmu' is specified")
        if mode == 'projected' and pimax is None:
            raise ValueError("'pimax' keyword is required when 'mode' is 'projected'")
        if pimax is not None and mode != 'projected':
            raise ValueError("mode should be 'projected' if 'projected' is specified")
        if mode == 'projected' and pimax < 1.0:
            raise ValueError("'pimax' must be at least 1.0 when 'mode' is 'projected'")

        self.first, self.second = first, second
        self.comm = first.comm
        self.attrs = {'mode': mode, 'edges': edges, 'Nmu': Nmu, 'pimax': pimax, 'show_progress': show_progress,
                      'N1': first.csize, 'N2': second.csize if second is not None else None}
        s1 = self.comm.allreduce(_weight_sum(first, weight, 1))
        if second is None or second is first:
            s2 = self.comm.allreduce(_weight_sum(first, weight, 2))
            # each unordered pair once, self-pairs excluded (the estimators only use ratios of these)
            self.attrs['total_wnpairs'] = 0.5 * (s1 ** 2 - s2)
            self.attrs['is_cross'] = False
        else:
            s2 = self.comm.allreduce(_weight_sum(second, weight, 1))
            self.attrs['total_wnpairs'] = 0.5 * s1 * s2
            self.attrs['is_cross'] = True
        self.attrs.update({'BoxSize': BoxSize, 'periodic': periodic, 'weight': weight, 'position': position,
                           'config': config, 'los': los})

        if periodic:
            min_box_side = 0.5 * BoxSize.min()
            if numpy.amax(edges) > min_box_side or mode == 'projected' and pimax > min_box_side:
                raise ValueError("periodic pair counts cannot be computed for Rmax > BoxSize/2")
            if not numpy.all(BoxSize == BoxSize[0]):
                raise NotImplementedError("periodic wrapping with non-cubic boxes not implemented yet")
        self.run()

    def run(self):
        """count the pairs: sets `pairs`"""
        a = self.attrs
        mode = a['mode']
        edges = numpy.asarray(a['edges'], dtype='f8').ravel()
        first, second = self.first, self.second
        pos1 = _column(first, a['position'], 'position')
        w1 = _column(first, a['weight'], 'weight')
        if second is None or second is first:
            pos2, w2 = pos1, w1
        else:
            pos2 = _column(second, a['position'], 'position')
            w2 = _column(second, a['weight'], 'weight')
        box = numpy.asarray(a['BoxSize'], dtype='f8') if a['periodic'] else None
        counter = _Counter(mode, edges, a['Nmu'], a['pimax'], a['los'], box)
        if self.comm.size > 1:
            pos1, w1, pos2, w2 = _distribute(pos1, w1, pos2, w2, counter.rmax, box, self.comm)
        nchunk = 10 if a['show_progress'] else 1
        npairs, wnpairs, sepsum = counter.count(pos1, w1, pos2, w2, nchunk, self.logger)
        with stage("pc_reduce"):
            npairs = self.comm.allreduce_tensor(npairs, "sum")
            wnpairs = self.comm.allreduce_tensor(wnpairs, "sum")
            sepsum = self.comm.allreduce_tensor(sepsum, "sum")
        self.pairs = _make_pairs(mode, a['edges'], a['Nmu'], a['pimax'], npairs.cpu().numpy(), wnpairs.cpu().numpy(),
                                 sepsum.cpu().numpy())
        self.pairs.attrs['total_wnpairs'] = a['total_wnpairs']

    def __getstate__(self):
        return {'pairs': self.pairs.data, 'attrs': self.attrs}

    def __setstate__(self, state):
        self.__dict__.update(state)
        a = self.attrs
        if a['mode'] not in _MODES:
            raise ValueError("mode = '%s' should be one of %s" % (a['mode'], list(_MODES)))
        dims, edges = _pair_edges(a['mode'], a['edges'], a['Nmu'], a['pimax'])
        self.pairs = BinnedStatistic(dims, edges, self.pairs, fields_to_sum=['npairs', 'wnpairs'])

    def save(self, output):
        """save the result as JSON (the reference's state layout: {'pairs': structured array, 'attrs': ...})"""
        _save(self, output)

    @classmethod
    @CurrentMPIComm.enable
    def load(cls, output, comm=None):
        """load a result written by `save`"""
        return _load(cls, output, comm)


def _save(obj, output):
    import json
    from ..utils import JSONEncoder
    if obj.comm.rank == 0:
        obj.logger.info('measurement done; saving result to %s' % output)
        with open(output, 'w') as ff:
            json.dump(obj.__getstate__(), ff, cls=JSONEncoder)


def _load(cls, output, comm):
    import json
    from ..utils import JSONDecoder
    if comm.rank == 0:
        with open(output, 'r') as ff:
            state = json.load(ff, cls=JSONDecoder)
    else:
        state = None
    state = comm.bcast(state)
    self = object.__new__(cls)
    self.__setstate__(state)
    self.comm = comm
    return self


def _make_pairs(mode, edges, Nmu, pimax, npairs, wnpairs, sepsum):
    """the `pairs` BinnedStatistic from the three flat histograms"""
    dims, bin_edges = _pair_edges(mode, edges, Nmu, pimax)
    shape = tuple(len(e) - 1 for e in bin_edges)
    data = numpy.zeros(shape, dtype=[(dims[0], 'f8'), ('npairs', 'u8'), ('wnpairs', 'f8')])
    n = npairs.view('u8').reshape(shape)
    data['npairs'] = n
    data['wnpairs'] = wnpairs.reshape(shape)
    nz = n > 0
    data[dims[0]][nz] = sepsum.reshape(shape)[nz] / n[nz]
    return BinnedStatistic(dims, bin_edges, data, fields_to_sum=['npairs', 'wnpairs'])


class _Counter(object):
    """one call of the count kernels: the grid (from n2, r_max and the box or bounds), bucketing, counting"""

    def __init__(self, mode, edges, Nmu, pimax, los, box):
        self.mode, self.code = mode, _MODES[mode]
        self.edges = edges
        self.nmu = int(Nmu) if mode == '2d' else 0
        self.pimax = float(pimax) if mode == 'projected' else 0.0
        self.los = los
        self.box = box
        self.rmax = _reach(mode, edges, self.pimax)
        dims, e = _pair_edges(mode, edges, Nmu, pimax)
        self.nbins = int(numpy.prod([len(x) - 1 for x in e]))

    def _bucket(self, pos, w, n2, bounds):
        n = int(pos.shape[0])
        dev = pos.device
        box_c, lo_c, hi_c = bounds
        ncell = (ctypes.c_int64 * 3)()
        wb = int(lib().nbk_pc_workspace(n, n2, self.rmax, box_c, lo_c, hi_c, ncell))
        check(min(wb, 0), "nbk_pc_workspace")
        C = int(ncell[0]) * int(ncell[1]) * int(ncell[2])
        work = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
        spos = torch.empty(3 * n, dtype=torch.float64, device=dev)
        sw = torch.empty(n, dtype=torch.float64, device=dev)
        scell = torch.empty(n, dtype=torch.int32, device=dev)
        cstart = torch.empty(C + 1, dtype=torch.int32, device=dev)
        check(lib().nbk_pc_bucket(_ptr(pos), _code(pos), _ptr(w), _code(w), n, n2, self.rmax, box_c, lo_c, hi_c,
                                  _ptr(work), wb, _ptr(spos), _ptr(sw), _ptr(scell), _ptr(cstart), _stream()),
              "nbk_pc_bucket")
        return spos, sw, scell, cstart

    def count(self, pos1, w1, pos2, w2, nchunk=1, logger=None):
        """(npairs int64, wnpairs f64, sepsum f64) device histograms of the ordered pairs (rows of pos1, rows of pos2)"""
        dev = pos1.device
        n1, n2 = int(pos1.shape[0]), int(pos2.shape[0])
        if self.box is not None:
            bounds = (darr(self.box), None, None)
        else:
            both = [p for p in (pos1, pos2) if p.shape[0]]
            if both:
                lo = torch.stack([p.min(dim=0).values.double() for p in both]).min(dim=0).values.tolist()
                hi = torch.stack([p.max(dim=0).values.double() for p in both]).max(dim=0).values.tolist()
            else:
                lo = hi = [0.0] * 3
            bounds = (None, darr(lo), darr(hi))
        npairs = torch.zeros(self.nbins, dtype=torch.int64, device=dev)
        wnpairs = torch.zeros(self.nbins, dtype=torch.float64, device=dev)
        sepsum = torch.zeros(self.nbins, dtype=torch.float64, device=dev)
        with stage("pc_bucket"):
            spos2, sw2, _, cstart2 = self._bucket(pos2, w2, n2, bounds)
        box_c, lo_c, hi_c = bounds
        stops = numpy.linspace(0, n1, nchunk + 1).astype('i8') if nchunk > 1 else [0, n1]
        for i in range(len(stops) - 1):
            a, b = int(stops[i]), int(stops[i + 1])
            with stage("pc_bucket"):
                spos1, sw1, scell1, cstart1 = self._bucket(pos1[a:b].contiguous(), w1[a:b].contiguous(), n2, bounds)
            with stage("pc_count"):
                check(lib().nbk_pc_count(self.code, darr(self.edges), len(self.edges), self.nmu, self.pimax, self.los,
                                         self.rmax, _ptr(spos1), _ptr(sw1), _ptr(scell1), _ptr(cstart1), b - a,
                                         _ptr(spos2), _ptr(sw2), _ptr(cstart2), n2, box_c, lo_c, hi_c, _ptr(npairs),
                                         _ptr(wnpairs), _ptr(sepsum), _stream()), "nbk_pc_count")
            if nchunk > 1 and logger is not None:
                logger.info("%d%% done" % (100 * (i + 1) // nchunk))
        return npairs, wnpairs, sepsum


def _distribute(pos1, w1, pos2, w2, rmax, box, comm):
    """(primaries, their weights, secondaries, their weights) of this rank: the primaries of its x slab, and every
    secondary within r_max of the slab.  Each ordered pair then meets on exactly one rank.  When a slab is not wider than
    2 r_max (or r_max > L/4) every rank keeps its own primaries and gathers all secondaries instead."""
    from ..utils import get_data_bounds
    from .fof import _routing_mesh
    P = comm.size
    dev = pos1.device
    p1, p2 = pos1.to(torch.float64), pos2.to(torch.float64)
    if box is not None:
        rbox, shift = box, None
    else:
        # route as if periodic in a box r_max wider than the data; copies that wrap around are only extra candidates
        lo1, hi1 = get_data_bounds(p1, comm)
        lo2, hi2 = get_data_bounds(p2, comm)
        lo, hi = numpy.minimum(lo1, lo2), numpy.maximum(hi1, hi2)
        if not numpy.all(numpy.isfinite(lo)):
            lo = hi = numpy.zeros(3)
        rbox = (hi - lo) + rmax
        shift = torch.as_tensor(lo, dtype=torch.float64, device=dev)
    pm = None
    if float(rbox[0]) / P > 2 * rmax and not (box is not None and rmax > 0.25 * float(numpy.min(box))):
        try:
            pm, smoothing = _routing_mesh(rmax * (1 + 1e-6), rbox, comm)
        except ValueError:
            pm = None
    if pm is None:
        parts = comm.allgather((p2.cpu(), w2.cpu()))
        return (pos1, w1, torch.cat([p[0] for p in parts]).to(dev).contiguous(),
                torch.cat([p[1] for p in parts]).to(dev).contiguous())
    r1 = p1 if shift is None else p1 - shift
    r2 = p2 if shift is None else p2 - shift
    with stage("pc_route"):
        lay1 = pm.decompose(r1, 0.0)
        q1, qw1 = lay1.route(p1, w1)
        own = torch.ones(p1.shape[0], dtype=torch.bool, device=dev)
        own[lay1.ghosts & 0xffffffff] = False
        lay2 = pm.decompose(r2, smoothing)
        q2, qw2 = lay2.route(p2, w2)
    return (torch.cat([p1[own], q1]).contiguous(), torch.cat([w1[own], qw1]).contiguous(),
            torch.cat([p2, q2]).contiguous(), torch.cat([w2, qw2]).contiguous())


# ---- correlation functions ----------------------------------------------------------------------------------------
class WedgeBinnedStatistic(BinnedStatistic):
    """a BinnedStatistic of xi(r, mu) wedges that converts to multipoles"""

    def to_poles(self, poles):
        r"""
        the multipoles :math:`\xi_\ell(r)` of the wedges: :math:`(2\ell+1) \sum \xi L_\ell(\mu_c) \Delta\mu /
        \sum \Delta\mu` with :math:`\mu_c` the bin centres (the reference's midpoint rule)
        """
        from scipy.special import legendre
        x = str(self.dims[0])
        data = numpy.zeros(self.shape[0], dtype=[(x, 'f8')] + [('corr_%d' % ell, 'f8') for ell in poles])
        mu = self.edges['mu']
        dmu = numpy.diff(mu)
        mid = 0.5 * (mu[1:] + mu[:-1])
        for ell in poles:
            data['corr_%d' % ell] = numpy.sum(self['corr'] * (2. * ell + 1.) * legendre(ell)(mid) * dmu,
                                              axis=-1) / numpy.sum(dmu)
        data[x] = numpy.mean(self[x], axis=-1)
        return BinnedStatistic(dims=[x], edges=[self.edges[x]], data=data, poles=poles)


def analytic_filling_factor(mode, edges, box):
    """fraction of the box volume in each bin for uniform randoms: sphere shells ('1d'), spherical sectors in |mu|
    ('2d'), cylinder shells of height 2 pi ('projected'); `edges` maps dim name -> edges"""
    V = float(numpy.prod(box))
    if mode == '1d':
        return numpy.diff(4. / 3. * numpy.pi * edges['r'] ** 3) / V
    if mode == '2d':
        vol = 2. * 2. / 3. * numpy.pi * numpy.outer(edges['r'] ** 3, edges['mu'])
        return numpy.diff(numpy.diff(vol, axis=0), axis=1) / V
    vol = numpy.pi * numpy.outer(edges['rp'] ** 2, 2. * edges['pi'])
    return numpy.diff(numpy.diff(vol, axis=0), axis=1) / V


def _corr_result(D1D2, CF):
    x = D1D2.dims[0]
    data = numpy.empty(CF.shape, dtype=[('corr', 'f8'), (x, 'f8')])
    data['corr'] = CF
    data[x] = D1D2[x]
    return WedgeBinnedStatistic(D1D2.dims, [D1D2.edges[d] for d in D1D2.dims], data)


def natural_estimator(D1D2, attrs):
    """(analytic R1R2 pairs, xi = DD f / RR - 1) for a periodic box; attrs of the D1D2 pair count"""
    N1 = attrs['N1']
    N2 = attrs['N2'] if attrs['is_cross'] else None
    f = analytic_filling_factor(attrs['mode'], D1D2.edges, numpy.asarray(attrs['BoxSize'], dtype='f8'))
    if N2 is None:
        RR, total = N1 ** 2 * f, N1 * (N1 - 1) * 0.5
    else:
        RR, total = N1 * N2 * f, N1 * N2 * 0.5
    data = numpy.empty(RR.shape, dtype=[('npairs', 'f8'), ('wnpairs', 'f8')])
    data['npairs'] = RR
    data['wnpairs'] = RR
    R1R2 = WedgeBinnedStatistic(D1D2.dims, [D1D2.edges[d] for d in D1D2.dims], data)
    R1R2.attrs['total_wnpairs'] = total
    CF = D1D2['wnpairs'] * (total / attrs['total_wnpairs']) / RR - 1.
    return R1R2, _corr_result(D1D2, CF)


def landy_szalay(D1D2, D1R2, D2R1, R1R2, totals, comm_rank=0):
    """xi = (fDD DD - fDR DR - fRD RD) / RR + 1 on the bins with RR > 0 (NaN elsewhere, with a warning); totals =
    total_wnpairs of (D1D2, D1R2, D2R1, R1R2)"""
    tDD, tDR, tRD, tRR = totals
    nonzero = R1R2['npairs'] > 0
    CF = numpy.full(D1D2.shape, numpy.nan)
    RR = R1R2['wnpairs'][nonzero]
    CF[nonzero] = (tRR / tDD * D1D2['wnpairs'][nonzero] - tRR / tDR * D1R2['wnpairs'][nonzero]
                   - tRR / tRD * D2R1['wnpairs'][nonzero]) / RR + 1
    if comm_rank == 0 and numpy.isnan(CF).any():
        warnings.warn("The RR calculation in the Landy-Szalay estimator contains separation bins with no bins. This "
                      "will result in NaN values in the resulting correlation function. Try increasing the number of "
                      "randoms and/or using broader bins.")
    return _corr_result(D1D2, CF)


def compute_wp(corr):
    r""":math:`w_p(r_p) = 2 \sum_\pi \xi(r_p, \pi) \Delta\pi`, as a BinnedStatistic over r_p"""
    dpi = numpy.diff(corr.edges['pi'])
    wp = (2 * corr['corr'] * dpi).sum(axis=-1)
    out = corr.copy()
    if len(out.dims) > 1:
        out = out.average(out.dims[-1])
    out['corr'] = wp
    return out


class SimulationBox2PCF(object):
    r"""
    The two-point correlation function of simulation-box data from GPU pair counts, as :math:`\xi(r)`,
    :math:`\xi(r,\mu)` or :math:`\xi(r_p,\pi)` (with :math:`w_p(r_p)`).

    Without randoms in a periodic box the natural estimator DD / RR - 1 is used with analytic RR (unweighted uniform
    randoms); with `randoms1` the Landy-Szalay estimator, each term scaled by the ratio of the total_wnpairs.
    Non-periodic data need randoms.  Parameters as :class:`SimulationBoxPairCount`; `randoms2` defaults to
    `randoms1` when `data2` is given, and a given `R1R2` pair count is reused.

    Results: D1D2, D1R2, D2R1, R1R2 (pair-count BinnedStatistics; D1R2 / D2R1 None with analytic randoms), corr (a
    WedgeBinnedStatistic with the variable 'corr') and, in projected mode, wp.
    """
    logger = logging.getLogger('SimulationBox2PCF')

    def __init__(self, mode, data1, edges, Nmu=None, pimax=None, data2=None, randoms1=None, randoms2=None, R1R2=None,
                 periodic=True, BoxSize=None, los='z', weight='Weight', position='Position', show_progress=False,
                 **config):
        _check_config(config)
        self.comm = data1.comm
        self.attrs = {'mode': mode, 'edges': numpy.array(edges), 'Nmu': Nmu, 'pimax': pimax, 'periodic': periodic,
                      'BoxSize': BoxSize, 'los': los, 'weight': weight, 'position': position,
                      'show_progress': show_progress, 'config': config}
        self.data1, self.data2 = data1, data2
        self.randoms1, self.randoms2 = randoms1, randoms2
        self.R1R2 = R1R2
        self.run()

    def run(self):
        """count the pairs and apply the estimator: sets D1D2, D1R2, D2R1, R1R2, corr (and wp)"""
        kws = self.attrs.copy()
        kws.update(kws.pop('config'))
        if kws['periodic'] and self.randoms1 is None:
            DD = SimulationBoxPairCount(first=self.data1, second=self.data2, **kws)
            self.R1R2, self.corr = natural_estimator(DD.pairs, DD.attrs)
            self.D1D2 = DD.pairs
            self.D1R2 = self.D2R1 = None
        else:
            if self.randoms1 is None:
                raise ValueError("a catalog of randoms must be specified as the ``randoms1`` keyword when the data is "
                                 "not in a simulation box with periodic boundary conditions")
            if self.data2 is not None and self.randoms2 is None:
                self.randoms2 = self.randoms1
            randoms2 = self.randoms2 if self.randoms2 is not None else self.randoms1
            log = self.comm.rank == 0
            if log:
                self.logger.info("computing randoms1 - randoms2 pair counts")
            RR = self.R1R2 if self.R1R2 else SimulationBoxPairCount(first=self.randoms1, second=randoms2, **kws)
            if log:
                self.logger.info("computing data1 - data2 pair counts")
            DD = SimulationBoxPairCount(first=self.data1, second=self.data2, **kws)
            if log:
                self.logger.info("computing data1 - randoms2 pair counts")
            DR = SimulationBoxPairCount(first=self.data1, second=randoms2, **kws)
            if self.data2 is not None:
                if log:
                    self.logger.info("computing data2 - randoms1 pair counts")
                RD = SimulationBoxPairCount(first=self.data2, second=self.randoms1, **kws)
            else:
                RD = DR
            totals = [c.attrs['total_wnpairs'] for c in (DD, DR, RD, RR)]
            self.corr = landy_szalay(DD.pairs, DR.pairs, RD.pairs, RR.pairs, totals, self.comm.rank)
            self.D1D2, self.D1R2, self.D2R1, self.R1R2 = DD.pairs, DR.pairs, RD.pairs, RR.pairs
        if self.attrs['mode'] == 'projected':
            self.wp = compute_wp(self.corr)

    def __getstate__(self):
        state = {'corr': self.corr.data, 'dims': self.corr.dims,
                 'edges': [self.corr.edges[d] for d in self.corr.dims]}
        for name in ('D1D2', 'D1R2', 'D2R1', 'R1R2', 'wp'):
            val = getattr(self, name, None)
            state[name] = val.data if val is not None else None
        state['attrs'] = self.attrs
        return state

    def __setstate__(self, state):
        state = dict(state)
        edges = state.pop('edges')
        dims = state.pop('dims')
        self.__dict__.update(state)
        self.corr = WedgeBinnedStatistic(dims, edges, self.corr)
        if self.wp is not None:
            self.wp = WedgeBinnedStatistic(dims[:1], edges[:1], self.wp)     # pi was summed over
        for name in ('D1D2', 'D1R2', 'D2R1', 'R1R2'):
            val = getattr(self, name)
            if val is not None:
                setattr(self, name, WedgeBinnedStatistic(dims, edges, val))

    def save(self, output):
        """save the result as JSON (the reference's state layout)"""
        _save(self, output)

    @classmethod
    @CurrentMPIComm.enable
    def load(cls, output, comm=None):
        """load a result written by `save`"""
        return _load(cls, output, comm)
