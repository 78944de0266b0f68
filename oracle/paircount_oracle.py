"""
CPU oracle of the simulation-box pair counts (SimulationBoxPairCount / SimulationBox2PCF).

The candidate pairs come from scipy's cKDTree (`sparse_distance_matrix`, with `boxsize` when periodic) at a slightly
larger radius; every component is then recomputed in float64 with the rules the GPU code follows, so that counts can be
compared exactly:
  * positions as float64, wrapped into [0, L] by x - floor(x / L) L when periodic; differences x2 - x1, minimum image
    x - L rint(x / L) per axis;
  * d^2 = (dx^2 + dy^2) + dz^2; separation bin k when edges[k]^2 <= d^2 < edges[k+1]^2;
  * '2d': mu = |d_los| / sqrt(d^2), dropped when mu >= 1, bin min(floor(mu Nmu), Nmu - 1);
  * 'projected': r_p^2 over the two other axes in axis order, pi = |d_los| < pimax, bin min(floor(pi npi / pimax),
    npi - 1), npi = int(pimax);
  * every ordered pair (i in pos1, j in pos2) counts, so an auto-correlation counts each unordered pair twice.
`near_ties` lists pairs within a relative tolerance of a boundary, where float64 rounding could decide the bin.
"""
import math

import numpy
from scipy.spatial import cKDTree


def wrap(pos, box):
    """float64 positions as the count sees them"""
    x = numpy.asarray(pos).astype('f8')
    if box is None:
        return x
    L = numpy.broadcast_to(numpy.asarray(box, dtype='f8'), (3,))
    return x - numpy.floor(x * (1.0 / L)) * L


def reach(mode, edges, pimax=None):
    emax = float(edges[-1])
    return math.sqrt(emax * emax + float(pimax) * float(pimax)) if mode == 'projected' else emax


def candidate_pairs(pos1, pos2, rmax, box):
    """(i, j) of every ordered pair with separation below rmax (plus a relative 1e-6 of slack); coincident points may
    be left out, since they never count"""
    u1, u2 = wrap(pos1, box), wrap(pos2, box)
    if len(u1) == 0 or len(u2) == 0:
        return numpy.zeros(0, 'i8'), numpy.zeros(0, 'i8')
    kw = {}
    if box is not None:
        L = numpy.broadcast_to(numpy.asarray(box, dtype='f8'), (3,))
        kw['boxsize'] = L
        u1, u2 = u1 % L, u2 % L
    m = cKDTree(u1, **kw).sparse_distance_matrix(cKDTree(u2, **kw), rmax * (1 + 1e-6), output_type='ndarray')
    return m['i'].astype('i8'), m['j'].astype('i8')


def components(pos1, pos2, i, j, box):
    """(dx, dy, dz) float64 of the pairs (i, j): x2[j] - x1[i], minimum image when periodic"""
    u1, u2 = wrap(pos1, box), wrap(pos2, box)
    d = u2[j] - u1[i]
    if box is not None:
        L = numpy.broadcast_to(numpy.asarray(box, dtype='f8'), (3,))
        d = d - L * numpy.rint(d * (1.0 / L))
    return d[:, 0], d[:, 1], d[:, 2]


def bin_pairs(mode, dx, dy, dz, edges, Nmu=None, pimax=None, los=2):
    """(keep mask, flat bin, first-dimension separation) of pairs given by their components"""
    edges = numpy.asarray(edges, dtype='f8')
    e2 = edges * edges
    nr = len(edges) - 1
    d = (dx, dy, dz)
    dl = d[los]
    if mode == 'projected':
        a, b = [d[k] for k in range(3) if k != los]
        x2 = a * a + b * b
    else:
        x2 = dx * dx + dy * dy + dz * dz
    keep = (x2 >= e2[0]) & (x2 < e2[-1])
    rb = numpy.clip(numpy.searchsorted(e2, x2, side='right') - 1, 0, nr - 1)
    sep = numpy.sqrt(x2)
    if mode == '1d':
        return keep, rb, sep
    if mode == '2d':
        with numpy.errstate(invalid='ignore', divide='ignore'):
            mu = numpy.abs(dl) / sep
        keep &= mu < 1.0
        mb = numpy.minimum(numpy.floor(numpy.where(keep, mu, 0) * Nmu).astype('i8'), Nmu - 1)
        return keep, rb * Nmu + mb, sep
    npi = int(pimax)
    pi = numpy.abs(dl)
    keep &= pi < pimax
    pb = numpy.minimum(numpy.floor(numpy.where(keep, pi, 0) * (npi / float(pimax))).astype('i8'), npi - 1)
    return keep, rb * npi + pb, sep


def nbins_of(mode, edges, Nmu=None, pimax=None):
    nr = len(edges) - 1
    return nr * (Nmu if mode == '2d' else (int(pimax) if mode == 'projected' else 1))


def shape_of(mode, edges, Nmu=None, pimax=None):
    nr = len(edges) - 1
    return (nr,) if mode == '1d' else (nr, Nmu if mode == '2d' else int(pimax))


def paircount(mode, pos1, edges, box=None, pos2=None, w1=None, w2=None, Nmu=None, pimax=None, los=2):
    """{'npairs' u8, 'wnpairs' f8, 'sep' f8 (unweighted mean, 0 when empty)} shaped like the result"""
    if pos2 is None:
        pos2, w2 = pos1, w1
    n1, n2 = len(pos1), len(pos2)
    w1 = numpy.ones(n1) if w1 is None else numpy.asarray(w1).astype('f8')
    w2 = numpy.ones(n2) if w2 is None else numpy.asarray(w2).astype('f8')
    i, j = candidate_pairs(pos1, pos2, reach(mode, edges, pimax), box)
    dx, dy, dz = components(pos1, pos2, i, j, box)
    keep, b, sep = bin_pairs(mode, dx, dy, dz, edges, Nmu, pimax, los)
    nb = nbins_of(mode, edges, Nmu, pimax)
    b = b[keep]
    npairs = numpy.bincount(b, minlength=nb).astype('u8')
    wn = numpy.bincount(b, weights=w1[i[keep]] * w2[j[keep]], minlength=nb)
    ss = numpy.bincount(b, weights=sep[keep], minlength=nb)
    mean = numpy.zeros(nb)
    nz = npairs > 0
    mean[nz] = ss[nz] / npairs[nz]
    shape = shape_of(mode, edges, Nmu, pimax)
    return {'npairs': npairs.reshape(shape), 'wnpairs': wn.reshape(shape), 'sep': mean.reshape(shape)}


def near_ties(mode, pos1, edges, box=None, pos2=None, Nmu=None, pimax=None, los=2, rtol=1e-9):
    """(i, j) of the pairs within a relative rtol of a squared edge, of mu = 1 (2d) or of pi = pimax (projected)"""
    if pos2 is None:
        pos2 = pos1
    e2 = numpy.asarray(edges, dtype='f8') ** 2
    i, j = candidate_pairs(pos1, pos2, reach(mode, edges, pimax) * (1 + 1e-6), box)
    dx, dy, dz = components(pos1, pos2, i, j, box)
    d = (dx, dy, dz)
    if mode == 'projected':
        a, b = [d[k] for k in range(3) if k != los]
        x2 = a * a + b * b
    else:
        x2 = dx * dx + dy * dy + dz * dz
    near = numpy.zeros(len(i), bool)
    for e in e2:
        near |= numpy.abs(x2 - e) <= rtol * e
    inside = (x2 >= e2[0] * (1 - rtol)) & (x2 < e2[-1] * (1 + rtol))
    if mode == '2d':
        near |= inside & (x2 > 0) & (numpy.abs(numpy.abs(d[los]) - numpy.sqrt(x2)) <= rtol * numpy.sqrt(x2))
    if mode == 'projected':
        near |= inside & (numpy.abs(numpy.abs(d[los]) - pimax) <= rtol * pimax)
    return i[near], j[near]


def total_wnpairs(w1, w2=None):
    """the reference's normalisation: 0.5 ((sum w)^2 - sum w^2) for an auto count, 0.5 sum w1 sum w2 for a cross"""
    w1 = numpy.asarray(w1, dtype='f8')
    if w2 is None:
        return 0.5 * (w1.sum() ** 2 - (w1 ** 2).sum())
    return 0.5 * w1.sum() * numpy.asarray(w2, dtype='f8').sum()


def filling_factor(mode, edges, box, Nmu=None, pimax=None):
    """expected fraction of uniform pairs per bin: shell volume over the box volume"""
    V = float(numpy.prod(numpy.broadcast_to(numpy.asarray(box, dtype='f8'), (3,))))
    r = numpy.asarray(edges, dtype='f8')
    if mode == '1d':
        return (4. / 3. * numpy.pi * (r[1:] ** 3 - r[:-1] ** 3)) / V
    if mode == '2d':
        mu = numpy.linspace(0, 1., Nmu + 1)
        # both signs of mu share a bin of |mu|
        return (4. / 3. * numpy.pi * numpy.outer(r[1:] ** 3 - r[:-1] ** 3, numpy.diff(mu))) / V
    pe = numpy.linspace(0, pimax, int(pimax + 1))
    return (numpy.pi * numpy.outer(r[1:] ** 2 - r[:-1] ** 2, 2. * numpy.diff(pe))) / V


def analytic_rr(mode, edges, box, N1, N2=None, Nmu=None, pimax=None):
    """(RR per bin, its total_wnpairs) for N1 (x N2) uniform randoms"""
    f = filling_factor(mode, edges, box, Nmu, pimax)
    if N2 is None:
        return N1 * N1 * f, 0.5 * N1 * (N1 - 1)
    return N1 * N2 * f, 0.5 * N1 * N2


def natural(DD_wn, DD_total, RR, RR_total):
    return DD_wn * (RR_total / DD_total) / RR - 1.


def landy_szalay(DD, DR, RD, RR, tDD, tDR, tRD, tRR):
    """(DD fDD - DR fDR - RD fRD) / RR + 1, NaN where RR == 0"""
    out = numpy.full(numpy.shape(DD), numpy.nan)
    nz = numpy.asarray(RR) > 0
    out[nz] = (DD[nz] * tRR / tDD - DR[nz] * tRR / tDR - RD[nz] * tRR / tRD) / RR[nz] + 1
    return out


def wp(xi, pimax):
    dpi = numpy.diff(numpy.linspace(0, pimax, int(pimax + 1)))
    return 2 * (xi * dpi).sum(axis=-1)


def to_poles(xi, Nmu, ells):
    """midpoint-rule Legendre moments of xi(r, mu) wedges over mu in [0, 1]"""
    from numpy.polynomial import legendre as L
    mu = numpy.linspace(0, 1., Nmu + 1)
    mid = 0.5 * (mu[1:] + mu[:-1])
    dmu = numpy.diff(mu)
    out = {}
    for ell in ells:
        P = L.legval(mid, [0] * ell + [1])
        out[ell] = (2 * ell + 1) * (xi * P * dmu).sum(axis=-1) / dmu.sum()
    return out
