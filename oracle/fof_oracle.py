"""
TEST INFRASTRUCTURE -- CPU oracle for FOF (nbodykit/algorithms/fof.py).  NOT product code.

A restatement, not the reference: kdcount and mpi4py are not needed.  Links come from scipy's cKDTree
(`query_pairs(ll)`: separation <= ll, periodic through `boxsize`), groups are the connected components of those links,
labels and the group catalogue follow FOF's documented rules (1..K by decreasing Length, ties by smallest row; label 0
for groups of nmin rows or fewer; centres of mass from the per-axis minimum with wrapped differences, in float64).
"""
import numpy as np


def components(pos, ll, boxsize=None):
    """minid of every row: the smallest row index of its friends-of-friends group"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    from scipy.spatial import cKDTree
    pos = np.asarray(pos, dtype='f8')
    n = len(pos)
    if boxsize is not None:
        L = np.broadcast_to(np.asarray(boxsize, dtype='f8'), (3,))
        tree = cKDTree(pos % L, boxsize=L)
    else:
        tree = cKDTree(pos)
    pairs = tree.query_pairs(ll, output_type='ndarray')
    g = coo_matrix((np.ones(len(pairs)), (pairs[:, 0], pairs[:, 1])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    minid = np.full(comp.max() + 1 if n else 0, n, dtype='i8')
    np.minimum.at(minid, comp, np.arange(n))
    return minid[comp]


def assign_labels(minid, nmin):
    """labels 1..K by decreasing group size, ties by increasing minid; 0 for groups of <= nmin rows"""
    u, inv, cnt = np.unique(minid, return_inverse=True, return_counts=True)
    keep = cnt > nmin
    order = np.lexsort((u[keep], -cnt[keep]))
    lab = np.zeros(len(u), dtype='i8')
    lab[np.flatnonzero(keep)[order]] = np.arange(1, keep.sum() + 1)
    return lab[inv.reshape(-1)]


def labels(pos, ll, nmin, boxsize=None):
    return assign_labels(components(pos, ll, boxsize), nmin)


def center_of_mass(label, val, ngroups, boxsize=None):
    """per-label mean of val; periodic: anchor at the per-axis minimum, differences wrapped into [-L/2, L/2)"""
    val = np.asarray(val, dtype='f8')
    N = np.bincount(label, minlength=ngroups).astype('f8')
    if boxsize is not None:
        L = np.broadcast_to(np.asarray(boxsize, dtype='f8'), (val.shape[1],))
        anchor = np.full((ngroups, val.shape[1]), np.inf)
        np.minimum.at(anchor, label, val)
        d = val - anchor[label]
        d = np.where(d < -0.5 * L, d + L, np.where(d >= 0.5 * L, d - L, d))
    else:
        d = val
    s = np.zeros((ngroups, val.shape[1]))
    np.add.at(s, label, d)
    with np.errstate(invalid='ignore', divide='ignore'):
        m = s / N[:, None]
        return (anchor + m) % L if boxsize is not None else m


def find_features(label, pos, vel, boxsize=None, peak=None, initpos=None):
    """dict of the find_features columns (float64 / int64), row 0 = label 0 with Length 0"""
    label = np.asarray(label, dtype='i8')
    K1 = int(label.max()) + 1 if len(label) else 1
    out = {'CMPosition': center_of_mass(label, pos, K1, boxsize),
           'CMVelocity': center_of_mass(label, vel, K1, None),
           'Length': np.bincount(label, minlength=K1)}
    out['Length'][0] = 0
    if initpos is not None:
        out['InitialPosition'] = center_of_mass(label, initpos, K1, boxsize)
    if peak is not None:
        peak = np.asarray(peak, dtype='f8')
        pmax = np.full(K1, -np.inf)
        np.maximum.at(pmax, label, peak)
        label1 = label * (peak >= pmax[label])
        out['PeakPosition'] = center_of_mass(label1, pos, K1, boxsize)
        out['PeakVelocity'] = center_of_mass(label1, vel, K1, None)
    return out


def near_ties(pos, ll, boxsize=None, rtol=1e-9):
    """pairs whose separation lies within a relative rtol of ll (where float rounding could flip a link)"""
    from scipy.spatial import cKDTree
    pos = np.asarray(pos, dtype='f8')
    if boxsize is not None:
        L = np.broadcast_to(np.asarray(boxsize, dtype='f8'), (3,))
        tree = cKDTree(pos % L, boxsize=L)
    else:
        tree = cKDTree(pos)
    outer = tree.query_pairs(ll * (1 + rtol), output_type='ndarray')
    if len(outer) == 0:
        return outer
    d = pos[outer[:, 0]] - pos[outer[:, 1]]
    if boxsize is not None:
        d -= L * np.rint(d / L)
    r = np.sqrt((d ** 2).sum(-1))
    return outer[r >= ll * (1 - rtol)]
