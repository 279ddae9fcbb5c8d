"""Point-cloud depth drivers on the B200 engine.

Same private seam as the reference (imported by name in statdepth/depth/depth.py:8):
    _pointwisedepth        statdepth/depth/calculations/_pointcloud.py:14-66
    _samplepointwisedepth  statdepth/depth/calculations/_pointcloud.py:68-123
"""
from typing import Union

import numpy as np
import pandas as pd
from scipy.spatial import ConvexHull
from scipy.special import binom

from . import _dist, settings
from ._engine import get_engine
from ._functional import _positions, _values
from ._helper import DepthDegeneracy

__all__ = ['_pointwisedepth', '_samplepointwisedepth', '_pointwisedepth_of']


def _pointwisedepth(
    data: pd.DataFrame,
    to_compute: Union[list, pd.Index] = None,
    containment='simplex',
    quiet=True,
) -> pd.Series:
    """Depth of each requested point w.r.t. the n x d cloud; mirrors _pointcloud.py:14-66."""
    n, d = data.shape
    if containment not in ('simplex', 'l1', 'mahalanobis', 'oja'):
        raise ValueError(f'{containment} is not a valid containment measure. ')
    if containment == 'mahalanobis':
        return _mahalanobis_depth(data=data, to_compute=to_compute)
    eng = get_engine()
    P = np.ascontiguousarray(_values(data))

    if containment == 'simplex':
        # #{(d+1)-subsets of the others containing p} / binom(n, d+1)      (_pointcloud.py:44-56)
        if to_compute is None:
            to_compute = data.index
        if d > 3:
            raise NotImplementedError('simplicial depth is implemented for d <= 3 on the B200 engine')
        q = _positions(to_compute, data.index, 'to_compute')
        tol = settings.get_simplex_tolerance()
        if d != 2 or n <= 64:  # 2-D clouds above 64 points are counted (tolerance band honoured), not enumerated
            settings.check_enumeration(float(len(q)) * binom(n - 1, d + 1), 'simplicial depth (d=%d, n=%d)' % (d, n))
        cnt = _dist.query_sharded(lambda qb: eng.simplicial_counts(P, qb, tol), q, np.int64)
        return pd.Series(index=to_compute, data=cnt.astype(np.float64) / binom(n, d + 1))
    elif containment == 'l1':
        # 1 - || sum_o (x_o - x_p)/||x_p - x_o|| || / n                       (_pointcloud.py:125-150)
        if to_compute is None:
            to_compute = list(data.index)
        if d > 16:
            raise NotImplementedError('L1 depth is implemented for d <= 16 on the B200 engine')
        q = _positions(to_compute, data.index, 'to_compute')
        dep = _dist.query_sharded(lambda qb: eng.l1_depth(P, qb), q, np.float64)
        return pd.Series(index=to_compute, data=dep)
    elif containment == 'oja':
        # sum over d-subsets of vol(conv(S u {p})) / vol(conv(data))          (_pointcloud.py:176-204)
        if d not in (2, 3):
            raise NotImplementedError('Oja depth is implemented for d in (2, 3) on the B200 engine')
        idx = data.index if to_compute is None else to_compute
        try:
            hull_volume = ConvexHull(P).volume  # once per call, host side (Qhull), as in the reference
        except Exception:
            raise DepthDegeneracy('Too many collinear points to compute depth of convex hull spanned by data. '
                                  'Try another depth method or remove collinearities.')
        q = _positions(idx, data.index, 'to_compute')
        # reference quirk (:182-183,191-193): with to_compute the subsets are drawn from to_compute only
        pool = None if to_compute is None else q
        npool = n if pool is None else len(pool)
        if d != 2 or npool <= 256:  # 2-D pools above 256 points are summed in O(n log n) per query, not enumerated
            settings.check_enumeration(float(len(q)) * binom(npool, d), 'Oja depth (d=%d)' % d)
        vals = _dist.query_sharded(lambda qb: eng.oja(P, hull_volume, qb, pool), q, np.float64)
        # reference quirk (:205): index=to_compute, i.e. a default RangeIndex when to_compute is None
        return pd.Series(index=to_compute, data=vals)
    else:
        raise ValueError(f'{containment} is not a valid containment measure. ')


def _pointwisedepth_of(
    data: pd.DataFrame,
    sample: pd.DataFrame,
    containment='simplex',
    quiet=True,
) -> pd.Series:
    """Depth of every row of data against the reference cloud sample, each point counted as if it alone were
    appended to the sample (population nS + 1).  Indexed by data.index."""
    if containment not in ('simplex', 'l1', 'mahalanobis', 'oja'):
        raise ValueError(f'{containment} is not a valid containment measure. ')
    if containment in ('mahalanobis', 'oja'):
        raise NotImplementedError(f'out-of-sample {containment} depth is not implemented; use \'simplex\' or \'l1\'')
    nY, d = data.shape
    nS, dS = sample.shape
    if d != dS:
        raise ValueError('data and sample must have the same number of dimensions.')
    S = np.ascontiguousarray(_values(sample))
    Y = np.ascontiguousarray(_values(data))
    ys = np.arange(nY, dtype=np.int64)
    eng = get_engine()
    if containment == 'simplex':
        if d > 3:
            raise NotImplementedError('simplicial depth is implemented for d <= 3 on the B200 engine')
        tol = settings.get_simplex_tolerance()
        if d != 2 or nS + 1 <= 64:  # as _pointwisedepth with n = nS + 1: larger 2-D samples are counted
            settings.check_enumeration(float(nY) * binom(nS, d + 1),
                                       'out-of-sample simplicial depth (d=%d, n=%d)' % (d, nS + 1))
        cnt = _dist.query_sharded(lambda qb: eng.simplicial_oos_counts(S, Y[qb], tol), ys, np.int64)
        return pd.Series(index=data.index, data=cnt.astype(np.float64) / binom(nS + 1, d + 1))
    if d > 16:
        raise NotImplementedError('L1 depth is implemented for d <= 16 on the B200 engine')
    dep = _dist.query_sharded(lambda qb: eng.l1_oos_depth(S, Y[qb]), ys, np.float64)
    return pd.Series(index=data.index, data=dep)


def _mahalanobis_depth(data: pd.DataFrame, to_compute=None) -> pd.Series:
    """_pointcloud.py:152-174.  Requires n == p; an n x n solve on the host (SURVEY 2: not a hot path)."""
    n, p = data.shape
    if n != p:
        raise ValueError('Mahalanobis depth requires equal number of dimensions and datapoints.')
    mu = data.mean()
    inv_cov = np.linalg.inv(np.cov(data, rowvar=True))
    idx = data.index if to_compute is None else to_compute
    depths = []
    for point in idx:
        x = data.loc[point, :]
        depths.append(np.dot((x - mu).T, np.dot(inv_cov, x)))
    return pd.Series(index=idx, data=depths)


def _samplepointwisedepth(
    data: pd.DataFrame,
    to_compute: pd.Index = None,
    K=2,
    containment='simplex',
    quiet=True,
) -> pd.Series:
    """Sampled point-cloud depth; mirrors _pointcloud.py:68-123 including its quirk that the inner loop runs
    ss = n // K times (not K) with blocks of ss rows drawn by `DataFrame.sample` from the global numpy RNG
    (same call sequence -> same stream as the reference).  The len(to_compute) * ss single-query blocks are
    evaluated by ONE engine call (sd_pointcloud_blocks_f64) for 'simplex' and 'l1'."""
    if K == 1:
        return _pointwisedepth(data=data, to_compute=to_compute, containment=containment)
    n, d = data.shape
    if to_compute is None:
        to_compute = data.index
    ss = n // K
    if containment not in ('simplex', 'l1') or d > 3 or (ss + 1) * d > 4096 or ss == 0:
        # 'oja' with to_compute=[point] enumerates subsets of that one point (reference quirk, :182-193) and
        # 'mahalanobis' is a host routine: both keep the reference's loop of single calls
        depths = []
        for time in to_compute:
            cd = []
            for _ in range(ss):
                sdata = data.sample(n=ss, axis=0)
                if time not in sdata.index:
                    sdata = pd.concat([sdata, data.loc[[time], :]])
                cd.append(_pointwisedepth(data=sdata, to_compute=[time], containment=containment))
            depths.append(np.mean(cd))
        return pd.Series(index=to_compute, data=depths)

    # label-level replay of the sampling (same pandas calls on a one-column frame with the same index)
    labels = pd.DataFrame(np.zeros((n, 1)), index=data.index)
    members, offsets, qpos = [], [0], []
    for time in to_compute:
        tpos = int(_positions([time], data.index, 'to_compute')[0])
        for _ in range(ss):
            pos = _positions(labels.sample(n=ss, axis=0).index, data.index, 'sampled rows')
            hit = np.flatnonzero(pos == tpos)
            if hit.size:
                qpos.append(int(hit[0]))
            else:  # the reference appends the point at the END of the sampled frame (:118)
                pos = np.append(pos, tpos)
                qpos.append(len(pos) - 1)
            members.append(pos)
            offsets.append(offsets[-1] + len(pos))
    P = np.ascontiguousarray(_values(data))
    eng = get_engine()
    sizes = np.diff(np.asarray(offsets, dtype=np.int64)).astype(np.float64)
    vals = eng.cloud_blocks(P, np.concatenate(members) if members else np.zeros(0, np.int64), offsets, qpos,
                            containment, settings.get_simplex_tolerance())
    if containment == 'simplex':
        vals = vals / binom(sizes, d + 1)  # _pointcloud.py:56 with n = len(sdata)
    depths = [np.mean(vals[i * ss:(i + 1) * ss]) for i in range(len(to_compute))]
    return pd.Series(index=to_compute, data=depths)
