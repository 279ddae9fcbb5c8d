"""Functional depth drivers on the B200 engine.

Same private seam as the reference (imported by name in statdepth/depth/depth.py:7):
    _functionaldepth        statdepth/depth/calculations/_functional.py:17-97
    _samplefunctionaldepth  statdepth/depth/calculations/_functional.py:99-196
The Python loops over curves and over J-subsets are gone: one call into libsdepth.so returns the
integer numerators for all requested curves, and the float64 depth is formed here with the
reference's own arithmetic (count / binom(n, j), summed over j = 2..J).
"""
from math import comb
from typing import List, Union

import numpy as np
import pandas as pd
from scipy.special import binom

from . import _dist, settings
from ._engine import get_engine
from ._helper import DepthDegeneracy, _check_containment, _handle_depth_errors

__all__ = ['_functionaldepth', '_samplefunctionaldepth', '_functionaldepth_of', '_relaxed_depths_of']


def _positions(labels, axis_index: pd.Index, what: str) -> np.ndarray:
    pos = axis_index.get_indexer(list(labels))
    if (pos < 0).any():
        missing = [lab for lab, p in zip(labels, pos) if p < 0]
        raise KeyError('%s not found in the data: %r' % (what, missing))
    return pos.astype(np.int64)


def _values(df: pd.DataFrame) -> np.ndarray:
    v = df.to_numpy()
    if v.dtype != np.float64:
        v = v.astype(np.float64)
    return v


def _univariate_depths(X: np.ndarray, queries, J: int, relax: bool) -> np.ndarray:
    """depth = sum_{j=2..J} S_nj / binom(n, j)  (_functional.py:238-253).  X is [T, n]."""
    eng = get_engine()
    T, n = X.shape
    nq = n if queries is None else len(queries)
    depth = np.zeros(nq, dtype=np.float64)
    ranks = None
    for j in range(2, J + 1):
        if j <= 3:
            if relax:
                cnt = _dist.relaxed_counts(lambda Xr, q, jj: eng.band_depth_counts(Xr, q, jj, True), X, queries, j, eng)
            else:
                qs = np.arange(n, dtype=np.int64) if queries is None else np.asarray(queries, dtype=np.int64)
                if j == 3:  # strict J = 3 enumerates the C(n-1, 3) triples of every query (bd_triple_kernel)
                    settings.check_enumeration(float(len(qs)) * binom(n - 1, 3), 'strict band depth with J=3 (n=%d)' % n)
                cnt = _dist.query_sharded(lambda qb: eng.band_depth_counts(X, qb, j, False), qs, np.int64)
            s_nj = cnt.astype(np.float64)
        elif relax:
            # j >= 4: closed form from the GPU's strict ranks, exact Python integers on the host
            if ranks is None:
                ranks = eng.band_ranks(X)
            below, above = ranks
            qs = range(n) if queries is None else queries
            full = comb(n - 1, j)
            s_nj = np.array([float(sum(full - comb(int(b), j) - comb(int(a), j)
                                       for b, a in zip(below[:, c], above[:, c]))) for c in qs])
        else:
            raise NotImplementedError('strict band depth with J >= 4 is not implemented on the B200 engine '
                                      '(the reference enumerates C(n-1, J) subsets in Python); use relax=True '
                                      'or J <= 3.')
        if relax:
            s_nj = s_nj / float(T)  # _containment.py:80 returns containment / len(curve)
        depth = depth + s_nj / binom(n, j)
    return depth


def _multivariate_depths(data: List[pd.DataFrame], queries: np.ndarray, relax: bool) -> np.ndarray:
    """_simplex_depth (_functional.py:257-286): count / binom(N - 1, d + 1); J is ignored there too."""
    eng = get_engine()
    F = np.stack([_values(df) for df in data])
    N, T, d = F.shape
    if d > 3:
        raise NotImplementedError('simplex containment is implemented for d <= 3 channels on the B200 engine')
    tol = settings.get_simplex_tolerance()
    if d == 2 and relax and N > 64:
        pass  # relaxed 2-D depth above 64 curves is COUNTED per (query, time point): O(N log N) each
    elif d == 2 and not relax:
        # strict 2-D depth is enumerated with first-row pruning in shared memory (~1.3 cheap tests per triple,
        # csrc/pointcloud.cu simplex2_strict_kernel): config 4 (5 000 queries x C(4999,3) triples) runs in minutes
        settings.check_enumeration(float(len(queries)) * binom(N - 1, 3) / 4.0,
                                   'strict multivariate simplex depth (d=2, N=%d)' % N)
    else:
        settings.check_enumeration(float(len(queries)) * binom(N - 1, d + 1) * (T if relax else 1.0),
                                   'multivariate simplex depth (d=%d, N=%d, relax=%s)' % (d, N, relax))
    cnt = _dist.query_sharded(lambda qb: eng.simplex_depth_counts(F, qb, relax, tol), queries, np.int64)
    s = cnt.astype(np.float64)
    if relax:
        s = s / float(T)
    return s / binom(N - 1, d + 1)


def _functionaldepth(
    data: List[pd.DataFrame],
    to_compute: Union[list, pd.Index] = None,
    J=2,
    containment='r2',
    relax=False,
    deep_check=False,
    quiet=True,
) -> Union[pd.Series, pd.DataFrame]:
    """Exact band depth of every requested curve.  Mirrors _functional.py:17-97 (same arguments, same
    validation, same pd.Series result: index = the columns / list positions requested)."""
    _handle_depth_errors(data=data, J=J, containment=containment, relax=relax, deep_check=deep_check)
    name = _check_containment(containment)

    if len(data) == 1:
        # 'simplex' on univariate data never gets here: _handle_depth_errors raised (_helper.py:92).
        if name == 'r2_enum':
            raise NotImplementedError  # _containment.py:103
        df = data[0]
        cols = df.columns
        queries = None
        if to_compute is not None:
            cols = to_compute
            queries = _positions(to_compute, df.columns, 'to_compute')
        depths = _univariate_depths(_values(df), queries, J, relax)
        return pd.Series(index=cols, data=depths)

    if name != 'simplex':
        # reference: `depths` is never assigned for 'r2_enum' / callables -> UnboundLocalError (_functional.py:97)
        raise NotImplementedError('multivariate data supports containment=\'simplex\' only')
    f = [i for i in range(len(data))]
    if to_compute is not None:
        f = to_compute
    queries = np.asarray([int(i) for i in f], dtype=np.int64)
    depths = _multivariate_depths(data, queries, relax)
    return pd.Series(index=f, data=depths)


def _univariate_depths_of(S: np.ndarray, Y: np.ndarray, J: int, relax: bool) -> np.ndarray:
    """Depth of every new curve (column of Y [T, nY]) inside S [T, nS] u {that curve}: the arithmetic of
    _univariate_depths with n = nS + 1, so the result is bit-identical to the in-sample call on the pooled frame."""
    eng = get_engine()
    T, nS = S.shape
    nY = Y.shape[1]
    depth = np.zeros(nY, dtype=np.float64)
    if nY == 0:
        return depth
    ys = np.arange(nY, dtype=np.int64)
    if relax:
        # additive over time rows: shard the rows of the pooled [S | Y] matrix, split it at nS per block
        X = np.ascontiguousarray(np.concatenate([S, Y], axis=1))
        return _relaxed_depths_of([_dist.relaxed_counts(
            lambda Xr, q, jj: eng.band_depth_oos_counts(Xr[:, :nS], Xr[:, nS:], jj, True)[q], X, ys, j)
            for j in range(2, J + 1)], T, nS)
    for j in range(2, J + 1):
        if j == 3:  # bd_triple_kernel enumerates the C(nS, 3) sample triples of every new curve
            settings.check_enumeration(float(nY) * binom(nS, 3),
                                       'out-of-sample strict band depth with J=3 (n=%d)' % (nS + 1))
        cnt = _dist.query_sharded(lambda qb: eng.band_depth_oos_counts(S, Y[:, qb], j, False), ys, np.int64)
        depth = depth + cnt.astype(np.float64) / binom(nS + 1, j)
    return depth


def _relaxed_depths_of(counts, T: int, nS: int) -> np.ndarray:
    """Relaxed out-of-sample depth from the numerators counts[j - 2] (j = 2..J): sum_j cnt_j / T / binom(nS + 1, j),
    the arithmetic of _univariate_depths with n = nS + 1.  Every out-of-sample path forms its floats here, so equal
    counts give bit-identical depths."""
    depth = np.zeros(len(counts[0]), dtype=np.float64)
    for j, cnt in enumerate(counts, start=2):
        depth = depth + (np.asarray(cnt).astype(np.float64) / float(T)) / binom(nS + 1, j)
    return depth


def _functionaldepth_of(
    data: List[pd.DataFrame],
    sample: List[pd.DataFrame],
    J=2,
    containment='r2',
    relax=False,
    deep_check=False,
    quiet=True,
) -> pd.Series:
    """Band depth of every curve of data[0] against the reference sample sample[0], each curve counted as if it
    alone were appended to the sample.  Indexed by data[0].columns (labels may repeat those of the sample)."""
    _handle_depth_errors(data=data, J=J, containment=containment, relax=relax, deep_check=deep_check)
    _handle_depth_errors(data=sample, J=J, containment=containment, relax=relax, deep_check=deep_check)
    name = _check_containment(containment)
    if len(data) != 1 or len(sample) != 1:
        raise NotImplementedError('out-of-sample depth is implemented for univariate data ([DataFrame] with '
                                  'containment=\'r2\'); multivariate simplex depth is not')
    if name == 'r2_enum':
        raise NotImplementedError  # as _functionaldepth (_containment.py:103)
    df, ref = data[0], sample[0]
    if df.shape[0] != ref.shape[0]:
        raise ValueError('data and sample must have the same number of time points.')
    if deep_check and not (len(df.index) == len(ref.index) and all(df.index == ref.index)):
        raise ValueError('DataFrames indices must be the same')
    if J > 3:
        raise NotImplementedError('out-of-sample band depth is implemented for J <= 3 on the B200 engine')
    depths = _univariate_depths_of(_values(ref), _values(df), J, relax)
    return pd.Series(index=df.columns, data=depths)


def _sample_blocks(df: pd.DataFrame, cols, K: int):
    """Label-level replay of the reference's sampling loop (_functional.py:159-183).

    Uses the same pandas calls (`DataFrame.sample(n, axis=1)` on the global numpy RNG, then `drop`)
    on a one-row frame carrying the same columns, so the RNG stream -- and therefore every block --
    is the one the reference would draw after the same `np.random.seed`.  Quirks kept: the block size
    is len(all columns) // K even when `to_compute` is given, and after the first curve the pool is
    rebuilt from the `to_compute` columns only (`df = orig.copy()`, :183).
    """
    orig_cols = list(df.loc[:, cols].columns)
    ss = df.shape[1] // K
    if ss == 0:
        raise DepthDegeneracy(f'Block size {K} is too large, not enough functions to sample.')
    pool = pd.DataFrame(np.zeros((1, df.shape[1])), columns=df.columns)
    blocks = []  # (query label, member labels)
    for col in orig_cols:
        for _ in range(K):
            t = pool.sample(n=ss, axis=1)
            pool = pool.drop(t.columns, axis=1)
            members = list(t.columns)
            if col not in members:
                members.append(col)
            blocks.append((col, members))
        pool = pd.DataFrame(np.zeros((1, len(orig_cols))), columns=orig_cols)
    return orig_cols, blocks


def _samplefunctionaldepth(
    data: List[pd.DataFrame],
    K: int,
    to_compute: Union[list, pd.Index] = None,
    J=2,
    containment='r2',
    relax=False,
    deep_check=False,
    quiet=True,
) -> Union[pd.Series, pd.DataFrame]:
    """K-block sampled band depth, mirrors _functional.py:99-196.  The K * len(cols) blocks are
    evaluated by ONE batched call (sd_band_depth_batched_f64)."""
    _handle_depth_errors(data=data, J=J, containment=containment, relax=relax, deep_check=deep_check)
    name = _check_containment(containment)

    if len(data) != 1:
        # the reference's multivariate branch is a stub that returns an empty list (:187-194)
        return pd.Series([], dtype=np.float64)
    if name == 'r2_enum':
        raise NotImplementedError
    if J > 3:
        raise NotImplementedError('sampled band depth is implemented for J <= 3 on the B200 engine')
    df = data[0]
    cols = df.columns if to_compute is None else to_compute
    orig_cols, blocks = _sample_blocks(df, cols, K)

    n = df.shape[1]
    membership = np.zeros((len(blocks), n), dtype=np.uint8)
    queries = np.zeros((len(blocks), 1), dtype=np.int64)
    sizes = np.zeros(len(blocks), dtype=np.int64)
    for b, (col, members) in enumerate(blocks):
        pos = _positions(members, df.columns, 'sampled columns')
        membership[b, pos] = 1
        sizes[b] = int(membership[b].sum())
        queries[b, 0] = _positions([col], df.columns, 'to_compute')[0]
    X = np.ascontiguousarray(_values(df))
    T = X.shape[0]
    eng = get_engine()
    depth = np.zeros(len(blocks), dtype=np.float64)
    for j in range(2, J + 1):
        s = eng.band_depth_counts_batched(X, membership, queries, j, relax)[:, 0].astype(np.float64)
        if relax:
            s = s / float(T)
        depth = depth + s / binom(sizes, j)
    samples = [np.mean(depth[i * K:(i + 1) * K]) for i in range(len(orig_cols))]
    return pd.Series(index=pd.Index(orig_cols), data=samples)
