"""Public API: FunctionalDepth / PointcloudDepth with the reference's signatures and result types.

Mirrors statdepth/depth/depth.py (factories :347-402, result wrappers :14-344) and
statdepth/depth/abstract.py.  The depth values come from the B200 engine; everything below is thin
pandas glue.  plotly is imported lazily inside the plot methods (the reference imports it at
module top, depth.py:4, which makes `import statdepth` fail where plotly is not installed).
"""
from abc import ABC, abstractmethod
from typing import List, Union

import numpy as np
import pandas as pd

from ._functional import _functionaldepth, _functionaldepth_of, _samplefunctionaldepth, _values
from ._helper import DepthDegeneracy  # noqa: F401  (re-exported like the reference's `from ._helper import *`)
from ._halfspace import _functional_halfspace, _pointcloud_halfspace
from ._outliers import (NO_FACTOR, _check_central, _check_extremal_rows, _checked_values, _extremal_depth,
                        _functional_boxplot, _outliergram)
from ._pointcloud import _pointwisedepth, _pointwisedepth_of, _samplepointwisedepth
from ._projection import KINDS, _functional_projection, _pointcloud_projection, draw_directions
from ._reference import _checked_reference, _curve_values, _ProjectedReference, _query_values, _SortedReference
from ._spatial import _functional_spatial, _functional_spatial_of, _spatial_curves, _SpatialReference

__all__ = ['FunctionalDepth', 'PointcloudDepth', 'FunctionalDepthOf', 'PointcloudDepthOf', 'ExtremalDepth',
           'HalfspaceDepth', 'FunctionalHalfspaceDepth', 'ProjectionDepth', 'FunctionalProjectionDepth',
           'FunctionalBoxplot', 'Outliergram', 'FunctionalReference', 'DepthClassifier',
           'FunctionalProjectionDepthOf', 'ProjectionDepthOf', 'FunctionalSpatialDepth', 'FunctionalSpatialDepthOf',
           'AbstractDepth']


def _go():
    try:
        import plotly.graph_objects as go
    except ImportError as exc:  # pragma: no cover - plotting is host-only convenience
        raise ImportError('the plot_* helpers need plotly (pip install plotly)') from exc
    return go


class AbstractDepth(ABC):
    """Interface every depth result implements (abstract.py:3-18)."""

    @abstractmethod
    def ordered(self, ascending=False):
        raise NotImplementedError

    @abstractmethod
    def deepest(self, n=1):
        raise NotImplementedError

    @abstractmethod
    def outlying(self, n=1):
        raise NotImplementedError


class _FunctionalDepthSeries(AbstractDepth, pd.Series):
    """pd.Series of depths that remembers the data it was computed from (depth.py:14-65)."""

    def __init__(self, df: pd.DataFrame, depths: pd.Series):
        super().__init__(data=depths)
        self._orig_data = df
        self._depths = depths
        self._ordered_depths = None

    def ordered(self, ascending=False) -> pd.Series:
        """Curves sorted from deepest to most outlying."""
        if self._ordered_depths is None:
            self._ordered_depths = self._depths.sort_values(ascending=ascending)
        return self._ordered_depths

    def _desc(self) -> pd.Series:
        if self._ordered_depths is None:
            self._ordered_depths = self._depths.sort_values(ascending=False)
        return self._ordered_depths

    def deepest(self, n=1) -> pd.Series:
        o = self._desc()
        if n == 1:
            return pd.Series(index=[list(o.index)[0]], data=[o.values[0]])
        return pd.Series(index=o.index[0:n], data=o.values[0:n])

    def outlying(self, n=1) -> pd.Series:
        o = self._desc()
        if n == 1:
            return pd.Series(index=[list(o.index)[-1]], data=[o.values[-1]])
        return pd.Series(index=o.index[-n:], data=o.values[-n:])

    def sorted(self, ascending=False):
        return self.ordered(ascending=ascending)

    def median(self):
        return self.deepest(n=1)

    def quartile(self, ratio=0.5):
        # the reference ignores `ratio` and always takes the lower half (depth.py:55-56); kept
        return self._depths.sort_values().head(int(self._depths.shape[0] * 0.5))

    def get_depths(self):
        return self._depths

    def get_data(self):
        return self._orig_data

    def depths(self):
        return self.get_depths()


class _FunctionalDepthMultivariateDataFrame(AbstractDepth, pd.DataFrame):
    """Placeholder result type of the reference (depth.py:67-83); never produced by the exact path."""

    def __init__(self, depths: pd.DataFrame):
        super().__init__(depths)
        self._depths = depths

    def ordered(self, ascending=False):
        pass

    def deepest(self, n=1):
        pass

    def outlying(self, n=1):
        pass


class _FunctionalDepthUnivariate(_FunctionalDepthSeries):
    """Real-valued curves: samples are COLUMNS of the original frame (depth.py:87-185)."""

    def __init__(self, df: pd.DataFrame, depths: pd.Series):
        super().__init__(df=df, depths=depths)

    def _plot(self, deep_or_outlying: pd.Series, title, xaxis_title, yaxis_title, return_plot, showlegend):
        go = _go()
        cols = self._orig_data.columns
        x = self._orig_data.index
        traces = [go.Scatter(x=x, y=self._orig_data.loc[:, y], mode='lines', name=y,
                             line=dict(color='#6ea8ff', width=.5))
                  for y in cols.difference(deep_or_outlying.index)]
        traces.extend(go.Scatter(x=x, y=self._orig_data.loc[:, y], mode='lines', name=y,
                                 line=dict(color='Red', width=1)) for y in deep_or_outlying.index)
        fig = go.Figure(data=traces, layout=go.Layout(
            title=dict(text=title, y=0.9, x=0.5, xanchor='center', yanchor='top'),
            xaxis=dict(title=xaxis_title), yaxis=dict(title=yaxis_title)))
        fig.update_layout(showlegend=showlegend)
        return fig if return_plot else fig.show()

    def plot_deepest(self, n=1, title=None, xaxis_title=None, yaxis_title=None, return_plot=False,
                     showlegend=False):
        """All curves in blue, the n deepest in red."""
        return self._plot(self.deepest(n=n), title, xaxis_title, yaxis_title, return_plot, showlegend)

    def plot_outlying(self, n=1, title=None, xaxis_title=None, yaxis_title=None, return_plot=False,
                      showlegend=False):
        """All curves in blue, the n most outlying in red."""
        return self._plot(self.outlying(n=n), title, xaxis_title, yaxis_title, return_plot, showlegend)

    def drop_outlying_data(self, n=1) -> pd.DataFrame:
        return self._orig_data.drop(self.outlying(n=n).index, axis=1)

    def get_deepest_data(self, n=1) -> pd.DataFrame:
        return self._orig_data.loc[:, self.deepest(n=n).index]

    def get_outlying_data(self, n=1) -> pd.DataFrame:
        return self._orig_data.loc[:, self.outlying(n=n).index]


class _PointwiseDepth(_FunctionalDepthSeries):
    """Depth of every point of a cloud: samples are ROWS of the original frame (depth.py:187-344)."""

    def __init__(self, df: pd.DataFrame, depths: pd.Series):
        super().__init__(df=df, depths=depths)

    def _scatter(self, go, frame, **marker):
        cols = self._orig_data.columns
        if len(cols) == 3:
            return go.Scatter3d(x=frame[cols[0]], y=frame[cols[1]], z=frame[cols[2]], mode='markers', **marker)
        return go.Scatter(x=frame[cols[0]], y=frame[cols[1]], mode='markers', **marker)

    def plot_depths(self, invert_colors=False, marker=None, return_plot=False, title='', xaxis_title=None,
                    yaxis_title=None):
        go = _go()
        d = 1 - self._depths if invert_colors else self._depths
        ncol = len(self._orig_data.columns)
        if marker is None:
            marker = dict(color=d, colorscale='viridis', size=7)
        if ncol > 3:
            return self._plot_parallel_axis()
        if ncol < 2:
            raise ValueError(f'Error: Dimensionality of data must be >=2. Value found is {ncol}')
        fig = go.Figure(data=[self._scatter(go, self._orig_data, marker=marker)],
                        layout=go.Layout(title=title, xaxis_title=xaxis_title, yaxis_title=yaxis_title))
        fig.update_layout(showlegend=False)
        return fig if return_plot else fig.show()

    def _plot_parallel_axis(self) -> None:
        pass

    def _plot(self, deep_or_outlying: pd.Series, return_plot, title, xaxis_title, yaxis_title):
        go = _go()
        ncol = len(self._orig_data.columns)
        select = self._orig_data.loc[deep_or_outlying.index, :]
        if ncol > 3:
            return self._plot_parallel_axis()
        if ncol < 2:
            raise ValueError(f'Error: Dimensionality of data must be >=2. Value found is {ncol}')
        fig = go.Figure(data=[self._scatter(go, self._orig_data, marker_color='blue', name=''),
                              self._scatter(go, select, marker_color='red', name='')],
                        layout=go.Layout(title=title, xaxis_title=xaxis_title, yaxis_title=yaxis_title))
        fig.update_layout(showlegend=False)
        return fig if return_plot else fig.show()

    def plot_deepest(self, n=1, return_plot=False, title='', xaxis_title=None, yaxis_title=None):
        return self._plot(self.deepest(n=n), return_plot, title, xaxis_title, yaxis_title)

    def plot_outlying(self, n=1, return_plot=False, title='', xaxis_title=None, yaxis_title=None):
        return self._plot(self.outlying(n=n), return_plot, title, xaxis_title, yaxis_title)

    def drop_outlying_data(self, n=1) -> pd.DataFrame:
        return self._orig_data.drop(self.outlying(n=n).index, axis=0)

    def get_deepest_data(self, n=1) -> pd.DataFrame:
        return self._orig_data.loc[self.deepest(n=n).index, :]

    def plot_distribution(self, invert_colors=False, marker=None) -> None:
        self.plot_depths(invert_colors, marker)


def PointcloudDepth(
    data: pd.DataFrame,
    to_compute: pd.Index = None,
    K=None,
    containment='simplex',
    quiet=True,
) -> _PointwiseDepth:
    """Depth of the rows of an n x d DataFrame.  containment in 'simplex' | 'l1' | 'oja' | 'mahalanobis'.
    Signature and result type of statdepth.PointcloudDepth (depth.py:347-359)."""
    if K is not None:
        depth = _samplepointwisedepth(data=data, to_compute=to_compute, K=K, containment=containment)
    else:
        depth = _pointwisedepth(data=data, to_compute=to_compute, containment=containment)
    return _PointwiseDepth(df=data, depths=depth)


def FunctionalDepth(
    data: List[pd.DataFrame],
    to_compute=None,
    K=None,
    J=2,
    containment='r2',
    relax=False,
    deep_check=False,
    quiet=True,
) -> Union[_FunctionalDepthSeries, _FunctionalDepthUnivariate, _FunctionalDepthMultivariateDataFrame]:
    """Band depth of curves.  `[df]` (T rows x n curve columns) is the univariate case; a list of N
    DataFrames (T rows x d channels) the multivariate one.  Signature and result types of
    statdepth.FunctionalDepth (depth.py:362-402)."""
    if K is not None:
        depth = _samplefunctionaldepth(data=data, to_compute=to_compute, K=K, J=J, containment=containment,
                                       relax=relax, deep_check=deep_check, quiet=quiet)
    else:
        depth = _functionaldepth(data=data, to_compute=to_compute, J=J, containment=containment, relax=relax,
                                 deep_check=deep_check, quiet=quiet)
    if isinstance(depth, pd.DataFrame):
        return _FunctionalDepthMultivariateDataFrame(depths=depth)
    elif len(data) == 1:
        return _FunctionalDepthUnivariate(df=data[0], depths=depth)
    else:
        return _FunctionalDepthSeries(df=data[0], depths=depth)


def FunctionalDepthOf(
    data: List[pd.DataFrame],
    sample: List[pd.DataFrame],
    J=2,
    containment='r2',
    relax=False,
    deep_check=False,
    quiet=True,
) -> _FunctionalDepthUnivariate:
    """Out-of-sample band depth: the depth of every curve (column) of data[0] against the reference sample
    sample[0] (both T x n DataFrames with the same T rows).  Each curve gets the depth FunctionalDepth would give it
    after it alone is appended to the sample; the other curves of data never take part.  The result is indexed by
    data[0].columns (positions decide, so a label may also occur in the sample).  J = 2 or 3, containment 'r2'."""
    depth = _functionaldepth_of(data=data, sample=sample, J=J, containment=containment, relax=relax,
                                deep_check=deep_check, quiet=quiet)
    return _FunctionalDepthUnivariate(df=data[0], depths=depth)


def PointcloudDepthOf(
    data: pd.DataFrame,
    sample: pd.DataFrame,
    containment='simplex',
    quiet=True,
) -> _PointwiseDepth:
    """Out-of-sample point-cloud depth: the depth of every row of data (m x d) against the reference cloud sample
    (n x d), as PointcloudDepth would give it after that row alone is appended to the sample.  containment is
    'simplex' (d <= 3) or 'l1' (d <= 16).  Indexed by data.index."""
    depth = _pointwisedepth_of(data=data, sample=sample, containment=containment, quiet=quiet)
    return _PointwiseDepth(df=data, depths=depth)


def ExtremalDepth(data: List[pd.DataFrame], deep_check=False) -> _FunctionalDepthUnivariate:
    """Extremal depth (Narisetty & Nair 2016) of the curves (columns) of data[0], a T x n DataFrame.

    At every time point a curve's extremity is |#curves strictly below - #curves strictly above|.  Curves are ordered
    by their extremities sorted from largest down, compared lexicographically, so a curve that is extreme somewhere,
    even for a short stretch, ranks as extreme (modified band depth averages such a stretch away).  The depth is the
    share of curves at least as extreme: the deepest curve has 1, equally extreme curves have equal depth.  Indexed
    by data[0].columns.  Univariate data with at most 16 384 time points; non-finite values are rejected."""
    X = _checked_values(data, NO_FACTOR, deep_check, what='extremal depth')
    _check_extremal_rows(X.shape[0])
    e = _extremal_depth(X)
    return _FunctionalDepthUnivariate(df=data[0], depths=pd.Series(index=data[0].columns,
                                                                   data=e.astype(np.float64) / X.shape[1]))


def HalfspaceDepth(data: pd.DataFrame, to_compute=None) -> _PointwiseDepth:
    """Halfspace (Tukey) depth of the rows of an n x d DataFrame, d = 1 or 2.

    A point's depth is the smallest share of the n points, itself included, that a closed half-plane (a half-line
    for d = 1) whose boundary passes through the point can hold: at least 1 / n, at most 1.  Directions are compared
    exactly in float64 (no tolerance band; set_simplex_tolerance does not apply).  Indexed by to_compute (row labels)
    or data.index.  Non-finite values are rejected."""
    return _PointwiseDepth(df=data, depths=_pointcloud_halfspace(data, to_compute))


def FunctionalHalfspaceDepth(data: List[pd.DataFrame],
                             to_compute=None) -> Union[_FunctionalDepthSeries, _FunctionalDepthUnivariate]:
    """Integrated halfspace depth of curves (Claeskens, Hubert, Slaets & Vakili 2014, uniform weights): the mean
    over time points of the halfspace depth of each curve's value among all curves' values at that time.

    `[df]` (T rows x n curve columns) is the univariate case, to_compute are column labels; a list of N DataFrames
    (T rows x 2 channels) the bivariate one, to_compute are list positions (as FunctionalDepth).  Other channel
    counts raise NotImplementedError.  Non-finite values are rejected."""
    depth = _functional_halfspace(data, to_compute)
    if len(data) == 1:
        return _FunctionalDepthUnivariate(df=data[0], depths=depth)
    return _FunctionalDepthSeries(df=data[0], depths=depth)


def ProjectionDepth(data: pd.DataFrame, kind='projection', directions=None, seed=0,
                    to_compute=None) -> _PointwiseDepth:
    """Random projection depth of the rows of an n x d DataFrame, any d.

    kind='projection': projection depth (Zuo & Serfling 2000), 1 / (1 + O) with O the largest |u.x - med| / MAD
    over the directions u (med and the unscaled MAD of the projected sample).  kind='tukey': random Tukey depth
    (Cuesta-Albertos & Nieto-Reyes 2008), the smallest share of points, the point included, in a closed half-line
    of one projection; an upper bound on the exact halfspace depth.  directions: None (1000), an int K (K random
    unit directions from np.random.default_rng(seed)) or an array [K, d] used as given (finite, non-zero rows).
    Indexed by to_compute (row labels) or data.index.  Non-finite values are rejected."""
    return _PointwiseDepth(df=data, depths=_pointcloud_projection(data, kind, directions, seed, to_compute))


def FunctionalProjectionDepth(data: List[pd.DataFrame], kind='projection', directions=None, seed=0,
                              to_compute=None) -> Union[_FunctionalDepthSeries, _FunctionalDepthUnivariate]:
    """Integrated random projection depth of curves: the mean over time points of ProjectionDepth of each curve's
    value among all curves' values at that time (kind='tukey': sum of numerators over time, divided once by T n).

    `[df]` (T rows x n curve columns) is the univariate case, with the single direction 1.0 (directions must be
    None; kind='tukey' is FunctionalHalfspaceDepth([df])), to_compute are column labels; a list of N DataFrames
    (T rows x d channels, any d) the multivariate one, to_compute are list positions.  directions and seed as for
    ProjectionDepth.  Non-finite values are rejected."""
    depth = _functional_projection(data, kind, directions, seed, to_compute)
    if len(data) == 1:
        return _FunctionalDepthUnivariate(df=data[0], depths=depth)
    return _FunctionalDepthSeries(df=data[0], depths=depth)


# ---------------------------------------------------------------------------------------------------------------
# functional outlier detection (drivers in _outliers.py)
# ---------------------------------------------------------------------------------------------------------------
class _OutlierResult:
    """What both outlier rules share: the curves' modified band depth."""

    def __init__(self, df: pd.DataFrame, r: dict):
        self._df = df
        self._r = r

    def _series(self, values) -> pd.Series:
        return pd.Series(index=self._df.columns, data=values)

    def _labels(self, positions) -> list:
        return [self._df.columns[p] for p in positions]

    def _rows(self, pair) -> pd.DataFrame:
        return pd.DataFrame({'lower': pair[0], 'upper': pair[1]}, index=self._df.index)

    def depths(self) -> _FunctionalDepthUnivariate:
        """Modified band depth of every curve, bit-identical to FunctionalDepth([df], J=2, relax=True) (the
        boxplot with depth='extremal': extremal depth, equal to ExtremalDepth([df]))."""
        return _FunctionalDepthUnivariate(df=self._df, depths=self._series(self._r['depth']))

    def outliers(self) -> list:
        """Labels of the flagged curves, in column order."""
        return self._labels(np.flatnonzero(self._outlier_mask()))


class _FunctionalBoxplot(_OutlierResult):
    """Functional boxplot (Sun & Genton 2011): central region, envelope, fences, whiskers, magnitude outliers."""

    def median(self):
        """Label of the deepest curve (first of the central region)."""
        return self._df.columns[self._r['central'][0]]

    def central_region(self) -> list:
        """Labels of the central curves, deepest first; ties in depth by column position."""
        return self._labels(self._r['central'])

    def envelope(self) -> pd.DataFrame:
        """Per time row, min ('lower') and max ('upper') of the central curves."""
        return self._rows(self._r['envelope'])

    def fences(self) -> pd.DataFrame:
        """The envelope inflated by factor x its width on both sides."""
        return self._rows(self._r['fences'])

    def whiskers(self) -> pd.DataFrame:
        """Per time row, min and max of the curves that are not outliers."""
        return self._rows(self._r['whiskers'])

    def outside_counts(self) -> pd.Series:
        """Per curve, the number of time rows at which it is strictly outside the fences."""
        return self._series(self._r['outside'])

    def _outlier_mask(self):
        return self._r['outside'] > 0


class _Outliergram(_OutlierResult):
    """Outliergram (Arribas-Gil & Romo 2014): MBD against the modified epigraph index, shape outliers."""

    def mei(self) -> pd.Series:
        """Modified epigraph index: the share of (curve, time) pairs at or above the curve, itself included."""
        return self._series(self._r['mei'])

    def distance(self) -> pd.Series:
        """How far below the parabola a0 + a1 MEI + a2 n^2 MEI^2 the curve's MBD lies (>= 0 without ties)."""
        return self._series(self._r['distance'])

    def _outlier_mask(self):
        return self._r['outlier']


def FunctionalBoxplot(data: List[pd.DataFrame], factor=1.5, central=0.5, deep_check=False,
                      depth='mbd') -> _FunctionalBoxplot:
    """Functional boxplot of the curves (columns) of data[0], a T x n DataFrame.

    The central region is the ceil(central * n) curves of largest depth (ties by column position; under ties this
    can differ from ordered(), whose sort is not stable): modified band depth with depth='mbd', extremal depth
    (ExtremalDepth) with depth='extremal', which keeps curves that leave the bulk for a short stretch out of the
    central region.  Its per-row envelope, inflated by factor x its width, gives the fences; a curve strictly
    outside them at any time point is a magnitude outlier.  depths() returns the depth the region was ranked by.
    Non-finite values are rejected."""
    X = _checked_values(data, factor, deep_check)
    _check_central(central)
    if not (isinstance(depth, str) and depth in ('mbd', 'extremal')):
        raise ValueError("depth must be 'mbd' or 'extremal'.")
    if depth == 'extremal':
        _check_extremal_rows(X.shape[0])
    return _FunctionalBoxplot(data[0], _functional_boxplot(X, float(factor), float(central), depth))


def Outliergram(data: List[pd.DataFrame], factor=1.5, deep_check=False) -> _Outliergram:
    """Outliergram of the curves (columns) of data[0], a T x n DataFrame: a curve whose distance below the
    MBD-MEI parabola is at least q3 + factor * (q3 - q1) of all distances is a shape outlier.
    Non-finite values are rejected."""
    X = _checked_values(data, factor, deep_check)
    return _Outliergram(data[0], _outliergram(X, float(factor)))


# ---------------------------------------------------------------------------------------------------------------
# fitted references and depth-based classification (driver in _reference.py)
# ---------------------------------------------------------------------------------------------------------------
def _check_reference_depth(depth, J, directions):
    if not (isinstance(depth, str) and depth in ('mbd', 'spatial') + KINDS):
        raise ValueError("depth must be 'mbd', 'projection', 'tukey' or 'spatial' (got %r)" % (depth,))
    if depth in ('mbd', 'spatial') and directions is not None:
        raise ValueError("directions apply to depth='projection' or 'tukey'")
    if depth != 'mbd' and J != 2:
        raise ValueError('J applies to depth=\'mbd\' only: leave it at 2 for depth=%r' % depth)


class FunctionalReference:
    """A reference sample fitted once; depth_of() scores new curves against it.

    depth='mbd' (relaxed band depth, J = 2 or 3, univariate sample[0], a T x n_S DataFrame): construction sorts every
    time row of the sample on the GPU and keeps only that index; each depth_of() call then uploads only the new curves
    and binary-searches them in the sorted rows.  depth_of([df]) equals FunctionalDepthOf([df], sample, J=J,
    relax=True) bit for bit.  A strict band must hold a curve at all T points jointly, which sorted rows cannot decide.

    depth='projection' or 'tukey' (J must stay 2): sample is [df] (univariate, directions must be None) or N
    DataFrames of T x d.  Construction draws the directions once (as FunctionalProjectionDepth: None gives 1000, an
    int K gives K random unit directions from seed, an array [K, d] is used as given; kept as .directions, None for
    univariate data) and sorts the sample's projections per (time point, direction) on the GPU: an index of T K n_S
    doubles (2.05 GB at n_S = 5 000, T = 256, K = 200) kept for as long as the reference.  A new curve g gets the depth
    FunctionalProjectionDepth(sample + [g], kind=depth, directions=.directions) gives it, bit for bit; the other new
    curves never take part.

    depth='spatial' (J must stay 2, directions None): sample is [df] or N DataFrames of T x d, as for the projection
    kinds.  The sample's n_S x T d values stay on the GPU for as long as the reference; a new curve g gets the depth
    FunctionalSpatialDepth(sample + [g]) gives it, bit for bit, and each depth_of() call uploads only the new curves.

    Non-finite values (and, for the projection kinds, projections that overflow) are rejected.  close() (or leaving a
    `with` block) frees the index."""

    def __init__(self, sample: List[pd.DataFrame], J=2, deep_check=False, depth='mbd', directions=None, seed=0):
        _check_reference_depth(depth, J, directions)
        self.J = J
        self.depth = depth
        self.directions = None
        if depth == 'mbd':
            _checked_reference(sample, J, deep_check)
            self._T = sample[0].shape[0]
            self._index = sample[0].index
            self._ref = _SortedReference(_values(sample[0]), J)
            return
        if depth == 'spatial':
            X, F = _spatial_curves(sample)
            self._T = sample[0].shape[0]
            self._index = sample[0].index
            self._d = None if F is None else F.shape[2]
            self._ref = _SpatialReference(X=X, F=F)
            return
        X, F = _curve_values(sample, directions)
        if X is not None and X.shape[1] == 0:
            raise ValueError('No data passed.')
        self._T = sample[0].shape[0]
        self._index = sample[0].index
        self._d = None if F is None else F.shape[2]
        if F is not None:
            self.directions = draw_directions(self._d, directions, seed)
        self._ref = _ProjectedReference(depth, X=X, F=F, U=self.directions)

    def depth_of(self, data: List[pd.DataFrame], deep_check=False) -> _FunctionalDepthSeries:
        """Depth of every new curve against the reference.  Univariate: the columns of data[0], indexed by
        data[0].columns (a label may repeat a sample label).  Multivariate (projection kinds, spatial): M DataFrames of
        T x d, indexed by list position, as FunctionalProjectionDepth."""
        if self._ref is None:
            raise ValueError('the reference is closed')
        if self.depth == 'mbd':
            Y = _query_values(data, self.J, deep_check, self._T, self._index)
            depth = pd.Series(index=data[0].columns, data=self._ref.depths(Y))
            return _FunctionalDepthUnivariate(df=data[0], depths=depth)
        X, F = _curve_values(data, frames=self._d is not None)
        if data[0].shape[0] != self._T:
            raise ValueError('data and sample must have the same number of time points.')
        if F is not None and F.shape[2] != self._d:
            raise ValueError('data and sample must have the same number of channels.')
        if deep_check and not all(len(df.index) == len(self._index) and all(df.index == self._index) for df in data):
            raise ValueError('DataFrames indices must be the same')
        if F is None:
            return _FunctionalDepthUnivariate(df=data[0], depths=pd.Series(index=data[0].columns,
                                                                           data=self._ref.depths(X)))
        return _FunctionalDepthSeries(df=data[0], depths=pd.Series(index=list(range(len(data))),
                                                                   data=self._ref.depths(F)))

    def close(self) -> None:
        if self._ref is not None:
            self._ref.close()
            self._ref = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


class DepthClassifier:
    """Maximum-depth classifier (Lopez-Pintado & Romo 2006): a curve belongs to the class in which it is deepest.

    references maps each class label to its training curves, each class fitted once as a FunctionalReference with
    the given depth.  depth='mbd': [DataFrame] T x n_k, the same T for every class; depths([df]) (one column per class)
    equal FunctionalDepthOf([df], references[label], J=J, relax=True).  depth='projection' or 'tukey': [df] for every
    class, or lists of T x d DataFrames with the same T and d for every class; one set of directions, drawn once from
    d and seed (or given), is shared by all classes (.directions), so that the DD-plot coordinates are comparable.
    depth='spatial': the same forms of data as the projection kinds, without directions.
    predict(data) takes the class of largest depth, ties going to the class listed first."""

    def __init__(self, references: dict, J=2, deep_check=False, depth='mbd', directions=None, seed=0):
        if not isinstance(references, dict) or len(references) < 2:
            raise ValueError('references must be a dict of at least two classes.')
        _check_reference_depth(depth, J, directions)
        for sample in references.values():
            if depth == 'mbd':
                _checked_reference(sample, J, deep_check)
            else:
                _curve_values(sample, directions)
        if len({sample[0].shape[0] for sample in references.values()}) > 1:
            raise ValueError('every class must have the same number of time points.')
        self.directions = None
        if depth != 'mbd':
            if len({len(sample) == 1 for sample in references.values()}) > 1:
                raise ValueError('every class must be univariate, or every class multivariate.')
            dims = {sample[0].shape[1] for sample in references.values() if len(sample) > 1}
            if len(dims) > 1:
                raise ValueError('every class must have the same number of channels.')
            if dims and depth in KINDS:
                self.directions = draw_directions(dims.pop(), directions, seed)
        self.labels = list(references)
        self._refs = []
        try:
            for label in self.labels:
                self._refs.append(FunctionalReference(references[label], J=J, deep_check=deep_check, depth=depth,
                                                      directions=self.directions))
        except BaseException:
            self.close()
            raise

    def depths(self, data: List[pd.DataFrame], deep_check=False) -> pd.DataFrame:
        """Depth of every new curve in every class: one column per class label, rows indexed as
        FunctionalReference.depth_of indexes them (data[0].columns, or list positions for multivariate curves)."""
        if not self._refs:
            raise ValueError('the classifier is closed')
        res = [ref.depth_of(data, deep_check=deep_check) for ref in self._refs]
        return pd.DataFrame(np.column_stack([r.values for r in res]), index=res[0].index,
                            columns=pd.Index(self.labels, tupleize_cols=False))

    def predict(self, data: List[pd.DataFrame], deep_check=False) -> pd.Series:
        """Label of the class of largest depth for every new curve (ties: the class listed first)."""
        d = self.depths(data, deep_check=deep_check)
        best = np.argmax(d.to_numpy(), axis=1)  # the first maximum
        return pd.Series([self.labels[k] for k in best], index=d.index, dtype=object)

    def close(self) -> None:
        for ref in self._refs:
            ref.close()
        self._refs = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


def FunctionalProjectionDepthOf(data: List[pd.DataFrame], sample: List[pd.DataFrame], kind='projection',
                                directions=None, seed=0) -> _FunctionalDepthSeries:
    """Out-of-sample integrated projection depth (kind='projection') or random Tukey depth ('tukey') of new curves
    against the reference curves sample: each new curve gets what FunctionalProjectionDepth(sample + [g], kind,
    directions, seed) gives it, bit for bit; the other new curves never take part.  Univariate [df] (T x n, indexed by
    data[0].columns; directions must be None) or lists of T x d DataFrames (indexed by list position).  One call of
    FunctionalReference(sample, depth=kind, ...).depth_of(data): to score many batches, keep the reference."""
    with FunctionalReference(sample, depth=kind, directions=directions, seed=seed) as ref:
        return ref.depth_of(data)


def ProjectionDepthOf(data: pd.DataFrame, sample: pd.DataFrame, kind='projection', directions=None,
                      seed=0) -> _PointwiseDepth:
    """Out-of-sample projection depth (kind='projection') or random Tukey depth ('tukey') of the rows of data (m x d)
    against the reference cloud sample (n x d): each row gets what ProjectionDepth(pd.concat([sample, row]), kind,
    directions, seed) gives it, bit for bit.  The sample's projections are sorted once on the GPU (K n doubles) and
    every row is binary-searched in them.  Indexed by data.index.  Non-finite values are rejected."""
    for name, df in (('data', data), ('sample', sample)):
        if not isinstance(df, pd.DataFrame):
            raise ValueError('%s must be a DataFrame (points x d columns).' % name)
    if sample.shape[0] == 0 or sample.shape[1] == 0:
        raise ValueError('No data passed.')
    if data.shape[1] != sample.shape[1]:
        raise ValueError('data and sample must have the same number of columns.')
    if kind not in KINDS:
        raise ValueError("kind must be one of %s (got %r)" % (KINDS, kind))
    U = draw_directions(sample.shape[1], directions, seed)
    ref = _ProjectedReference(kind, F=np.ascontiguousarray(_values(sample))[:, None, :], U=U, cloud=True)
    try:
        depth = ref.depths(np.ascontiguousarray(_values(data))[:, None, :])
    finally:
        ref.close()
    return _PointwiseDepth(df=data, depths=pd.Series(index=data.index, data=depth))


# ---------------------------------------------------------------------------------------------------------------
# functional spatial depth (driver in _spatial.py)
# ---------------------------------------------------------------------------------------------------------------
def FunctionalSpatialDepth(data: List[pd.DataFrame],
                           to_compute=None) -> Union[_FunctionalDepthSeries, _FunctionalDepthUnivariate]:
    """Functional spatial depth (Chakraborty & Chaudhuri 2014; depth.FSD in fda.usc): a curve is the vector of its
    T d values, and its depth is 1 - || sum_j u(x_j - x) || / n with u(v) = v / ||v|| (Euclidean norm over all values,
    (t, c) order, no time weight, channels as given) and u(0) = 0, so duplicates of x contribute nothing; n counts x.
    Unlike the pointwise depths it sees a curve as one object: a shape that is slightly wrong at every time point
    gets a low depth.

    `[df]` (T rows x n curve columns) is the univariate case, to_compute are column labels; a list of N DataFrames
    (T rows x d channels, any d) the multivariate one, to_compute are list positions.  Non-finite values are
    rejected, and so (EngineError, SD_ERR_OVERFLOW) are curves whose squared distance overflows float64."""
    depth = _functional_spatial(data, to_compute)
    if len(data) == 1:
        return _FunctionalDepthUnivariate(df=data[0], depths=depth)
    return _FunctionalDepthSeries(df=data[0], depths=depth)


def FunctionalSpatialDepthOf(data: List[pd.DataFrame],
                             sample: List[pd.DataFrame]) -> Union[_FunctionalDepthSeries, _FunctionalDepthUnivariate]:
    """Out-of-sample functional spatial depth: each new curve g gets what FunctionalSpatialDepth(sample + [g]) gives
    it (divisor n_S + 1), bit for bit; the other new curves never take part.  Univariate [df] (T x n, indexed by
    data[0].columns) or lists of T x d DataFrames (indexed by list position).  To score many batches against one
    sample, keep a FunctionalReference(sample, depth='spatial'), which keeps the sample on the GPU."""
    depth = _functional_spatial_of(data, sample)
    if len(sample) == 1:
        return _FunctionalDepthUnivariate(df=data[0], depths=depth)
    return _FunctionalDepthSeries(df=data[0], depths=depth)
