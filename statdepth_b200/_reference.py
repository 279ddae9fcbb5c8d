"""Fitted reference driver: a reference sample indexed once on the device (csrc/reference.cu, DESIGN.md K9).

Modified band depth (K9).  Relaxed out-of-sample band depth needs, per new curve and time row, only the number of sample values strictly below
and strictly above the new value.  Both come from binary searches in the sorted row, so the sample's rows are sorted
once on the device and kept there (the index); every later call uploads only the new curves.  The counts are the
integers sd_band_depth_oos_f64 returns and the floats are formed by _functional._relaxed_depths_of, so the depths are
bit-identical to FunctionalDepthOf(relax=True).

On one GPU the index lives in a torch tensor on the engine's device.  An engine without the `_dev` entry points (the
CPU test double) keeps a host index from its `band_sort_rows` and answers `band_depth_sorted_counts`.  Under
`enable_distributed()` every rank indexes its block of time rows; each call scores the same rows of the new curves and
all-reduces the counts, so construction and every call are collectives.

Projection and random Tukey depth (csrc/reference_proj.cu, DESIGN.md K13).  The reference's projections along the
directions U are sorted once per (time point, direction): an index of T K n_S doubles (K9's sorted rows for univariate
curves, whose single direction is 1.0).  A new observation g gets the depth FunctionalProjectionDepth /
ProjectionDepth give it after g alone is appended to the reference, with the same U: the engine returns the integer
numerators or the outlyingness rows of that pooled call, and the floats are formed here with the expressions
_projection.py uses, so the depths are bit-identical.  Under `enable_distributed()` this mirrors _projection.py: curves
split the time rows (numerators summed, outlyingness rows all-gathered), point clouds split the directions (MIN / MAX
all-reduced); a rank without rows or directions contributes the identity.
"""
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import device_rows, get_engine
from ._functional import _relaxed_depths_of, _values
from ._helper import _handle_depth_errors
from ._projection import _depth_from_rows

__all__ = ['_checked_reference', '_query_values', '_SortedReference', '_curve_values', '_ProjectedReference']


def _checked_reference(data: List[pd.DataFrame], J, deep_check) -> None:
    """The checks FunctionalDepthOf(relax=True) runs on one of its arguments, for univariate data and J <= 3."""
    if isinstance(data, list) and len(data) > 1:
        raise NotImplementedError('a fitted reference is implemented for univariate data ([DataFrame])')
    _handle_depth_errors(data=data, J=J, containment='r2', relax=True, deep_check=deep_check)
    if J > 3:
        raise NotImplementedError('a fitted reference is implemented for J <= 3 on the B200 engine')


class _SortedReference:
    """This rank's time rows of a reference sample S [T, nS], sorted once."""

    def __init__(self, S: np.ndarray, J: int):
        self.T, self.nS = S.shape
        self.J = J
        rank, self.size = _dist.world()
        self.lo, self.hi = _dist.block(self.T, rank, self.size)
        self.eng = get_engine()
        self.on_device = hasattr(self.eng, 'band_sort_rows_dev')
        rows = S[self.lo:self.hi]
        self.index = None
        if self.hi == self.lo:
            return
        if not self.on_device:
            self.index = np.asarray(self.eng.band_sort_rows(rows), dtype=np.float64)
            return
        import torch
        self.torch = torch
        stream, dX = device_rows(self.eng, rows)
        with torch.cuda.stream(stream):
            index = torch.empty((self.hi - self.lo, self.nS), dtype=torch.float64, device=dX.device)
            self.eng.band_sort_rows_dev(dX.data_ptr(), self.hi - self.lo, self.nS, self.nS, index.data_ptr())
        self.index = index  # the raw rows are dropped on return

    def counts(self, Y: np.ndarray) -> np.ndarray:
        """int64 [J - 1, nY]: row j - 2 holds the relaxed numerators of subset size j, summed over the ranks."""
        nY = Y.shape[1]
        rows = Y[self.lo:self.hi]
        if self.index is None:
            local = np.zeros((self.J - 1, nY), dtype=np.int64)
        elif not self.on_device:
            local = np.asarray(self.eng.band_depth_sorted_counts(self.index, rows, self.J), dtype=np.int64)
        else:
            torch = self.torch
            stream, dY = device_rows(self.eng, rows)
            with torch.cuda.stream(stream):
                out = torch.empty((self.J - 1, nY), dtype=torch.int64, device=dY.device)
                self.eng.band_depth_sorted_counts_dev(self.index.data_ptr(), self.hi - self.lo, self.nS, dY.data_ptr(),
                                                      nY, nY, self.J, out.data_ptr())
                local = out.cpu().numpy()
        return local if self.size == 1 else _dist.allreduce(local)

    def depths(self, Y: np.ndarray) -> np.ndarray:
        """Relaxed depth of every new curve (column of Y [T, nY]), bit-identical to FunctionalDepthOf(relax=True)."""
        if Y.shape[1] == 0:
            return np.zeros(0, dtype=np.float64)
        return _relaxed_depths_of(list(self.counts(Y)), self.T, self.nS)

    def close(self) -> None:
        self.index = None


def _query_values(data: List[pd.DataFrame], J: int, deep_check, T: int, index: pd.Index) -> np.ndarray:
    """FunctionalDepthOf's checks of the new curves against a fitted sample; their values [T, nY]."""
    _checked_reference(data, J, deep_check)
    df = data[0]
    if df.shape[0] != T:
        raise ValueError('data and sample must have the same number of time points.')
    if deep_check and not (len(df.index) == len(index) and all(df.index == index)):
        raise ValueError('DataFrames indices must be the same')
    return _values(df)


def _curve_values(data: List[pd.DataFrame], directions=None, frames=None):
    """(X [T, n], None) of univariate curves [df] (directions must be None) or (None, F [N, T, d]) of N DataFrames of
    T x d, checked as FunctionalProjectionDepth checks them.  frames=True takes even one DataFrame as one curve of
    T x d (new curves against a multivariate reference), frames=False requires [df]."""
    if not isinstance(data, list):
        raise ValueError('data must be passed as a list.')
    if len(data) == 0:
        raise ValueError('No data passed.')
    if frames is False and len(data) != 1:
        raise ValueError('the reference is univariate: pass the new curves as [DataFrame].')
    if len(data) == 1 and not frames:
        if directions is not None:
            raise ValueError('univariate curves have the single direction 1.0: directions must be None')
        if data[0].shape[0] == 0:
            raise ValueError('No data passed.')
        return _values(data[0]), None
    if len({df.shape[1] for df in data}) > 1:
        raise ValueError('every curve must have the same number of channels.')
    if len({df.shape[0] for df in data}) > 1:
        raise ValueError('every curve must have the same number of time points.')
    if data[0].shape[0] == 0 or data[0].shape[1] == 0:
        raise ValueError('No data passed.')
    return None, np.stack([_values(df) for df in data])


class _ProjectedReference:
    """This rank's share of a reference fitted for projection (kind='projection') or random Tukey depth ('tukey'):
    univariate curves X [T, nS] (U None), or curves F [nS, T, d] along U [K, d]; cloud=True (F [nS, 1, d]) shards the
    directions instead of the time rows.  The device index is a torch tensor of T K nS doubles that lives as long as
    the reference."""

    def __init__(self, kind: str, X=None, F=None, U=None, cloud=False):
        self.kind, self.U, self.cloud = kind, U, cloud
        if U is None:
            self.T, self.nS = X.shape
        else:
            self.nS, self.T, self.d = F.shape
        rank, self.size = _dist.world()
        self.lo, self.hi = _dist.block(len(U) if cloud else self.T, rank, self.size)
        self.eng = get_engine()
        self.on_device = hasattr(self.eng, 'projection_sort_rows_dev')
        self.index = None
        if self.hi == self.lo:
            return
        if U is None:
            rows = X[self.lo:self.hi]
        else:
            F = np.ascontiguousarray(F if cloud else F[:, self.lo:self.hi], dtype=np.float64)
            self.Ul = np.ascontiguousarray(U[self.lo:self.hi] if cloud else U)
        if not self.on_device:
            self.index = np.asarray(self.eng.band_sort_rows(rows) if U is None
                                    else self.eng.projection_sort_rows(F, self.Ul), dtype=np.float64)
            return
        import torch
        self.torch = torch
        if U is None:
            stream, dX = device_rows(self.eng, rows)
            with torch.cuda.stream(stream):
                index = torch.empty((self.hi - self.lo, self.nS), dtype=torch.float64, device=dX.device)
                self.eng.band_sort_rows_dev(dX.data_ptr(), self.hi - self.lo, self.nS, self.nS, index.data_ptr())
        else:
            tb = F.shape[1]
            stream, dF = device_rows(self.eng, F.reshape(self.nS, -1))
            with torch.cuda.stream(stream):
                index = torch.empty((tb, len(self.Ul), self.nS), dtype=torch.float64, device=dF.device)
                self.eng.projection_sort_rows_dev(dF.data_ptr(), self.nS, tb, self.d, self.Ul, index.data_ptr())
        self.index = index  # the raw reference is dropped on return

    def _local(self, Y):
        """This rank's numerators [nY] (Tukey) or outlyingness rows [rows, nY] of the new observations."""
        tukey = self.kind == 'tukey'
        if self.U is None:
            nY = Y.shape[1]
            rows = Y[self.lo:self.hi]
        else:
            nY = Y.shape[0]
            rows = np.ascontiguousarray(Y if self.cloud else Y[:, self.lo:self.hi], dtype=np.float64)
        eng = self.eng
        if not self.on_device:
            if self.U is None:
                out = (eng.band_halfspace_sorted_counts(self.index, rows) if tukey
                       else eng.band_outlyingness_sorted(self.index, rows))
            else:
                out = (eng.projection_tukey_sorted_counts(self.index, rows, self.Ul) if tukey
                       else eng.projection_outlyingness_sorted(self.index, rows, self.Ul))
            return np.asarray(out, dtype=np.int64 if tukey else np.float64)
        torch = self.torch
        tb = self.index.shape[0]
        stream, dY = device_rows(eng, rows if self.U is None else rows.reshape(nY, -1))
        with torch.cuda.stream(stream):
            if tukey:
                out = torch.empty(nY, dtype=torch.int64, device=dY.device)
            else:
                out = torch.empty((tb, nY), dtype=torch.float64, device=dY.device)
            if self.U is None:
                fn = eng.band_halfspace_sorted_counts_dev if tukey else eng.band_outlyingness_sorted_dev
                fn(self.index.data_ptr(), tb, self.nS, dY.data_ptr(), nY, nY, out.data_ptr())
            else:
                fn = eng.projection_tukey_sorted_counts_dev if tukey else eng.projection_outlyingness_sorted_dev
                fn(self.index.data_ptr(), self.nS, tb, dY.data_ptr(), nY, self.d, self.Ul, out.data_ptr())
            return out.cpu().numpy()

    def depths(self, Y: np.ndarray) -> np.ndarray:
        """Depth of every new observation (columns of Y [T, nY] for univariate curves, else Y [nY, T, d]), bit-identical
        to the in-sample depth of the reference with that observation appended."""
        nY = Y.shape[1] if self.U is None else Y.shape[0]
        if nY == 0:
            return np.zeros(0, dtype=np.float64)
        n = self.nS + 1
        empty = self.hi == self.lo
        if self.kind == 'tukey':
            if empty:
                cnt = np.full(nY, n, dtype=np.int64) if self.cloud else np.zeros(nY, dtype=np.int64)
            else:
                cnt = self._local(Y)
            if self.size > 1:
                cnt = _dist.allreduce(cnt, 'min' if self.cloud else 'sum')
            return cnt.astype(np.float64) / (self.T * n)
        if self.cloud:
            o = np.zeros(nY) if empty else self._local(Y)[0]
            if self.size > 1:
                o = _dist.allreduce(o, 'max')
            return 1.0 / (1.0 + o)
        return _depth_from_rows(self.T, nY, lambda lo, hi: self._local(Y))

    def close(self) -> None:
        self.index = None
