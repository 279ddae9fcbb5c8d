"""Fitted reference driver: a reference sample indexed once on the device (csrc/reference.cu, DESIGN.md K9).

Relaxed out-of-sample band depth needs, per new curve and time row, only the number of sample values strictly below
and strictly above the new value.  Both come from binary searches in the sorted row, so the sample's rows are sorted
once on the device and kept there (the index); every later call uploads only the new curves.  The counts are the
integers sd_band_depth_oos_f64 returns and the floats are formed by _functional._relaxed_depths_of, so the depths are
bit-identical to FunctionalDepthOf(relax=True).

On one GPU the index lives in a torch tensor on the engine's device.  An engine without the `_dev` entry points (the
CPU test double) keeps a host index from its `band_sort_rows` and answers `band_depth_sorted_counts`.  Under
`enable_distributed()` every rank indexes its block of time rows; each call scores the same rows of the new curves and
all-reduces the counts, so construction and every call are collectives.
"""
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import device_rows, get_engine
from ._functional import _relaxed_depths_of, _values
from ._helper import _handle_depth_errors

__all__ = ['_checked_reference', '_query_values', '_SortedReference']


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
