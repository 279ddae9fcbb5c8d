"""ctypes binding of libsdepth.so (include/statdepth_b200.h) -- the only way the host reaches the GPU.

There is NO CPU fallback: if the CUDA library is missing or no sm_100 device is visible, every
compute entry point raises :class:`EngineUnavailable`.
"""
import ctypes as C
import os
import threading
import warnings

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STATDEPTH_B200_LIB", os.path.join(_HERE, "libsdepth.so"))  # override: tuning builds

SD_OK = 0
STATUS_NAMES = {1: "SD_ERR_INVALID", 2: "SD_ERR_CUDA", 3: "SD_ERR_NO_DEVICE", 4: "SD_ERR_NONFINITE",
                5: "SD_ERR_OVERFLOW", 6: "SD_ERR_UNSUPPORTED"}
LAYOUT_TN, LAYOUT_NT = 0, 1
BD_AUTO, BD_BITS, BD_GEMM, BD_MATCH = 0, 1, 2, 3
OPT_BD_IMPL, OPT_MBD_FORCE_FALLBACK, OPT_PROFILE, OPT_SIMPLICIAL_IMPL, OPT_ASYNC_DEVICE = 1, 2, 3, 4, 5
SIMPLICIAL_AUTO, SIMPLICIAL_ENUMERATE, SIMPLICIAL_COUNT = 0, 1, 2
PHASES = ("mbd_splitters", "mbd_partition", "mbd_rank", "mbd_generic", "bd_masks", "bd_pairs", "mbd_slab_hist",
          "mbd_slab_rank")


class EngineUnavailable(RuntimeError):
    """The CUDA extension or the GPU is missing; the B200 engine has no CPU path."""


class EngineError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("%s: %s" % (STATUS_NAMES.get(status, status), message))
        self.status = status


class Timings(C.Structure):
    _fields_ = [("h2d_ns", C.c_int64), ("kernel_ns", C.c_int64), ("d2h_ns", C.c_int64),
                ("launches", C.c_int64), ("fallback_rows", C.c_int64), ("bd_impl_used", C.c_int64)]


class DevInfo(C.Structure):
    _fields_ = [("device", C.c_int), ("sm_count", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int),
                ("total_mem", C.c_int64), ("name", C.c_char * 128)]


_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_f64p = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)

# name -> (restype, argtypes); must list every symbol include/statdepth_b200.h declares
SIGNATURES = {
    "sd_abi_version": (C.c_int, []),
    "sd_last_error": (C.c_char_p, []),
    "sd_init": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "sd_destroy": (C.c_int, [C.c_void_p]),
    "sd_device_info": (C.c_int, [C.c_void_p, C.POINTER(DevInfo)]),
    "sd_set_option": (C.c_int, [C.c_void_p, C.c_int, C.c_int64]),
    "sd_get_timings": (C.c_int, [C.c_void_p, C.POINTER(Timings)]),
    "sd_get_phase_ns": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sd_probe_int8_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "sd_stream": (C.c_void_p, [C.c_void_p]),
    "sd_sync": (C.c_int, [C.c_void_p]),
    "sd_mbd_plan": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p]),
    "sd_band_depth_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                    C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "sd_band_depth_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "sd_band_ranks_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                    C.c_void_p]),
    "sd_simplex_depth_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                       C.c_int64, C.c_int, C.c_double, C.c_void_p]),
    "sd_pointcloud_simplicial_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                               C.c_double, C.c_void_p]),
    "sd_pointcloud_l1_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                       C.c_void_p]),
    "sd_pointcloud_oja_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                        C.c_void_p, C.c_int64, C.c_double, C.c_void_p]),
    "sd_pointcloud_blocks_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_void_p, C.c_void_p]),
    "sd_band_depth_oos_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "sd_band_depth_oos_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                            C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "sd_band_sort_rows_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "sd_band_depth_sorted_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                               C.c_int64, C.c_int, C.c_void_p]),
    "sd_pointcloud_simplicial_oos_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                                   C.c_int64, C.c_double, C.c_void_p]),
    "sd_pointcloud_l1_oos_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                           C.c_void_p]),
    "sd_band_rank_sums_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "sd_band_rank_sums_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                            C.c_void_p, C.c_void_p]),
    "sd_band_envelope_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                       C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sd_band_envelope_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                           C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sd_band_extremity_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "sd_extremal_depth_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "sd_pointcloud_halfspace_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                              C.c_void_p]),
    "sd_functional_halfspace_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                              C.c_int64, C.c_void_p]),
    "sd_band_halfspace_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                        C.c_void_p]),
    "sd_band_halfspace_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "sd_projection_tukey_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                          C.c_int64, C.c_void_p]),
    "sd_projection_outlyingness_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                                 C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sd_band_outlyingness_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "sd_projection_tukey_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                              C.c_int64, C.c_void_p]),
    "sd_projection_outlyingness_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int,
                                                     C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sd_band_outlyingness_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                               C.c_void_p, C.c_void_p]),
    "sd_projection_sort_rows_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                                  C.c_int64, C.c_void_p]),
    "sd_projection_tukey_sorted_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                                     C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "sd_projection_outlyingness_sorted_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                                            C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "sd_band_halfspace_sorted_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                                   C.c_int64, C.c_int64, C.c_void_p]),
    "sd_band_outlyingness_sorted_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                                      C.c_int64, C.c_int64, C.c_void_p]),
    "sd_spatial_norms_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p,
                                       C.c_int64, C.c_void_p]),
    "sd_spatial_norms_of_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64,
                                          C.c_int, C.c_void_p]),
    "sd_spatial_norms_of_f64_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64,
                                              C.c_void_p]),
    "sd_band_depth_batched_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                            C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None
_lib_lock = threading.Lock()


def load_library(path: str = None):
    """dlopen libsdepth.so and attach prototypes.  Works without a GPU (symbol check only)."""
    global _lib
    with _lib_lock:
        if _lib is not None and path is None:
            return _lib
        p = path or LIB_PATH
        if not os.path.exists(p):
            raise EngineUnavailable(
                "%s not found: build it with `python -m statdepth_b200.build` (nvcc, sm_100a). "
                "The B200 engine has no CPU fallback." % p)
        lib = C.CDLL(p)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the ABI and this table ever drift apart
            fn.restype = res
            fn.argtypes = args
        if path is None:
            _lib = lib
        return lib


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _dptr(p):
    """A device (or raw host) address as passed to the C ABI: 0 and None are NULL."""
    return C.c_void_p(int(p)) if p else None


def mbd_plan(n: int, ld: int = None) -> dict:
    """Rank pipeline relaxed depth takes for rows of n curves (host arithmetic of the library, no GPU needed)."""
    out = np.zeros(6, dtype=np.int64)
    lib = load_library()
    if lib.sd_mbd_plan(int(n), int(n if ld is None else ld), _ptr(out)) != 0:
        raise ValueError(lib.sd_last_error().decode())
    keys = ("slab", "ctas_per_row", "bins_per_cta", "entries_per_cta", "smem_rank", "smem_hist")
    return dict(zip(keys, (int(v) for v in out)))


class Engine:
    """One context (stream + workspace) on one GPU.  Not thread-safe; use one per thread."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self._ctx = C.c_void_p()
        st = self.lib.sd_init(int(device), C.byref(self._ctx))
        if st != SD_OK:
            msg = self.lib.sd_last_error().decode()
            self._ctx = C.c_void_p()
            if st == 3:
                raise EngineUnavailable("no usable B200: %s (the engine has no CPU fallback)" % msg)
            raise EngineError(st, msg)
        self.device = int(device)

    # -- plumbing ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self.lib.sd_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st):
        if st != SD_OK:
            raise EngineError(st, self.lib.sd_last_error().decode())

    def info(self) -> dict:
        di = DevInfo()
        self._check(self.lib.sd_device_info(self._ctx, C.byref(di)))
        return dict(device=di.device, sm_count=di.sm_count, cc=(di.cc_major, di.cc_minor),
                    total_mem=di.total_mem, name=di.name.decode())

    def timings(self) -> dict:
        t = Timings()
        self._check(self.lib.sd_get_timings(self._ctx, C.byref(t)))
        return dict(h2d_ns=t.h2d_ns, kernel_ns=t.kernel_ns, d2h_ns=t.d2h_ns, launches=t.launches,
                    fallback_rows=t.fallback_rows, bd_impl_used=t.bd_impl_used)

    def phase_ns(self) -> dict:
        """Per-phase device time of the last call (needs set_option(OPT_PROFILE, 1))."""
        out = np.zeros(len(PHASES), dtype=np.int64)
        self._check(self.lib.sd_get_phase_ns(self._ctx, _ptr(out)))
        return {k: int(v) for k, v in zip(PHASES, out) if v}

    def probe_int8_peak(self) -> float:
        """Measured tcgen05 kind::i8 rate of this GPU, int8 ops/s."""
        v = C.c_double()
        self._check(self.lib.sd_probe_int8_peak(self._ctx, C.byref(v)))
        return float(v.value)

    def set_option(self, option: int, value: int):
        self._check(self.lib.sd_set_option(self._ctx, int(option), int(value)))

    def stream(self) -> int:
        return int(self.lib.sd_stream(self._ctx) or 0)

    def sync(self):
        """Wait for the engine's stream; completes a call made under OPT_ASYNC_DEVICE (raises its error)."""
        self._check(self.lib.sd_sync(self._ctx))

    @staticmethod
    def _queries(queries, n):
        if queries is None:
            return None, n
        q = np.ascontiguousarray(queries, dtype=np.int64)
        return q, int(q.size)

    @staticmethod
    def _matrix(X):
        """(X, ld, layout) of a 2-D float64 array [T, n]: a C-order X is SD_LAYOUT_TN with ld = n; an F-order X (what a
        column-built DataFrame gives) is passed as-is, its memory [n, T] row-major: SD_LAYOUT_NT with ld = T."""
        X = np.asarray(X)
        if X.dtype != np.float64:
            X = X.astype(np.float64)
        if X.ndim != 2:
            raise ValueError("expected a 2-D array")
        if X.flags.f_contiguous and not X.flags.c_contiguous:
            return X, X.shape[0], LAYOUT_NT
        X = np.ascontiguousarray(X)
        return X, X.shape[1], LAYOUT_TN

    # -- band depth -------------------------------------------------------------------------------
    def band_depth_counts(self, X, queries=None, j=2, relax=False):
        """Integer numerators for subset size j.  X is [T, n] (rows = time points, columns = curves);
        an F-ordered X (what a column-built DataFrame gives) is passed as-is with SD_LAYOUT_NT."""
        X, ld, layout = self._matrix(X)
        T, n = X.shape
        q, nq = self._queries(queries, n)
        out = np.empty(nq, dtype=np.int64)
        self._check(self.lib.sd_band_depth_f64(self._ctx, _ptr(X), T, n, ld, layout, _ptr(q), nq, int(j),
                                               int(bool(relax)), _ptr(out)))
        return out

    def band_depth_counts_ptr(self, host_ptr, T, n, ld, queries=None, j=2, relax=False, out=None):
        """Same, from a raw host pointer (e.g. pinned memory) in SD_LAYOUT_TN."""
        q, nq = self._queries(queries, n)
        if out is None:
            out = np.empty(nq, dtype=np.int64)
        self._check(self.lib.sd_band_depth_f64(self._ctx, _dptr(host_ptr), int(T), int(n), int(ld), LAYOUT_TN,
                                               _ptr(q), nq, int(j), int(bool(relax)), _ptr(out)))
        return out

    def band_depth_counts_dev(self, dX_ptr, T, n, ld, d_out_ptr, d_query_ptr=None, nq=None, j=2, relax=False):
        """Device-pointer variant: no copies; result stays on the device."""
        nq = int(n if nq is None else nq)
        self._check(self.lib.sd_band_depth_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(n), int(ld),
                                                   _dptr(d_query_ptr), nq, int(j), int(bool(relax)), _dptr(d_out_ptr)))

    def band_ranks(self, X):
        """(below, above) int32 [T, n]: strict ranks of every curve at every time point."""
        X, ld, layout = self._matrix(X)
        T, n = X.shape
        below = np.empty((T, n), dtype=np.int32)
        above = np.empty((T, n), dtype=np.int32)
        self._check(self.lib.sd_band_ranks_f64(self._ctx, _ptr(X), T, n, ld, layout, _ptr(below), _ptr(above)))
        return below, above

    def band_depth_counts_batched(self, X, membership, queries, j=2, relax=False):
        """membership [B, n] (bool/uint8), queries [B, nqb] global curve ids -> counts [B, nqb]."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        T, n = X.shape
        mem = np.ascontiguousarray(membership, dtype=np.uint8)
        qs = np.ascontiguousarray(queries, dtype=np.int64)
        B, nqb = qs.shape
        assert mem.shape == (B, n)
        out = np.empty((B, nqb), dtype=np.int64)
        self._check(self.lib.sd_band_depth_batched_f64(self._ctx, _ptr(X), T, n, n, _ptr(mem), B, _ptr(qs), nqb,
                                                       int(j), int(bool(relax)), _ptr(out)))
        return out

    # -- outlier detection ------------------------------------------------------------------------------
    def band_rank_sums(self, X, want_above=False):
        """(Q, B[, A]) int64 [n]: the relaxed J = 2 numerator and the per-curve sums over time rows of the curves
        strictly below (and above) each curve.  X is [T, n]; an F-ordered X is passed with SD_LAYOUT_NT."""
        X, ld, layout = self._matrix(X)
        T, n = X.shape
        q, b = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64)
        a = np.empty(n, dtype=np.int64) if want_above else None
        self._check(self.lib.sd_band_rank_sums_f64(self._ctx, _ptr(X), T, n, ld, layout, _ptr(q), _ptr(b), _ptr(a)))
        return (q, b, a) if want_above else (q, b)

    def band_rank_sums_dev(self, dX_ptr, T, n, ld, d_q_ptr, d_b_ptr, d_a_ptr=None):
        """Device-pointer variant (SD_LAYOUT_TN): int64 [n] outputs stay on the device."""
        self._check(self.lib.sd_band_rank_sums_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(n), int(ld),
                                                       _dptr(d_q_ptr), _dptr(d_b_ptr), _dptr(d_a_ptr)))

    def band_envelope(self, X, member, factor, want_outside=True):
        """(lo [T], hi [T], outside [n] or None): per-row min / max of the member curves, and per curve the number of
        rows outside the fences lo - factor * (hi - lo), hi + factor * (hi - lo)."""
        X, ld, layout = self._matrix(X)
        T, n = X.shape
        mem = np.ascontiguousarray(member, dtype=np.uint8)
        if mem.shape != (n,):
            raise ValueError("member must have one entry per curve")
        lower, upper = np.empty(T), np.empty(T)
        outside = np.empty(n, dtype=np.int64) if want_outside else None
        self._check(self.lib.sd_band_envelope_f64(self._ctx, _ptr(X), T, n, ld, layout, _ptr(mem), float(factor),
                                                  _ptr(lower), _ptr(upper), _ptr(outside)))
        return lower, upper, outside

    def band_envelope_dev(self, dX_ptr, T, n, ld, d_member_ptr, factor, d_lower_ptr, d_upper_ptr,
                          d_outside_ptr=None):
        """Device-pointer variant (SD_LAYOUT_TN): member uint8 [n], lo / hi float64 [T], outside int64 [n]."""
        self._check(self.lib.sd_band_envelope_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(n), int(ld),
                                                      _dptr(d_member_ptr), float(factor), _dptr(d_lower_ptr),
                                                      _dptr(d_upper_ptr), _dptr(d_outside_ptr)))

    # -- extremal depth ---------------------------------------------------------------------------------
    def band_extremity_dev(self, dX_ptr, T, n, ld, d_m_ptr):
        """Pointwise extremities |b - a| of the rows X [T, n] (SD_LAYOUT_TN): int32 [T, n] on the device."""
        self._check(self.lib.sd_band_extremity_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(n), int(ld),
                                                       _dptr(d_m_ptr)))

    def extremal_depth_dev(self, d_m_ptr, T, n, d_num_ptr):
        """Extremal-depth numerators int64 [n] from the full extremity matrix int32 [T, n], on the device."""
        self._check(self.lib.sd_extremal_depth_dev(self._ctx, _dptr(d_m_ptr), int(T), int(n), _dptr(d_num_ptr)))

    # -- halfspace (Tukey) depth -----------------------------------------------------------------------
    def halfspace_counts(self, P, queries=None):
        """Numerators h in [1, n] of the points of the cloud P [n, d], d = 1 or 2: the fewest points, p itself
        included, in a closed half-plane (half-line) whose boundary passes through p.  HD = h / n."""
        P = np.ascontiguousarray(P, dtype=np.float64)
        n, d = P.shape
        q, nq = self._queries(queries, n)
        out = np.empty(nq, dtype=np.int64)
        self._check(self.lib.sd_pointcloud_halfspace_f64(self._ctx, _ptr(P), n, d, _ptr(q), nq, _ptr(out)))
        return out

    def functional_halfspace_counts(self, F, queries=None):
        """sum over t of the numerator of curve c at time t among the N values F[:, t] (F [N, T, 2]), per query."""
        F = np.ascontiguousarray(F, dtype=np.float64)
        N, T, d = F.shape
        q, nq = self._queries(queries, N)
        out = np.empty(nq, dtype=np.int64)
        self._check(self.lib.sd_functional_halfspace_f64(self._ctx, _ptr(F), N, T, d, _ptr(q), nq, _ptr(out)))
        return out

    def band_halfspace_counts(self, X):
        """int64 [n]: sum over the time rows of X [T, n] of n - max(b_t, a_t), b_t / a_t the other curves strictly
        below / above.  An F-ordered X is passed with SD_LAYOUT_NT."""
        X, ld, layout = self._matrix(X)
        T, n = X.shape
        out = np.empty(n, dtype=np.int64)
        self._check(self.lib.sd_band_halfspace_f64(self._ctx, _ptr(X), T, n, ld, layout, _ptr(out)))
        return out

    def band_halfspace_counts_dev(self, dX_ptr, T, n, ld, d_out_ptr):
        """Device-pointer variant (SD_LAYOUT_TN): int64 [n] stays on the device."""
        self._check(self.lib.sd_band_halfspace_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(n), int(ld),
                                                       _dptr(d_out_ptr)))

    # -- random projection depths --------------------------------------------------------------------------
    @staticmethod
    def _curves_and_directions(F, U):
        F = np.ascontiguousarray(F, dtype=np.float64)
        U = np.ascontiguousarray(U, dtype=np.float64)
        if F.ndim != 3 or U.ndim != 2 or U.shape[1] != F.shape[2]:
            raise ValueError("expected curves F [N, T, d] and directions U [K, d]")
        return F, U

    def projection_tukey_counts(self, F, U):
        """Random Tukey numerators int64 [N] of the curves F [N, T, d] (a cloud is T = 1) along the directions
        U [K, d]: sum over t of min over k of N - max(b, a), b / a the other projections strictly below / above."""
        F, U = self._curves_and_directions(F, U)
        N, T, d = F.shape
        out = np.empty(N, dtype=np.int64)
        self._check(self.lib.sd_projection_tukey_f64(self._ctx, _ptr(F), N, T, d, _ptr(U), U.shape[0], _ptr(out)))
        return out

    def projection_outlyingness(self, F, U, want_medmad=False):
        """O [T, N]: per time point the max over the directions U [K, d] of |u.x - med| / MAD of the curves
        F [N, T, d]; with want_medmad also med and MAD [T, K] of every projected row."""
        F, U = self._curves_and_directions(F, U)
        N, T, d = F.shape
        K = U.shape[0]
        o = np.empty((T, N))
        med, mad = (np.empty((T, K)), np.empty((T, K))) if want_medmad else (None, None)
        self._check(self.lib.sd_projection_outlyingness_f64(self._ctx, _ptr(F), N, T, d, _ptr(U), K, _ptr(o),
                                                            _ptr(med), _ptr(mad)))
        return (o, med, mad) if want_medmad else o

    def band_outlyingness(self, X, want_medmad=False):
        """O [T, n] = |x - med_t| / MAD_t of the univariate curves X [T, n] (and med, MAD [T]).  An F-ordered X is
        passed with SD_LAYOUT_NT."""
        X, ld, layout = self._matrix(X)
        T, n = X.shape
        o = np.empty((T, n))
        med, mad = (np.empty(T), np.empty(T)) if want_medmad else (None, None)
        self._check(self.lib.sd_band_outlyingness_f64(self._ctx, _ptr(X), T, n, ld, layout, _ptr(o), _ptr(med),
                                                      _ptr(mad)))
        return (o, med, mad) if want_medmad else o

    def projection_tukey_counts_dev(self, dF_ptr, N, T, d, U, d_out_ptr):
        """Device-pointer variant (F and the int64 [N] output on the device; U is host memory)."""
        U = np.ascontiguousarray(U, dtype=np.float64)
        self._check(self.lib.sd_projection_tukey_f64_dev(self._ctx, _dptr(dF_ptr), int(N), int(T), int(d), _ptr(U),
                                                         U.shape[0], _dptr(d_out_ptr)))

    def projection_outlyingness_dev(self, dF_ptr, N, T, d, U, d_o_ptr, d_med_ptr=None, d_mad_ptr=None):
        """Device-pointer variant (F, O [T, N] and med / MAD [T, K] on the device; U is host memory)."""
        U = np.ascontiguousarray(U, dtype=np.float64)
        self._check(self.lib.sd_projection_outlyingness_f64_dev(self._ctx, _dptr(dF_ptr), int(N), int(T), int(d),
                                                                _ptr(U), U.shape[0], _dptr(d_o_ptr), _dptr(d_med_ptr),
                                                                _dptr(d_mad_ptr)))

    def band_outlyingness_dev(self, dX_ptr, T, n, ld, d_o_ptr, d_med_ptr=None, d_mad_ptr=None):
        """Device-pointer variant (SD_LAYOUT_TN): O [T, n] and med / MAD [T] stay on the device."""
        self._check(self.lib.sd_band_outlyingness_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(n), int(ld),
                                                          _dptr(d_o_ptr), _dptr(d_med_ptr), _dptr(d_mad_ptr)))

    # -- out-of-sample depth ----------------------------------------------------------------------------
    @staticmethod
    def _rows(A):
        """float64 [rows, cols] with unit column stride (a column slice of a C-order matrix stays a view) and its
        leading dimension in elements."""
        A = np.asarray(A, dtype=np.float64)
        if A.ndim != 2:
            raise ValueError("expected a 2-D array")
        if A.shape[1] > 0 and not (A.strides[1] == 8 and A.strides[0] % 8 == 0 and A.strides[0] >= 8 * A.shape[1]):
            A = np.ascontiguousarray(A)
        return A, (A.strides[0] // 8 if A.shape[0] > 1 else max(A.shape[1], 1))

    def band_depth_oos_counts(self, S, Y, j=2, relax=False):
        """Numerators of the new curves Y [T, nY] against the sample S [T, nS] (each new curve alone appended)."""
        S, ldS = self._rows(S)
        Y, ldY = self._rows(Y)
        T, nS = S.shape
        if Y.shape[0] != T:
            raise ValueError("S and Y must have the same number of rows (time points)")
        nY = Y.shape[1]
        out = np.empty(nY, dtype=np.int64)
        if nY == 0:
            return out
        self._check(self.lib.sd_band_depth_oos_f64(self._ctx, _ptr(S), T, nS, ldS, _ptr(Y), nY, ldY, int(j),
                                                   int(bool(relax)), _ptr(out)))
        return out

    def band_depth_oos_counts_dev(self, dS_ptr, T, nS, ldS, dY_ptr, nY, ldY, d_out_ptr, j=2, relax=False):
        """Device-pointer variant: no host copies; int64 counts [nY] stay on the device."""
        self._check(self.lib.sd_band_depth_oos_f64_dev(self._ctx, _dptr(dS_ptr), int(T), int(nS), int(ldS),
                                                       _dptr(dY_ptr), int(nY), int(ldY), int(j), int(bool(relax)),
                                                       _dptr(d_out_ptr)))

    def band_sort_rows_dev(self, dX_ptr, T, nS, ld, d_sorted_ptr):
        """The index of a fitted reference: float64 [T, nS] rows of X (SD_LAYOUT_TN) sorted ascending, on the device."""
        self._check(self.lib.sd_band_sort_rows_f64_dev(self._ctx, _dptr(dX_ptr), int(T), int(nS), int(ld),
                                                       _dptr(d_sorted_ptr)))

    def band_depth_sorted_counts_dev(self, d_sorted_ptr, T, nS, dY_ptr, nY, ldY, J, d_out_ptr):
        """Relaxed numerators of the new curves Y [T, nY] against sorted rows: int64 [(J - 1), nY] on the device,
        row j - 2 equal to band_depth_oos_counts_dev(relax=True) for j."""
        self._check(self.lib.sd_band_depth_sorted_f64_dev(self._ctx, _dptr(d_sorted_ptr), int(T), int(nS),
                                                          _dptr(dY_ptr), int(nY), int(ldY), int(J), _dptr(d_out_ptr)))

    # -- fitted references for random projection depths ----------------------------------------------------------
    def projection_sort_rows_dev(self, dF_ptr, nS, T, d, U, d_sorted_ptr):
        """The index of a projected reference: float64 [T, K, nS], the projections of the curves F [nS, T, d] (on the
        device) along U [K, d] (host memory) sorted ascending per (t, k), on the device."""
        U = np.ascontiguousarray(U, dtype=np.float64)
        self._check(self.lib.sd_projection_sort_rows_f64_dev(self._ctx, _dptr(dF_ptr), int(nS), int(T), int(d), _ptr(U),
                                                             U.shape[0], _dptr(d_sorted_ptr)))

    def projection_tukey_sorted_counts_dev(self, d_sorted_ptr, nS, T, dF_ptr, nY, d, U, d_out_ptr):
        """Random Tukey numerators int64 [nY] of the new curves F [nY, T, d] against a projected index, each equal to
        projection_tukey_counts of the reference with that curve appended (its entry nS)."""
        U = np.ascontiguousarray(U, dtype=np.float64)
        self._check(self.lib.sd_projection_tukey_sorted_f64_dev(self._ctx, _dptr(d_sorted_ptr), int(nS), int(T),
                                                                _dptr(dF_ptr), int(nY), int(d), _ptr(U), U.shape[0],
                                                                _dptr(d_out_ptr)))

    def projection_outlyingness_sorted_dev(self, d_sorted_ptr, nS, T, dF_ptr, nY, d, U, d_o_ptr):
        """O [T, nY] of the new curves F [nY, T, d] against a projected index, each column equal to
        projection_outlyingness of the reference with that curve appended (its column nS)."""
        U = np.ascontiguousarray(U, dtype=np.float64)
        self._check(self.lib.sd_projection_outlyingness_sorted_f64_dev(self._ctx, _dptr(d_sorted_ptr), int(nS),
                                                                       int(T), _dptr(dF_ptr), int(nY), int(d),
                                                                       _ptr(U), U.shape[0], _dptr(d_o_ptr)))

    def band_halfspace_sorted_counts_dev(self, d_sorted_ptr, T, nS, dY_ptr, nY, ldY, d_out_ptr):
        """Integrated halfspace numerators int64 [nY] of the univariate new curves Y [T, nY] against sorted rows
        (band_sort_rows_dev), each equal to band_halfspace_counts of [S | g] (its entry nS)."""
        self._check(self.lib.sd_band_halfspace_sorted_f64_dev(self._ctx, _dptr(d_sorted_ptr), int(T), int(nS),
                                                              _dptr(dY_ptr), int(nY), int(ldY), _dptr(d_out_ptr)))

    def band_outlyingness_sorted_dev(self, d_sorted_ptr, T, nS, dY_ptr, nY, ldY, d_o_ptr):
        """O [T, nY] of the univariate new curves Y [T, nY] against sorted rows, each column equal to
        band_outlyingness of [S | g] (its column nS)."""
        self._check(self.lib.sd_band_outlyingness_sorted_f64_dev(self._ctx, _dptr(d_sorted_ptr), int(T), int(nS),
                                                                 _dptr(dY_ptr), int(nY), int(ldY), _dptr(d_o_ptr)))

    # -- functional spatial depth ----------------------------------------------------------------------
    @staticmethod
    def _curves(A):
        """(A, layout) of curves as the rows of a 2-D float64 array [n, F]: a C-order A is SD_LAYOUT_NT; an F-order A
        (the transpose of a univariate DataFrame's C-order values [T, n]) is passed as-is with SD_LAYOUT_TN."""
        A = np.asarray(A)
        if A.dtype != np.float64:
            A = A.astype(np.float64)
        if A.ndim != 2:
            raise ValueError("expected curves as a 2-D array [n, F]")
        if A.flags.f_contiguous and not A.flags.c_contiguous:
            return A, LAYOUT_TN
        return np.ascontiguousarray(A), LAYOUT_NT

    def spatial_norms(self, X, queries=None):
        """r [nq] = || sum_j u(x_j - x_q) || of the curves X [n, F] (rows; u(0) = 0) for the queries (all when None);
        spatial depth is 1 - r / n."""
        X, layout = self._curves(X)
        n, F = X.shape
        q, nq = self._queries(queries, n)
        out = np.empty(nq, dtype=np.float64)
        self._check(self.lib.sd_spatial_norms_f64(self._ctx, _ptr(X), n, F, layout, _ptr(q), nq, _ptr(out)))
        return out

    def spatial_norms_of(self, S, Y):
        """r [nY] of the new curves Y [nY, F] against the sample S [nS, F] (rows); the depth is 1 - r / (nS + 1)."""
        S, ls = self._curves(S)
        Y = np.asarray(Y, dtype=np.float64)
        Y = np.asfortranarray(Y) if ls == LAYOUT_TN else np.ascontiguousarray(Y)  # in S's layout
        if Y.ndim != 2 or S.shape[1] != Y.shape[1]:
            raise ValueError("S and Y must have the same number of values per curve")
        out = np.empty(Y.shape[0], dtype=np.float64)
        if Y.shape[0] == 0:
            return out
        self._check(self.lib.sd_spatial_norms_of_f64(self._ctx, _ptr(S), S.shape[0], _ptr(Y), Y.shape[0], S.shape[1],
                                                     ls, _ptr(out)))
        return out

    def spatial_norms_of_dev(self, dS_ptr, nS, dY_ptr, nY, F, d_r_ptr):
        """Device-pointer variant (curves as rows: S [nS, F], Y [nY, F]); r [nY] stays on the device."""
        self._check(self.lib.sd_spatial_norms_of_f64_dev(self._ctx, _dptr(dS_ptr), int(nS), _dptr(dY_ptr), int(nY),
                                                         int(F), _dptr(d_r_ptr)))

    def simplicial_oos_counts(self, S, Y, tol=1e-7):
        S = np.ascontiguousarray(S, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        nS, d = S.shape
        out = np.empty(Y.shape[0], dtype=np.int64)
        if Y.shape[0] == 0:
            return out
        self._check(self.lib.sd_pointcloud_simplicial_oos_f64(self._ctx, _ptr(S), nS, d, _ptr(Y), Y.shape[0],
                                                              float(tol), _ptr(out)))
        return out

    def l1_oos_depth(self, S, Y):
        S = np.ascontiguousarray(S, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        nS, d = S.shape
        out = np.empty(Y.shape[0], dtype=np.float64)
        if Y.shape[0] == 0:
            return out
        self._check(self.lib.sd_pointcloud_l1_oos_f64(self._ctx, _ptr(S), nS, d, _ptr(Y), Y.shape[0], _ptr(out)))
        return out

    # -- multivariate / point clouds -----------------------------------------------------------------
    def simplex_depth_counts(self, F, queries=None, relax=False, tol=1e-7):
        F = np.ascontiguousarray(F, dtype=np.float64)
        N, T, d = F.shape
        q, nq = self._queries(queries, N)
        out = np.empty(nq, dtype=np.int64)
        self._check(self.lib.sd_simplex_depth_f64(self._ctx, _ptr(F), N, T, d, _ptr(q), nq, int(bool(relax)),
                                                  float(tol), _ptr(out)))
        return out

    def simplicial_counts(self, P, queries=None, tol=1e-7):
        P = np.ascontiguousarray(P, dtype=np.float64)
        n, d = P.shape
        q, nq = self._queries(queries, n)
        out = np.empty(nq, dtype=np.int64)
        self._check(self.lib.sd_pointcloud_simplicial_f64(self._ctx, _ptr(P), n, d, _ptr(q), nq, float(tol),
                                                          _ptr(out)))
        return out

    def l1_depth(self, P, queries=None):
        P = np.ascontiguousarray(P, dtype=np.float64)
        n, d = P.shape
        q, nq = self._queries(queries, n)
        out = np.empty(nq, dtype=np.float64)
        self._check(self.lib.sd_pointcloud_l1_f64(self._ctx, _ptr(P), n, d, _ptr(q), nq, _ptr(out)))
        return out

    def oja(self, P, hull_volume, queries=None, pool=None):
        P = np.ascontiguousarray(P, dtype=np.float64)
        n, d = P.shape
        q, nq = self._queries(queries, n)
        pl = None if pool is None else np.ascontiguousarray(pool, dtype=np.int64)
        npool = n if pl is None else int(pl.size)
        out = np.empty(nq, dtype=np.float64)
        self._check(self.lib.sd_pointcloud_oja_f64(self._ctx, _ptr(P), n, d, _ptr(q), nq, _ptr(pl), npool,
                                                   float(hull_volume), _ptr(out)))
        return out


    BLOCK_KINDS = {"simplex": 0, "l1": 1, "oja": 2}

    def cloud_blocks(self, P, members, offsets, query_pos, kind, tol=1e-7, hull_volumes=None):
        """One single-query depth per block of member points (K-sampled point-cloud depth), one launch for all.
        members: concatenated point ids; offsets [B+1]; query_pos [B] position of the query inside its block.
        Returns float64 [B]: simplicial COUNT (exact), L1 depth, or Oja sum / hull_volumes[b]."""
        P = np.ascontiguousarray(P, dtype=np.float64)
        n, d = P.shape
        mem = np.ascontiguousarray(members, dtype=np.int64)
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        qp = np.ascontiguousarray(query_pos, dtype=np.int64)
        B = int(qp.size)
        hv = None if hull_volumes is None else np.ascontiguousarray(hull_volumes, dtype=np.float64)
        out = np.empty(B, dtype=np.float64)
        self._check(self.lib.sd_pointcloud_blocks_f64(self._ctx, _ptr(P), n, d, _ptr(mem), _ptr(off), _ptr(qp), B,
                                                      int(self.BLOCK_KINDS[kind]), float(tol), _ptr(hv), _ptr(out)))
        return out


def device_rows(eng, X):
    """(stream, dX): the rows X [T, n] as a C-order float64 tensor on eng's device, uploaded on eng's stream (so the
    upload, later outputs and the engine's kernels are ordered on it).  A DataFrame's values are usually curve-major
    (F order): that memory is uploaded as it is and transposed on the device, as sd_band_depth_f64 does with
    SD_LAYOUT_NT (a host transpose of 819 MB takes over a second)."""
    import torch
    device = torch.device("cuda", eng.device)
    stream = torch.cuda.ExternalStream(eng.stream(), device=device)
    curve_major = X.strides[0] == X.itemsize and X.strides[1] != X.itemsize
    host = np.ascontiguousarray(X.T if curve_major else X, dtype=np.float64)
    with warnings.catch_warnings():
        warnings.filterwarnings("ignore", message="The given NumPy array is not writable")  # only read here
        with torch.cuda.stream(stream):
            d = torch.from_numpy(host).to(device)
            return stream, (d.t().contiguous() if curve_major else d)


_engines = {}


def get_engine(device: int = None) -> Engine:
    """Process-wide engine for `device` (default: $LOCAL_RANK or $STATDEPTH_DEVICE or 0)."""
    if device is None:
        device = int(os.environ.get("STATDEPTH_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        if "STATDEPTH_DEVICE" not in os.environ:
            # LOCAL_RANK is out of range when CUDA_VISIBLE_DEVICES is narrowed to one device per rank
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis is not None and device >= len([v for v in vis.split(",") if v.strip()]):
                device = 0
    eng = _engines.get(device)
    if eng is None:
        eng = Engine(device)
        _engines[device] = eng
    return eng
