"""GPU: parity of the CUDA path (through the C ABI) with the CPU oracle and the reference's golden vectors.

Bar (north star): integer counts, ranks and depth orderings bit-exact; float64 depths within 1e-12
relative.  All inputs are seeded; sizes are chosen so the oracle finishes in seconds; BASELINE's full
sizes are covered by size-independent properties (additivity over time rows, the closed-form
checksum of tie-free ranks, depth bounds) plus an oracle comparison on a row slice.
"""
from math import comb

import numpy as np
import pandas as pd
import pytest

from api_cases import check_case

pytestmark = pytest.mark.gpu

RTOL = 1e-12  # float64 proportions / L1 / Oja (north star); counts are compared with ==


def walks(seed, T, n):
    return np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)


# ------------------------------------------------------------------------------------------------
# modified band depth (relax=True)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,n,seed", [(100, 200, 0), (5, 6, 1), (3, 2, 2), (1, 1, 3), (64, 513, 4), (17, 1000, 5),
                                      (256, 4096, 6), (33, 12345, 7)])
def test_mbd_counts_bit_exact(engine, oracle, T, n, seed):
    X = walks(seed, T, n)
    for j in (2, 3):
        got = engine.band_depth_counts(X, None, j, True)
        assert (got == oracle.mbd_counts_all(X, j=j)).all()
    assert engine.timings()["fallback_rows"] == 0  # well-spread data never needs the generic path


@pytest.mark.parametrize("maker", ["round", "few", "constant", "half_constant", "outliers", "sorted", "negzero",
                                   "far_reference"])
def test_mbd_ties_and_skew(engine, oracle, maker):
    rng = np.random.default_rng(11)
    T, n = 24, 6000
    X = rng.standard_normal((T, n)).cumsum(0)
    if maker == "round":
        X = np.round(X)
    elif maker == "few":
        X = rng.integers(0, 3, size=(T, n)).astype(np.float64)
    elif maker == "constant":
        X = np.full((T, n), 2.5)
    elif maker == "half_constant":
        X[:, : n // 2] = 1.0
    elif maker == "outliers":
        X[:, :5] = 1e300
        X[:, 5:9] = -1e300
    elif maker == "sorted":
        X = np.sort(X, axis=1)
    elif maker == "negzero":
        X = np.where(rng.random((T, n)) < 0.5, 0.0, -0.0)
    elif maker == "far_reference":  # outliers where the offsets' reference is taken from (first / middle / last)
        X[:, 0] = 1e13
        X[::2, n - 1] = -1e13
        X += 1e7
    got = engine.band_depth_counts(X, None, 2, True)
    assert (got == oracle.mbd_counts_all(X)).all()


def test_mbd_generic_path_forced(engine, oracle):
    """SD_OPT_MBD_FORCE_FALLBACK: the one-CTA-per-row bitonic path alone must give the same counts."""
    from statdepth_b200 import _engine as E
    X = walks(21, 19, 5000)
    X[:, 100:200] = np.round(X[:, 100:200])
    try:
        engine.set_option(E.OPT_MBD_FORCE_FALLBACK, 1)
        for j in (2, 3):
            assert (engine.band_depth_counts(X, None, j, True) == oracle.mbd_counts_all(X, j=j)).all()
        assert engine.timings()["fallback_rows"] == 19
        Xs = walks(22, 7, 300)
        assert (engine.band_depth_counts(Xs, None, 2, True) == oracle.mbd_counts_all(Xs)).all()
    finally:
        engine.set_option(E.OPT_MBD_FORCE_FALLBACK, 0)


def test_ranks_bit_exact(engine, oracle):
    X = walks(31, 9, 3000)
    X[:, :50] = np.round(X[:, :50])
    below, above = engine.band_ranks(X)
    _, rb, ra = oracle.mbd_counts_all(X, want_ranks=True)
    assert (below == rb).all() and (above == ra).all()


def test_layouts_queries_and_ld(engine, oracle):
    X = walks(41, 40, 700)
    ref = oracle.mbd_counts_all(X)
    q = np.array([5, 699, 0, 5, 333])
    assert (engine.band_depth_counts(X, q, 2, True) == ref[q]).all()
    Xf = np.asfortranarray(X)  # what a column-built DataFrame hands over: SD_LAYOUT_NT + device transpose
    assert (engine.band_depth_counts(Xf, None, 2, True) == ref).all()
    sref = oracle.bd_counts(X, q)
    assert (engine.band_depth_counts(Xf, q, 2, False) == sref).all()
    wide = np.zeros((40, 900))
    wide[:, :700] = X
    out = engine.band_depth_counts_ptr(wide.ctypes.data, 40, 700, 900, None, 2, True)
    assert (out == ref).all()


def test_pipelined_host_path(engine, oracle):
    """Inputs >= 64 MB take the row-block pipeline (H2D of block k+1 overlaps ranking of block k); also
    with a padded leading dimension and with J = 3."""
    T, n, ld = 70, 150_000, 150_016
    wide = np.zeros((T, ld))
    wide[:, :n] = walks(43, T, n)
    X = np.ascontiguousarray(wide[:, :n])
    exp = oracle.mbd_counts_all(X)
    assert (engine.band_depth_counts(X, None, 2, True) == exp).all()
    assert engine.timings()["launches"] > 12  # several row blocks
    q = np.array([149_999, 3, 77_777])
    out = engine.band_depth_counts_ptr(wide.ctypes.data, T, n, ld, q, 2, True)
    assert (out == exp[q]).all()
    assert (engine.band_depth_counts(X, q, 3, True) == oracle.mbd_counts_all(X, j=3)[q]).all()


def test_nonfinite_is_rejected(engine):
    from statdepth_b200 import EngineError
    X = walks(51, 8, 1200)
    X[3, 77] = np.nan
    for relax in (True, False):
        with pytest.raises(EngineError, match="NONFINITE"):
            engine.band_depth_counts(X, None, 2, relax)
    X[3, 77] = np.inf
    with pytest.raises(EngineError, match="NONFINITE"):
        engine.band_depth_counts(X, None, 2, True)


def test_mbd_full_size_properties(engine, oracle):
    """BASELINE config 2 (100k curves x 1024 points): additivity over row blocks, the tie-free checksum
    sum_c count_c = T * (n*C(n-1,2) - 2*C(n,3)), depth <= (n-2)/n, and the oracle on a 48-row slice."""
    T, n = 1024, 100_000
    X = walks(1, T, n)
    full = engine.band_depth_counts(X, None, 2, True)
    assert engine.timings()["fallback_rows"] == 0
    assert int(full.sum()) == T * (n * comb(n - 1, 2) - 2 * comb(n, 3))
    a = engine.band_depth_counts(X[:500], None, 2, True)
    b = engine.band_depth_counts(X[500:], None, 2, True)
    assert (a + b == full).all()
    sl = engine.band_depth_counts(X[500:548], None, 2, True)
    assert (sl == oracle.mbd_counts_all(X[500:548])).all()
    depth = full / T / comb(n, 2)
    assert depth.max() <= (n - 2) / n and depth.min() > 0
    # tie stress at full width: integers -> value classes of thousands of curves overflow their parts; they are
    # recognised as single-value classes (no sorting); only rows where an overflowing part mixes several
    # values still take the generic path
    Xr = np.round(X[:16])
    assert (engine.band_depth_counts(Xr, None, 2, True) == oracle.mbd_counts_all(Xr)).all()
    assert engine.timings()["fallback_rows"] < 16
    Xc = np.round(X[:8] / 50.0)  # a handful of classes, each far above the part capacity
    assert (engine.band_depth_counts(Xc, None, 2, True) == oracle.mbd_counts_all(Xc)).all()
    # an adversarial row: 3000 DISTINCT values squeezed between two sample quantiles cannot be a single class
    Xa = X[:4].copy()
    Xa[:, :3000] = Xa[:, [3000]] + np.arange(3000) * 1e-13
    assert (engine.band_depth_counts(Xa, None, 2, True) == oracle.mbd_counts_all(Xa)).all()


def _slab_rows(rng, kind, T, n):
    if kind == "normal":
        return rng.standard_normal((T, n))
    if kind == "walk":
        return rng.standard_normal((T, n)).cumsum(0)
    if kind == "expo":
        return rng.standard_exponential((T, n))
    if kind == "t3":
        return rng.standard_t(3, (T, n))
    if kind == "round4":     # moderately tied: the table kernel's sample sees the ties and the part pipeline takes over
        return np.round(rng.standard_normal((T, n)), 4)
    if kind == "sparse_ties":  # ties too rare for the sample: the slab path ranks them on the exact values
        X = rng.standard_normal((T, n))
        X[:, 1::97] = X[:, 0:-1:97][:, : X[:, 1::97].shape[1]]
        return X
    if kind == "shifted":    # spread far below the magnitude
        return 1e6 + 1e-3 * rng.standard_normal((T, n))
    if kind == "outliers":   # a few huge values: they clamp into the end buckets and are ranked exactly
        X = rng.standard_normal((T, n))
        X[:, ::997] *= 1e9
        return X
    if kind == "tail_all":   # heavy tails: every row fails the hist kernel's validation -> masked part pipeline
        return rng.standard_cauchy((T, n))
    if kind == "tail_many":  # 10 of 40 rows unfit: the slab path ranks 30 rows, the part pipeline the other 10
        X = rng.standard_normal((T, n))
        X[5:15] = rng.standard_cauchy((10, n))
        return X
    if kind == "tail_few":   # 2 of 40 rows unfit: generic path for those
        X = rng.standard_normal((T, n))
        X[7] = rng.standard_cauchy(n)
        X[30] = rng.standard_cauchy(n)
        return X
    if kind == "mixed":      # a constant row and a rounded row among continuous ones
        X = rng.standard_normal((T, n))
        X[1] = np.round(X[1] * 10)
        X[2] = 7.0
        return X
    raise ValueError(kind)


@pytest.mark.parametrize("kind,n", [("normal", 16384), ("walk", 20000), ("expo", 50000), ("t3", 100000),
                                    ("normal", 131072), ("round4", 100000), ("sparse_ties", 65536),
                                    ("shifted", 40000), ("outliers", 100000), ("tail_all", 20000),
                                    ("tail_many", 100000), ("tail_few", 20000), ("mixed", 30000), ("walk", 16386)])
def test_mbd_slab_path(engine, oracle, monkeypatch, kind, n):
    """Rows of 16384 .. 131072 curves take the slab path (csrc/mbd_slab.cuh): counts (j = 2, 3) and ranks equal the
    oracle's AND the part pipeline's (SD_MBD_PATH=parts) on fit rows, unfit rows and mixtures of both."""
    rng = np.random.default_rng(4000 + n + len(kind))
    T = 40 if kind.startswith("tail_") or kind == "mixed" else 5
    X = _slab_rows(rng, kind, T, n)
    want2, wb, wa = oracle.mbd_counts_all(X, j=2, want_ranks=True)
    want3 = oracle.mbd_counts_all(X, j=3)
    for path in ("slab", "parts"):
        if path == "parts":
            monkeypatch.setenv("SD_MBD_PATH", "parts")
        else:
            monkeypatch.delenv("SD_MBD_PATH", raising=False)
        assert (engine.band_depth_counts(X, None, 2, True) == want2).all(), path
        assert (engine.band_depth_counts(X, None, 3, True) == want3).all(), path
        below, above = engine.band_ranks(X)
        assert (below == wb).all() and (above == wa).all(), path
    q = rng.choice(n, size=7, replace=False)
    monkeypatch.delenv("SD_MBD_PATH", raising=False)
    assert (engine.band_depth_counts(X, q, 2, True) == want2[q]).all()


def test_mbd_slab_path_is_taken(engine, monkeypatch):
    """Launch counts tell the paths apart: table + hist + rank + finish on fit data (no generic launch)."""
    monkeypatch.delenv("SD_MBD_PATH", raising=False)
    X = walks(5, 8, 50_000)
    engine.band_depth_counts(X, None, 2, True)
    tm = engine.timings()
    assert tm["launches"] <= 5 and tm["fallback_rows"] == 0
    monkeypatch.setenv("SD_MBD_PATH", "parts")
    engine.band_depth_counts(X, None, 2, True)
    assert engine.timings()["launches"] >= 7


def _random_matrix(rng, T, n):
    """Random shapes of trouble: continuous, rounded, few classes, constant rows, point masses, tiny spreads."""
    kind = rng.integers(0, 7)
    X = rng.standard_normal((T, n)).cumsum(0)
    if kind == 1:
        X = np.round(X * rng.choice([0.2, 1.0, 5.0]))
    elif kind == 2:
        X = rng.integers(0, int(rng.integers(1, 6)), size=(T, n)).astype(np.float64)
    elif kind == 3:
        X[rng.integers(0, T)] = 7.0
    elif kind == 4:  # zero-inflated
        X[rng.random((T, n)) < rng.choice([0.1, 0.5, 0.9])] = 0.0
    elif kind == 5:  # spreads far below the magnitude: float offsets collapse, exact compares must decide
        X = 1e6 + X * 1e-9
    elif kind == 6:  # a few huge outliers stretch the first / last part
        X[:, rng.integers(0, n, size=3)] *= 1e200
    return X


@pytest.mark.parametrize("seed", range(24))
def test_mbd_randomized_differential(engine, oracle, seed):
    """Seeded random shapes, tie structures and query subsets: counts (j = 2, 3) and ranks equal the oracle's."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.choice([3, 17, 200, 1024, 1025, 1500, 4000, 9000, 20_000]))
    T = int(rng.integers(1, 12))
    X = _random_matrix(rng, T, n)
    want2, wb, wa = oracle.mbd_counts_all(X, j=2, want_ranks=True)
    assert (engine.band_depth_counts(X, None, 2, True) == want2).all()
    assert (engine.band_depth_counts(X, None, 3, True) == oracle.mbd_counts_all(X, j=3)).all()
    below, above = engine.band_ranks(X)
    assert (below == wb).all() and (above == wa).all()
    q = rng.choice(n, size=min(n, 5), replace=False)
    assert (engine.band_depth_counts(X, q, 2, True) == want2[q]).all()
    assert (engine.band_depth_counts(np.asfortranarray(X), q, 2, True) == want2[q]).all()


@pytest.mark.parametrize("seed", range(12))
def test_bd_randomized_differential(engine, oracle, seed):
    """Strict band depth: every implementation against the oracle on random shapes with and without ties."""
    from statdepth_b200._engine import BD_AUTO, BD_BITS, BD_GEMM, BD_MATCH, OPT_BD_IMPL
    rng = np.random.default_rng(2000 + seed)
    n = int(rng.choice([3, 9, 64, 130, 300, 700]))
    T = int(rng.choice([1, 5, 31, 32, 33, 100]))
    X = _random_matrix(rng, T, n)
    want = oracle.bd_counts(X)
    try:
        for impl in (BD_AUTO, BD_BITS, BD_GEMM, BD_MATCH):
            engine.set_option(OPT_BD_IMPL, impl)
            assert (engine.band_depth_counts(X, None, 2, False) == want).all(), impl
    finally:
        engine.set_option(OPT_BD_IMPL, BD_AUTO)


def test_device_entry_point_async(engine, oracle):
    """sd_band_depth_f64_dev on device buffers: synchronous by default; with SD_OPT_ASYNC_DEVICE it only enqueues and
    sd_sync() completes the call -- result, timings and errors (a NaN in the input) all surface there."""
    import torch
    from statdepth_b200 import EngineError
    from statdepth_b200._engine import OPT_ASYNC_DEVICE
    X = walks(61, 40, 3000)
    want = oracle.mbd_counts_all(X)
    dX = torch.from_numpy(X).cuda()
    out = torch.zeros(3000, dtype=torch.int64, device="cuda")
    engine.band_depth_counts_dev(dX.data_ptr(), 40, 3000, 3000, out.data_ptr(), None, 3000, 2, True)
    assert (out.cpu().numpy() == want).all()
    try:
        engine.set_option(OPT_ASYNC_DEVICE, 1)
        out.zero_()
        engine.band_depth_counts_dev(dX.data_ptr(), 40, 3000, 3000, out.data_ptr(), None, 3000, 2, True)
        engine.sync()
        assert (out.cpu().numpy() == want).all() and engine.timings()["kernel_ns"] > 0
        # two calls back to back without a sync in between: the second call completes the first
        engine.band_depth_counts_dev(dX.data_ptr(), 40, 3000, 3000, out.data_ptr(), None, 3000, 2, True)
        engine.band_depth_counts_dev(dX.data_ptr(), 40, 3000, 3000, out.data_ptr(), None, 3000, 2, True)
        engine.sync()
        assert (out.cpu().numpy() == want).all()
        dX[3, 77] = float("nan")
        engine.band_depth_counts_dev(dX.data_ptr(), 40, 3000, 3000, out.data_ptr(), None, 3000, 2, True)  # queued
        with pytest.raises(EngineError, match="NONFINITE"):
            engine.sync()
    finally:
        engine.set_option(OPT_ASYNC_DEVICE, 0)
        engine.sync()


def test_mbd_heavy_parts_edge_cases(engine, oracle):
    """Parts over capacity: value tables (<= 8 distinct values per part, <= 128 such parts per row), -0.0 == +0.0,
    a mix of heavy classes and a continuous remainder, and the hand-over to the generic path beyond the limits."""
    rng = np.random.default_rng(31)
    n = 200_000
    # 150 value classes of ~1333 copies: more heavy parts than the tables hold -> generic path, same counts
    Xm = np.stack([rng.permutation(np.arange(n) % 150).astype(np.float64) for _ in range(2)])
    assert (engine.band_depth_counts(Xm, None, 2, True) == oracle.mbd_counts_all(Xm)).all()
    assert engine.timings()["fallback_rows"] == 2
    # zero-inflated rows: a few heavy classes (each far above the part capacity, one of them +-0.0) inside a
    # continuous sample -> each class gets a part of its own next to normally sorted parts, no generic rows
    n = 120_000
    Xh = rng.standard_normal((3, n))
    Xh[:, : n // 2] = np.round(Xh[:, : n // 2] * 2.0)
    Xh[1, :5000] = -0.0
    Xh[1, 5000:9000] = 0.0
    for r in range(3):
        Xh[r] = rng.permutation(Xh[r])
    assert (engine.band_depth_counts(Xh, None, 2, True) == oracle.mbd_counts_all(Xh)).all()
    assert engine.timings()["fallback_rows"] == 0
    # many mid-sized classes (hundreds to ~2400 copies) inside a continuous sample: any route, same counts
    Xg = rng.standard_normal((3, n))
    Xg[:, : n // 2] = np.round(Xg[:, : n // 2] * 10.0)
    for r in range(3):
        Xg[r] = rng.permutation(Xg[r])
    assert (engine.band_depth_counts(Xg, None, 2, True) == oracle.mbd_counts_all(Xg)).all()
    # J = 3 and the rank output go through the same emit path
    cnt3 = engine.band_depth_counts(Xh, None, 3, True)
    assert (cnt3 == oracle.mbd_counts_all(Xh, j=3)).all()


# ------------------------------------------------------------------------------------------------
# strict band depth (relax=False)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,n,seed", [(100, 200, 0), (5, 6, 1), (2, 3, 2), (31, 300, 3), (32, 257, 4), (33, 256, 5),
                                      (64, 1000, 6), (97, 777, 7)])
def test_strict_counts_bit_exact(engine, oracle, T, n, seed):
    X = walks(seed, T, n)
    assert (engine.band_depth_counts(X, None, 2, False) == oracle.bd_counts(X)).all()


@pytest.mark.parametrize("maker", ["round", "noncrossing", "constant"])
def test_strict_ties_and_many_survivors(engine, oracle, maker):
    """Rounded curves tie with the query; non-crossing curves (the reference's own generator) make
    about half of all pairs survive every word, which exercises the survivor queue drain."""
    rng = np.random.default_rng(13)
    T, n = 70, 600
    if maker == "round":
        X = np.round(rng.standard_normal((T, n)).cumsum(0))
    elif maker == "noncrossing":
        X = np.outer(rng.random(T) + 0.1, rng.random(n))
    else:
        X = np.full((T, n), 1.0)
    assert (engine.band_depth_counts(X, None, 2, False) == oracle.bd_counts(X)).all()


@pytest.mark.parametrize("T,n,seed,maker", [(64, 128, 0, "walk"), (100, 200, 1, "walk"), (5, 6, 2, "walk"),
                                            (130, 300, 3, "round"), (512, 1000, 4, "walk"), (70, 600, 5, "noncrossing"),
                                            (200, 129, 6, "walk")])
def test_strict_tcgen05_gram_bit_exact(engine, oracle, T, n, seed, maker):
    """SD_BD_GEMM: the int8 violation Gram on tcgen05 / TMEM gives the same counts as the oracle."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((T, n)).cumsum(0)
    if maker == "round":
        X = np.round(X)
    elif maker == "noncrossing":
        X = np.outer(rng.random(T) + 0.1, rng.random(n))
    try:
        engine.set_option(E.OPT_BD_IMPL, E.BD_GEMM)
        assert (engine.band_depth_counts(X, None, 2, False) == oracle.bd_counts(X)).all()
        q = [n - 1, 0, n // 2]
        assert (engine.band_depth_counts(X, q, 2, False) == oracle.bd_counts(X, q)).all()
    finally:
        engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)


def test_strict_auto_policy(engine, oracle):
    """SD_BD_AUTO: tie-free queries are answered by sign-vector matching; queries with ties fall back to an
    enumerating kernel -- the bit kernel, or the tcgen05 Gram when a probe shows that the bit kernel would
    drown in survivors.  Every route gives the oracle's counts."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(23)
    T, n = 96, 1300
    q = np.arange(0, n, 13)  # 100 queries
    walk = rng.standard_normal((T, n)).cumsum(0)
    smooth = np.outer(rng.random(T) + 0.1, rng.random(n))           # non-crossing, tie-free
    cases = [(walk, E.BD_MATCH), (smooth, E.BD_MATCH),
             (np.round(walk), E.BD_BITS),                            # ties, few survivors
             (np.round(smooth * 8.0), E.BD_GEMM)]                    # ties, ~half of all pairs survive
    for X, used in cases:
        exp = oracle.bd_counts(X, q)
        assert (engine.band_depth_counts(X, q, 2, False) == exp).all()
        assert engine.timings()["bd_impl_used"] == used
    for impl in (E.BD_BITS, E.BD_GEMM, E.BD_MATCH):
        try:
            engine.set_option(E.OPT_BD_IMPL, impl)
            for X, _ in cases[:3]:
                assert (engine.band_depth_counts(X, q[:40], 2, False) == oracle.bd_counts(X, q[:40])).all()
        finally:
            engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)
    assert (engine.band_depth_counts(smooth, None, 2, False)[q] == oracle.bd_counts(smooth, q)).all()


def test_strict_null_queries(engine):
    """queries=None means the ids 0 .. n-1, written once on the device before the strict route is chosen: on every
    route the counts and the route equal those of an explicit np.arange(n), at exactly one launch more.  n = 8200 is
    above the matcher's limit, so SD_BD_AUTO reaches the probe of the enumerating path, which offsets that list."""
    from statdepth_b200 import _engine as E
    walk = walks(31, 96, 1300)
    cases = [(walk, E.BD_BITS, (E.BD_BITS,)), (walk, E.BD_GEMM, (E.BD_GEMM,)), (walk, E.BD_MATCH, (E.BD_MATCH,)),
             (walks(37, 8, 8200), E.BD_AUTO, (E.BD_BITS, E.BD_GEMM))]
    for X, impl, used in cases:
        try:
            engine.set_option(E.OPT_BD_IMPL, impl)
            got = engine.band_depth_counts(X, None, 2, False)
            t_null = engine.timings()
            exp = engine.band_depth_counts(X, np.arange(X.shape[1]), 2, False)
            t_list = engine.timings()
        finally:
            engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)
        assert (got == exp).all()
        assert t_null["bd_impl_used"] == t_list["bd_impl_used"] and t_list["bd_impl_used"] in used
        assert t_null["launches"] == t_list["launches"] + 1


def test_strict_match_edge_shapes(engine, oracle):
    """Sign-vector matcher on ragged shapes: T not a multiple of 32, n = 3 .. 8193, a few tied curves (set Z)."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(29)
    try:
        engine.set_option(E.OPT_BD_IMPL, E.BD_MATCH)
        for T, n in ((1, 3), (5, 6), (33, 70), (100, 513), (37, 1025), (64, 2500)):
            X = rng.standard_normal((T, n)).cumsum(0)
            assert (engine.band_depth_counts(X, None, 2, False) == oracle.bd_counts(X)).all()
            X[:, 1] = X[:, 0]                    # curve 1 duplicates curve 0: ties for queries 0 and 1 only
            X[T // 2, 2::7] = X[T // 2, 0]       # a few curves touch curve 0 once
            assert (engine.band_depth_counts(X, None, 2, False) == oracle.bd_counts(X)).all()
        X = rng.standard_normal((40, 8193)).cumsum(0)  # largest n the matcher takes
        qs = [0, 4096, 8192]
        assert (engine.band_depth_counts(X, qs, 2, False) == oracle.bd_counts(X, qs)).all()
        assert engine.timings()["bd_impl_used"] == E.BD_MATCH
    finally:
        engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)


def test_strict_j3(engine, oracle):
    X = walks(61, 40, 60)
    assert (engine.band_depth_counts(X, None, 3, False) == oracle.bd_counts(X, j=3)).all()
    Xr = np.round(X)
    assert (engine.band_depth_counts(Xr, [0, 7, 59], 3, False) == oracle.bd_counts(Xr, [0, 7, 59], j=3)).all()


def test_strict_full_size_sample(engine, oracle):
    """BASELINE config 3 (8192 curves x 512 points): all 8192 queries on the GPU (sign-vector matcher), 48 of
    them checked against the oracle, and three independent GPU algorithms cross-checked on larger samples:
    matcher == bit kernel on 256 queries == tcgen05 Gram on 64 queries; plus the bound count <= C(n-1,2)."""
    from statdepth_b200 import _engine as E
    T, n = 512, 8192
    X = walks(2, T, n)
    got = engine.band_depth_counts(X, None, 2, False)
    assert engine.timings()["bd_impl_used"] == E.BD_MATCH
    rng = np.random.default_rng(0)
    q = rng.choice(n, 48, replace=False)
    assert (got[q] == oracle.bd_counts(X, q)).all()
    assert got.max() <= comb(n - 1, 2) and got.min() >= 0
    q2 = rng.choice(n, 256, replace=False)
    try:
        engine.set_option(E.OPT_BD_IMPL, E.BD_BITS)
        assert (engine.band_depth_counts(X, q2, 2, False) == got[q2]).all()
        engine.set_option(E.OPT_BD_IMPL, E.BD_GEMM)
        assert (engine.band_depth_counts(X, q2[:64], 2, False) == got[q2[:64]]).all()
    finally:
        engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)


# ------------------------------------------------------------------------------------------------
# public API against the reference's golden vectors
# ------------------------------------------------------------------------------------------------
def test_golden_vectors_through_public_api(golden):
    from statdepth_b200 import FunctionalDepth, PointcloudDepth
    n = 0
    for case in golden.values():
        if case["kind"] in ("functional", "multivariate", "pointcloud"):
            check_case(case, FunctionalDepth, PointcloudDepth, rtol=RTOL)
            n += 1
    assert n >= 30


def test_cfg1_reference_values(golden):
    """BASELINE config 1: the two curves the reference itself computed (88 s of CPU) -- strict bit-exact."""
    from statdepth_b200 import FunctionalDepth
    df = pd.DataFrame(walks(0, 100, 200))
    s = FunctionalDepth([df], to_compute=[0, 1], relax=False)
    assert s.values.tolist() == golden["cfg1_200x100_strict"]["depths"]
    r = FunctionalDepth([df], to_compute=[0, 1], relax=True)
    np.testing.assert_allclose(r.values, golden["cfg1_200x100_relax"]["depths"], rtol=RTOL)


def test_k_sampled_and_batched(engine, oracle, golden):
    from statdepth_b200 import FunctionalDepth
    case = golden["walk_K3_seed123"]
    np.random.seed(case["np_seed"])
    res = FunctionalDepth([pd.DataFrame(np.array(case["X"]))], K=case["K"], **case["kwargs"])
    np.testing.assert_allclose(res.values, case["depths"], rtol=RTOL)
    # batched ABI directly: random sub-populations of one matrix
    rng = np.random.default_rng(71)
    X = walks(72, 30, 90)
    B = 7
    mem = (rng.random((B, 90)) < 0.6).astype(np.uint8)
    qs = np.stack([rng.choice(np.flatnonzero(mem[b]), 3, replace=False) for b in range(B)])
    for relax in (True, False):
        got = engine.band_depth_counts_batched(X, mem, qs, 2, relax)
        for b in range(B):
            cols = np.flatnonzero(mem[b])
            loc = [int(np.searchsorted(cols, g)) for g in qs[b]]
            sub = np.ascontiguousarray(X[:, cols])
            exp = oracle.mbd_counts_all(sub)[loc] if relax else oracle.bd_counts(sub, loc)
            assert (got[b] == exp).all()
    # equally sized batches (what a permutation test asks for): relaxed depth runs all batches as ONE grouped pass
    B, m = 9, 40
    members = np.stack([np.sort(rng.choice(90, m, replace=False)) for _ in range(B)])
    mem = np.zeros((B, 90), dtype=np.uint8)
    for b in range(B):
        mem[b, members[b]] = 1
    qs = np.stack([rng.permutation(members[b])[:11] for b in range(B)])
    Xt = np.round(X)  # with ties
    for Xm in (X, Xt):
        for j in (2, 3):
            got = engine.band_depth_counts_batched(Xm, mem, qs, j, True)
            for b in range(B):
                loc = [int(np.searchsorted(members[b], g)) for g in qs[b]]
                exp = oracle.mbd_counts_all(np.ascontiguousarray(Xm[:, members[b]]), j=j)[loc]
                assert (got[b] == exp).all(), (b, j)
        # strict: one rank pass + one signature / match launch pair for all batches; tied queries are re-enumerated
        got = engine.band_depth_counts_batched(Xm, mem, qs, 2, False)
        for b in range(B):
            loc = [int(np.searchsorted(members[b], g)) for g in qs[b]]
            exp = oracle.bd_counts(np.ascontiguousarray(Xm[:, members[b]]), loc)
            assert (got[b] == exp).all(), b


def test_reference_test_suite_types():
    """The reference's own 5 tests (tests/test_statdepth.py:22-73), same calls, same assertions."""
    from statdepth_b200 import FunctionalDepth, PointcloudDepth
    from statdepth_b200.testing import (generate_noisy_multivariate, generate_noisy_pointcloud,
                                        generate_noisy_univariate)
    df = generate_noisy_univariate()
    bd = FunctionalDepth([df], containment='r2')
    for obj in (bd, bd.ordered(), bd.median(), bd.deepest(n=2), bd.outlying(n=2)):
        assert isinstance(obj, pd.Series)
    assert isinstance(FunctionalDepth([df], K=5, containment='r2'), pd.Series)
    for c, npts in (('l1', 10), ('simplex', 10), ('oja', 20)):
        pc = generate_noisy_pointcloud(n=npts, d=2)
        r = PointcloudDepth(pc, containment=c)
        for obj in (r, r.ordered(), r.median(), r.deepest(n=2), r.outlying(n=2)):
            assert isinstance(obj, pd.Series)
        assert isinstance(PointcloudDepth(pc, K=2, containment=c), pd.Series)
    mv = FunctionalDepth(generate_noisy_multivariate(), containment='simplex')
    assert isinstance(mv, pd.Series) and isinstance(mv.ordered(), pd.Series)


# ------------------------------------------------------------------------------------------------
# point clouds and multivariate simplex depth
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,seed", [(300, 2, 0), (257, 3, 1), (64, 1, 2), (100, 5, 3), (1500, 2, 4)])
def test_l1_depth(engine, oracle, n, d, seed):
    P = np.random.default_rng(seed).standard_normal((n, d))
    got = engine.l1_depth(P)
    exp = oracle.l1_depth(P)
    np.testing.assert_allclose(got, exp, rtol=RTOL)
    # same IEEE operations per term; the sum runs over 4 interleaved lanes per query instead of one sequence,
    # which moves 1 - |sum|/n by a few ulp of 1 (observed <= 3e-14 relative; bar: 1e-12)
    np.testing.assert_allclose(got, exp, rtol=1e-13, atol=0)
    q = [3, 0, n - 1]
    assert (engine.l1_depth(P, q) == got[q]).all()  # independent of which queries are asked for


def test_l1_duplicates_propagate_nan(engine, oracle):
    P = np.random.default_rng(5).standard_normal((20, 2))
    P[7] = P[3]
    got, exp = engine.l1_depth(P), oracle.l1_depth(P)
    assert np.isnan(got[[3, 7]]).all() and np.isnan(exp[[3, 7]]).all()  # 0/0, as in the reference


@pytest.mark.parametrize("n,d,seed", [(40, 2, 0), (18, 3, 1), (30, 1, 2), (120, 2, 3)])
def test_simplicial_counts(engine, oracle, n, d, seed):
    P = np.random.default_rng(seed).standard_normal((n, d))
    assert (engine.simplicial_counts(P) == oracle.simplicial_counts(P)).all()
    assert (engine.simplicial_counts(P, [1, 0], 0.0) == oracle.simplicial_counts(P, [1, 0], 0.0)).all()


def test_simplicial_degenerate_inputs(engine, oracle):
    rng = np.random.default_rng(8)
    P = rng.integers(0, 4, size=(25, 2)).astype(np.float64)  # lattice: collinear triples, duplicates
    for tol in (0.0, 1e-7):
        assert (engine.simplicial_counts(P, None, tol) == oracle.simplicial_counts(P, None, tol)).all()
    L = np.outer(rng.random(12), [1.0, 2.0, -1.0])  # all points on one line in 3-D
    assert (engine.simplicial_counts(L) == oracle.simplicial_counts(L)).all()


def test_simplicial_angular_counting(engine, oracle):
    """SD_SIMPLICIAL_COUNT: the O(n log n) angular counting gives exactly the enumeration's counts
    (closed triangles, tolerance 0) -- general position, lattice data with collinear / duplicate /
    antipodal points, and a larger cloud checked against the GPU enumeration."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(17)
    try:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_COUNT)
        for n, lattice in ((37, False), (30, True), (64, True), (5, False), (4, False), (3, False), (200, False)):
            P = rng.integers(0, 5, size=(n, 2)).astype(np.float64) if lattice else rng.standard_normal((n, 2))
            assert (engine.simplicial_counts(P, None, 0.0) == oracle.simplicial_counts(P, None, 0.0)).all()
        P = rng.standard_normal((1500, 2))
        q = [0, 777, 1499]
        got = engine.simplicial_counts(P, q, 0.0)
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_ENUMERATE)
        assert (got == engine.simplicial_counts(P, q, 0.0)).all()
    finally:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_AUTO)


def test_simplicial_full_size_properties(engine):
    """BASELINE config 5: 2-D simplicial depth of 50 000 points (generate_noisy_pointcloud(n, 2, seed=4)).
    Size-independent checks: 0 <= count <= C(n-1,3); translating / scaling by powers of two leaves every
    count unchanged; the deepest point is near the centre, hull vertices have count 0."""
    from statdepth_b200.testing import generate_noisy_pointcloud
    n = 50_000
    P = generate_noisy_pointcloud(n=n, d=2, seed=4).values
    q = np.arange(0, n, 97)
    c = engine.simplicial_counts(P, q, 0.0)
    assert c.min() >= 0 and c.max() <= comb(n - 1, 3)
    assert (engine.simplicial_counts(P * 4.0, q, 0.0) == c).all()
    far = int(np.argmax((P ** 2).sum(1)))
    assert engine.simplicial_counts(P, [far], 0.0)[0] == 0
    deepest = q[int(np.argmax(c))]
    assert np.hypot(*P[deepest]) < 0.2 and c.max() / comb(n, 3) > 0.24  # max simplicial depth in 2-D is 1/4


def test_relaxed_simplex_depth_counting(engine, oracle):
    """Relaxed multivariate simplex depth (d = 2) through the counting path, per (query, time point)."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(19)
    try:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_COUNT)
        for N, T in ((12, 9), (30, 5), (7, 3)):
            F = rng.standard_normal((N, T, 2)).cumsum(1)
            assert (engine.simplex_depth_counts(F, None, True, 0.0) == oracle.simplex_depth_counts(F, None, True, 0.0)).all()
            assert (engine.simplex_depth_counts(F, [N - 1, 1], True, 0.0) ==
                    oracle.simplex_depth_counts(F, [N - 1, 1], True, 0.0)).all()
        Fl = rng.integers(0, 4, size=(15, 6, 2)).astype(np.float64)
        assert (engine.simplex_depth_counts(Fl, None, True, 0.0) == oracle.simplex_depth_counts(Fl, None, True, 0.0)).all()
    finally:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_AUTO)
    # AUTO switches to counting above 64 curves
    F = rng.standard_normal((80, 4, 2)).cumsum(1)
    assert (engine.simplex_depth_counts(F, [0, 41], True, 0.0) == oracle.simplex_depth_counts(F, [0, 41], True, 0.0)).all()


def test_counting_honours_the_tolerance_band(engine, oracle):
    """Above the enumerate -> count switch (64 curves / points) the counting kernels keep the reference's
    semantics, dist(p, triangle) <= tol with tol = 1e-7 (the LP's band, _containment.py:164-176): AUTO equals
    the oracle's enumeration on the reference's own 100 % collinear fixture (round-1 verdict: depths jumped by
    up to 0.43 at 65 curves), on clouds with many collinear points, on lattices, and for large tolerances."""
    from statdepth_b200.testing import generate_noisy_multivariate
    for N in (64, 65, 70):  # 64: still enumerated; 65, 70: counted -- no jump
        data = generate_noisy_multivariate(num_curves=N, n=6, d=2, seed=0)
        F = np.stack([x.values for x in data])
        got = engine.simplex_depth_counts(F, None, True)
        assert (got == oracle.simplex_depth_counts(F, None, True)).all(), N
        if N == 70:
            assert got[:3].tolist() == [233160, 75978, 52260]  # the reference's semantics, not tolerance 0
    rng = np.random.default_rng(70)
    p0 = np.array([0.25, -0.5])
    d1, d2 = np.array([1.0, 2.0]) / np.sqrt(5.0), np.array([3.0, -1.0]) / np.sqrt(10.0)
    P = np.vstack([p0[None, :], p0 + rng.uniform(-2, 2, 60)[:, None] * d1, p0 + rng.uniform(-2, 2, 40)[:, None] * d2,
                   rng.standard_normal((59, 2))])
    q = [0, 1, 61, 101, 159]
    assert (engine.simplicial_counts(P, q) == oracle.simplicial_counts(P, q)).all()
    Lt = rng.integers(0, 9, size=(100, 2)).astype(np.float64)
    for tol in (1e-7, 1e-3, 0.25):
        assert (engine.simplicial_counts(Lt, None, tol) == oracle.simplicial_counts(Lt, None, tol)).all(), tol
    G = rng.standard_normal((150, 2))
    for tol in (1e-7, 0.05, 0.6):
        assert (engine.simplicial_counts(G, None, tol) == oracle.simplicial_counts(G, None, tol)).all(), tol


def test_angular_key_wraps_at_two_pi(engine, oracle):
    """Round-1 advisor finding: a direction a hair below the +x axis got the key 16.0, the sentinel range of the
    exact (tolerance 0) counting path, and was counted as a point coincident with the query (counts off by O(n^2)).
    It now folds onto the +x axis class.  Directions within one rounding of each other are ONE class for the
    exact path (their ratio rounds to the same double), so on this deliberately near-degenerate cloud it equals
    the enumeration with a hair of tolerance (1e-12), not the enumeration's own rounding of orient2 at 0."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(3)
    P = rng.standard_normal((90, 2))
    P[0] = (0.0, 0.1 + 0.2)
    P[1] = (1.0, 0.3)              # dy = -5.6e-17: rounds onto the axis from below
    P[2] = (2.0, 0.1 + 0.2 - 1e-16)
    P[3] = (-1.5, 0.1 + 0.2)       # exact antipode on the axis
    q = [0, 1, 2, 3, 50]
    try:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_COUNT)
        got = engine.simplicial_counts(P, q, 0.0)
    finally:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_AUTO)
    assert got.tolist() == [28278, 13587, 336, 4551, 23673]  # numpy emulation of the key formulas
    assert (got == oracle.simplicial_counts(P, q, 1e-12)).all()
    assert (engine.simplicial_counts(P, q) == oracle.simplicial_counts(P, q)).all()  # default band: arcs


def test_large_golden_through_public_api():
    """Outputs of the UNMODIFIED reference on samples above the switch (tests/golden/make_golden_large.py:
    66 collinear curves, 66 random-walk curves, clouds of 70 / 130 points with collinear structure)."""
    import json
    import os
    from statdepth_b200 import FunctionalDepth, PointcloudDepth
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors_large.json")) as fh:
        cases = json.load(fh)["cases"]
    assert len(cases) >= 6
    for case in cases:
        check_case(case, FunctionalDepth, PointcloudDepth, rtol=RTOL)


def test_config_sized_counts_pinned_by_the_oracle(engine, oracle):
    """BASELINE configs 4 and 5 at FULL size against an independent computation (round-1 verdict: properties
    only): three queries each, the oracle's O(n^2)-per-(query, time point) arc counter."""
    from statdepth_b200.testing import generate_noisy_pointcloud
    P = generate_noisy_pointcloud(n=50_000, d=2, seed=4).values
    q = [0, 12_345, 49_999]
    assert (engine.simplicial_counts(P, q) == oracle.triangle_counts_arcs(P, q)).all()
    F = np.random.default_rng(3).standard_normal((5000, 256, 2)).cumsum(1)
    q = [0, 2500, 4999]
    assert (engine.simplex_depth_counts(F, q, True) == oracle.simplex2_relaxed_counts_arcs(F, q)).all()
    Lq = [7, 25_000, 49_998]
    np.testing.assert_allclose(engine.l1_depth(P, Lq), oracle.l1_depth(P, Lq), rtol=RTOL)


@pytest.mark.parametrize("n,d,seed", [(60, 2, 0), (20, 3, 1)])
def test_oja(engine, oracle, n, d, seed):
    from scipy.spatial import ConvexHull
    P = np.random.default_rng(seed).standard_normal((n, d))
    hv = ConvexHull(P).volume
    np.testing.assert_allclose(engine.oja(P, hv), oracle.oja(P, hv), rtol=RTOL)
    pool = np.array([0, 3, 5, 9, 11, 12])
    np.testing.assert_allclose(engine.oja(P, hv, pool, pool), oracle.oja(P, hv, pool, pool), rtol=RTOL)


def test_oja_angular_sums(engine, oracle):
    """Oja depth in 2-D by angular prefix sums (O(n log n) per query; AUTO above 256 points) against the
    oracle's pair enumeration: general position, a lattice (collinear pairs have area 0), a pool, and the size
    at which AUTO switches.  Different summation order: 1e-12 relative, as for every float64 result."""
    from scipy.spatial import ConvexHull
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(23)
    try:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_COUNT)
        for n, lattice in ((3, False), (4, False), (37, False), (60, True), (300, False)):
            P = rng.integers(0, 6, size=(n, 2)).astype(np.float64) if lattice else rng.standard_normal((n, 2))
            hv = ConvexHull(P).volume if n > 3 else 1.0
            np.testing.assert_allclose(engine.oja(P, hv), oracle.oja(P, hv), rtol=RTOL, atol=1e-13)
        P = rng.standard_normal((80, 2))
        pool = np.array([5, 0, 33, 79, 12, 40, 41, 7])
        np.testing.assert_allclose(engine.oja(P, 2.5, pool, pool), oracle.oja(P, 2.5, pool, pool), rtol=RTOL)
        np.testing.assert_allclose(engine.oja(P, 2.5, [3, 5], pool), oracle.oja(P, 2.5, [3, 5], pool), rtol=RTOL)
    finally:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_AUTO)
    P = rng.standard_normal((1200, 2))  # AUTO: counted; 50 queries against the enumeration
    q = rng.choice(1200, 50, replace=False)
    np.testing.assert_allclose(engine.oja(P, 7.0, q), oracle.oja(P, 7.0, q), rtol=RTOL)


@pytest.mark.parametrize("N,T,d,seed", [(12, 9, 2, 0), (9, 5, 3, 1), (10, 7, 1, 2), (30, 16, 2, 3)])
def test_simplex_depth_counts(engine, oracle, N, T, d, seed):
    F = np.random.default_rng(seed).standard_normal((N, T, d)).cumsum(1)
    for relax in (False, True):
        assert (engine.simplex_depth_counts(F, None, relax) == oracle.simplex_depth_counts(F, None, relax)).all()
    assert (engine.simplex_depth_counts(F, [2, 0], True, 0.0) == oracle.simplex_depth_counts(F, [2, 0], True, 0.0)).all()


def test_simplex_depth_reference_fixture(engine, oracle):
    """The reference's multivariate generator makes 100% degenerate simplices (all curves are scalar
    multiples of one base curve): containment reduces to 'r between min r_i and max r_i'."""
    from statdepth_b200.testing import generate_noisy_multivariate
    for seed, d in ((0, 3), (1, 3), (5, 2)):
        data = generate_noisy_multivariate(num_curves=7, n=6, d=d, seed=seed)
        F = np.stack([x.values for x in data])
        for relax in (False, True):
            assert (engine.simplex_depth_counts(F, None, relax) == oracle.simplex_depth_counts(F, None, relax)).all()


def test_homogeneity_and_permutation_test(golden):
    from statdepth_b200.homogeneity import FunctionalHomogeneity, permutation_test
    for m in ("p1", "p2", "p3"):
        case = golden["functional_%s" % m]
        F = pd.DataFrame(np.array(case["F"]), columns=["F%d" % i for i in range(7)])
        G = pd.DataFrame(np.array(case["G"]), columns=["G%d" % i for i in range(6)])
        h = FunctionalHomogeneity([F], [G], method=m, quiet=True).homogeneity()
        np.testing.assert_allclose(float(np.asarray(h).ravel()[0]), case["value"], rtol=RTOL)
    rng = np.random.default_rng(5)
    F = pd.DataFrame(rng.standard_normal((32, 24)).cumsum(0))
    G = pd.DataFrame(rng.standard_normal((32, 24)).cumsum(0) + 6.0)
    out = permutation_test(F, G, method='p1', B=20, seed=5)
    assert out["null"].shape == (20,) and 0.0 < out["p_value"] <= 1.0
    assert out["p_value"] < 0.2  # a 6-sigma shift is not exchangeable
    loop = permutation_test(F, G, method='p1', B=20, seed=5, batched=False)
    assert loop["null"].tolist() == out["null"].tolist() and loop["observed"] == out["observed"]
    for method in ("p2",):
        a = permutation_test(F, G, method=method, B=10, seed=6, relax=False)
        b = permutation_test(F, G, method=method, B=10, seed=6, relax=False, batched=False)
        assert a["null"].tolist() == b["null"].tolist()


def test_next_rows_against_the_reference_on_gpu():
    """SURVEY 8(f): K-sampled point-cloud depth through sd_pointcloud_blocks_f64, point-cloud homogeneity p1..p3,
    Mahalanobis -- the unmodified reference's outputs (tests/golden/make_golden_next.py)."""
    from api_cases import check_next_case, load_next_cases
    from statdepth_b200 import PointcloudDepth
    from statdepth_b200.homogeneity import PointcloudHomogeneity
    for case in load_next_cases():
        check_next_case(case, PointcloudDepth, PointcloudHomogeneity, rtol=RTOL)


def test_cloud_blocks_abi(engine, oracle):
    """sd_pointcloud_blocks_f64: ragged blocks, all three kinds, d = 2 and 3, against single-cloud oracle calls."""
    rng = np.random.default_rng(61)
    for d in (2, 3):
        P = rng.standard_normal((40, d))
        members, offsets, qpos, hv = [], [0], [], []
        for b in range(23):
            m = int(rng.integers(d + 2, 15))
            ids = rng.choice(40, m, replace=False)
            members.append(ids)
            offsets.append(offsets[-1] + m)
            qpos.append(int(rng.integers(0, m)))
            hv.append(float(rng.uniform(0.5, 2.0)))
        mem = np.concatenate(members)
        for kind in ("simplex", "l1", "oja"):
            got = engine.cloud_blocks(P, mem, offsets, qpos, kind, 1e-7, hv)
            for b in range(23):
                sub = np.ascontiguousarray(P[members[b]])
                if kind == "simplex":
                    assert got[b] == oracle.simplicial_counts(sub, [qpos[b]])[0]
                elif kind == "l1":
                    assert got[b] == oracle.l1_depth(sub, [qpos[b]])[0]  # same operations in the same order
                else:
                    np.testing.assert_allclose(got[b], oracle.oja(sub, hv[b], [qpos[b]])[0], rtol=RTOL)


def test_permutation_test_p3_batched(engine):
    from statdepth_b200.homogeneity import permutation_test
    rng = np.random.default_rng(8)
    F = pd.DataFrame(rng.standard_normal((24, 14)).cumsum(0))
    G = pd.DataFrame(rng.standard_normal((24, 14)).cumsum(0) + 1.0)
    for relax in (True, False):
        a = permutation_test(F, G, method="p3", B=6, seed=2, relax=relax)
        b = permutation_test(F, G, method="p3", B=6, seed=2, relax=relax, batched=False)
        np.testing.assert_allclose(a["null"], b["null"], rtol=RTOL)
        assert a["observed"] == b["observed"]


def test_strict_simplex_depth_d2_pruned_kernel(engine, oracle):
    """Strict multivariate simplex depth, d = 2 (first-row pruning in shared memory, exact pre-test, reference
    predicate inside the band): equals the oracle's plain enumeration on random walks, a lattice (collinear and
    on-edge cases), the reference's collinear fixture, several tolerances and query subsets."""
    from statdepth_b200.testing import generate_noisy_multivariate
    rng = np.random.default_rng(4)
    for N, T in ((4, 1), (5, 3), (9, 2), (12, 5), (33, 1), (40, 3), (90, 6), (150, 4)):
        F = rng.standard_normal((N, T, 2)).cumsum(1) * (0.2 if N == 150 else 1.0)
        for tol in (0.0, 1e-7, 0.05):
            assert (engine.simplex_depth_counts(F, None, False, tol) == oracle.simplex_depth_counts(F, None, False, tol)).all()
    Fl = rng.integers(0, 4, size=(25, 4, 2)).astype(np.float64)
    assert (engine.simplex_depth_counts(Fl, None, False) == oracle.simplex_depth_counts(Fl, None, False)).all()
    data = generate_noisy_multivariate(num_curves=70, n=5, d=2, seed=1)
    Fd = np.stack([x.values for x in data])
    got = engine.simplex_depth_counts(Fd, None, False)
    assert (got == oracle.simplex_depth_counts(Fd, None, False)).all() and got.max() > 0
    q = [3, 0, 69]
    assert (engine.simplex_depth_counts(Fd, q, False) == got[q]).all()
    F = rng.standard_normal((600, 16, 2)).cumsum(1)   # mid size against the oracle's pre-tested enumeration
    q = [0, 299, 599]
    assert (engine.simplex_depth_counts(F, q, False) == oracle.simplex2_strict_fast(F, q)).all()


def _config4_strict_data():
    """5 000 curves x 256 points x 2 channels: random walks, plus 14 far 'anchor' curves on a big circle so that the
    strict depth of an inner curve is not simply 0 (only anchor triangles contain it at all 256 rows)."""
    rng = np.random.default_rng(3)
    F = rng.standard_normal((5000, 256, 2)).cumsum(1)
    ang = np.sort(rng.uniform(0, 2 * np.pi, 14))
    F[:14] = 2000.0 * np.stack([np.cos(ang), np.sin(ang)], axis=1)[:, None, :] + rng.standard_normal((14, 256, 2))
    return F


def test_config4_strict_depth_full_size(engine, oracle):
    """BASELINE config 4, strict, d = 2, FULL size: one query (C(4999,3) = 2.1e10 triples) pinned by the oracle's
    multi-threaded enumeration (about a minute of host time), plus 16 more queries for bounds and timing."""
    F = _config4_strict_data()
    got = engine.simplex_depth_counts(F, [2500], False)
    exp = oracle.simplex2_strict_fast(F, [2500])
    assert got.tolist() == exp.tolist() and got[0] > 0
    more = engine.simplex_depth_counts(F, list(range(100, 4900, 300)), False)
    assert more.min() >= 0 and more.max() <= comb(13, 3) + comb(13, 2) * 4986  # at most: triangles with >= 2 anchors


def _random_cloud(rng, n):
    """2-D clouds of trouble: general position, lattices, points on a few lines through a query, clusters within the
    tolerance band of each other, duplicates, widely different scales."""
    kind = int(rng.integers(0, 6))
    P = rng.standard_normal((n, 2))
    if kind == 1:
        P = rng.integers(0, int(rng.integers(3, 9)), size=(n, 2)).astype(np.float64)
    elif kind == 2:  # half of the points on two lines through point 0
        d = rng.standard_normal((2, 2))
        k = n // 2
        P[1:k] = P[0] + rng.uniform(-3, 3, k - 1)[:, None] * d[rng.integers(0, 2, k - 1)]
    elif kind == 3:  # clusters tighter than the band: members lie within 1e-7 of each other
        c = rng.standard_normal((max(2, n // 8), 2))
        P = c[rng.integers(0, len(c), n)] + rng.uniform(-4e-8, 4e-8, (n, 2))
    elif kind == 4:  # duplicates
        P[rng.integers(0, n, n // 4)] = P[rng.integers(0, n, n // 4)]
    elif kind == 5:
        P = P * rng.choice([1e-3, 1e3]) + rng.choice([0.0, 1e4])
    return np.ascontiguousarray(P)


@pytest.mark.parametrize("seed", range(16))
def test_counting_randomized_differential(engine, oracle, seed):
    """Seeded random clouds / curve sets with degenerate structure: the counting kernels (arcs with a tolerance,
    exact keys at tolerance 0 on integer data), the strict pruned kernel and the Oja prefix sums against the
    oracle's enumeration.  Cases within rounding of the band's edge are excluded by construction: structure is exact
    (lattice, duplicates) or far from the band (1e-7 vs >= 1e-3), except kind 3, which sits INSIDE the band."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(7000 + seed)
    n = int(rng.choice([65, 80, 130, 200]))
    P = _random_cloud(rng, n)
    q = rng.choice(n, size=6, replace=False)
    tol = float(rng.choice([1e-7, 1e-7, 1e-3]))
    assert (engine.simplicial_counts(P, q, tol) == oracle.simplicial_counts(P, q, tol)).all()  # AUTO: counted
    N, T = int(rng.choice([66, 90])), int(rng.integers(2, 6))
    F = np.stack([_random_cloud(rng, N) for _ in range(T)], axis=1)  # [N, T, 2]: every row a troubled cloud
    qf = rng.choice(N, size=4, replace=False)
    assert (engine.simplex_depth_counts(F, qf, True, tol) == oracle.simplex_depth_counts(F, qf, True, tol)).all()
    assert (engine.simplex_depth_counts(F, qf, False, tol) == oracle.simplex_depth_counts(F, qf, False, tol)).all()
    try:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_COUNT)
        L = rng.integers(0, 7, size=(n, 2)).astype(np.float64)
        assert (engine.simplicial_counts(L, q, 0.0) == oracle.simplicial_counts(L, q, 0.0)).all()  # exact keys
        np.testing.assert_allclose(engine.oja(P, 3.0, q), oracle.oja(P, 3.0, q), rtol=1e-10, atol=1e-12)
    finally:
        engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_AUTO)
