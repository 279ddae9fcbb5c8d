"""The Engine's host-array calls against the CPU test doubles that stand in for it.

The CPU suite drives the outlier, fitted-reference and spatial drivers with test doubles in place of the Engine.  This
file holds the real Engine to those doubles at every call the drivers make, on the same seeded inputs: rows given in C
order, curve-major (F order) and as a tensor from Engine.upload, with ties, one time point and one sample curve.  So a
host-layer test that passes on a double speaks for the GPU path.  Integers and every float a kernel pins bit for bit
must be equal; spatial norms meet test_spatial's bar."""
import numpy as np
import pytest

from test_extremal import ExtremalOracleEngine
from test_outliers import OutlierOracleEngine
from test_reference import SortedOracleEngine
from test_reference_projection import ReferenceOracleEngine
from test_spatial import SpatialOracleEngine, assert_depths

pytestmark = pytest.mark.gpu


def _tied(rng, shape):
    """Values on 7 levels, zeros of both signs."""
    X = rng.integers(-3, 4, size=shape).astype(np.float64) * 0.5
    X[(X == 0) & (rng.random(shape) < 0.5)] = -0.0
    return X


def _host(engine, a):
    if a is None or isinstance(a, np.ndarray):
        return a
    engine.sync()  # a tensor the engine wrote on its stream
    return a.cpu().numpy()


def _equal(engine, got, exp, where):
    got, exp = _host(engine, got), _host(engine, exp)
    if got is None or exp is None:
        assert got is None and exp is None, where
        return
    exp = np.asarray(exp)
    assert got.dtype == exp.dtype and got.shape == exp.shape, (where, got.dtype, exp.dtype, got.shape, exp.shape)
    assert np.array_equal(got, exp), where


def _forms(engine, X):
    """X as a driver may hand it to the engine."""
    return {"C": np.ascontiguousarray(X), "F": np.asfortranarray(X), "uploaded C": engine.upload(X),
            "uploaded F": engine.upload(np.asfortranarray(X))}


def _rows_cases():
    """Time rows X [T, n]: walks, tie-heavy with a repeated curve, one time point, two curves."""
    rng = np.random.default_rng(0)
    tied = _tied(rng, (7, 33))
    tied[:, 5] = tied[:, 2]
    return {"walks": rng.standard_normal((9, 40)).cumsum(0), "tied": tied, "T1": rng.standard_normal((1, 25)),
            "n2": rng.standard_normal((6, 2))}


def test_upload_gives_c_order_rows(engine):
    import torch
    for name, X in _rows_cases().items():
        for A in (X, np.asfortranarray(X), X[:, ::2], X.astype(np.float32)):
            d = engine.upload(A)
            assert d.dtype == torch.float64 and d.is_contiguous() and d.device == torch.device("cuda", engine.device)
            assert np.array_equal(_host(engine, d), A), name
    m = np.arange(12, dtype=np.int32).reshape(3, 4)
    assert np.array_equal(_host(engine, engine.upload(m, np.int32)), m)


def test_outlier_calls_equal_the_doubles(engine, oracle):
    doubles = OutlierOracleEngine(), ExtremalOracleEngine()
    ext = doubles[1]
    rng = np.random.default_rng(1)
    for name, X in _rows_cases().items():
        member = rng.random(X.shape[1]) < 0.4
        member[0] = True
        for form, A in _forms(engine, X).items():
            where = (name, form)
            for dbl in doubles:
                _equal(engine, engine.band_depth_counts(A, None, 2, True), dbl.band_depth_counts(X, None, 2, True),
                       where)
                for factor, want_outside in ((1.5, True), (0.0, False), (0.25, True)):
                    got = engine.band_envelope(A, member, factor, want_outside)
                    for g, e in zip(got, dbl.band_envelope(X, member, factor, want_outside)):
                        _equal(engine, g, e, where + (factor,))
            for want_above in (False, True):
                got, exp = engine.band_rank_sums(A, want_above), doubles[0].band_rank_sums(X, want_above)
                assert len(got) == len(exp) == 2 + want_above
                for g, e in zip(got, exp):
                    _equal(engine, g, e, where + (want_above,))
            m = engine.band_extremity(A)  # on the device for uploaded rows, where extremal_depth reads it
            _equal(engine, m, ext.band_extremity(X), where)
            _equal(engine, engine.extremal_depth(m), ext.extremal_depth(ext.band_extremity(X)), where)
        m = ext.band_extremity(X)
        _equal(engine, engine.extremal_depth(m), ext.extremal_depth(m), name)


def _reference_cases():
    """(S [T, nS], Y [T, nY]): new curves tied to sample curves, repeated and outside the sample's range; tie-heavy;
    one time point; one sample curve."""
    rng = np.random.default_rng(2)
    S = rng.standard_normal((8, 30)).cumsum(0)
    Y = rng.standard_normal((8, 6)).cumsum(0)
    Y[:, 0] = S[:, 4]
    Y[:, 2] = Y[:, 1]
    Y[0, 3], Y[-1, 3] = S[0].min() - 1.0, S[-1].max() + 1.0
    St, Yt = _tied(rng, (6, 21)), _tied(rng, (6, 9))
    Yt[:, 0] = St[:, 3]
    return {"walks": (S, Y), "tied": (St, Yt), "T1": (rng.standard_normal((1, 12)), rng.standard_normal((1, 5))),
            "nS1": (rng.standard_normal((5, 1)), rng.standard_normal((5, 4)))}


def test_fitted_reference_calls_equal_the_doubles(engine, oracle):
    srt, ref = SortedOracleEngine(), ReferenceOracleEngine()
    for name, (S, Y) in _reference_cases().items():
        for form in ("C", "F"):
            mk = np.asfortranarray if form == "F" else np.ascontiguousarray
            where = (name, form)
            index = engine.band_sort_rows(mk(S))
            _equal(engine, index, srt.band_sort_rows(S), where)
            for J in (2, 3):
                _equal(engine, engine.band_depth_sorted_counts(index, mk(Y), J),
                       srt.band_depth_sorted_counts(srt.band_sort_rows(S), Y, J), where + (J,))
                _equal(engine, engine.band_depth_oos_counts(mk(S), mk(Y), J, True),
                       srt.band_depth_oos_counts(S, Y, J, True), where + (J,))
            host_index = ref.band_sort_rows(S)
            _equal(engine, engine.band_halfspace_sorted_counts(index, mk(Y)),
                   ref.band_halfspace_sorted_counts(host_index, Y), where)
            _equal(engine, engine.band_outlyingness_sorted(index, mk(Y)), ref.band_outlyingness_sorted(host_index, Y),
                   where)
            _equal(engine, engine.band_halfspace_counts(mk(S)), ref.band_halfspace_counts(S), where)
            _equal(engine, engine.band_outlyingness(mk(S)), ref.band_outlyingness(S), where)


def _projection_cases():
    """(S [nS, T, d], Y [nY, T, d], U [K, d]): tie-heavy curves along integer directions, walks along unit directions,
    a point cloud (T = 1), one sample curve, and d = 1."""
    rng = np.random.default_rng(3)

    def unit(K, d):
        U = rng.standard_normal((K, d))
        return U / np.linalg.norm(U, axis=1, keepdims=True)

    Ui = rng.integers(-2, 3, size=(6, 2)).astype(np.float64)
    Ui[(Ui == 0).all(axis=1), 0] = 1.0
    St, Yt = _tied(rng, (7, 5, 2)), _tied(rng, (4, 5, 2))
    Yt[0] = St[3]
    Sw = rng.standard_normal((20, 4, 3)).cumsum(1)
    Yw = rng.standard_normal((5, 4, 3)).cumsum(1)
    Yw[1] = Sw[0]
    Sc = _tied(rng, (15, 1, 3))
    return {"tied": (St, Yt, Ui), "walks": (Sw, Yw, unit(5, 3)), "cloud": (Sc, _tied(rng, (6, 1, 3)), unit(9, 3)),
            "nS1": (rng.standard_normal((1, 3, 2)), rng.standard_normal((3, 3, 2)), unit(4, 2)),
            "d1": (rng.standard_normal((9, 6, 1)), rng.standard_normal((2, 6, 1)), np.array([[1.0]]))}


def test_projected_reference_calls_equal_the_doubles(engine):
    ref = ReferenceOracleEngine()
    for name, (S, Y, U) in _projection_cases().items():
        for form in ("C", "F"):
            mk = np.asfortranarray if form == "F" else np.ascontiguousarray
            where = (name, form)
            index, host_index = engine.projection_sort_rows(mk(S), U), ref.projection_sort_rows(S, U)
            _equal(engine, index, host_index, where)
            _equal(engine, engine.projection_tukey_sorted_counts(index, mk(Y), U),
                   ref.projection_tukey_sorted_counts(host_index, Y, U), where)
            _equal(engine, engine.projection_outlyingness_sorted(index, mk(Y), U),
                   ref.projection_outlyingness_sorted(host_index, Y, U), where)
            _equal(engine, engine.projection_tukey_counts(mk(S), U), ref.projection_tukey_counts(S, U), where)
            _equal(engine, engine.projection_outlyingness(mk(S), U), ref.projection_outlyingness(S, U), where)


def test_spatial_calls_equal_the_double(engine):
    sp = SpatialOracleEngine()
    rng = np.random.default_rng(4)
    X = rng.standard_normal((8, 30)).cumsum(0)   # univariate [T, n]: its curves as rows are X.T, curve-major
    G = _tied(rng, (25, 6))                      # duplicate curves
    cases = {"univariate": (X.T[:24], X.T[24:]), "tied": (G[:20], G[19:]), "T1": (X[:1].T[:20], X[:1].T[20:]),
             "nS1": (G[:1], G[1:5])}
    for name, (S, Y) in cases.items():
        nS, F = S.shape
        host = engine.spatial_norms_of(S, Y)
        exp = sp.spatial_norms_of(S, Y)
        assert_depths(1 - host / (nS + 1), 1 - exp / (nS + 1), nS + 1, F)
        for form, A in _forms(engine, S).items():
            for Yf in (np.ascontiguousarray(Y), np.asfortranarray(Y)):
                got = engine.spatial_norms_of(A, Yf)
                assert got.dtype == np.float64 and got.tolist() == host.tolist(), (name, form)  # bit-identical
        P = np.concatenate([S, Y])
        q = np.arange(0, len(P), 3)
        assert_depths(1 - engine.spatial_norms(P, q) / len(P), 1 - sp.spatial_norms(P, q) / len(P), len(P), F)
