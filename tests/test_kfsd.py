"""Kernelized functional spatial depth (FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf,
FunctionalReference / DepthClassifier with depth='kfsd', sd_kfsd_*): KFSD(x) = 1 - r / n, r the norm of the sum of
the unit vectors (phi(x) - phi(x_j)) / ||.|| in the feature space of k(x, y) = exp(-||x - y||^2 / sigma^2).

The CPU part pins a numpy oracle in the E form the engine evaluates (r^2 = 2 A B - Q) against the per-pair definition
at 50 digits and against closed forms, and drives the host layer with a numpy test double.  The GPU part holds the
engine to the oracle within DESIGN K16's bound and checks the bit-identities K16 promises."""
import math
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
N_MAX = 32768


# ---------------------------------------------------------------------------------------------------------------
# oracles
# ---------------------------------------------------------------------------------------------------------------
def np_d2(S, Q):
    """d2[q, s] = sum_f (Q[q, f] - S[s, f])^2 by direct differences, in blocks of queries."""
    S = np.asarray(S, dtype=np.float64)
    Q = np.asarray(Q, dtype=np.float64)
    out = np.empty((len(Q), len(S)))
    blk = max(1, (1 << 24) // max(1, S.size))
    for b in range(0, len(Q), blk):
        D = S[None, :, :] - Q[b:b + blk, None, :]
        out[b:b + blk] = np.einsum('qsf,qsf->qs', D, D)
    return out


def np_bandwidth(A, quantile=0.15):
    A = np.asarray(A, dtype=np.float64)
    return float(np.quantile(np.sqrt(np_d2(A, A)[np.triu_indices(len(A), k=1)]), quantile))


def weights(e):
    return np.where(e > 0, 1.0 / np.sqrt(2.0 * np.where(e > 0, e, 1.0)), 0.0)


def kfsd_parts(S, Y, c, E=None, d2=None):
    """(A, B, Q, r) of the curves Y against the sample S in the E form: e = -expm1(c d2), w = 1 / sqrt(2 e) on e > 0,
    r = sqrt(max(2 A B - Q, 0)).  d2: the squared distances of Y to S, when known exactly."""
    S = np.asarray(S, dtype=np.float64)
    if E is None:
        E = -np.expm1(c * np_d2(S, S))
    e = -np.expm1(c * (np_d2(S, Y) if d2 is None else d2))
    w = weights(e)
    A, B = w.sum(axis=1), (w * e).sum(axis=1)
    Q = np.einsum('qj,qj->q', w @ E, w)
    return A, B, Q, np.sqrt(np.maximum(2.0 * A * B - Q, 0.0))


def np_kfsd(A, queries=None, quantile=0.15, bandwidth=None):
    A = np.asarray(A, dtype=np.float64)
    q = np.arange(len(A)) if queries is None else np.asarray(queries)
    h = np_bandwidth(A, quantile) if bandwidth is None else bandwidth
    return 1.0 - kfsd_parts(A, A[q], -1.0 / (h * h))[3] / len(A)


def mp_kfsd(A, q, h):
    """The per-pair definition at 50 digits: r^2 = sum_{i, j in J} (e_qi + e_qj - e_ij) / (2 sqrt(e_qi e_qj))."""
    import mpmath
    with mpmath.workdps(50):
        X = [[mpmath.mpf(float(v)) for v in row] for row in A]
        c = -1 / (mpmath.mpf(h) ** 2)

        def e(a, b):
            return -mpmath.expm1(c * sum((s - t) ** 2 for s, t in zip(X[a], X[b])))
        J = [j for j in range(len(A)) if e(q, j) > 0]
        eq = {j: e(q, j) for j in J}
        r2 = mpmath.mpf(0)
        for i in J:
            for j in J:
                r2 += (eq[i] + eq[j] - e(i, j)) / (2 * mpmath.sqrt(eq[i] * eq[j]))
        return float(1 - mpmath.sqrt(max(r2, 0)) / len(A))


def depth_bound(A, B, r, n_pop, F, n_sample):
    """DESIGN K16: |error| of one depth, kernel or oracle, is at most (1 / n_pop) min(sqrt(D), D / r) + u, with
    D = 2 A B (4 F + 4 n + 35) u the bound on the error of r^2."""
    D = 2.0 * A * B * (4 * F + 4 * n_sample + 35) * U
    with np.errstate(divide='ignore', invalid='ignore'):
        dr = np.where(r > 0, np.minimum(np.sqrt(D), D / np.where(r > 0, r, 1.0)), np.sqrt(D))
    return dr / n_pop + U


def assert_depths(got, exp, bound):
    got, exp = np.asarray(got), np.asarray(exp)
    err = np.abs(got - exp)
    tol = np.maximum(2 * bound, 1e-12 * np.abs(exp))
    assert (err <= tol).all(), (err.max(), tol[np.argmax(err - tol)])


def check_in_sample(got, A, h, queries=None):
    A = np.asarray(A, dtype=np.float64)
    q = np.arange(len(A)) if queries is None else np.asarray(queries)
    a, b, _, r = kfsd_parts(A, A[q], -1.0 / (h * h))
    assert_depths(got, 1.0 - r / len(A), depth_bound(a, b, r, len(A), A.shape[1], len(A)))


def _frames(F):
    return [pd.DataFrame(F[i]) for i in range(F.shape[0])]


class KfsdOracleEngine:
    """TEST DOUBLE: the engine methods the KFSD drivers call, answered by the numpy oracle, refusing non-finite input
    with SD_ERR_NONFINITE as the engine does (not an Engine, so the reference keeps a host sample and a host E).  An
    out-of-sample norm is that of the sample with the query appended, as the in-sample norm of that pooled set."""

    def __init__(self):
        self.calls = 0

    def _finite(self, *arrays):
        from statdepth_b200 import EngineError
        self.calls += 1
        for A in arrays:
            if not np.isfinite(A).all():
                raise EngineError(4, 'non-finite input')

    def modal_pair_select(self, X, k):
        self._finite(X)
        X = np.asarray(X, dtype=np.float64)
        d2 = np.sort(np_d2(X, X)[np.triu_indices(len(X), k=1)])
        return np.array([d2[k], d2[min(k + 1, len(d2) - 1)]])

    def kfsd_gram(self, S, c):
        self._finite(S)
        S = np.asarray(S, dtype=np.float64)
        return -np.expm1(c * np_d2(S, S))

    def kfsd_norms(self, X, c, queries=None):
        self._finite(X)
        X = np.asarray(X, dtype=np.float64)
        q = np.arange(len(X)) if queries is None else np.asarray(queries, dtype=np.int64)
        return kfsd_parts(X, X[q], c)[3]

    def kfsd_norms_of(self, S, E, Y, c):
        self._finite(S, Y)
        S = np.asarray(S, dtype=np.float64)
        return np.array([kfsd_parts(np.vstack([S, y[None]]), y[None], c)[3][0]
                         for y in np.asarray(Y, dtype=np.float64)])


def _install(fake, setter):
    import statdepth_b200._kfsd as kf
    setter(kf, "get_engine", lambda device=None: fake)


@pytest.fixture()
def kf_oracle(monkeypatch):
    import statdepth_b200._spatial as sp
    fake = KfsdOracleEngine()
    _install(fake, monkeypatch.setattr)
    monkeypatch.setattr(sp, "get_engine", lambda device=None: fake)  # a spatial reference holds its sample only
    return fake


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracle
# ---------------------------------------------------------------------------------------------------------------
def test_oracle_equals_50_digit_pair_loop():
    rng = np.random.default_rng(0)
    general = rng.standard_normal((9, 5))
    dups = rng.standard_normal((10, 3))
    dups[4] = dups[7]
    dups[1] = dups[7]  # three copies in the sample
    query_dup = rng.integers(-1, 2, size=(11, 2)).astype(np.float64)
    query_dup[3] = query_dup[0]  # queries 0 and 3 equal sample curves
    shifted = rng.standard_normal((8, 4)) * 1e-3 + 5.0
    for A in (general, dups, query_dup, shifted, rng.standard_normal((3, 1))):
        h = np_bandwidth(A)
        got = np_kfsd(A, bandwidth=h)
        a, b, _, r = kfsd_parts(A, A, -1.0 / (h * h))
        bound = depth_bound(a, b, r, len(A), A.shape[1], len(A))
        for q in range(len(A)):
            exp = mp_kfsd(A, q, h)
            assert abs(got[q] - exp) <= max(bound[q], 1e-15), (q, got[q], exp, bound[q])


def test_closed_forms():
    for m in (1, 2, 5, 40):
        A = np.arange(m + 1, dtype=np.float64)[:, None] * 100.0  # every pair 100 sigma apart: e = 1 exactly
        a, b, Q, r = kfsd_parts(A, A, -1.0)
        assert np.allclose(r ** 2, m + m * (m - 1) / 2, rtol=4 * U, atol=0), (m, r ** 2)  # w = 1 / sqrt(2) rounded
        assert np.allclose(np_kfsd(A, bandwidth=1.0), 1.0 - math.sqrt(m + m * (m - 1) / 2) / (m + 1), rtol=0,
                           atol=1e-15)
        B = np.zeros((m + 1, 3))
        B[0] = [0.3, -0.2, 0.1]  # one query, m identical other curves: r = m
        for h in (0.05, 1.0, 30.0):
            assert kfsd_parts(B, B[:1], -1.0 / (h * h))[3][0] == pytest.approx(m, rel=1e-14)
    assert np_kfsd(np.ones((4, 2)), bandwidth=1.0).tolist() == [1.0] * 4  # all duplicates: J empty
    assert np_kfsd(np.zeros((1, 5)), bandwidth=1.0).tolist() == [1.0]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the host layer on the test double
# ---------------------------------------------------------------------------------------------------------------
def test_univariate_frames_and_to_compute(kf_oracle):
    from statdepth_b200 import FunctionalKernelSpatialDepth
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(2)
    X = rng.standard_normal((9, 6))
    df = pd.DataFrame(X, columns=list('abcdef'))
    res = FunctionalKernelSpatialDepth([df])
    assert type(res) is _FunctionalDepthUnivariate and list(res.index) == list('abcdef')
    assert np.allclose(res.values, np_kfsd(X.T), rtol=1e-14, atol=0)
    sub = FunctionalKernelSpatialDepth([df], to_compute=['e', 'a'])
    assert list(sub.index) == ['e', 'a'] and sub.values.tolist() == res[['e', 'a']].values.tolist()
    for q in (0.0, 0.5, 1.0):
        assert np.allclose(FunctionalKernelSpatialDepth([df], quantile=q).values, np_kfsd(X.T, quantile=q),
                           rtol=1e-14, atol=0)
    assert np.allclose(FunctionalKernelSpatialDepth([df], bandwidth=0.8).values, np_kfsd(X.T, bandwidth=0.8),
                       rtol=1e-14, atol=0)
    F = rng.standard_normal((7, 5, 3))
    res = FunctionalKernelSpatialDepth(_frames(F))
    assert type(res) is _FunctionalDepthSeries and list(res.index) == list(range(7))
    assert np.allclose(res.values, np_kfsd(F.reshape(7, -1)), rtol=1e-14, atol=0)  # (t, c) order
    sub = FunctionalKernelSpatialDepth(_frames(F), to_compute=[6, 2])
    assert list(sub.index) == [6, 2] and sub.values.tolist() == res.values[[6, 2]].tolist()
    assert FunctionalKernelSpatialDepth([df.iloc[:, [0]]], bandwidth=2.0).values.tolist() == [1.0]  # n = 1


def test_refusals(kf_oracle):
    from statdepth_b200 import (DepthClassifier, FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf,
                                FunctionalReference)
    rng = np.random.default_rng(4)
    df = pd.DataFrame(rng.standard_normal((5, 4)), columns=list('wxyz'))
    wide = pd.DataFrame(np.zeros((1, N_MAX + 1)))
    bad = [
        (ValueError, lambda: FunctionalKernelSpatialDepth(df)),
        (ValueError, lambda: FunctionalKernelSpatialDepth([])),
        (ValueError, lambda: FunctionalKernelSpatialDepth([pd.DataFrame(np.zeros((4, 0)))])),
        (KeyError, lambda: FunctionalKernelSpatialDepth([df], to_compute=['q'])),
        (KeyError, lambda: FunctionalKernelSpatialDepth(_frames(np.zeros((3, 4, 2))), to_compute=[3])),
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], quantile=-0.1)),
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], quantile=float('nan'))),
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], quantile=0.3, bandwidth=1.0)),
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], bandwidth=0.0)),
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], bandwidth=float('inf'))),
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], bandwidth=1e-160)),  # sigma^2 is not normal
        (ValueError, lambda: FunctionalKernelSpatialDepth([df], bandwidth=1e160)),   # sigma^2 overflows
        (ValueError, lambda: FunctionalKernelSpatialDepth([df.iloc[:, [0]]])),       # n = 1: no pairs
        (ValueError, lambda: FunctionalKernelSpatialDepth([wide], bandwidth=1.0)),   # n above the cap
        (ValueError, lambda: FunctionalKernelSpatialDepthOf([wide.iloc[:, :2]], [wide], bandwidth=1.0)),
        (ValueError, lambda: FunctionalKernelSpatialDepthOf([pd.DataFrame(np.zeros((6, 2)))], [df])),
        (ValueError, lambda: FunctionalReference([wide], depth='kfsd', bandwidth=1.0)),
        (ValueError, lambda: FunctionalReference([df], J=3, depth='kfsd')),
        (ValueError, lambda: FunctionalReference([df], depth='kfsd', directions=4)),
        (ValueError, lambda: FunctionalReference([df], depth='kfsd', quantile=2.0)),
        (ValueError, lambda: FunctionalReference([df], depth='kfsd', quantile=0.2, bandwidth=1.0)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [df]}, depth='kfsd', directions=4)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [pd.DataFrame(np.zeros((6, 3)))]}, depth='kfsd')),
    ]
    for exc, fn in bad:
        with pytest.raises(exc):
            fn()
    for fn in (lambda: FunctionalReference([df], depth='spatial', quantile=0.2),
               lambda: FunctionalReference([df], depth='projection', bandwidth=1.0),
               lambda: DepthClassifier({0: [df], 1: [df]}, depth='mbd', bandwidth=1.0)):
        with pytest.raises(ValueError, match="'kfsd'"):
            fn()
    with pytest.raises(ValueError, match="'kfsd'"):
        FunctionalReference([df], depth='kernel')
    assert kf_oracle.calls == 0
    dup = pd.DataFrame(np.tile(rng.standard_normal((5, 1)), (1, 6)))
    with pytest.raises(ValueError, match='bandwidth='):  # every pair a duplicate: sigma = 0
        FunctionalKernelSpatialDepth([dup])
    X = rng.standard_normal((5, 4))
    X[1, 2] = np.nan
    from statdepth_b200 import EngineError
    with pytest.raises(EngineError) as ei:
        FunctionalKernelSpatialDepth([pd.DataFrame(X)])
    assert ei.value.status == 4


def test_reference_and_classifier_on_the_double(kf_oracle):
    from statdepth_b200 import (DepthClassifier, FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf,
                                FunctionalReference)
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(5)
    S = rng.standard_normal((8, 11))
    Y = rng.standard_normal((8, 3))
    Y[:, 1] = S[:, 4]  # a new curve that duplicates a sample curve
    sdf, ydf = pd.DataFrame(S), pd.DataFrame(Y, columns=['p', 'q', 'r'])
    with FunctionalReference([sdf], depth='kfsd') as ref:
        h = ref.bandwidth
        assert ref.directions is None and h == np_bandwidth(S.T)
        res = ref.depth_of([ydf])
    one = FunctionalKernelSpatialDepthOf([ydf], [sdf])
    assert type(res) is _FunctionalDepthUnivariate and list(res.index) == ['p', 'q', 'r']
    assert type(one) is _FunctionalDepthUnivariate and res.values.tolist() == one.values.tolist()
    for k in range(3):  # the out-of-sample identity, with the sample's bandwidth given
        pooled = FunctionalKernelSpatialDepth([pd.concat([sdf, ydf.iloc[:, [k]]], axis=1)], bandwidth=h)
        assert pooled.values[-1] == res.values[k]
        assert FunctionalKernelSpatialDepthOf([ydf.iloc[:, [k]]], [sdf], bandwidth=h).values[0] == res.values[k]
    with FunctionalReference([sdf], depth='kfsd', quantile=0.5) as ref:
        assert ref.bandwidth == np_bandwidth(S.T, 0.5)
    with FunctionalReference([sdf], depth='kfsd', bandwidth=0.25) as ref:
        assert ref.bandwidth == 0.25
    Fs, Fy = rng.standard_normal((6, 4, 2)), rng.standard_normal((2, 4, 2))
    with FunctionalReference(_frames(Fs), depth='kfsd') as ref:
        res = ref.depth_of(_frames(Fy))
        one = ref.depth_of(_frames(Fy[1:]))
        h = ref.bandwidth
    assert type(res) is _FunctionalDepthSeries and list(res.index) == [0, 1]
    assert one.values[0] == res.values[1]
    assert FunctionalKernelSpatialDepth(_frames(np.concatenate([Fs, Fy[:1]])), bandwidth=h).values[-1] == res.values[0]
    # two shifted classes, each with its own bandwidth
    A = rng.standard_normal((30, 16)) * 0.3
    B = A[:15] * 3.0 + np.linspace(0, 3, 16)
    refs = {'a': [pd.DataFrame(A[:15].T)], 'b': [pd.DataFrame(B.T)]}
    with DepthClassifier(refs, depth='kfsd') as clf:
        assert clf.bandwidths == {'a': np_bandwidth(A[:15]), 'b': np_bandwidth(B)}
        test = np.vstack([A[15:], A[15:] * 3.0 + np.linspace(0, 3, 16)])
        pred = clf.predict([pd.DataFrame(test.T)])
        d = clf.depths([pd.DataFrame(test.T)])
    assert pred.tolist() == ['a'] * 15 + ['b'] * 15
    exp = FunctionalKernelSpatialDepthOf([pd.DataFrame(test.T)], refs['b']).values
    assert d['b'].tolist() == exp.tolist()
    with DepthClassifier(refs, depth='kfsd', bandwidth=0.9) as clf:
        assert clf.bandwidths == {'a': 0.9, 'b': 0.9}


def test_kfsd_is_local_where_spatial_depth_is_global(kf_oracle, monkeypatch):
    """A curve midway between two tight clusters: spatial depth ranks it deepest, KFSD shallowest."""
    import statdepth_b200._spatial as sp
    from statdepth_b200 import FunctionalKernelSpatialDepth, FunctionalSpatialDepth
    rng = np.random.default_rng(6)
    A = np.vstack([rng.standard_normal((20, 8)) * 0.1 - 3.0, rng.standard_normal((20, 8)) * 0.1 + 3.0,
                   np.zeros((1, 8))])
    monkeypatch.setattr(sp, "get_engine", lambda device=None: _SpatialDouble())
    spatial = FunctionalSpatialDepth([pd.DataFrame(A.T)]).values
    kfsd = FunctionalKernelSpatialDepth([pd.DataFrame(A.T)], bandwidth=1.0).values
    assert np.argmax(spatial) == 40 and np.argmin(kfsd) == 40


class _SpatialDouble:
    """TEST DOUBLE: spatial norms by the definition (u(0) = 0)."""

    def spatial_norms(self, X, queries=None):
        X = np.asarray(X, dtype=np.float64)
        q = np.arange(len(X)) if queries is None else np.asarray(queries)
        out = []
        for i in q:
            D = X - X[i]
            nrm = np.sqrt((D * D).sum(axis=1))
            out.append(np.linalg.norm((D[nrm > 0] / nrm[nrm > 0, None]).sum(axis=0)))
        return np.array(out)


# ---------------------------------------------------------------------------------------------------------------
# CPU: two ranks (gloo) shard the queries
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _results():
    from statdepth_b200 import FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf, FunctionalReference
    rng = np.random.default_rng(11)
    uni = pd.DataFrame(rng.integers(-2, 3, size=(6, 13)).astype(np.float64))  # 13 curves: 7 + 6
    F = rng.standard_normal((9, 4, 2))
    new = pd.DataFrame(rng.standard_normal((6, 5)))
    with FunctionalReference([uni], depth='kfsd') as ref:
        ref_vals = ref.depth_of([new]).values
        one = ref.depth_of([new.iloc[:, [0]]]).values  # one new curve: one rank scores nothing
        h = np.array([ref.bandwidth])
    return dict(uni=FunctionalKernelSpatialDepth([uni]).values, frames=FunctionalKernelSpatialDepth(_frames(F)).values,
                tc=FunctionalKernelSpatialDepth(_frames(F), to_compute=[8, 0, 3]).values,
                of=FunctionalKernelSpatialDepthOf([new], [uni]).values, ref=ref_vals, one=one, h=h)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(KfsdOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(KfsdOracleEngine(), monkeypatch.setattr)
    exp = _results()
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the engine against the double and the oracle
# ---------------------------------------------------------------------------------------------------------------
def _selected(engine, A, quantile=0.15):
    from statdepth_b200._modal import _selected_bandwidth
    return _selected_bandwidth(engine, A, len(A), quantile)


@pytest.mark.gpu
def test_engine_calls_held_to_the_double(engine):
    rng = np.random.default_rng(20)
    S = rng.standard_normal((300, 37)).cumsum(axis=1)
    Y = rng.standard_normal((45, 37)).cumsum(axis=1)
    Y[3] = S[17]
    fake = KfsdOracleEngine()
    h = _selected(engine, S)
    c = -1.0 / (h * h)
    E = engine.kfsd_gram(S, c)
    Eh = E.cpu().numpy()
    assert E.is_cuda and Eh.shape == (300, 300)
    assert (Eh == Eh.T).all() and (np.diag(Eh) == 0).all()
    Ef = fake.kfsd_gram(S, c)
    assert (np.abs(Eh - Ef) <= 2 * (37 + 5) * U * Ef + 1e-300).all()
    q = [299, 0, 17, 150]
    a, b, _, r = kfsd_parts(S, S[q], c)
    bound = depth_bound(a, b, r, 1, 37, 300)  # on r itself
    assert_depths(engine.kfsd_norms(S, c, q), fake.kfsd_norms(S, c, q), bound)
    assert engine.kfsd_norms(np.asfortranarray(S), c, q).tolist() == engine.kfsd_norms(S, c, q).tolist()
    dS = engine.upload(S)
    assert engine.kfsd_norms(dS, c, q).tolist() == engine.kfsd_norms(S, c, q).tolist()
    got = engine.kfsd_norms_of(dS, E, Y, c)
    assert engine.kfsd_norms_of(S, None, Y, c).tolist() == got.tolist()  # one-shot host call
    a, b, _, r = kfsd_parts(S, Y, c)
    assert_depths(got, fake.kfsd_norms_of(S, None, Y, c), depth_bound(a, b, r, 1, 37, 301))
    assert engine.kfsd_norms_of(dS, E, Y[:0], c).shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("F", [1, 7, 256, 1024])
@pytest.mark.parametrize("n", [2, 3, 129, 2000])
def test_depths_against_oracle(engine, n, F):
    from statdepth_b200 import FunctionalKernelSpatialDepth
    A = np.random.default_rng(300 + n + F).standard_normal((n, F)).cumsum(axis=1)
    res = FunctionalKernelSpatialDepth([pd.DataFrame(A.T)]).values
    check_in_sample(res, A, _selected(engine, A))
    assert (res <= 1.0).all() and np.isfinite(res).all()


@pytest.mark.gpu
def test_multichannel_query_subset(engine):
    from statdepth_b200 import FunctionalKernelSpatialDepth
    rng = np.random.default_rng(7)
    F = rng.standard_normal((5000, 256, 3)).cumsum(axis=1)
    A = F.reshape(5000, -1)
    q = sorted(rng.choice(5000, 40, replace=False).tolist())
    res = FunctionalKernelSpatialDepth(_frames(F), to_compute=q).values
    check_in_sample(res, A, _selected(engine, A), q)


@pytest.mark.gpu
def test_far_outlier(engine):
    from statdepth_b200 import FunctionalKernelSpatialDepth
    rng = np.random.default_rng(8)
    A = rng.standard_normal((500, 8))
    A[123] += 1e8
    res = FunctionalKernelSpatialDepth([pd.DataFrame(A.T)]).values
    check_in_sample(res, A, _selected(engine, A))
    assert np.argmin(res) == 123
    # e = 1 to every other curve and Q <= m (m - 1) / 2: r^2 >= m + m (m - 1) / 2
    assert res[123] <= 1.0 - math.sqrt(499 * 500 / 2) / 500 + 1e-12


# ---------------------------------------------------------------------------------------------------------------
# GPU: bit identities, integer curves, errors
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_out_of_sample_and_query_identities(engine):
    from statdepth_b200 import FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf, FunctionalReference
    rng = np.random.default_rng(10)
    X = rng.standard_normal((96, 700)).cumsum(axis=0)
    df = pd.DataFrame(X)
    full = FunctionalKernelSpatialDepth([df]).values
    assert FunctionalKernelSpatialDepth([df]).values.tolist() == full.tolist()  # deterministic
    tc = [699, 3, 64, 65, 0, 300]
    assert FunctionalKernelSpatialDepth([df], to_compute=tc).values.tolist() == full[tc].tolist()
    S, new = df.iloc[:, :600], df.iloc[:, 600:]
    with FunctionalReference([S], depth='kfsd') as ref:
        b = ref.bandwidth
        got = ref.depth_of([new]).values
        single = [ref.depth_of([new.iloc[:, [k]]]).values[0] for k in (0, 57, 99)]
    assert got.tolist() == FunctionalKernelSpatialDepthOf([new], [S]).values.tolist()
    assert single == got[[0, 57, 99]].tolist()
    for k in (0, 57, 99):
        assert FunctionalKernelSpatialDepth([pd.concat([S, new.iloc[:, [k]]], axis=1)],
                                            bandwidth=b).values[-1] == got[k]
    F = rng.standard_normal((300, 5, 3))
    Fs, Fn = F[:280], F[280:]
    with FunctionalReference(_frames(Fs), depth='kfsd') as ref:
        got = ref.depth_of(_frames(Fn)).values
        b = ref.bandwidth
    assert got.tolist() == FunctionalKernelSpatialDepthOf(_frames(Fn), _frames(Fs)).values.tolist()
    assert FunctionalKernelSpatialDepth(_frames(np.concatenate([Fs, Fn[:1]])), bandwidth=b).values[-1] == got[0]


@pytest.mark.gpu
def test_scaling_by_powers_of_two(engine):
    from statdepth_b200 import FunctionalKernelSpatialDepth, FunctionalReference
    rng = np.random.default_rng(9)
    A = rng.standard_normal((260, 130))
    base = FunctionalKernelSpatialDepth([pd.DataFrame(A.T)]).values
    with FunctionalReference([pd.DataFrame(A.T)], depth='kfsd') as ref:
        h = ref.bandwidth
    for k in (-300, -40, 37, 400):
        As = A * 2.0 ** k
        assert FunctionalKernelSpatialDepth([pd.DataFrame(As.T)]).values.tolist() == base.tolist(), k
        with FunctionalReference([pd.DataFrame(As.T)], depth='kfsd') as ref:
            assert ref.bandwidth == h * 2.0 ** k, k


def int_kfsd_r(S, Y, c, blk=2000):
    """r of the integer-valued curves Y against the integer-valued sample S: every d2 exact through float64 Gram
    products (all integers below 2^53), E built in row blocks."""
    S = np.asarray(S, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    sqS, sqY = (S * S).sum(axis=1), (Y * Y).sum(axis=1)
    e = -np.expm1(c * ((sqY[:, None] + sqS[None, :]) - 2.0 * (Y @ S.T)))
    w = weights(e)
    A, B = w.sum(axis=1), (w * e).sum(axis=1)
    Q = np.zeros(len(Y))
    for b0 in range(0, len(S), blk):
        Eb = -np.expm1(c * ((sqS[b0:b0 + blk, None] + sqS[None, :]) - 2.0 * (S[b0:b0 + blk] @ S.T)))
        Q += np.einsum('qj,qj->q', w[:, b0:b0 + blk] @ Eb, w)
    return A, B, np.sqrt(np.maximum(2.0 * A * B - Q, 0.0))


@pytest.mark.gpu
def test_integer_curves_and_a_reference_of_20000(engine):
    from statdepth_b200 import FunctionalKernelSpatialDepth, FunctionalReference
    rng = np.random.default_rng(13)
    A = rng.integers(-4, 5, size=(3000, 24)).astype(np.float64)
    q = [0, 1, 1500, 2999]
    res = FunctionalKernelSpatialDepth([pd.DataFrame(A.T)], to_compute=q, bandwidth=6.0).values
    a, b, r = int_kfsd_r(A, A[q], -1.0 / 36.0)
    assert_depths(res, 1.0 - r / 3000, depth_bound(a, b, r, 3000, 24, 3000))
    # 20 000 sample curves: W row blocks of 6 656 queries, so 14 000 new curves span three of them
    S = rng.integers(-4, 5, size=(20_000, 16)).astype(np.float64)
    Y = rng.integers(-5, 6, size=(14_000, 16)).astype(np.float64)
    with FunctionalReference([pd.DataFrame(S.T)], depth='kfsd') as ref:
        h = ref.bandwidth
        got = ref.depth_of([pd.DataFrame(Y.T)]).values
        ks = (0, 6655, 6656, 13_312, 13_999)
        for k in ks:
            assert ref.depth_of([pd.DataFrame(Y[[k]].T)]).values[0] == got[k], k
        again = ref.depth_of([pd.DataFrame(Y[list(ks)].T)]).values
    assert again.tolist() == got[list(ks)].tolist()
    a, b, r = int_kfsd_r(S, Y[list(ks)], -1.0 / (h * h))
    assert_depths(got[list(ks)], 1.0 - r / 20_001, depth_bound(a, b, r, 20_001, 16, 20_000))


@pytest.mark.gpu
def test_errors(engine):
    from statdepth_b200 import EngineError
    rng = np.random.default_rng(14)
    A = rng.standard_normal((260, 13))
    for call in (lambda: engine.kfsd_norms(A * 1e160, -1.0), lambda: engine.kfsd_gram(A * 1e160, -1.0),
                 lambda: engine.kfsd_norms_of(A, None, A[:2] * 1e160, -1.0)):
        with pytest.raises(EngineError) as ei:
            call()
        assert ei.value.status == 5
    B = A.copy()
    B[3, 3] = np.nan
    for call in (lambda: engine.kfsd_norms(B, -1.0), lambda: engine.kfsd_gram(B, -1.0),
                 lambda: engine.kfsd_norms_of(A, None, B[2:4], -1.0),
                 lambda: engine.kfsd_norms_of(B, None, A[:2], -1.0)):
        with pytest.raises(EngineError) as ei:
            call()
        assert ei.value.status == 4
    wide = np.zeros((N_MAX + 1, 1))
    for call in (lambda: engine.kfsd_norms(wide, -1.0, [0]), lambda: engine.kfsd_norms_of(wide, None, wide[:1], -1.0),
                 lambda: engine.kfsd_gram(wide, -1.0)):
        with pytest.raises(EngineError) as ei:
            call()
        assert ei.value.status == 6
    for c in (0.0, 1.0, -math.inf, math.nan):
        with pytest.raises(EngineError) as ei:
            engine.kfsd_norms(A, c, [0])
        assert ei.value.status == 1
