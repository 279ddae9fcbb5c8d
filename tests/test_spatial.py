"""Functional spatial depth (FunctionalSpatialDepth, FunctionalSpatialDepthOf, FunctionalReference / DepthClassifier
with depth='spatial', sd_spatial_norms_*): SD(x) = 1 - || sum_{x_j != x} u(x_j - x) || / n_pop, u(v) = v / ||v||,
a curve being the vector of its T d values.

The CPU part pins a numpy oracle against a per-pair loop and against the point-cloud L1 oracle, and drives the host
layer with a numpy test double.  The GPU part pins the CUDA engine to the oracle within DESIGN K14's bar: relative
1e-12, or the absolute bound 2 (n + F / 2 + 3) 2^-53 (twice the worst-case error of either side) where depths are
near 0; and it checks the bit-identities K14 promises."""
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------
# oracles
# ---------------------------------------------------------------------------------------------------------------
def np_spatial_r(S, Q, block=8192):
    """r of every row of Q against the rows of S (rows of S equal to q contribute 0), float64 numpy."""
    S = np.asarray(S, dtype=np.float64)
    Q = np.asarray(Q, dtype=np.float64)
    out = np.empty(len(Q))
    for i, q in enumerate(Q):
        v = np.zeros(S.shape[1])
        for b in range(0, len(S), block):
            D = S[b:b + block] - q
            nrm = np.sqrt(np.einsum('ij,ij->i', D, D))
            w = np.divide(1.0, nrm, out=np.zeros_like(nrm), where=nrm > 0)
            v += w @ D
        out[i] = np.sqrt(v @ v)
    return out


def loop_spatial_r(A, q):
    """The definition, one pair at a time."""
    x = A[q]
    s = np.zeros(A.shape[1])
    for j in range(A.shape[0]):
        d = A[j] - x
        nrm = float(np.sqrt(sum(float(t) * float(t) for t in d)))
        if nrm > 0:
            s += d / nrm
    return float(np.sqrt(s @ s))


def np_spatial_depth(A, queries=None):
    A = np.asarray(A, dtype=np.float64)
    q = np.arange(len(A)) if queries is None else np.asarray(queries)
    return 1.0 - np_spatial_r(A, A[q]) / len(A)


def assert_depths(got, exp, n, F):
    """K14's bar: relative 1e-12, or the absolute bound for depths near 0."""
    got, exp = np.asarray(got), np.asarray(exp)
    bound = np.maximum(1e-12 * np.abs(exp), 2 * (n + F / 2 + 3) * 2.0 ** -53)
    err = np.abs(got - exp)
    assert (err <= bound).all(), (err.max(), bound[np.argmax(err - bound)])


def _frames(F):
    return [pd.DataFrame(F[i]) for i in range(F.shape[0])]


class SpatialOracleEngine:
    """TEST DOUBLE: the engine methods the spatial drivers call, answered by the numpy oracle, refusing non-finite
    input with SD_ERR_NONFINITE as the engine does (no `_dev` methods: the reference keeps a host sample)."""

    def __init__(self):
        self.calls = 0

    def _finite(self, *arrays):
        from statdepth_b200 import EngineError
        self.calls += 1
        for A in arrays:
            if not np.isfinite(A).all():
                raise EngineError(4, 'non-finite input')

    def spatial_norms(self, X, queries=None):
        self._finite(X)
        X = np.asarray(X, dtype=np.float64)
        q = np.arange(len(X)) if queries is None else np.asarray(queries, dtype=np.int64)
        return np_spatial_r(X, X[q])

    def spatial_norms_of(self, S, Y):
        self._finite(S, Y)
        return np_spatial_r(S, Y)


def _install(fake, setter):
    import statdepth_b200._spatial as sp
    setter(sp, "get_engine", lambda device=None: fake)


@pytest.fixture()
def sp_oracle(monkeypatch):
    fake = SpatialOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracle
# ---------------------------------------------------------------------------------------------------------------
def test_oracle_equals_pairwise_loop():
    rng = np.random.default_rng(0)
    cases = [rng.standard_normal((1, 5)), rng.standard_normal((2, 3)), np.zeros((2, 4)),
             rng.integers(-1, 2, size=(12, 3)).astype(np.float64), rng.standard_normal((9, 1)),
             rng.standard_normal((15, 7)) * 1e-3 + 5.0]
    dup = rng.standard_normal((6, 4))
    cases.append(np.vstack([dup, dup[:3], dup[:1]]))
    for A in cases:
        r = np_spatial_r(A, A)
        for q in range(len(A)):
            assert abs(r[q] - loop_spatial_r(A, q)) <= 1e-13 * max(1.0, len(A))
    assert np_spatial_depth(np.ones((1, 3))).tolist() == [1.0]          # n = 1: only itself
    assert np_spatial_depth(np.array([[0.0], [2.0]])).tolist() == [0.5, 0.5]  # n = 2: one unit vector each
    assert np_spatial_depth(np.zeros((5, 2))).tolist() == [1.0] * 5      # all duplicates


def test_oracle_equals_pointcloud_l1_depth():
    from oracle import np_oracle
    rng = np.random.default_rng(1)
    for n, F in [(5, 1), (40, 3), (64, 16), (2, 7)]:
        A = rng.standard_normal((n, F))
        assert np.allclose(np_spatial_depth(A), np_oracle.l1_depth(A), rtol=1e-12, atol=0)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the host layer on the test double
# ---------------------------------------------------------------------------------------------------------------
def test_univariate_labels_and_to_compute(sp_oracle):
    from statdepth_b200 import FunctionalSpatialDepth
    from statdepth_b200.depth import _FunctionalDepthUnivariate
    rng = np.random.default_rng(2)
    X = rng.standard_normal((9, 6))
    df = pd.DataFrame(X, columns=list('abcdef'))
    res = FunctionalSpatialDepth([df])
    assert type(res) is _FunctionalDepthUnivariate and list(res.index) == list('abcdef')
    assert np.allclose(res.values, np_spatial_depth(X.T), rtol=1e-14)
    sub = FunctionalSpatialDepth([df], to_compute=['e', 'a'])
    assert list(sub.index) == ['e', 'a'] and np.allclose(sub.values, res[['e', 'a']].values, rtol=1e-14)


def test_frames_labels_and_to_compute(sp_oracle):
    from statdepth_b200 import FunctionalSpatialDepth
    from statdepth_b200.depth import _FunctionalDepthSeries
    rng = np.random.default_rng(3)
    F = rng.standard_normal((7, 5, 3))
    res = FunctionalSpatialDepth(_frames(F))
    assert type(res) is _FunctionalDepthSeries and list(res.index) == list(range(7))
    assert np.allclose(res.values, np_spatial_depth(F.reshape(7, -1)), rtol=1e-14)  # (t, c) order
    sub = FunctionalSpatialDepth(_frames(F), to_compute=[6, 2])
    assert list(sub.index) == [6, 2] and np.allclose(sub.values, res.values[[6, 2]], rtol=1e-14)


def test_refusals_make_no_engine_call(sp_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalReference, FunctionalSpatialDepth, FunctionalSpatialDepthOf
    rng = np.random.default_rng(4)
    df = pd.DataFrame(rng.standard_normal((5, 4)), columns=list('wxyz'))
    bad = [
        (ValueError, lambda: FunctionalSpatialDepth(df)),
        (ValueError, lambda: FunctionalSpatialDepth([])),
        (ValueError, lambda: FunctionalSpatialDepth([pd.DataFrame(np.zeros((0, 3)))])),
        (ValueError, lambda: FunctionalSpatialDepth([pd.DataFrame(np.zeros((4, 0)))])),
        (ValueError, lambda: FunctionalSpatialDepth([pd.DataFrame(np.zeros((4, 2))), pd.DataFrame(np.zeros((5, 2)))])),
        (ValueError, lambda: FunctionalSpatialDepth([pd.DataFrame(np.zeros((4, 2))), pd.DataFrame(np.zeros((4, 3)))])),
        (KeyError, lambda: FunctionalSpatialDepth([df], to_compute=['q'])),
        (KeyError, lambda: FunctionalSpatialDepth(_frames(np.zeros((3, 4, 2))), to_compute=[3])),
        (ValueError, lambda: FunctionalSpatialDepthOf([pd.DataFrame(np.zeros((6, 2)))], [df])),
        (ValueError, lambda: FunctionalSpatialDepthOf(_frames(np.zeros((2, 5, 3))), _frames(np.zeros((3, 5, 2))))),
        (ValueError, lambda: FunctionalReference([df], J=3, depth='spatial')),
        (ValueError, lambda: FunctionalReference([df], depth='spatial', directions=4)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [df]}, depth='spatial', directions=4)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [pd.DataFrame(np.zeros((6, 3)))]}, depth='spatial')),
    ]
    for exc, fn in bad:
        with pytest.raises(exc):
            fn()
    assert sp_oracle.calls == 0
    with FunctionalReference([df], depth='spatial') as ref:
        with pytest.raises(ValueError):
            ref.depth_of([pd.DataFrame(np.zeros((6, 2)))])
        with pytest.raises(ValueError):
            ref.depth_of(_frames(np.zeros((2, 5, 1))))
    assert sp_oracle.calls == 0
    X = rng.standard_normal((5, 4))
    X[1, 2] = np.nan
    from statdepth_b200 import EngineError
    with pytest.raises(EngineError) as ei:
        FunctionalSpatialDepth([pd.DataFrame(X)])
    assert ei.value.status == 4


def test_reference_and_classifier_on_the_double(sp_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalReference, FunctionalSpatialDepth, FunctionalSpatialDepthOf
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(5)
    S = rng.standard_normal((8, 11))
    Y = rng.standard_normal((8, 3))
    Y[:, 1] = S[:, 4]  # a new curve that duplicates a sample curve
    sdf, ydf = pd.DataFrame(S), pd.DataFrame(Y, columns=['p', 'q', 'r'])
    with FunctionalReference([sdf], depth='spatial') as ref:
        assert ref.directions is None
        res = ref.depth_of([ydf])
    one = FunctionalSpatialDepthOf([ydf], [sdf])
    assert type(res) is _FunctionalDepthUnivariate and list(res.index) == ['p', 'q', 'r']
    assert type(one) is _FunctionalDepthUnivariate and res.values.tolist() == one.values.tolist()
    for k in range(3):
        pooled = FunctionalSpatialDepth([pd.concat([sdf, ydf.iloc[:, [k]]], axis=1)])
        assert np.isclose(pooled.values[-1], res.values[k], rtol=1e-14, atol=0)
    Fs, Fy = rng.standard_normal((6, 4, 2)), rng.standard_normal((2, 4, 2))
    with FunctionalReference(_frames(Fs), depth='spatial') as ref:
        res = ref.depth_of(_frames(Fy))
        one = ref.depth_of(_frames(Fy[1:]))  # one frame against a multivariate reference is one curve
    assert type(res) is _FunctionalDepthSeries and list(res.index) == [0, 1]
    assert one.values[0] == res.values[1]
    exp = 1.0 - np_spatial_r(Fs.reshape(6, -1), Fy.reshape(2, -1)) / 7
    assert np.allclose(res.values, exp, rtol=1e-14)
    # two shifted classes: every curve goes to its own class
    A = rng.standard_normal((30, 16)) * 0.3
    B = A[:15] + np.linspace(0, 3, 16)
    clf = DepthClassifier({'a': [pd.DataFrame(A[:15].T)], 'b': [pd.DataFrame(B.T)]}, depth='spatial')
    test = np.vstack([A[15:], A[15:] + np.linspace(0, 3, 16)])
    pred = clf.predict([pd.DataFrame(test.T)])
    assert clf.directions is None and pred.tolist() == ['a'] * 15 + ['b'] * 15
    clf.close()


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
    from statdepth_b200 import FunctionalReference, FunctionalSpatialDepth, FunctionalSpatialDepthOf
    rng = np.random.default_rng(11)
    uni = pd.DataFrame(rng.integers(-2, 3, size=(6, 13)).astype(np.float64))  # 13 curves: 7 + 6
    F = rng.standard_normal((9, 4, 2))
    new = pd.DataFrame(rng.standard_normal((6, 5)))
    with FunctionalReference([uni], depth='spatial') as ref:
        ref_vals = ref.depth_of([new]).values
        one = ref.depth_of([new.iloc[:, [0]]]).values  # one new curve: one rank scores nothing
    return dict(uni=FunctionalSpatialDepth([uni]).values, frames=FunctionalSpatialDepth(_frames(F)).values,
                tc=FunctionalSpatialDepth(_frames(F), to_compute=[8, 0, 3]).values,
                of=FunctionalSpatialDepthOf([new], [uni]).values, ref=ref_vals, one=one)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(SpatialOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(SpatialOracleEngine(), monkeypatch.setattr)
    exp = _results()
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("F", [1, 7, 1024])
@pytest.mark.parametrize("n", [1, 2, 3, 257, 2000])
def test_sizes_against_oracle(engine, n, F):
    A = np.random.default_rng(100 + n + F).standard_normal((n, F)).cumsum(axis=1)
    q = np.arange(n) if n * F <= 300_000 else np.random.default_rng(n).choice(n, 64, replace=False)
    r = engine.spatial_norms(A, q)
    assert_depths(1 - r / n, 1 - np_spatial_r(A, A[q]) / n, n, F)
    if n == 1:
        assert r.tolist() == [0.0]


@pytest.mark.gpu
def test_multichannel_public_api(engine):
    from statdepth_b200 import FunctionalSpatialDepth
    rng = np.random.default_rng(7)
    F = rng.standard_normal((500, 64, 3)).cumsum(axis=1)
    res = FunctionalSpatialDepth(_frames(F))
    assert_depths(res.values, np_spatial_depth(F.reshape(500, -1)), 500, 192)
    F = rng.standard_normal((5000, 256, 3)).cumsum(axis=1)
    q = sorted(rng.choice(5000, 40, replace=False).tolist())
    res = FunctionalSpatialDepth(_frames(F), to_compute=q)
    A = F.reshape(5000, -1)
    assert_depths(res.values, 1 - np_spatial_r(A, A[q]) / 5000, 5000, 768)


@pytest.mark.gpu
def test_univariate_20000_x_1024_sampled(engine):
    from statdepth_b200 import FunctionalSpatialDepth
    rng = np.random.default_rng(8)
    X = rng.standard_normal((1024, 20_000)).cumsum(axis=0)  # C order [T, n]: SD_LAYOUT_TN, transposed on the device
    cols = sorted(rng.choice(20_000, 48, replace=False).tolist())
    res = FunctionalSpatialDepth([pd.DataFrame(X)], to_compute=cols)
    assert_depths(res.values, 1 - np_spatial_r(X.T, X.T[cols]) / 20_000, 20_000, 1024)
    # the F-ordered memory of a column-built DataFrame (SD_LAYOUT_NT) gives the same bits
    assert engine.spatial_norms(np.ascontiguousarray(X.T), cols).tolist() == engine.spatial_norms(X.T, cols).tolist()


@pytest.mark.gpu
def test_data_shapes(engine):
    rng = np.random.default_rng(9)
    G = rng.integers(-1, 2, size=(400, 6)).astype(np.float64)  # 729 cells: many duplicates
    assert_depths(1 - engine.spatial_norms(G) / 400, np_spatial_depth(G), 400, 6)
    assert (1 - engine.spatial_norms(np.full((50, 33), 2.5)) / 50).tolist() == [1.0] * 50
    B = rng.standard_normal((300, 40))
    B[17] += 1e8  # far outlier: W X - (sum W) x_q would cancel here
    exp = np_spatial_depth(B)
    got = 1 - engine.spatial_norms(B) / 300
    assert_depths(got, exp, 300, 40)
    assert got[17] < 2.0 / 300 and exp[17] < 2.0 / 300  # every unit vector points back to the bulk: r = n - 1
    A = rng.standard_normal((260, 130))
    base = engine.spatial_norms(A)
    for k in (-300, -40, 37, 400):
        assert engine.spatial_norms(A * 2.0 ** k).tolist() == base.tolist(), k
    for scale in (1e150, 1e-150):
        assert_depths(1 - engine.spatial_norms(A * scale) / 260, 1 - np_spatial_r(A, A) / 260, 260, 130)
    from statdepth_b200 import EngineError
    with pytest.raises(EngineError) as ei:
        engine.spatial_norms(A * 1e160)
    assert ei.value.status == 5
    A[3, 3] = np.nan
    for call in (lambda: engine.spatial_norms(A), lambda: engine.spatial_norms_of(A, A[:2] * 0),
                 lambda: engine.spatial_norms_of(A * 0, A[:2])):
        with pytest.raises(EngineError) as ei:
            call()
        assert ei.value.status == 4


@pytest.mark.gpu
def test_determinism_and_bit_identities(engine):
    from statdepth_b200 import (FunctionalReference, FunctionalSpatialDepth, FunctionalSpatialDepthOf,
                                PointcloudDepth)
    rng = np.random.default_rng(10)
    X = rng.standard_normal((96, 700)).cumsum(axis=0)
    df = pd.DataFrame(X)
    full = FunctionalSpatialDepth([df]).values
    assert FunctionalSpatialDepth([df]).values.tolist() == full.tolist()
    tc = [699, 3, 64, 65, 0, 300]
    assert FunctionalSpatialDepth([df], to_compute=tc).values.tolist() == full[tc].tolist()
    S, new = df.iloc[:, :600], df.iloc[:, 600:]
    with FunctionalReference([S], depth='spatial') as ref:
        got = ref.depth_of([new]).values
        single = [ref.depth_of([new.iloc[:, [k]]]).values[0] for k in (0, 57, 99)]
    assert got.tolist() == FunctionalSpatialDepthOf([new], [S]).values.tolist()
    assert single == got[[0, 57, 99]].tolist()
    for k in (0, 57, 99):
        pooled = FunctionalSpatialDepth([pd.concat([S, new.iloc[:, [k]]], axis=1)]).values[-1]
        assert pooled == got[k]
    F = rng.standard_normal((300, 5, 3))
    Fs, Fn = F[:280], F[280:]
    with FunctionalReference(_frames(Fs), depth='spatial') as ref:
        got = ref.depth_of(_frames(Fn)).values
    assert got.tolist() == FunctionalSpatialDepthOf(_frames(Fn), _frames(Fs)).values.tolist()
    assert FunctionalSpatialDepth(_frames(np.concatenate([Fs, Fn[:1]]))).values[-1] == got[0]
    P = rng.standard_normal((400, 12))
    l1 = PointcloudDepth(pd.DataFrame(P), containment='l1').values
    sp = FunctionalSpatialDepth(_frames(P.reshape(400, 4, 3))).values
    assert np.allclose(sp, l1, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_classifier_separates_shifted_classes(engine):
    from statdepth_b200 import DepthClassifier
    rng = np.random.default_rng(12)
    t = np.linspace(0, 1, 128)
    a = rng.standard_normal((128, 400)).cumsum(axis=0) * 0.02
    b = rng.standard_normal((128, 400)).cumsum(axis=0) * 0.02 + 0.5 * np.sin(6 * t)[:, None]
    with DepthClassifier({'a': [pd.DataFrame(a[:, :300])], 'b': [pd.DataFrame(b[:, :300])]}, depth='spatial') as clf:
        pred = clf.predict([pd.DataFrame(np.hstack([a[:, 300:], b[:, 300:]]))])
    acc = (np.array(pred.tolist()) == np.array(['a'] * 100 + ['b'] * 100)).mean()
    assert acc >= 0.95, acc


@pytest.mark.gpu
def test_reference_spans_several_w_row_blocks(engine):
    from statdepth_b200 import FunctionalReference
    rng = np.random.default_rng(13)
    S = rng.standard_normal((1024, 100_000)).astype(np.float64)
    Y = rng.standard_normal((1024, 2000)) * 1.1
    with FunctionalReference([pd.DataFrame(S)], depth='spatial') as ref:
        got = ref.depth_of([pd.DataFrame(Y)]).values  # W: 2000 x 100 000 doubles = 1.6 GB, two row blocks
        last = ref.depth_of([pd.DataFrame(Y[:, [1999]])]).values[0]
    assert last == got[1999]  # the second row block gives the bits a call of its own gives
    q = [0, 1, 1279, 1280, 1281, 1999]
    assert_depths(got[q], 1 - np_spatial_r(S.T, Y.T[q]) / 100_001, 100_001, 1024)
