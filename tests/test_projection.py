"""Random projection depths (ProjectionDepth, FunctionalProjectionDepth and the sd_projection_* / sd_band_outlyingness
entry points).

The contract: curves F [N, T, d] (a cloud is T = 1) and directions U [K, d] give the rows
y_k(i, t) = (...(U[k,0] F[i,t,0]) + U[k,1] F[i,t,1]) + ...) + U[k,d-1] F[i,t,d-1], correctly rounded in this order.
Random Tukey: R(i) = sum_t min_k (N - max(b, a)), b / a the other projections strictly below / above; depth
R / (T N).  Projection: O_t(i) = max_k |y - med| / MAD with med = np.median of the row and MAD = np.median(|y - med|)
(MAD = 0: 0 where y == med, else inf); depth 1 / (1 + O), averaged over t for curves.

The CPU part pins the numpy oracle to brute-force definitions, checks the kernel's selection of the MAD and that
random Tukey depth with cell-interior directions is the exact halfspace depth, and drives the host layer with an
engine answering from numpy; the GPU part pins the CUDA engine to the oracle bit for bit and to invariants."""
import math
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

from test_halfspace import np_band_halfspace, np_halfspace_exact

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------
# numpy oracle
# ---------------------------------------------------------------------------------------------------------------
def np_project(F, U):
    """Y [T, K, N] in the engine's fixed order."""
    F = np.asarray(F, dtype=np.float64)
    U = np.asarray(U, dtype=np.float64)
    Y = U[None, :, 0, None] * F[:, :, 0].T[:, None, :]
    for c in range(1, U.shape[1]):
        Y = Y + U[None, :, c, None] * F[:, :, c].T[:, None, :]
    return Y


def np_tukey_counts(F, U):
    Y = np_project(F, U)
    T, K, N = Y.shape
    R = np.zeros(N, dtype=np.int64)
    for t in range(T):
        m = np.full(N, N, dtype=np.int64)
        for k in range(K):
            s = np.sort(Y[t, k])
            b = np.searchsorted(s, Y[t, k], 'left')
            a = N - np.searchsorted(s, Y[t, k], 'right')
            m = np.minimum(m, N - np.maximum(b, a))
        R += m
    return R


def np_medmad(Y):
    """med, MAD along the last axis."""
    med = np.median(Y, axis=-1)
    return med, np.median(np.abs(Y - med[..., None]), axis=-1)


def np_outlyingness_rows(Y, med, mad):
    with np.errstate(divide='ignore', invalid='ignore'):
        O = np.abs(Y - med[..., None]) / mad[..., None]
    return np.where(mad[..., None] == 0, np.where(Y == med[..., None], 0.0, np.inf), O)


def np_outlyingness(F, U):
    """O [T, N], med [T, K], MAD [T, K]."""
    Y = np_project(F, U)
    med, mad = np_medmad(Y)
    return np_outlyingness_rows(Y, med, mad).max(axis=1), med, mad


def cell_directions(P):
    """Integer directions, one strictly inside every cell of the arrangement of the normals (-v_y, v_x) of all
    differences v of the integer cloud P [n, 2]: sums of angularly consecutive primitive normals."""
    P = np.asarray(np.round(P), dtype=np.int64)
    V = np.unique((P[:, None, :] - P[None, :, :]).reshape(-1, 2), axis=0)
    V = V[(V != 0).any(axis=1)]
    if len(V) == 0:
        return np.array([[1.0, 0.0]])
    V = V // np.gcd(V[:, 0], V[:, 1])[:, None]
    Nrm = np.unique(np.concatenate([np.stack([-V[:, 1], V[:, 0]], 1), np.stack([V[:, 1], -V[:, 0]], 1)]), axis=0)
    Nrm = Nrm[np.argsort(np.arctan2(Nrm[:, 1], Nrm[:, 0]))]
    if len(Nrm) == 2:  # one line: the two half-planes' directions
        a = Nrm[0]
        return np.array([[-a[1], a[0]], [a[1], -a[0]]], dtype=np.float64)
    return (Nrm + np.roll(Nrm, -1, axis=0)).astype(np.float64)


def kernel_medmad(s):
    """medmad_kernel (csrc/projection.cu) restated: the median, then the MAD by a binary search over how many of
    the k + 1 smallest deviations come from L = |s[m-1..0] - med|."""
    n = len(s)
    h = n // 2
    med = s[h] if n % 2 else (s[h - 1] + s[h]) / 2.0
    m = int(np.searchsorted(s, med, 'left'))

    def kth(k):
        lo, hi = max(0, k + 1 - (n - m)), min(k + 1, m)
        while lo < hi:
            i = (lo + hi) // 2
            j = k + 1 - i
            if j > 0 and i < m and abs(s[m + j - 1] - med) > abs(s[m - 1 - i] - med):
                lo = i + 1
            else:
                hi = i
        j = k + 1 - lo
        v = abs(s[m - lo] - med) if lo > 0 else None
        if j > 0:
            r = abs(s[m + j - 1] - med)
            if v is None or r > v:
                v = r
        return v

    return med, (kth(h) if n % 2 else (kth(h - 1) + kth(h)) / 2.0)


def _tied(rng, shape):
    X = rng.integers(-4, 4, size=shape).astype(np.float64) * 0.5
    X[(X == 0) & (rng.random(shape) < 0.5)] = -0.0
    return X


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracle
# ---------------------------------------------------------------------------------------------------------------
def test_oracle_equals_brute_force():
    rng = np.random.default_rng(1)
    for case in range(120):
        N, T, d, K = (int(v) for v in rng.integers(1, [12, 4, 5, 6]))
        F = _tied(rng, (N, T, d)) if case % 2 else rng.standard_normal((N, T, d))
        U = rng.integers(-2, 3, size=(K, d)).astype(np.float64)
        U[(U == 0).all(axis=1), 0] = 1.0
        Y = np_project(F, U)
        R = np.zeros(N, dtype=np.int64)
        O = np.zeros((T, N))
        for t in range(T):
            for k in range(K):
                y = np.empty(N)
                for i in range(N):  # the fixed-order sum
                    acc = U[k, 0] * F[i, t, 0]
                    for c in range(1, d):
                        acc = acc + U[k, c] * F[i, t, c]
                    y[i] = acc
                assert np.array_equal(Y[t, k], y)
            h = [min(min(sum(Y[t, k, j] <= Y[t, k, i] for j in range(N)),
                         sum(Y[t, k, j] >= Y[t, k, i] for j in range(N))) for k in range(K)) for i in range(N)]
            R += np.array(h, dtype=np.int64)
            for k in range(K):  # sort-based median and MAD
                s = sorted(Y[t, k])
                med = s[N // 2] if N % 2 else (s[N // 2 - 1] + s[N // 2]) / 2
                dev = sorted(abs(v - med) for v in Y[t, k])
                mad = dev[N // 2] if N % 2 else (dev[N // 2 - 1] + dev[N // 2]) / 2
                for i in range(N):
                    o = abs(Y[t, k, i] - med) / mad if mad else (0.0 if Y[t, k, i] == med else math.inf)
                    O[t, i] = max(O[t, i], o)
        assert np_tukey_counts(F, U).tolist() == R.tolist()
        assert np.array_equal(np_outlyingness(F, U)[0], O)


def test_kernel_selection_equals_np_median():
    rng = np.random.default_rng(2)
    for it in range(1500):
        n = int(rng.integers(1, 60))
        kind = it % 3
        y = (rng.standard_normal(n) if kind == 0 else rng.integers(-3, 4, n).astype(float) if kind == 1
             else rng.standard_normal(n) * 10.0 ** rng.integers(-300, 300))
        med, mad = kernel_medmad(np.sort(y))
        em = np.median(y)
        assert med == em and mad == np.median(np.abs(y - em)) and not np.signbit(mad), y


def _grid_cloud(rng, n, lo=-3, hi=3):
    P = rng.integers(lo, hi + 1, size=(n, 2)).astype(np.float64)
    P[:n // 3, 1] = 2 * P[:n // 3, 0] + 1
    return P


def test_tukey_with_cell_directions_is_exact_halfspace():
    rng = np.random.default_rng(3)
    for case in range(300):
        n = int(rng.integers(1, 25))
        if case % 3 == 0:  # collinear, duplicates
            x = rng.integers(-3, 4, n)
            P = np.stack([x, 2 * x - 1], 1).astype(np.float64)
        else:
            P = _grid_cloud(rng, n)
        U = cell_directions(P)
        assert np_tukey_counts(P[:, None, :], U).tolist() == np_halfspace_exact(P).tolist(), P
        Ur = rng.standard_normal((5, 2))
        assert (np_tukey_counts(P[:, None, :], Ur) >= np_halfspace_exact(P)).all()  # an upper bound


# ---------------------------------------------------------------------------------------------------------------
# CPU: host layer on a test double
# ---------------------------------------------------------------------------------------------------------------
class ProjectionOracleEngine:
    """TEST DOUBLE: the engine methods the projection drivers call, answered by numpy, refusing non-finite input
    with SD_ERR_NONFINITE as the engine does."""

    def __init__(self):
        self.calls = 0

    def _finite(self, A):
        from statdepth_b200 import EngineError
        self.calls += 1
        if not np.isfinite(A).all():
            raise EngineError(4, 'non-finite input')

    def projection_tukey_counts(self, F, U):
        self._finite(F)
        return np_tukey_counts(F, U)

    def projection_outlyingness(self, F, U):
        self._finite(F)
        return np_outlyingness(F, U)[0]

    def band_outlyingness(self, X):
        X = np.asarray(X, dtype=np.float64)
        self._finite(X)
        med, mad = np_medmad(X)
        return np_outlyingness_rows(X, med, mad)

    def band_halfspace_counts(self, X):
        self._finite(X)
        return np_band_halfspace(X)


def _install(fake, setter):
    import statdepth_b200._halfspace as h
    import statdepth_b200._projection as p
    setter(h, "get_engine", lambda device=None: fake)
    setter(p, "get_engine", lambda device=None: fake)


@pytest.fixture()
def pj_oracle(monkeypatch):
    fake = ProjectionOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _unit(U):
    return np.stack([u / np.linalg.norm(u) for u in U])


def test_pointcloud_kinds_labels_and_draw(pj_oracle):
    from statdepth_b200 import ProjectionDepth
    from statdepth_b200._projection import draw_directions
    from statdepth_b200.depth import _PointwiseDepth
    rng = np.random.default_rng(5)
    P = rng.standard_normal((40, 4))
    labels = ['p%d' % i for i in range(40)]
    df = pd.DataFrame(P, index=labels)
    U = draw_directions(4, 25, seed=7)
    assert np.array_equal(U, _unit(np.random.default_rng(7).standard_normal((25, 4))))
    assert draw_directions(4).shape == (1000, 4)
    assert np.array_equal(draw_directions(4), _unit(np.random.default_rng(0).standard_normal((1000, 4))))
    d = ProjectionDepth(df, directions=25, seed=7)
    assert isinstance(d, _PointwiseDepth) and list(d.index) == labels
    assert np.array_equal(d.values, 1.0 / (1.0 + np_outlyingness(P[:, None, :], U)[0][0]))
    assert np.array_equal(ProjectionDepth(df, directions=U).values, d.values)
    assert np.array_equal(ProjectionDepth(df, directions=25, seed=7).values, d.values)  # same seed, same depths
    assert not np.array_equal(ProjectionDepth(df, directions=25, seed=8).values, d.values)
    t = ProjectionDepth(df, kind='tukey', directions=U)
    assert t.values.tolist() == (np_tukey_counts(P[:, None, :], U) / 40.0).tolist()
    sub = ProjectionDepth(df, kind='tukey', directions=U, to_compute=['p7', 'p0', 'p7'])
    assert list(sub.index) == ['p7', 'p0', 'p7'] and sub.values.tolist() == t.loc[['p7', 'p0', 'p7']].values.tolist()
    assert d.deepest().values[0] == d.values.max()
    Q = _grid_cloud(rng, 30)  # integer cloud, cell directions: the exact halfspace depth
    assert (ProjectionDepth(pd.DataFrame(Q), kind='tukey', directions=cell_directions(Q)).values.tolist()
            == (np_halfspace_exact(Q) / 30.0).tolist())


def test_functional_kinds(pj_oracle):
    from statdepth_b200 import FunctionalHalfspaceDepth, FunctionalProjectionDepth
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(6)
    X = _tied(rng, (11, 23))
    cols = ['c%d' % k for k in range(23)]
    df = pd.DataFrame(X, columns=cols)
    d = FunctionalProjectionDepth([df])
    assert isinstance(d, _FunctionalDepthUnivariate) and list(d.index) == cols
    med, mad = np_medmad(X)
    exp = np.sum(1.0 / (1.0 + np_outlyingness_rows(X, med, mad)), axis=0) / 11
    assert np.array_equal(d.values, exp)
    # u = 1.0 is the only direction: the engine path for curves with d = 1 gives the same bits
    assert np.array_equal(np_outlyingness(X.T[:, :, None], [[1.0]])[0], np_outlyingness_rows(X, med, mad))
    sub = FunctionalProjectionDepth([df], to_compute=['c4', 'c1'])
    assert list(sub.index) == ['c4', 'c1'] and sub.values.tolist() == d.loc[['c4', 'c1']].values.tolist()
    t = FunctionalProjectionDepth([df], kind='tukey')
    assert isinstance(t, _FunctionalDepthUnivariate)
    assert t.values.tolist() == FunctionalHalfspaceDepth([df]).values.tolist()
    assert (FunctionalProjectionDepth([df], kind='tukey', to_compute=['c3']).values.tolist()
            == FunctionalHalfspaceDepth([df], to_compute=['c3']).values.tolist())
    data = [pd.DataFrame(rng.standard_normal((6, 3)).cumsum(0), columns=list('xyz')) for _ in range(30)]
    F = np.stack([x.values for x in data])
    U = rng.standard_normal((17, 3))
    m = FunctionalProjectionDepth(data, directions=U)
    assert type(m) is _FunctionalDepthSeries and list(m.index) == list(range(30))
    assert np.array_equal(m.values, np.sum(1.0 / (1.0 + np_outlyingness(F, U)[0]), axis=0) / 6)
    mt = FunctionalProjectionDepth(data, kind='tukey', directions=U, to_compute=[29, 3])
    assert list(mt.index) == [29, 3]
    assert mt.values.tolist() == (np_tukey_counts(F, U)[[29, 3]] / (6.0 * 30)).tolist()
    assert np.array_equal(FunctionalProjectionDepth(data, directions=12, seed=3).values,
                          FunctionalProjectionDepth(data, directions=_unit(
                              np.random.default_rng(3).standard_normal((12, 3)))).values)


def test_refusals(pj_oracle):
    from statdepth_b200 import EngineError, FunctionalProjectionDepth, ProjectionDepth
    rng = np.random.default_rng(8)
    df = pd.DataFrame(rng.standard_normal((20, 3)))
    curves = [pd.DataFrame(rng.standard_normal((5, 3))) for _ in range(6)]
    uni = pd.DataFrame(rng.standard_normal((5, 9)))
    for bad in ('halfspace', 'Tukey', None):
        with pytest.raises(ValueError):
            ProjectionDepth(df, kind=bad)
        with pytest.raises(ValueError):
            FunctionalProjectionDepth(curves, kind=bad)
    for dirs in (0, -3, np.zeros((4, 3)), np.ones((4, 2)), np.ones(3), np.ones((0, 3)), [[1.0, np.nan, 0.0]],
                 [[1.0, 0.0, 0.0], [0.0, 0.0, 0.0]], [[np.inf, 1.0, 1.0]]):
        with pytest.raises(ValueError):
            ProjectionDepth(df, directions=dirs)
        with pytest.raises(ValueError):
            FunctionalProjectionDepth(curves, kind='tukey', directions=dirs)
    for dirs in (5, [[1.0]], np.ones((1, 1))):
        with pytest.raises(ValueError):
            FunctionalProjectionDepth([uni], directions=dirs)
    with pytest.raises(ValueError):
        FunctionalProjectionDepth(curves[:3] + [pd.DataFrame(rng.standard_normal((5, 2)))])
    with pytest.raises(ValueError):
        FunctionalProjectionDepth(curves[:3] + [pd.DataFrame(rng.standard_normal((4, 3)))])
    for empty in (pd.DataFrame(np.zeros((0, 3))), pd.DataFrame(np.zeros((4, 0)))):
        with pytest.raises(ValueError):
            ProjectionDepth(empty)
    with pytest.raises(ValueError):
        FunctionalProjectionDepth([])
    with pytest.raises(ValueError):
        FunctionalProjectionDepth(uni)
    with pytest.raises(ValueError):
        ProjectionDepth(rng.standard_normal((5, 2)))
    with pytest.raises(KeyError):
        ProjectionDepth(df, to_compute=['nope'])
    with pytest.raises(KeyError):
        FunctionalProjectionDepth(curves, to_compute=[6])
    with pytest.raises(KeyError):
        FunctionalProjectionDepth([uni], to_compute=[9])
    assert pj_oracle.calls == 0  # every refusal above happens before any engine call
    P = df.values.copy()
    P[4, 1] = np.nan
    for kind in ('projection', 'tukey'):
        with pytest.raises(EngineError) as ei:
            ProjectionDepth(pd.DataFrame(P), kind=kind, directions=4)
        assert ei.value.status == 4
        X = uni.values.copy()
        X[2, 2] = np.inf
        with pytest.raises(EngineError) as ei:
            FunctionalProjectionDepth([pd.DataFrame(X)], kind=kind)
        assert ei.value.status == 4


# ---------------------------------------------------------------------------------------------------------------
# CPU: two ranks (gloo)
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _results():
    from statdepth_b200 import FunctionalProjectionDepth, ProjectionDepth
    rng = np.random.default_rng(11)
    cloud = pd.DataFrame(_tied(rng, (31, 3)))
    U = rng.integers(-2, 3, size=(7, 3)).astype(np.float64)
    U[(U == 0).all(axis=1), 2] = 1.0
    uni = pd.DataFrame(_tied(rng, (13, 17)))  # 13 rows: uneven split 7 + 6
    curves = [pd.DataFrame(rng.standard_normal((5, 4))) for _ in range(9)]
    one_row = [pd.DataFrame(rng.standard_normal((1, 2))) for _ in range(6)]  # T = 1: one rank holds no rows
    out = {}
    for kind in ('projection', 'tukey'):
        out[kind + '_cloud'] = ProjectionDepth(cloud, kind=kind, directions=U).values
        out[kind + '_cloud_tc'] = ProjectionDepth(cloud, kind=kind, directions=U, to_compute=[30, 2]).values
        out[kind + '_k1'] = ProjectionDepth(cloud, kind=kind, directions=U[:1]).values  # one rank has no direction
        out[kind + '_uni'] = FunctionalProjectionDepth([uni], kind=kind).values
        out[kind + '_curves'] = FunctionalProjectionDepth(curves, kind=kind, directions=6, seed=2).values
        out[kind + '_t1'] = FunctionalProjectionDepth(one_row, kind=kind, directions=5).values
    return out


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(ProjectionOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(ProjectionOracleEngine(), monkeypatch.setattr)
    exp = _results()
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert np.array_equal(got[k], exp[k]), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the oracle
# ---------------------------------------------------------------------------------------------------------------
def _check_parity(engine, F, U):
    R = engine.projection_tukey_counts(F, U)
    assert R.tolist() == np_tukey_counts(F, U).tolist()
    O, med, mad = engine.projection_outlyingness(F, U, want_medmad=True)
    eO, emed, emad = np_outlyingness(F, U)
    assert np.array_equal(med, emed) and np.array_equal(mad, emad)
    assert np.array_equal(O, eO)
    return R, O


@pytest.mark.gpu
@pytest.mark.parametrize("N", [20_000, 5_000])
def test_cloud_parity_both_rank_pipelines(engine, N):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(N, N)["slab"] == (1 if N == 20_000 else 0)
    rng = np.random.default_rng(20)
    P = rng.standard_normal((N, 3)) @ rng.standard_normal((3, 3))
    _check_parity(engine, P[:, None, :], rng.standard_normal((48, 3)))


@pytest.mark.gpu
def test_integer_grids_with_ties(engine):
    rng = np.random.default_rng(21)
    for N, d in ((7, 2), (300, 3), (4000, 4), (20_001, 2)):
        P = rng.integers(-3, 4, size=(N, d)).astype(np.float64)
        P[rng.permutation(N)[:N * 6 // 10 + 1]] = 0.0  # most points equal: MAD = 0, O = inf
        P[(P == 0) & (rng.random(P.shape) < 0.5)] = -0.0
        U = rng.integers(-2, 3, size=(25, d)).astype(np.float64)
        U[(U == 0).all(axis=1), 0] = 1.0
        R, O = _check_parity(engine, P[:, None, :], U)
        assert np.isinf(O).any() and (O == 0).any(), N


@pytest.mark.gpu
def test_edge_shapes(engine):
    rng = np.random.default_rng(22)
    cases = [(rng.standard_normal((1, 1, 3)), rng.standard_normal((4, 3))),  # N = 1
             (rng.standard_normal((2, 3, 2)), rng.standard_normal((5, 2))),  # N = 2
             (rng.standard_normal((300, 7, 2)).cumsum(1), rng.standard_normal((33, 2))),  # partial time tiles
             (rng.standard_normal((900, 1, 5)), rng.standard_normal((1, 5))),  # K = 1
             (_tied(rng, (700, 4, 1)), np.array([[1.0], [-2.5]])),  # d = 1
             (rng.standard_normal((700, 2, 300)), rng.standard_normal((40, 300))),  # d >= 256, chunks of 32
             (rng.standard_normal((500, 1, 3)),
              rng.standard_normal((12, 3)) * 10.0 ** rng.integers(-150, 150, size=(12, 1)))]  # scales
    zeros = np.zeros((64, 1, 2))
    zeros[::2] = -0.0
    zeros[5] = [1.0, -1.0]
    cases.append((zeros, np.array([[1.0, 1.0], [1.0, 0.0]])))
    for F, U in cases:
        _check_parity(engine, np.ascontiguousarray(F), U)


@pytest.mark.gpu
def test_cloud_50000x8_k1000(engine):
    rng = np.random.default_rng(23)
    P = rng.standard_normal((50_000, 8)) * np.linspace(0.5, 3.0, 8)
    U = _unit(rng.standard_normal((1000, 8)))
    _check_parity(engine, P[:, None, :], U)


@pytest.mark.gpu
def test_curves_5000x256x3_k200(engine):
    rng = np.random.default_rng(24)
    F = rng.standard_normal((5000, 256, 3)).cumsum(1)
    U = _unit(rng.standard_normal((200, 3)))
    R = engine.projection_tukey_counts(F, U)
    parts = sum(engine.projection_tukey_counts(np.ascontiguousarray(F[:, a:b]), U)
                for a, b in ((0, 100), (100, 101), (101, 256)))
    assert R.tolist() == parts.tolist()
    assert ((R >= 256) & (R <= 256 * 5000)).all()
    O = engine.projection_outlyingness(F, U)
    ts = [0, 1, 9, 10, 133, 134, 200, 255]  # both time blocks, both sides of the projection's time tiles
    assert np.array_equal(O[ts], np_outlyingness(F[:, ts], U)[0])


@pytest.mark.gpu
def test_univariate_outlyingness_100000x1024(engine):
    rng = np.random.default_rng(25)
    T, n = 1024, 100_000
    X = rng.standard_normal((T, n)).cumsum(0)
    O, med, mad = engine.band_outlyingness(X, want_medmad=True)
    rows = rng.choice(T, 12, replace=False)
    emed, emad = np_medmad(X[rows])
    assert np.array_equal(med[rows], emed) and np.array_equal(mad[rows], emad)
    assert np.array_equal(O[rows], np_outlyingness_rows(X[rows], emed, emad))
    Of = engine.band_outlyingness(np.asfortranarray(X[:64]))  # the transposing upload
    assert np.array_equal(Of, O[:64])


@pytest.mark.gpu
def test_device_variants(engine):
    import torch
    rng = np.random.default_rng(26)
    F = rng.standard_normal((3000, 5, 3))
    U = rng.standard_normal((20, 3))
    dF = torch.from_numpy(F).cuda()
    cnt = torch.zeros(3000, dtype=torch.int64, device='cuda')
    engine.projection_tukey_counts_dev(dF.data_ptr(), 3000, 5, 3, U, cnt.data_ptr())
    assert cnt.cpu().numpy().tolist() == engine.projection_tukey_counts(F, U).tolist()
    o = torch.empty((5, 3000), dtype=torch.float64, device='cuda')
    med = torch.empty((5, 20), dtype=torch.float64, device='cuda')
    mad = torch.empty((5, 20), dtype=torch.float64, device='cuda')
    engine.projection_outlyingness_dev(dF.data_ptr(), 3000, 5, 3, U, o.data_ptr(), med.data_ptr(), mad.data_ptr())
    eO, emed, emad = engine.projection_outlyingness(F, U, want_medmad=True)
    assert np.array_equal(o.cpu().numpy(), eO) and np.array_equal(med.cpu().numpy(), emed)
    assert np.array_equal(mad.cpu().numpy(), emad)
    X = rng.standard_normal((9, 4001))
    dX = torch.from_numpy(X).cuda()
    ox = torch.empty((9, 4001), dtype=torch.float64, device='cuda')
    engine.band_outlyingness_dev(dX.data_ptr(), 9, 4001, 4001, ox.data_ptr())
    assert np.array_equal(ox.cpu().numpy(), engine.band_outlyingness(X))


@pytest.mark.gpu
def test_public_calls(engine):
    from statdepth_b200 import FunctionalProjectionDepth, ProjectionDepth
    rng = np.random.default_rng(27)
    P = rng.standard_normal((3000, 6))
    df = pd.DataFrame(P, index=['p%d' % i for i in range(3000)])
    U = _unit(np.random.default_rng(0).standard_normal((1000, 6)))
    d = ProjectionDepth(df)
    assert np.array_equal(d.values, 1.0 / (1.0 + np_outlyingness(P[:, None, :], U)[0][0]))
    t = ProjectionDepth(df, kind='tukey', to_compute=['p5', 'p0'])
    assert t.values.tolist() == (np_tukey_counts(P[:, None, :], U)[[5, 0]] / 3000.0).tolist()
    X = rng.standard_normal((30, 500)).cumsum(0)
    u = FunctionalProjectionDepth([pd.DataFrame(X)])
    med, mad = np_medmad(X)
    assert np.array_equal(u.values, np.sum(1.0 / (1.0 + np_outlyingness_rows(X, med, mad)), axis=0) / 30)
    data = [pd.DataFrame(rng.standard_normal((8, 4)).cumsum(0)) for _ in range(400)]
    F = np.stack([x.values for x in data])
    m = FunctionalProjectionDepth(data, kind='tukey', directions=50, seed=4)
    U4 = _unit(np.random.default_rng(4).standard_normal((50, 4)))
    assert m.values.tolist() == (np_tukey_counts(F, U4) / (8.0 * 400)).tolist()


# ---------------------------------------------------------------------------------------------------------------
# GPU: invariants that need no oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cell_directions_give_exact_halfspace(engine):
    rng = np.random.default_rng(28)
    for n, lo, hi in ((2000, -6, 6), (1999, -3, 3)):
        P = _grid_cloud(rng, n, lo, hi)
        U = cell_directions(P)
        assert engine.projection_tukey_counts(P[:, None, :], U).tolist() == engine.halfspace_counts(P).tolist()


@pytest.mark.gpu
def test_unit_direction_is_band_halfspace(engine):
    rng = np.random.default_rng(29)
    for X in (rng.standard_normal((40, 3000)).cumsum(0), _tied(rng, (16, 20_000))):
        F = np.ascontiguousarray(X.T[:, :, None])
        assert engine.projection_tukey_counts(F, [[1.0]]).tolist() == engine.band_halfspace_counts(X).tolist()
        assert np.array_equal(engine.projection_outlyingness(F, [[1.0]]), engine.band_outlyingness(X))


@pytest.mark.gpu
def test_direction_and_point_invariants(engine):
    rng = np.random.default_rng(30)
    F = rng.standard_normal((6000, 3, 4))
    U = rng.standard_normal((30, 4))
    R, O = engine.projection_tukey_counts(F, U), engine.projection_outlyingness(F, U)
    for V in (np.concatenate([U, U[[3, 3, 0]]]), U * 2.0, U[::-1]):
        assert engine.projection_tukey_counts(F, V).tolist() == R.tolist()
        assert np.array_equal(engine.projection_outlyingness(F, V), O)
    p = rng.permutation(6000)
    assert engine.projection_tukey_counts(F[p], U).tolist() == R[p].tolist()
    assert np.array_equal(engine.projection_outlyingness(F[p], U), O[:, p])
    # one call equals the min / max of two calls on disjoint direction sets: the cloud form, per time point
    P = F[:, :1]
    a, b = engine.projection_tukey_counts(P, U[:11]), engine.projection_tukey_counts(P, U[11:])
    assert np.minimum(a, b).tolist() == engine.projection_tukey_counts(P, U).tolist()
    oa, ob = engine.projection_outlyingness(F, U[:11]), engine.projection_outlyingness(F, U[11:])
    assert np.array_equal(np.maximum(oa, ob), O)


@pytest.mark.gpu
def test_direction_blocks_continue_the_running_value(engine):
    """2 000 000 points: 67 rows fit the 1 GB row budget, so K = 150 runs in three direction blocks."""
    rng = np.random.default_rng(31)
    P = rng.standard_normal((2_000_000, 1, 2))
    U = rng.standard_normal((150, 2))
    R = engine.projection_tukey_counts(P, U)
    O = engine.projection_outlyingness(P, U)
    Rs = [engine.projection_tukey_counts(P, U[k:k + 50]) for k in (0, 50, 100)]
    Os = [engine.projection_outlyingness(P, U[k:k + 50]) for k in (0, 50, 100)]
    assert R.tolist() == np.minimum.reduce(Rs).tolist()
    assert np.array_equal(O, np.maximum.reduce(Os))


@pytest.mark.gpu
def test_more_directions_than_one_launch_holds(engine):
    """40 points: all 2 200 000 directions fit the row budget, but one projection launch takes at most
    65 535 x 32 of them, so the call runs in two direction blocks."""
    rng = np.random.default_rng(33)
    P = rng.standard_normal((40, 1, 2))
    U = rng.standard_normal((2_200_000, 2))
    halves = (U[:1_100_000], U[1_100_000:])
    assert (engine.projection_tukey_counts(P, U).tolist()
            == np.minimum(*[engine.projection_tukey_counts(P, V) for V in halves]).tolist())
    assert np.array_equal(engine.projection_outlyingness(P, U),
                          np.maximum(*[engine.projection_outlyingness(P, V) for V in halves]))


@pytest.mark.gpu
def test_errors(engine):
    from statdepth_b200 import EngineError
    rng = np.random.default_rng(32)
    F = rng.standard_normal((100, 3, 2))
    U = rng.standard_normal((5, 2))
    X = rng.standard_normal((12, 90))
    calls = (lambda A: engine.projection_tukey_counts(A, U), lambda A: engine.projection_outlyingness(A, U))
    for bad in (np.nan, np.inf, -np.inf):
        for call in calls:
            B = F.copy()
            B[17, 2, 1] = bad
            with pytest.raises(EngineError) as ei:
                call(B)
            assert ei.value.status == 4
        B = X.copy()
        B[7, 33] = bad
        with pytest.raises(EngineError) as ei:
            engine.band_outlyingness(B)
        assert ei.value.status == 4
    big = np.full((50, 1, 2), 1.5e308) * np.sign(rng.standard_normal((50, 1, 2)))
    big[3] = 1.5e308  # finite data; 1.5e308 + 1.5e308 overflows
    for call in (engine.projection_tukey_counts, engine.projection_outlyingness):
        with pytest.raises(EngineError) as ei:
            call(big, [[1.0, 1.0]])
        assert ei.value.status == 4
    for V in (np.array([[1.0, 0.0], [0.0, 0.0]]), np.array([[np.nan, 1.0]]), np.zeros((0, 2))):
        for call in (engine.projection_tukey_counts, engine.projection_outlyingness):
            with pytest.raises(EngineError) as ei:
                call(F, V)
            assert ei.value.status == 1
    for call in (engine.projection_tukey_counts, engine.projection_outlyingness):
        with pytest.raises(EngineError) as ei:
            call(np.zeros((10, 2, 0)), np.zeros((3, 0)))
        assert ei.value.status == 1
    assert engine.projection_tukey_counts(F, U).tolist() == np_tukey_counts(F, U).tolist()  # still usable
    assert np.array_equal(engine.projection_outlyingness(F, U), np_outlyingness(F, U)[0])
