"""Halfspace (Tukey) depth (HalfspaceDepth, FunctionalHalfspaceDepth and the sd_*_halfspace_f64 entry points).

The contract: for a point p among n points, h(p) = the fewest points, p included, in a closed half-plane (half-line
for d = 1) whose boundary passes through p; HD = h / n.  d = 1: h = n - max(b, a).  d = 2: with z = #points equal to
p (p included), the m non-zero directions v_i = x_i - p and k_i = #{directions in (phi_i, phi_i + pi]},
h = z + min_i min(k_i, m - k_i), and h = n when m = 0.  Curves: H(c) = sum_t h_t(c), depth H / (T n).

The CPU part pins two numpy oracles (exact integer cross products; the engine's angular keys with searchsorted) to a
definitional brute force and drives the host layer with an engine of its own answering from numpy; the GPU part pins
the CUDA engine to the oracles and to invariants that need none."""
import math
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------
# numpy oracles
# ---------------------------------------------------------------------------------------------------------------
def np_halfspace_1d(x, queries=None):
    """h = n - max(b, a) of the values x [n] (b / a = other values strictly below / above)."""
    x = np.asarray(x, dtype=np.float64).ravel()
    n = x.size
    s = np.sort(x)
    q = np.arange(n) if queries is None else np.asarray(queries, dtype=np.int64)
    b = np.searchsorted(s, x[q], side='left')
    a = n - np.searchsorted(s, x[q], side='right')
    return (n - np.maximum(b, a)).astype(np.int64)


def np_halfspace_exact(P, queries=None):
    """The closed form with exact integer cross products, O(m^2) per query; P [n, 2] integer-valued."""
    P = np.asarray(P)
    n = len(P)
    V0 = np.asarray(np.round(P), dtype=np.int64)
    assert (V0 == P).all()
    out = []
    for q in (range(n) if queries is None else queries):
        V = V0 - V0[q]
        W = V[(V != 0).any(axis=1)]
        m = len(W)
        if m == 0:
            out.append(n)
            continue
        cr = W[:, None, 0] * W[None, :, 1] - W[:, None, 1] * W[None, :, 0]   # cross(v_i, v_j)
        dot = W[:, None, 0] * W[None, :, 0] + W[:, None, 1] * W[None, :, 1]
        k = ((cr > 0) | ((cr == 0) & (dot < 0))).sum(axis=1)
        out.append(n - m + int(np.minimum(k, m - k).min()))
    return np.array(out, dtype=np.int64)


def sc_keys(dx, dy):
    """The engine's angular key of every direction (csrc/angular_key.cuh sc_key), float64 operation for operation;
    the zero vector gets 17 (SC_ZERO)."""
    dx = np.asarray(dx, dtype=np.float64)
    dy = np.asarray(dy, dtype=np.float64)
    lower = (dy < 0) | ((dy == 0) & (dx < 0))
    add = np.where(lower, 12.0, 8.0)
    dx = np.where(lower, -dx, dx)
    dy = np.where(lower, -dy, dy)
    ax = -dx
    with np.errstate(divide='ignore', invalid='ignore'):
        f = np.where(dx > 0, np.where(dy < dx, dy / dx, 1.0 - dx / dy),
                     np.where(ax < dy, ax / dy, 1.0 - dy / ax))
    octant = np.where(dx > 0, np.where(dy < dx, 0.0, 1.0), np.where(ax < dy, 2.0, 3.0))
    k = (add + octant) + f
    k = np.where(k >= 16.0, 8.0, k)
    return np.where((dx == 0) & (dy == 0), 17.0, k)


def np_halfspace_keys(PX, PY, qx, qy):
    """h of the points (qx[r], qy[r]) among the rows PX[r], PY[r] (each holding the point itself), by the engine's
    keys and one searchsorted per row block: rows are offset by 32 so that one sorted array serves all of them."""
    R, n = PX.shape
    K = sc_keys(PX - qx[:, None], PY - qy[:, None])
    m = (K < 16.0).sum(axis=1)
    off = 32.0 * np.arange(R)[:, None]
    G = np.sort(K, axis=1) + off
    flat = G.ravel()
    start = (np.arange(R) * n)[:, None]
    le_u = np.searchsorted(flat, K + off, side='right') - start              # keys <= u in the row
    w = np.where(K < 12.0, K + 4.0, K - 4.0)
    le_w = np.searchsorted(flat, w + off, side='right') - start
    k = np.where(K < 12.0, le_w - le_u, (m[:, None] - le_u) + le_w)
    side = np.where(K < 16.0, np.minimum(k, m[:, None] - k), n)
    return (n - m + np.minimum(side.min(axis=1), m)).astype(np.int64)


def np_halfspace_sorted(P, queries=None, block=256):
    """h of the queries of the cloud P [n, 2] by the engine's keys, O(n log n) per query."""
    P = np.asarray(P, dtype=np.float64)
    q = np.arange(len(P)) if queries is None else np.asarray(queries, dtype=np.int64)
    out = []
    for i in range(0, len(q), block):
        qb = q[i:i + block]
        R = len(qb)
        out.append(np_halfspace_keys(np.broadcast_to(P[:, 0], (R, len(P))), np.broadcast_to(P[:, 1], (R, len(P))),
                                     P[qb, 0], P[qb, 1]))
    return np.concatenate(out) if out else np.zeros(0, dtype=np.int64)


def np_functional_sorted(F, queries=None):
    """sum_t h_t of the curves F [N, T, 2] by the engine's keys."""
    F = np.asarray(F, dtype=np.float64)
    N, T, _ = F.shape
    q = np.arange(N) if queries is None else np.asarray(queries, dtype=np.int64)
    return sum(np_halfspace_sorted(F[:, t, :], q) for t in range(T)).astype(np.int64)


def np_band_halfspace(X):
    """H [n] of the curves of X [T, n]."""
    X = np.asarray(X, dtype=np.float64)
    return sum(np_halfspace_1d(X[t]) for t in range(X.shape[0])).astype(np.int64)


def brute_halfspace(P, q):
    """The definition: the fewest points in a closed half-plane through p, over one direction between every two
    consecutive critical angles phi_i +- pi / 2."""
    p = P[q]
    V = P - p
    nz = (V != 0).any(axis=1)
    z = int((~nz).sum())
    if not nz.any():
        return len(P)
    ang = np.arctan2(V[nz, 1], V[nz, 0])
    crit = np.unique(np.mod(np.concatenate([ang + np.pi / 2, ang - np.pi / 2]), 2 * np.pi))
    nxt = np.append(crit[1:], crit[0] + 2 * np.pi)
    best = len(P)
    for th in (crit + nxt) / 2:
        d = V[nz] @ np.array([math.cos(th), math.sin(th)])
        best = min(best, int((d >= 0).sum()) + z)
    return best


def _grid_cloud(rng, n, lo=-3, hi=3):
    """Integers in [lo, hi], a third of the points on one line, duplicates by construction."""
    P = rng.integers(lo, hi + 1, size=(n, 2)).astype(np.float64)
    k = n // 3
    P[:k, 1] = 2 * P[:k, 0] + 1
    return P


def _tied(rng, shape):
    """Values on 8 levels, zeros of both signs."""
    X = rng.integers(-4, 4, size=shape).astype(np.float64) * 0.5
    X[(X == 0) & (rng.random(shape) < 0.5)] = -0.0
    return X


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracles
# ---------------------------------------------------------------------------------------------------------------
def test_oracles_equal_brute_force():
    rng = np.random.default_rng(1)
    for case in range(300):
        n = int(rng.integers(1, 25))
        P = _grid_cloud(rng, n)
        exp = [brute_halfspace(P, q) for q in range(n)]
        assert np_halfspace_exact(P).tolist() == exp, P
        assert np_halfspace_sorted(P).tolist() == exp, P
        assert all(1 <= h <= n for h in exp)


def test_oracles_equal_on_larger_clouds():
    rng = np.random.default_rng(2)
    P = _grid_cloud(rng, 400, -6, 6)
    assert np_halfspace_sorted(P).tolist() == np_halfspace_exact(P).tolist()
    P = rng.standard_normal((300, 2))
    assert np_halfspace_sorted(P).tolist() == [brute_halfspace(P, q) for q in range(300)]
    x = rng.integers(-3, 4, size=60).astype(np.float64)
    exp = [min(int((x <= v).sum()), int((x >= v).sum())) for v in x]
    assert np_halfspace_1d(x).tolist() == exp
    # a line through the cloud: the 2-D numerator is the 1-D one of the coordinate along it
    assert np_halfspace_exact(np.column_stack([x, 3 * x - 2])).tolist() == exp


def test_sc_keys_are_monotone_and_antipodal():
    rng = np.random.default_rng(3)
    v = rng.integers(-50, 51, size=(4000, 2)).astype(np.float64)
    v = v[(v != 0).any(axis=1)]
    k = sc_keys(v[:, 0], v[:, 1])
    ang = np.mod(np.arctan2(v[:, 1], v[:, 0]), 2 * np.pi)
    o = np.argsort(ang, kind='stable')
    assert (np.diff(k[o]) >= 0).all()
    kw = sc_keys(-v[:, 0], -v[:, 1])
    assert (kw == np.where(k < 12, k + 4, k - 4)).all()


# ---------------------------------------------------------------------------------------------------------------
# CPU: host layer on a test double
# ---------------------------------------------------------------------------------------------------------------
class HalfspaceOracleEngine:
    """TEST DOUBLE: the engine methods the halfspace drivers call, answered by numpy, refusing non-finite input with
    SD_ERR_NONFINITE as the engine does."""

    def __init__(self):
        self.calls = 0

    def _finite(self, A):
        from statdepth_b200 import EngineError
        self.calls += 1
        if not np.isfinite(A).all():
            raise EngineError(4, 'non-finite input')

    def halfspace_counts(self, P, queries=None):
        P = np.ascontiguousarray(P, dtype=np.float64)
        self._finite(P)
        q = np.arange(len(P)) if queries is None else np.asarray(queries, dtype=np.int64)
        return np_halfspace_1d(P[:, 0], q) if P.shape[1] == 1 else np_halfspace_sorted(P, q)

    def functional_halfspace_counts(self, F, queries=None):
        self._finite(F)
        return np_functional_sorted(F, queries)

    def band_halfspace_counts(self, X):
        self._finite(X)
        return np_band_halfspace(X)


def _install(fake, setter):
    import statdepth_b200._halfspace as h
    setter(h, "get_engine", lambda device=None: fake)


@pytest.fixture()
def hs_oracle(monkeypatch):
    fake = HalfspaceOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _curves2(rng, N, T, grid=True):
    if grid:
        return [pd.DataFrame(rng.integers(-3, 4, size=(T, 2)).astype(np.float64), columns=['x', 'y'])
                for _ in range(N)]
    return [pd.DataFrame(rng.standard_normal((T, 2)).cumsum(0), columns=['x', 'y']) for _ in range(N)]


def test_pointcloud_labels_and_to_compute(hs_oracle):
    from statdepth_b200 import HalfspaceDepth
    from statdepth_b200.depth import _PointwiseDepth
    rng = np.random.default_rng(5)
    P = _grid_cloud(rng, 40)
    labels = ['p%d' % i for i in range(40)]
    df = pd.DataFrame(P, index=labels, columns=['a', 'b'])
    d = HalfspaceDepth(df)
    assert isinstance(d, _PointwiseDepth)
    assert list(d.index) == labels
    assert d.values.tolist() == (np_halfspace_exact(P) / 40.0).tolist()
    sub = HalfspaceDepth(df, to_compute=['p7', 'p0', 'p39'])
    assert list(sub.index) == ['p7', 'p0', 'p39']
    assert sub.values.tolist() == d.loc[['p7', 'p0', 'p39']].values.tolist()
    assert d.deepest().values[0] == d.values.max()
    x = pd.DataFrame({'v': [0.0, 1.0, 1.0, -2.0, 5.0]}, index=list('abcde'))
    assert HalfspaceDepth(x).values.tolist() == [2 / 5, 3 / 5, 3 / 5, 1 / 5, 1 / 5]
    with pytest.raises(KeyError):
        HalfspaceDepth(df, to_compute=['nope'])


def test_functional_univariate(hs_oracle):
    from statdepth_b200 import FunctionalHalfspaceDepth
    from statdepth_b200.depth import _FunctionalDepthUnivariate
    rng = np.random.default_rng(6)
    X = _tied(rng, (11, 23))
    cols = ['c%d' % k for k in range(23)]
    df = pd.DataFrame(X, columns=cols)
    d = FunctionalHalfspaceDepth([df])
    assert isinstance(d, _FunctionalDepthUnivariate)
    assert list(d.index) == cols
    assert d.values.tolist() == (np_band_halfspace(X) / (11.0 * 23)).tolist()
    sub = FunctionalHalfspaceDepth([df], to_compute=['c4', 'c1'])
    assert list(sub.index) == ['c4', 'c1'] and sub.values.tolist() == d.loc[['c4', 'c1']].values.tolist()
    one = FunctionalHalfspaceDepth([pd.DataFrame(X[:1])])  # a single time point is the 1-D cloud
    assert one.values.tolist() == (np_halfspace_1d(X[0]) / 23.0).tolist()


def test_functional_bivariate(hs_oracle):
    from statdepth_b200 import FunctionalHalfspaceDepth
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(7)
    data = _curves2(rng, 30, 6)
    F = np.stack([df.values for df in data])
    d = FunctionalHalfspaceDepth(data)
    assert type(d) is _FunctionalDepthSeries and not isinstance(d, _FunctionalDepthUnivariate)
    assert list(d.index) == list(range(30))
    exp = sum(np_halfspace_exact(F[:, t, :]) for t in range(6)) / (6.0 * 30)
    assert d.values.tolist() == exp.tolist()
    sub = FunctionalHalfspaceDepth(data, to_compute=[29, 3])
    assert list(sub.index) == [29, 3] and sub.values.tolist() == [exp[29], exp[3]]


def test_refusals(hs_oracle):
    from statdepth_b200 import EngineError, FunctionalHalfspaceDepth, HalfspaceDepth
    rng = np.random.default_rng(8)
    with pytest.raises(NotImplementedError):
        HalfspaceDepth(pd.DataFrame(rng.standard_normal((20, 3))))
    with pytest.raises(NotImplementedError):
        FunctionalHalfspaceDepth([pd.DataFrame(rng.standard_normal((5, 3))) for _ in range(6)])
    with pytest.raises(NotImplementedError):
        FunctionalHalfspaceDepth([pd.DataFrame(rng.standard_normal((5, 1))) for _ in range(6)])
    ragged = _curves2(rng, 5, 4) + [pd.DataFrame(rng.standard_normal((4, 3)))]
    with pytest.raises(NotImplementedError):
        FunctionalHalfspaceDepth(ragged)
    with pytest.raises(ValueError):
        FunctionalHalfspaceDepth(_curves2(rng, 5, 4) + _curves2(rng, 1, 5))
    with pytest.raises(ValueError):
        FunctionalHalfspaceDepth(pd.DataFrame(rng.standard_normal((5, 4))))
    with pytest.raises(ValueError):
        FunctionalHalfspaceDepth([])
    with pytest.raises(KeyError):
        FunctionalHalfspaceDepth(_curves2(rng, 5, 4), to_compute=[5])
    assert hs_oracle.calls == 0  # every refusal above happens before any engine call
    P = rng.standard_normal((20, 2))
    P[4, 1] = np.nan
    with pytest.raises(EngineError) as ei:
        HalfspaceDepth(pd.DataFrame(P))
    assert ei.value.status == 4
    X = rng.standard_normal((6, 9))
    X[2, 2] = np.inf
    with pytest.raises(EngineError) as ei:
        FunctionalHalfspaceDepth([pd.DataFrame(X)])
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
    from statdepth_b200 import FunctionalHalfspaceDepth, HalfspaceDepth
    rng = np.random.default_rng(11)
    cloud = pd.DataFrame(_grid_cloud(rng, 31))
    uni = pd.DataFrame(_tied(rng, (13, 17)))  # 13 rows: uneven split 7 + 6
    biv = _curves2(rng, 9, 5)
    one_row = pd.DataFrame(rng.standard_normal((1, 6)))  # T = 1: one rank holds no rows
    return dict(cloud=HalfspaceDepth(cloud).values, cloud_tc=HalfspaceDepth(cloud, to_compute=[30, 2, 5]).values,
                uni=FunctionalHalfspaceDepth([uni]).values, biv=FunctionalHalfspaceDepth(biv).values,
                biv_tc=FunctionalHalfspaceDepth(biv, to_compute=[8, 0]).values,
                t1=FunctionalHalfspaceDepth([one_row]).values)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(HalfspaceOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(HalfspaceOracleEngine(), monkeypatch.setattr)
    exp = _results()
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the oracles
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cloud_normal_3000_all_queries(engine):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(6000)["slab"] == 0  # rows of n and 2n take the part pipeline
    P = np.random.default_rng(20).standard_normal((3000, 2))
    h = engine.halfspace_counts(P)
    assert h.tolist() == np_halfspace_sorted(P).tolist()
    assert h.max() >= math.ceil(3000 / 3)  # centerpoint theorem


@pytest.mark.gpu
def test_cloud_20000_sampled_queries(engine):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(20_000)["slab"] == 1 and mbd_plan(40_000)["slab"] == 1
    rng = np.random.default_rng(21)
    P = rng.standard_normal((20_000, 2)) * [1.0, 3.0]
    q = rng.choice(20_000, 512, replace=False)
    assert engine.halfspace_counts(P, q).tolist() == np_halfspace_sorted(P, q).tolist()


@pytest.mark.gpu
def test_integer_grids(engine):
    rng = np.random.default_rng(22)
    for n, lo, hi in ((7, -1, 1), (64, -3, 3), (1500, -3, 3), (5000, -20, 20)):
        P = _grid_cloud(rng, n, lo, hi)
        h = engine.halfspace_counts(P)
        assert h.tolist() == np_halfspace_sorted(P).tolist(), n
        q = rng.choice(n, min(n, 150 if n <= 1500 else 20), replace=False)
        assert h[q].tolist() == np_halfspace_exact(P, q).tolist(), n
    P = np.zeros((9, 2))  # every point equal: h = n
    assert engine.halfspace_counts(P).tolist() == [9] * 9
    assert engine.halfspace_counts(np.array([[1.0, 2.0]])).tolist() == [1]
    assert engine.halfspace_counts(np.array([[0.0, 0.0], [-0.0, 1.0]])).tolist() == [1, 1]


@pytest.mark.gpu
def test_d1_clouds_with_ties(engine):
    rng = np.random.default_rng(23)
    for n in (1, 2, 33, 3000, 50_000):
        x = _tied(rng, (n, 1))
        assert engine.halfspace_counts(x).tolist() == np_halfspace_1d(x).tolist(), n
        q = rng.integers(0, n, size=7)
        assert engine.halfspace_counts(x, q).tolist() == np_halfspace_1d(x, q).tolist(), n


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["walks", "tied"])
def test_univariate_full_size(engine, kind):
    from statdepth_b200 import FunctionalHalfspaceDepth
    rng = np.random.default_rng(24)
    T, n = 1024, 100_000
    X = rng.standard_normal((T, n)).cumsum(0) if kind == "walks" else _tied(rng, (T, n))
    exp = np_band_halfspace(X)
    assert engine.band_halfspace_counts(X).tolist() == exp.tolist()
    d = FunctionalHalfspaceDepth([pd.DataFrame(X)])  # F-ordered values: the transposing upload
    assert d.values.tolist() == (exp.astype(np.float64) / (T * n)).tolist()


@pytest.mark.gpu
def test_bivariate_grid_all_curves(engine):
    rng = np.random.default_rng(25)
    F = rng.integers(-4, 5, size=(300, 32, 2)).astype(np.float64)
    h = engine.functional_halfspace_counts(F)
    assert h.tolist() == np_functional_sorted(F).tolist()
    q = rng.choice(300, 20, replace=False)
    assert h[q].tolist() == sum(np_halfspace_exact(F[:, t, :], q) for t in range(32)).tolist()


@pytest.mark.gpu
def test_bivariate_5000x256_sampled(engine):
    rng = np.random.default_rng(26)
    F = rng.standard_normal((5000, 256, 2)).cumsum(1)
    q = rng.choice(5000, 16, replace=False)
    assert engine.functional_halfspace_counts(F, q).tolist() == np_functional_sorted(F, q).tolist()


# ---------------------------------------------------------------------------------------------------------------
# GPU: invariants that need no oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collinear_equals_1d(engine):
    rng = np.random.default_rng(27)
    for n in (50, 4000):
        x = rng.integers(-30, 31, size=n).astype(np.float64)
        one = engine.halfspace_counts(x[:, None])
        for a, b in ((1.0, 0.0), (0.0, 1.0), (2.0, -3.0)):
            assert engine.halfspace_counts(np.column_stack([a * x, b * x + 7.0])).tolist() == one.tolist()


@pytest.mark.gpu
def test_unimodular_map_keeps_counts(engine):
    rng = np.random.default_rng(28)
    for A in (np.array([[1, 3], [0, 1]]), np.array([[2, 1], [1, 1]]), np.array([[0, -1], [1, 0]])):
        P = _grid_cloud(rng, 2000, -10, 10)
        assert engine.halfspace_counts(P @ A.T.astype(np.float64)).tolist() == engine.halfspace_counts(P).tolist()


@pytest.mark.gpu
def test_centerpoint_bound(engine):
    """The centerpoint theorem gives a point of the plane of depth >= ceil(n / 3); it need not be a sample point (10
    points in convex position all have h = 1), but in a large random cloud the deepest sample point lies near the
    middle, with h close to n / 2."""
    rng = np.random.default_rng(29)
    for n in (999, 10_000):
        P = rng.standard_normal((n, 2)) @ rng.standard_normal((2, 2))
        assert engine.halfspace_counts(P).max() >= math.ceil(n / 3), n


@pytest.mark.gpu
def test_identical_rows_scale_cloud_counts(engine):
    rng = np.random.default_rng(30)
    for P in (rng.standard_normal((500, 2)), _grid_cloud(rng, 300)):
        F = np.repeat(P[:, None, :], 7, axis=1)
        assert engine.functional_halfspace_counts(F).tolist() == (7 * engine.halfspace_counts(P)).tolist()


@pytest.mark.gpu
def test_to_compute_subsets(engine):
    from statdepth_b200 import FunctionalHalfspaceDepth, HalfspaceDepth
    rng = np.random.default_rng(31)
    df = pd.DataFrame(rng.standard_normal((800, 2)), index=['p%d' % i for i in range(800)])
    full = HalfspaceDepth(df)
    tc = ['p5', 'p799', 'p0', 'p5']
    assert HalfspaceDepth(df, to_compute=tc).values.tolist() == full.loc[tc].values.tolist()
    uni = pd.DataFrame(rng.standard_normal((40, 300)))
    fu = FunctionalHalfspaceDepth([uni])
    assert FunctionalHalfspaceDepth([uni], to_compute=[299, 3]).values.tolist() == fu.loc[[299, 3]].values.tolist()
    data = _curves2(rng, 120, 9, grid=False)
    fb = FunctionalHalfspaceDepth(data)
    assert FunctionalHalfspaceDepth(data, to_compute=[7, 119, 0]).values.tolist() == fb.loc[[7, 119, 0]].values.tolist()


@pytest.mark.gpu
def test_errors(engine):
    from statdepth_b200 import EngineError
    rng = np.random.default_rng(32)
    P = rng.standard_normal((100, 2))
    F = rng.standard_normal((80, 6, 2))
    X = rng.standard_normal((12, 90))
    for bad in (np.nan, np.inf, -np.inf):
        for call, A, idx in ((lambda A: engine.halfspace_counts(A), P, (17, 1)),
                             (lambda A: engine.halfspace_counts(A, [0]), P, (99, 0)),
                             (lambda A: engine.halfspace_counts(A[:, :1], []), P, (3, 0)),
                             (lambda A: engine.functional_halfspace_counts(A, [5]), F, (70, 4, 1)),
                             (lambda A: engine.band_halfspace_counts(A), X, (7, 33))):
            B = A.copy()
            B[idx] = bad
            with pytest.raises(EngineError) as ei:
                call(B)
            assert ei.value.status == 4
    for A in (rng.standard_normal((10, 3)), rng.standard_normal((10, 4))):
        with pytest.raises(EngineError) as ei:
            engine.halfspace_counts(A)
        assert ei.value.status == 6
    with pytest.raises(EngineError) as ei:
        engine.functional_halfspace_counts(rng.standard_normal((10, 4, 3)))
    assert ei.value.status == 6
    assert engine.halfspace_counts(P).tolist() == np_halfspace_sorted(P).tolist()  # the context stays usable
