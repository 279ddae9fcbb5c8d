"""2-D triangle counting (K3 / K4, csrc/simplicial_count.cu) at multi-million-point scale, where its int64 counts
approach 2^63, against an exact count.

Every count is C(m, 3) minus the non-containing triples of m other points, so it grows as n^3: C(m, 3) fits in int64
up to m = 3 810 779, and curves add T counts into one int64.  The engine must give exact counts up to the largest
size whose T * C(m, 3) fits, and refuse with SD_ERR_OVERFLOW from the next size on.

The reference (`tri_count`) is the tolerance-0 count of one query against a set of other points, by the engine's
angular keys (`test_halfspace.sc_keys`), one sort and two searchsorted per query: with the keys sorted into classes of
g equal directions and c = #keys strictly inside the open half-turn after the class (antipodes excluded), the
non-containing triples are sum g C(c, 2) + C(g, 2) c + C(g, 3), each term at most C(m, 3).  The CPU part pins it to
the C oracle's enumeration on small clouds; the GPU part compares exact integers with it, and with a closed form: the
center of a regular p-gon (p odd) lies in C(p, 3) - p C((p - 1) / 2, 2) triangles of its vertices."""
import math

import numpy as np
import pandas as pd
import pytest

from test_halfspace import np_halfspace_sorted, sc_keys

I64_MAX = 2 ** 63 - 1


# ---------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------
def c3(m):
    """C(m, 3) of an int64 array as csrc/simplicial_count.cu forms it: the even factor halved and the multiple of 3
    divided by 3 before the product."""
    m = np.asarray(m, dtype=np.int64)
    a, b, c = m, m - 1, m - 2
    even = a % 2 == 0
    a, b = np.where(even, a // 2, a), np.where(even, b, b // 2)
    da = a % 3 == 0
    db = ~da & (b % 3 == 0)
    a, b, c = np.where(da, a // 3, a), np.where(db, b // 3, b), np.where(da | db, c, c // 3)
    return np.where(m < 3, 0, a * b * c)


def tri_count(others, p):
    """#closed triangles of the points `others` [m, 2] that contain p, tolerance 0, by the engine's keys (exact)."""
    K = sc_keys(others[:, 0] - p[0], others[:, 1] - p[1])
    K = np.sort(K[K < 16.0])  # directions equal to zero take part only in containing triangles
    u, g = np.unique(K, return_counts=True)
    w = np.where(u < 12.0, u + 4.0, u - 4.0)  # the antipode, exact (same binade)
    le_u = np.searchsorted(K, u, 'right')
    lt_w = np.searchsorted(K, w, 'left')
    c = np.where(u < 12.0, lt_w - le_u, (len(K) - le_u) + lt_w).astype(np.int64)
    g = g.astype(np.int64)
    noncontaining = g * (c * (c - 1) // 2) + (g * (g - 1) // 2) * c + c3(g)
    return math.comb(len(others), 3) - int(noncontaining.sum(dtype=np.int64))


def tri_count_in(P, q):
    """In-sample form: point q of the cloud P against the n - 1 others."""
    return tri_count(np.delete(P, q, axis=0), P[q])


def polygon(p):
    """The p vertices of a regular p-gon on the unit circle [p, 2]."""
    t = 2.0 * np.pi * np.arange(p) / p
    return np.stack([np.cos(t), np.sin(t)], axis=1)


def center_count(p):
    """#triangles of the vertices of a regular p-gon (p odd) that contain its center: the non-containing ones are
    the triples within one open half-turn, (p - 1) / 2 vertices after their first."""
    assert p % 2 == 1
    return math.comb(p, 3) - p * math.comb((p - 1) // 2, 2)


def rotations(P):
    """P and its three exact quarter turns (x, y) -> (-y, x)."""
    out = [P]
    for _ in range(3):
        out.append(np.stack([-out[-1][:, 1], out[-1][:, 0]], axis=1))
    return out


# Largest accepted size and the first refused one (T * C(m, 3) > 2^63 - 1): (call, T, m_others - size, last ok)
EDGES = [("in-sample", 1, -1, 3_810_780), ("out-of-sample", 1, 0, 3_810_779),
         ("curves", 1, -1, 3_810_780), ("curves", 2, -1, 3_024_618), ("curves", 64, -1, 952_696)]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the references against the C oracle and math.comb
# ---------------------------------------------------------------------------------------------------------------
def _small_cloud(rng, kind, n):
    if kind == "general":
        return rng.standard_normal((n, 2))
    if kind == "lattice":  # ties of direction, duplicates of the query and of each other
        return rng.integers(-3, 4, size=(n, 2)).astype(np.float64)
    q = rng.integers(-2, 3, size=2).astype(np.float64)
    if kind == "lines":  # points on lines through the query, on both sides of it
        dirs = rng.integers(-3, 4, size=(4, 2)).astype(np.float64)
        dirs[(dirs == 0).all(axis=1)] = (1.0, 2.0)
        t = rng.integers(-4, 5, size=n - 1).astype(np.float64)
        rest = q + t[:, None] * dirs[rng.integers(0, 4, size=n - 1)]
    else:  # "antipodes": exact pairs q + v, q - v
        v = rng.integers(-5, 6, size=((n - 1) // 2, 2)).astype(np.float64) * 0.5
        rest = np.concatenate([q + v, q - v, rng.standard_normal(((n - 1) % 2, 2))])
    return np.concatenate([q[None, :], rest])


@pytest.mark.parametrize("kind", ["general", "lattice", "lines", "antipodes"])
def test_reference_equals_oracle(oracle, kind):
    rng = np.random.default_rng(["general", "lattice", "lines", "antipodes"].index(kind))
    for _ in range(8):
        n = int(rng.integers(4, 40))
        P = _small_cloud(rng, kind, n)
        got = [tri_count_in(P, q) for q in range(n)]
        assert got == oracle.simplicial_counts(P, None, 0.0).tolist(), P


@pytest.mark.parametrize("kind", ["general", "lattice", "lines", "antipodes"])
def test_out_of_sample_reference_equals_oracle(oracle, kind):
    """others = S for a new point y: the in-sample count of y in S + [y]."""
    rng = np.random.default_rng(10 + ["general", "lattice", "lines", "antipodes"].index(kind))
    for _ in range(8):
        n = int(rng.integers(5, 40))
        P = _small_cloud(rng, kind, n)
        S = P[1:]
        for y in (P[0], S[int(rng.integers(0, n - 1))], rng.integers(-3, 4, size=2).astype(np.float64)):
            assert tri_count(S, y) == oracle.simplicial_counts(np.vstack([S, y]), [n - 1], 0.0)[0], (S, y)


@pytest.mark.parametrize("p", [3, 5, 7, 9, 21, 41])
def test_polygon_closed_form(oracle, p):
    V = polygon(p)
    P = np.vstack([V, [[0.0, 0.0]]])
    assert center_count(p) == tri_count(V, P[p])
    assert center_count(p) == oracle.simplicial_counts(P, [p])[0]  # the default tolerance band
    assert center_count(p) == oracle.simplicial_counts(P, [p], 0.0)[0]
    assert tri_count_in(P, 0) == 0 == oracle.simplicial_counts(P, [0], 0.0)[0]


def test_c3_is_exact_wherever_the_result_fits():
    ms = np.array([0, 1, 2, 3, 4, 5, 6, 7, 2_642_246, 2_642_247, 2_642_248, 3_000_000, 3_810_778, 3_810_779]
                  + np.random.default_rng(1).integers(3, 3_810_780, size=1000).tolist(), dtype=np.int64)
    assert c3(ms).tolist() == [math.comb(int(m), 3) for m in ms]
    assert math.comb(3_810_779, 3) <= I64_MAX < math.comb(3_810_780, 3)
    # the former (m (m - 1) / 2) (m - 2) / 3 wraps first at m = 2 642 247 (in-sample clouds of 2 642 248 points)
    old = lambda m: (m * (m - 1) // 2) * (m - 2)  # noqa: E731
    assert old(2_642_246) <= I64_MAX < old(2_642_247)


def test_edges_are_where_the_count_stops_fitting():
    for _, T, off, last in EDGES:
        assert T * math.comb(last + off, 3) <= I64_MAX < T * math.comb(last + 1 + off, 3)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
N_MAX = 3_810_781  # one standard-normal cloud; every size below takes a prefix of it
_REFS = {}


def _ref(tag, P, q):
    """tri_count_in, once per (data, size, query)."""
    key = (tag, len(P), int(q))
    if key not in _REFS:
        _REFS[key] = tri_count_in(P, int(q))
    return _REFS[key]


@pytest.fixture(scope="module")
def cloud():
    return np.random.default_rng(2026).standard_normal((N_MAX, 2))


@pytest.fixture()
def count_impl(engine):
    """Set SD_OPT_SIMPLICIAL_IMPL for one test, AUTO again afterwards."""
    from statdepth_b200 import _engine as E
    yield lambda impl: engine.set_option(E.OPT_SIMPLICIAL_IMPL, impl)
    engine.set_option(E.OPT_SIMPLICIAL_IMPL, E.SIMPLICIAL_AUTO)


def _queries(P, rng, k=3):
    """The point nearest the origin, a hull vertex (the largest x) and k random points."""
    return [int(np.argmin((P * P).sum(axis=1))), int(np.argmax(P[:, 0]))] + rng.choice(len(P), k, False).tolist()


def _overflows(call):
    from statdepth_b200 import EngineError
    with pytest.raises(EngineError) as ei:
        call()
    assert ei.value.status == 5, ei.value
    assert "overflows int64" in str(ei.value)


def _still_usable(engine, oracle):
    P = np.random.default_rng(5).standard_normal((200, 2))
    q = [0, 77, 199]
    assert (engine.simplicial_counts(P, q, 0.0) == oracle.simplicial_counts(P, q, 0.0)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("data,n", [("normal", 2_642_247), ("normal", 2_642_248), ("normal", 3_000_001),
                                    ("normal", 3_810_780), ("lattice", 3_000_001)])
def test_in_sample_counts_across_the_edges(engine, count_impl, cloud, data, n):
    """C(n - 1, 3) wrapped in the former c3 from n = 2 642 248; n = 3 810 780 is the largest accepted cloud.  The
    lattice gives large tied classes and coincident points.  24 queries: more than one batch of instances
    (3 GiB / 56 n bytes: 19 at 3 M points)."""
    from statdepth_b200 import _engine as E
    rng = np.random.default_rng(n)
    P = cloud[:n] if data == "normal" else rng.integers(-1000, 1001, size=(n, 2)).astype(np.float64)
    qs = _queries(P, rng)
    ref = {q: _ref(data, P, q) for q in qs}
    if data == "normal":
        assert ref[qs[1]] == 0  # a hull vertex
    assert ref[qs[0]] > math.comb(n - 1, 3) // 8  # the deepest point: about a quarter of all triangles
    ql = (qs * 5)[:24]
    exp = np.array([ref[q] for q in ql], dtype=np.int64)
    for impl in (E.SIMPLICIAL_COUNT, E.SIMPLICIAL_AUTO):
        count_impl(impl)
        assert engine.simplicial_counts(P, ql, 0.0).tolist() == exp.tolist(), impl


@pytest.mark.gpu
@pytest.mark.parametrize("p", [3_000_001, 3_810_779])
def test_polygon_center_at_both_tolerances(engine, p):
    """No antipodes, angular gaps >= 2 pi / p and every non-containing triangle at least sin(pi / 2p) >= 4.1e-7 from
    the center: the arcs of the default band (1e-7) and the exact keys (0) give the closed form.  Cloud n = p + 1:
    p = 3 810 779 is the largest accepted."""
    P = np.vstack([polygon(p), [[0.0, 0.0]]])
    exp = center_count(p)
    assert engine.simplicial_counts(P, [p]).tolist() == [exp]
    assert engine.simplicial_counts(P, [p, 0, p // 2], 0.0).tolist() == [exp, 0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("nS", [2_642_247, 3_810_779])
def test_out_of_sample_counts(engine, nS):
    """Against the nS vertices of a p-gon (m = nS others; C(nS, 3) wrapped from nS = 2 642 247): its center, two
    random points of the disk and two duplicates of sample points."""
    S = polygon(nS)
    rng = np.random.default_rng(nS)
    Y = np.vstack([[[0.0, 0.0]], rng.uniform(-0.7, 0.7, size=(2, 2)), S[[5, nS // 3]]])
    exp = [center_count(nS)] + [tri_count(S, y) for y in Y[1:]]
    assert exp[3] == exp[4] == math.comb(nS - 1, 2)  # a vertex duplicate: exactly the triangles through it
    assert engine.simplicial_oos_counts(S, Y, 0.0).tolist() == exp
    assert engine.simplicial_oos_counts(S, Y[:1]).tolist() == exp[:1]


@pytest.mark.gpu
@pytest.mark.parametrize("T,N", [(2, 3_000_001), (64, 952_696)])
def test_relaxed_curves(engine, cloud, T, N):
    """Curves F [N, T, 2] whose row t is the cloud turned t quarter turns: the count is sum_t tri_count(row t), from
    the four distinct rows.  T = 2 at 3 M curves wrapped in every row; T = 64, N = 952 696 is the largest accepted,
    and the 128 instances of two queries take three batches (60 per batch at this N)."""
    R = rotations(cloud[:N])
    F = np.stack([R[t % 4] for t in range(T)], axis=1)
    qs = [int(np.argmin((R[0] * R[0]).sum(axis=1))), int(np.random.default_rng(T).integers(N))]
    exp = [sum(_ref("rot%d" % (t % 4), R[t % 4], q) for t in range(T)) for q in qs]
    assert engine.simplex_depth_counts(F, qs, True, 0.0).tolist() == exp


@pytest.mark.gpu
def test_refusals_at_the_first_size_that_overflows(engine, oracle, cloud):
    """SD_ERR_OVERFLOW one past each largest accepted size, on every entry point that counts triangles, and through
    PointcloudDepth; the context stays usable.  Halfspace depth reduces the same keys to numerators <= T n and is
    not refused on the same cloud."""
    from statdepth_b200 import PointcloudDepth
    P = cloud  # 3 810 781 points
    _overflows(lambda: engine.simplicial_counts(P, [0], 0.0))
    _still_usable(engine, oracle)
    _overflows(lambda: engine.simplicial_counts(P, [1, 2]))
    _still_usable(engine, oracle)
    _overflows(lambda: PointcloudDepth(pd.DataFrame(P), to_compute=[3]))
    _still_usable(engine, oracle)
    _overflows(lambda: engine.simplicial_oos_counts(P[:3_810_780], np.zeros((1, 2))))
    _still_usable(engine, oracle)
    _overflows(lambda: engine.simplex_depth_counts(P.reshape(-1, 1, 2), [0], True, 0.0))
    _still_usable(engine, oracle)
    R = rotations(P[:3_024_619])
    _overflows(lambda: engine.simplex_depth_counts(np.stack(R[:2], axis=1), [0], True))
    _still_usable(engine, oracle)
    R = rotations(P[:952_697])
    _overflows(lambda: engine.simplex_depth_counts(np.stack([R[t % 4] for t in range(64)], axis=1), [0], True, 0.0))
    _still_usable(engine, oracle)
    for q in (0, int(np.argmin((P * P).sum(axis=1))), N_MAX - 1):
        assert engine.halfspace_counts(P, [q]).tolist() == np_halfspace_sorted(P, [q]).tolist()
