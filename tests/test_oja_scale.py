"""2-D Oja depth by angular prefix sums (csrc/simplicial_count.cu::oja2_reduce_kernel) against an exact rational
reference: the BASELINE config-5 cloud at full size, every route of the rank pipeline that ranks its keys, tie-heavy
lattices, ill-conditioned clouds (far outliers, a large shift, very different axis scales), the pool route, and
bit-identity between calls.

The reference takes the same float64 differences v = fl(x - p) as the engine, scales them to Python integers and
sums det(v_a, S_a) / 2 exactly, S_a = sum of the v_b strictly inside the half-turn counter-clockwise of a.  The bar is
DESIGN §4's float64 bar: |got - exact| <= 1e-12 * exact.

One approximation of the kernel is not modelled: its angular keys are correctly rounded, so two directions less than
about 2^-48 rad apart can share a key and then add 0 instead of det(v_a, v_b) <= |v_a| |v_b| 2^-48.  On the clouds
below such pairs are rare (about one per query on the 1e-3 x 1e3 cloud) and each is worth less than 1e-20 of the
value, far inside the bar."""
from fractions import Fraction

import numpy as np
import pytest

RTOL = 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# exact reference
# ---------------------------------------------------------------------------------------------------------------------
def _as_ints(V):
    """float64 [m, 2] -> (object array of Python ints [m, 2], E) with V == I * 2**E exactly."""
    mant, ex = np.frexp(V)
    mant = (mant * 2.0 ** 53).astype(np.int64)  # exact: every significand has 53 bits
    nz = mant != 0
    E = int(ex[nz].min()) - 53 if nz.any() else 0
    sh = np.where(nz, ex - 53 - E, 0)
    out = np.empty(V.shape, dtype=object)
    out.ravel()[:] = [m << s for m, s in zip(mant.ravel().tolist(), sh.ravel().tolist())]
    return out, E


def _exact_sum(V):
    """sum over pairs of |det(v_a, v_b)| / 2 of the rows of V, exactly (a Fraction)."""
    V = V[(V[:, 0] != 0.0) | (V[:, 1] != 0.0)]  # the query itself and its duplicates
    if len(V) < 2:
        return Fraction(0)
    # canonical direction c = v in the upper half-plane (angle in [0, pi)), c = -v in the lower one
    upper = (V[:, 1] > 0) | ((V[:, 1] == 0) & (V[:, 0] > 0))
    C = np.where(upper[:, None], V, -V)
    order = np.argsort(np.arctan2(C[:, 1], C[:, 0]), kind="stable")  # float presort; the order is made exact below
    I, E = _as_ints(V[order])
    lower = ~upper[order]
    sgn = np.where(lower, -1, 1)
    cx, cy = (I[:, 0] * sgn).tolist(), (I[:, 1] * sgn).tolist()
    perm = list(range(len(cx)))
    for k in range(1, len(perm)):  # insertion sort by exact cross products: only near-collinear neighbours move
        j = k
        while j > 0:
            a, b = perm[j - 1], perm[j]
            if cx[a] * cy[b] - cy[a] * cx[b] >= 0:
                break
            perm[j - 1], perm[j] = b, a
            j -= 1
    I, lower = I[perm], lower[perm]
    cxs, cys = np.array(cx, dtype=object)[perm], np.array(cy, dtype=object)[perm]
    # classes of equal canonical direction: the same direction, or exactly opposite ones (one in each half-plane)
    starts = np.flatnonzero(np.concatenate(([True], cxs[:-1] * cys[1:] - cys[:-1] * cxs[1:] != 0)))
    zero = np.zeros(len(I), dtype=object)

    def class_sums(mask, col):
        return np.add.reduceat(np.where(mask, I[:, col], zero), starts)

    X = [[class_sums(~lower, 0), class_sums(~lower, 1)], [class_sums(lower, 0), class_sums(lower, 1)]]
    pre = [[np.cumsum(x) - x for x in h] for h in X]  # exclusive prefix sums over the classes
    tot = [[int(np.sum(x)) for x in h] for h in X]
    acc = 0
    for h in (0, 1):
        # the half-turn after a class: the rest of its own half-plane, then the other half-plane's classes before it
        S = [(tot[h][c] - pre[h][c] - X[h][c]) + pre[1 - h][c] for c in (0, 1)]
        acc += int(np.sum(X[h][0] * S[1] - X[h][1] * S[0]))
    return Fraction(acc, 2) * Fraction(2) ** (2 * E)


def exact_oja2(P, queries, pool=None):
    """Oja sums of `queries` (ids into P) over the pairs of `pool` (ids into P; default: all points) without the
    query: (list of exact Fractions, their correctly rounded float64 values)."""
    P = np.ascontiguousarray(P, dtype=np.float64)
    members = np.arange(len(P)) if pool is None else np.asarray(pool, dtype=np.int64)
    ex = [_exact_sum(P[members[members != q]] - P[q]) for q in np.asarray(queries, dtype=np.int64).tolist()]
    return ex, np.array([float(x) for x in ex])


def _pair_loop(P, q, pool=None):
    """The definition, with Fractions: sum over pairs {a, b} of pool \\ {q} of |det(x_a - p, x_b - p)| / 2."""
    members = range(len(P)) if pool is None else pool
    V = [(Fraction(float(P[j, 0] - P[q, 0])), Fraction(float(P[j, 1] - P[q, 1]))) for j in members if j != q]
    s = Fraction(0)
    for i, (ax, ay) in enumerate(V):
        for bx, by in V[i + 1:]:
            s += abs(ax * by - ay * bx)
    return s / 2


def _small_clouds():
    rng = np.random.default_rng(41)
    yield "general", rng.standard_normal((40, 2)), None
    yield "lattice", rng.integers(0, 5, (60, 2)).astype(np.float64), None  # collinear, duplicate, antipodal points
    P = rng.standard_normal((45, 2))
    P[5:12] = P[0]  # duplicates of query 0
    P[12:24] = P[0] + rng.integers(-3, 4, (12, 1)) * (P[1] - P[0])  # a line through query 0, both sides
    yield "duplicates_and_a_line", P, None
    yield "n3", rng.standard_normal((3, 2)), None
    yield "n4", rng.integers(-2, 3, (4, 2)).astype(np.float64), None
    P = rng.integers(-4, 5, (50, 2)).astype(np.float64)
    yield "pool", P, np.array([3, 0, 17, 40, 41, 9, 22, 30, 31, 2, 6])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference against the definition
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,P,pool", list(_small_clouds()), ids=[c[0] for c in _small_clouds()])
def test_reference_equals_the_pair_loop(name, P, pool):
    qs = range(len(P)) if pool is None else list(pool[:6]) + [1, 4]  # 1 and 4 are not pool members
    ex, _ = exact_oja2(P, qs, pool)
    assert ex == [_pair_loop(P, q, pool) for q in qs]


@pytest.mark.parametrize("name,P,pool", list(_small_clouds()), ids=[c[0] for c in _small_clouds()])
def test_reference_agrees_with_the_oracle(oracle, name, P, pool):
    qs = np.arange(len(P)) if pool is None else pool[:6]
    _, f = exact_oja2(P, qs, pool)
    got = oracle.oja(P, 1.0, qs, pool)
    np.testing.assert_allclose(got, f, rtol=1e-14, atol=0)


def test_reference_symmetries():
    rng = np.random.default_rng(5)
    P = rng.standard_normal((300, 2))
    P[10:20] = P[3]
    qs = [0, 3, 7, 150, 299]
    base, _ = exact_oja2(P, qs)
    assert base == exact_oja2(P[:, ::-1], qs)[0]  # swap x and y (a reflection)
    assert base == exact_oja2(-P, qs)[0]
    assert base == exact_oja2(np.stack([-P[:, 1], P[:, 0]], axis=1), qs)[0]  # rotation by 90 degrees
    for k in (-30, 7, 200):
        assert [x * Fraction(2) ** (2 * k) for x in base] == exact_oja2(np.ldexp(P, k), qs)[0]


def test_cases_cover_the_rank_routes():
    """The sizes of test_rank_pipeline_routes put row A (n keys) and row B (2n keys) on either side of every switch
    of the rank pipeline: the slab path takes even rows of 16 384 .. 131 072 values, the part pipeline the rest."""
    from statdepth_b200 import build
    from statdepth_b200._engine import mbd_plan
    build.build()
    slab = {n: (mbd_plan(n)["slab"], mbd_plan(2 * n)["slab"]) for n in ROUTE_SIZES}
    assert slab == {257: (0, 0), 8191: (0, 0), 8192: (0, 1), 16383: (0, 1), 16384: (1, 1), 50000: (1, 1),
                    50001: (0, 1), 65536: (1, 1), 65537: (0, 0), 131072: (1, 0), 131074: (0, 0)}


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
ROUTE_SIZES = (257, 8191, 8192, 16383, 16384, 50000, 50001, 65536, 65537, 131072, 131074)


def oja_batch(n):
    """Queries per batch of oja2_count_device (its IB for a pool of n points)."""
    return max(1, min(32768, (3 << 30) // (88 * n)))


def cfg5_cloud():
    from statdepth_b200.testing import generate_noisy_pointcloud
    return np.ascontiguousarray(generate_noisy_pointcloud(n=50_000, d=2, seed=4).values)


def bench_queries():
    return np.arange(2048, dtype=np.int64) * 24  # bench.py's cfg5_oja_depth sample


def lattice_cloud():
    return np.random.default_rng(8).integers(0, 40, (50_000, 2)).astype(np.float64)


def outlier_cloud():
    """Normal bulk and one far point at each of R = 1e2 .. 1e6 (ids 0 .. 4)."""
    rng = np.random.default_rng(9)
    P = rng.standard_normal((50_000, 2))
    for i, R in enumerate((1e2, 1e3, 1e4, 1e5, 1e6)):
        t = rng.uniform(0, 2 * np.pi)
        P[i] = R * np.cos(t), R * np.sin(t)
    return P, [0, 1, 2, 3, 4, 5, 25_000, 49_999]


def shifted_cloud():
    return 1e6 + 1e-3 * np.random.default_rng(10).standard_normal((50_000, 2)), [0, 7, 31_000, 49_999]


def anisotropic_cloud():
    return np.random.default_rng(11).standard_normal((50_000, 2)) * [1e-3, 1e3], [0, 7, 31_000, 49_999]


def max_rel_err(got, exact):
    return float(np.max(np.abs(np.asarray(got) - exact) / np.abs(exact)))


def check_exact(engine, P, queries, pool=None, got=None):
    """engine.oja with hull volume 1 (the bare sums) against the exact reference; returns the largest relative error."""
    if got is None:
        got = engine.oja(P, 1.0, queries, pool)
    _, exact = exact_oja2(P, queries, pool)
    err = max_rel_err(got, exact)
    assert err <= RTOL, "largest relative error %.3e" % err
    return err


def extreme_queries(P, val):
    """The farthest point from the mean and the deepest point (smallest Oja sum)."""
    return [int(np.argmax(((P - P.mean(0)) ** 2).sum(1))), int(np.argmin(val))]


@pytest.mark.gpu
def test_config5_cloud_exact(engine):
    """BASELINE config 5 at full size (the cloud bench.py times): the farthest and the deepest point and every 64th
    query of the bench's sample, pinned by the exact reference."""
    P = cfg5_cloud()
    allv = engine.oja(P, 1.0)
    q = extreme_queries(P, allv) + bench_queries()[::64].tolist()
    check_exact(engine, P, q, got=allv[q])


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROUTE_SIZES)
def test_rank_pipeline_routes(engine, n):
    """Pool sizes on either side of every switch of the rank pipeline (see test_cases_cover_the_rank_routes)."""
    P = np.random.default_rng(n).standard_normal((n, 2))
    check_exact(engine, P, [0, n // 3, n - 1])


@pytest.mark.gpu
def test_several_batches(engine):
    """n = 300 000 with more queries than one batch holds: the queries on either side of the batch boundary against
    the exact reference, every query bit-identical to the same query asked alone."""
    n = 300_000
    ib = oja_batch(n)
    nq = ib + 38
    P = np.random.default_rng(12).standard_normal((n, 2))
    q = np.random.default_rng(13).choice(n, nq, replace=False)
    got = engine.oja(P, 1.0, q)
    pick = [0, ib - 1, ib, nq - 1]
    check_exact(engine, P, q[pick], got=got[pick])
    alone = np.array([engine.oja(P, 1.0, [int(x)])[0] for x in q])
    assert got.tobytes() == alone.tobytes()


@pytest.mark.gpu
def test_tie_heavy_lattice(engine):
    """50 000 points of the 40 x 40 integer lattice: about 31 copies of every query (zero vectors), collinear classes
    that share a rank bucket, exact antipodes, and key rows too tie-heavy for the slab path."""
    P = lattice_cloud()
    q = [0, 1, 2, 3, 4, 17, 25_000, 49_999]
    check_exact(engine, P, q)


@pytest.mark.gpu
@pytest.mark.parametrize("make", [outlier_cloud, shifted_cloud, anisotropic_cloud])
def test_ill_conditioned_clouds(engine, make):
    """Far outliers (R = 1e2 .. 1e6: at such a query every direction is nearly parallel to the half-turn sums), a
    cloud shifted by 1e6 with spread 1e-3, and axes scaled by 1e-3 and 1e3."""
    P, q = make()
    check_exact(engine, P, q)


@pytest.mark.gpu
def test_pool_route(engine):
    """A 5 000-member pool of a 50 000-point cloud with its queries inside it (counted), and a query outside a
    300-member pool (the enumeration kernel)."""
    rng = np.random.default_rng(14)
    P = rng.standard_normal((50_000, 2))
    pool = rng.choice(50_000, 5000, replace=False)
    check_exact(engine, P, pool[[0, 1, 2500, 4999]], pool)
    small = pool[:300]
    check_exact(engine, P, [int(pool[300]), int(small[7])], small)


@pytest.mark.gpu
@pytest.mark.parametrize("make", [cfg5_cloud, lattice_cloud])
def test_bit_identical_across_calls(engine, make):
    """Two identical calls return identical bits, and a query's value does not depend on the other queries of the
    call or on the batch it lands in (2048 queries of 50 000 points take several batches)."""
    P = make()
    q = bench_queries()
    a = engine.oja(P, 1.0, q)
    b = engine.oja(P, 1.0, q)
    assert a.tobytes() == b.tobytes()
    sub = q[::-97]
    assert engine.oja(P, 1.0, sub).tobytes() == a[::-97].tobytes()
    assert engine.oja(P, 1.0, q[-1:]).tobytes() == a[-1:].tobytes()
