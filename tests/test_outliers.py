"""Functional outlier detection (FunctionalBoxplot / Outliergram and the sd_band_rank_sums / sd_band_envelope
entry points).

The contract: b_t(c) / a_t(c) = other curves strictly below / above curve c at row t; per curve
Q = sum_t [C(n-1,2) - C(b,2) - C(a,2)], B = sum_t b, A = sum_t a; the outliergram's D = (n+1) U T - U^2 - T Q - n T^2
with U = n T - B; the boxplot's central region is the ceil(central n) curves of largest Q (ties by position), its
fences lo - f / hi + f with f = factor (hi - lo).  The CPU part pins a numpy oracle to the C oracle and drives the host
layer with an engine of its own answering from numpy; the GPU part pins the CUDA engine to the same oracle."""
import math
import os
import socket
import sys
from fractions import Fraction

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp
from scipy.special import binom

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------
# numpy oracle
# ---------------------------------------------------------------------------------------------------------------
def np_ranks(X):
    """(b, a) int64 [T, n] by searchsorted on each sorted row."""
    X = np.asarray(X, dtype=np.float64)
    T, n = X.shape
    b = np.empty((T, n), dtype=np.int64)
    a = np.empty((T, n), dtype=np.int64)
    for t in range(T):
        s = np.sort(X[t])
        b[t] = np.searchsorted(s, X[t], side='left')
        a[t] = n - np.searchsorted(s, X[t], side='right')
    return b, a


def np_rank_sums(X):
    """(Q, B, A) int64 [n], row by row (full-size inputs never hold a [T, n] rank matrix)."""
    X = np.asarray(X, dtype=np.float64)
    T, n = X.shape
    q = np.zeros(n, dtype=np.int64)
    bs = np.zeros(n, dtype=np.int64)
    as_ = np.zeros(n, dtype=np.int64)
    full = (n - 1) * (n - 2) // 2
    for t in range(T):
        b, a = np_ranks(X[t:t + 1])
        b, a = b[0], a[0]
        q += full - b * (b - 1) // 2 - a * (a - 1) // 2
        bs += b
        as_ += a
    return q, bs, as_


def np_envelope(X, member, factor, want_outside=True):
    """(lo, hi, outside) with the fences formed as three separately rounded numpy operations."""
    X = np.asarray(X, dtype=np.float64)
    sel = X[:, np.asarray(member, dtype=bool)]
    lo, hi = sel.min(axis=1), sel.max(axis=1)
    f = factor * (hi - lo)
    lower, upper = lo - f, hi + f
    outside = ((X < lower[:, None]) | (X > upper[:, None])).sum(axis=0).astype(np.int64) if want_outside else None
    return lo, hi, outside


def np_distance_ints(q, b, T, n):
    """D in Python integers."""
    return [(n + 1) * (n * T - int(bb)) * T - (n * T - int(bb)) ** 2 - T * int(qq) - n * T * T for qq, bb in zip(q, b)]


def np_boxplot(X, factor=1.5, central=0.5):
    X = np.asarray(X, dtype=np.float64)
    T, n = X.shape
    q, _, _ = np_rank_sums(X)
    k = max(1, math.ceil(Fraction(central) * n))
    order = sorted(range(n), key=lambda c: (-int(q[c]), c))
    member = np.zeros(n, dtype=np.uint8)
    member[order[:k]] = 1
    lo, hi, outside = np_envelope(X, member, factor)
    f = factor * (hi - lo)
    wlo, whi, _ = np_envelope(X, outside == 0, 0.0, False)
    depth = np.zeros(n) + (q.astype(np.float64) / float(T)) / binom(n, 2)
    return dict(q=q, central=order[:k], envelope=(lo, hi), fences=(lo - f, hi + f), whiskers=(wlo, whi),
                outside=outside, depth=depth)


def np_outliergram(X, factor=1.5):
    X = np.asarray(X, dtype=np.float64)
    T, n = X.shape
    q, b, _ = np_rank_sums(X)
    D = np_distance_ints(q, b, T, n)
    denom = T * T * (n * (n - 1) // 2)
    d = np.array([float(v) for v in D]) / float(denom)
    mei = (n * T - b).astype(np.float64) / float(n * T)
    q1, q3 = np.percentile(d, [25, 75])
    depth = np.zeros(n) + (q.astype(np.float64) / float(T)) / binom(n, 2)
    return dict(q=q, D=D, distance=d, mei=mei, outlier=d >= q3 + factor * (q3 - q1), depth=depth)


# ---------------------------------------------------------------------------------------------------------------
# CPU test double
# ---------------------------------------------------------------------------------------------------------------
class OutlierOracleEngine:
    """TEST DOUBLE: the Engine methods the outlier drivers call, answered by numpy (not an Engine, so the drivers hand
    it the host rows)."""

    def __init__(self):
        from oracle import cpu_oracle
        self.o = cpu_oracle
        self.calls = 0

    def band_depth_counts(self, X, queries=None, j=2, relax=False):
        assert queries is None and j == 2 and relax
        self.calls += 1
        return self.o.mbd_counts_all(np.ascontiguousarray(X, dtype=np.float64))

    def band_rank_sums(self, X, want_above=False):
        self.calls += 1
        q, b, a = np_rank_sums(X)
        return (q, b, a) if want_above else (q, b)

    def band_envelope(self, X, member, factor, want_outside=True):
        self.calls += 1
        return np_envelope(X, member, factor, want_outside)


def _install(fake, setter):
    import statdepth_b200._functional as f
    import statdepth_b200._outliers as o
    setter(o, "get_engine", lambda device=None: fake)
    setter(f, "get_engine", lambda device=None: fake)  # FunctionalDepth, for the bit-identity checks


@pytest.fixture()
def outlier_oracle(monkeypatch):
    fake = OutlierOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _walks(T, n, seed, labels=None, index=None):
    X = np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)
    return pd.DataFrame(X, columns=labels if labels is not None else range(n), index=index)


def _planted(seed=0, T=120, n=60):
    """Noisy level-shifted copies of one trend; curve 7 (level in the lower tenth, so outside the central half) lifted
    by 10x the spread over a window (magnitude), curve 11 a half-period phase shift of the trend at level 0 (shape,
    inside the range of the others).  A lift on a mid-level curve can leave it among the deepest half, since MBD
    averages over time, and the central envelope then includes it."""
    rng = np.random.default_rng(seed)
    t = np.arange(T) / T
    trend = 0.5 * np.sin(2 * np.pi * t)
    levels = rng.uniform(-1.25, 1.25, n)
    levels[7] = -1.05
    X = trend[:, None] + levels[None, :] + 0.05 * rng.standard_normal((T, n))
    spread = X.max() - X.min()
    X[50:60, 7] += 10 * spread
    X[:, 11] = 0.5 * np.sin(2 * np.pi * t + np.pi)
    return pd.DataFrame(X, columns=['c%d' % k for k in range(n)])


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracle and the arithmetic
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tied", [False, True])
def test_numpy_oracle_matches_c_oracle(oracle, tied):
    X = np.random.default_rng(1).standard_normal((23, 41)).cumsum(0)
    if tied:
        X = np.round(X)
        X[:, 3] = X[:, 9]
    q, bs, as_ = np_rank_sums(X)
    cnt, rb, ra = oracle.mbd_counts_all(X, want_ranks=True)
    b, a = np_ranks(X)
    assert (b == rb).all() and (a == ra).all()
    assert (q == cnt).all()
    assert (bs == rb.sum(0)).all() and (as_ == ra.sum(0)).all()


def test_distance_equals_papers_float_formula():
    from statdepth_b200._outliers import outliergram_distance
    for seed, (T, n) in enumerate(((30, 50), (200, 17), (64, 300))):
        X = np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)
        q, b, _ = np_rank_sums(X)
        mei, d = outliergram_distance(q, b, T, n)
        mbd_paper = q / T / binom(n, 2) + 2.0 / n
        a0 = a2 = -2.0 / (n * (n - 1))
        a1 = 2.0 * (n + 1) / (n - 1)
        np.testing.assert_allclose(mei, (n * T - b) / (n * T), rtol=0)
        paper = a0 + a1 * mei + a2 * n * n * mei ** 2 - mbd_paper
        np.testing.assert_allclose(d, paper, rtol=1e-9, atol=1e-12)
        assert (d >= 0).all()


def test_distance_zero_on_shifted_copies_positive_on_crossing():
    from statdepth_b200._outliers import outliergram_distance
    T, n = 40, 12
    base = np.random.default_rng(0).standard_normal(T).cumsum()
    X = base[:, None] + np.arange(n)[None, :] * 3.0
    q, b, _ = np_rank_sums(X)
    D = np_distance_ints(q, b, T, n)
    assert D == [0] * n
    assert (outliergram_distance(q, b, T, n)[1] == 0).all()
    X[:, 5] = X[:, 0] + np.linspace(0, 3.0 * (n - 1), T)  # climbs from the bottom to the top: crosses every curve
    q, b, _ = np_rank_sums(X)
    D = np_distance_ints(q, b, T, n)
    assert D[5] > 0
    assert outliergram_distance(q, b, T, n)[1][5] > 0


def test_distance_python_int_path_matches_int64_path():
    from statdepth_b200._outliers import outliergram_distance
    T, n = 50, 30
    X = np.random.default_rng(3).standard_normal((T, n)).cumsum(0)
    q, b, _ = np_rank_sums(X)
    mei, d = outliergram_distance(q, b, T, n)
    exact = np.array([float(v) for v in np_distance_ints(q, b, T, n)]) / float(T * T * (n * (n - 1) // 2))
    assert d.tolist() == exact.tolist()
    # the same sums past the int64 bound: (n + 1) n T^2 >= 2^63 takes Python integers
    Tb = 3 * 10 ** 6
    nb = 10 ** 6
    qb = np.full(2, (nb - 1) * (nb - 2) // 2 * Tb // 2, dtype=np.int64)
    bb = np.array([Tb * (nb - 1) // 2, Tb * (nb - 1) // 3], dtype=np.int64)
    assert (nb + 1) * nb * Tb * Tb >= 2 ** 63
    _, db = outliergram_distance(qb, bb, Tb, nb)
    exp = np.array([float(v) for v in np_distance_ints(qb, bb, Tb, nb)]) / float(Tb * Tb * (nb * (nb - 1) // 2))
    assert db.tolist() == exp.tolist()


# ---------------------------------------------------------------------------------------------------------------
# CPU: host layer on the test double
# ---------------------------------------------------------------------------------------------------------------
def test_boxplot_equals_oracle_with_labels(outlier_oracle):
    from statdepth_b200 import FunctionalBoxplot, FunctionalDepth
    from statdepth_b200.depth import _FunctionalDepthUnivariate
    idx = pd.Index(['t%02d' % k for k in range(19)])
    df = _walks(19, 25, 4, labels=['c%d' % k for k in range(24)] + [('tuple', 1)], index=idx)
    df.iloc[3:6, 4] += 40.0
    res = FunctionalBoxplot([df])
    exp = np_boxplot(df.values)
    cols = list(df.columns)
    assert res.central_region() == [cols[c] for c in exp['central']]
    assert res.median() == cols[exp['central'][0]]
    for name in ('envelope', 'fences', 'whiskers'):
        frame = getattr(res, name)()
        assert list(frame.columns) == ['lower', 'upper'] and frame.index.equals(idx)
        assert frame['lower'].tolist() == exp[name][0].tolist(), name
        assert frame['upper'].tolist() == exp[name][1].tolist(), name
    assert res.outside_counts().tolist() == exp['outside'].tolist()
    assert list(res.outside_counts().index) == cols
    assert res.outliers() == [cols[c] for c in np.flatnonzero(exp['outside'] > 0)]
    assert 'c4' in res.outliers()
    d = res.depths()
    assert isinstance(d, _FunctionalDepthUnivariate)
    assert d.values.tolist() == FunctionalDepth([df], J=2, relax=True).values.tolist()
    assert list(d.index) == cols


def test_boxplot_central_region_tie_rule(outlier_oracle):
    from statdepth_b200 import FunctionalBoxplot
    # curves 1 and 3 and curves 0 and 4 are equal pairs: equal depth; the middle curves 2 / 5 are deepest ties too
    T = 6
    base = np.random.default_rng(0).standard_normal(T).cumsum()
    X = np.column_stack([base - 2, base + 1, base + 3, base + 1, base - 2, base + 3, base - 5, base + 7])
    df = pd.DataFrame(X, columns=list('abcdefgh'))
    q, _, _ = np_rank_sums(X)
    assert q[1] == q[3] and q[2] == q[5] and q[0] == q[4]
    res = FunctionalBoxplot([df], central=0.5)
    order = sorted(range(8), key=lambda c: (-int(q[c]), c))
    assert res.central_region() == [df.columns[c] for c in order[:4]]
    for c1, c2 in ((1, 3), (2, 5), (0, 4)):  # within a tie, the earlier column comes first
        labels = [df.columns[c] for c in order]
        assert labels.index(df.columns[c1]) < labels.index(df.columns[c2])
    assert res.median() == df.columns[order[0]]
    one = FunctionalBoxplot([df], central=0.01)  # ceil(0.08) = 1 curve
    assert one.central_region() == [df.columns[order[0]]]
    assert one.envelope()['lower'].tolist() == X[:, order[0]].tolist()


def test_boxplot_factor_zero_and_full_central(outlier_oracle):
    from statdepth_b200 import FunctionalBoxplot
    df = _walks(15, 20, 7)
    for factor, central in ((0.0, 0.5), (1.5, 1.0), (0, 1), (3, 0.3)):
        res = FunctionalBoxplot([df], factor=factor, central=central)
        exp = np_boxplot(df.values, factor=float(factor), central=central)
        assert res.fences()['lower'].tolist() == exp['fences'][0].tolist()
        assert res.fences()['upper'].tolist() == exp['fences'][1].tolist()
        assert res.outside_counts().tolist() == exp['outside'].tolist()
        assert res.whiskers()['upper'].tolist() == exp['whiskers'][1].tolist()
        if central == 1:  # every curve is central: nothing is outside
            assert res.outliers() == [] and len(res.central_region()) == 20
        if factor == 0:
            assert res.fences().equals(res.envelope())
    assert len(FunctionalBoxplot([df], central=0.3).central_region()) == 6  # exact ceil(0.3 * 20)


def test_outliergram_equals_oracle(outlier_oracle):
    from statdepth_b200 import FunctionalDepth, Outliergram
    df = _walks(31, 27, 5, labels=['x%d' % k for k in range(27)], index=pd.RangeIndex(100, 131))
    res = Outliergram([df])
    exp = np_outliergram(df.values)
    assert res.mei().tolist() == exp['mei'].tolist()
    assert res.distance().tolist() == exp['distance'].tolist()
    assert list(res.distance().index) == list(df.columns)
    assert res.outliers() == [df.columns[c] for c in np.flatnonzero(exp['outlier'])]
    assert res.depths().values.tolist() == FunctionalDepth([df], J=2, relax=True).values.tolist()
    res0 = Outliergram([df], factor=0)
    assert res0.outliers() == [df.columns[c] for c in np.flatnonzero(np_outliergram(df.values, 0.0)['outlier'])]


def test_planted_outliers():
    """On the oracle engine: the lifted curve is a magnitude outlier, the phase-shifted one a shape outlier only."""
    fake = OutlierOracleEngine()
    import statdepth_b200._outliers as o
    from statdepth_b200 import FunctionalBoxplot, Outliergram
    saved = o.get_engine
    o.get_engine = lambda device=None: fake
    try:
        df = _planted()
        box = FunctionalBoxplot([df])
        og = Outliergram([df])
    finally:
        o.get_engine = saved
    assert 'c7' in box.outliers()
    assert 'c11' not in box.outliers()
    assert 'c11' in og.outliers()
    lo, hi = df.drop(columns='c11').min(axis=1), df.drop(columns='c11').max(axis=1)
    assert ((df['c11'] >= lo) & (df['c11'] <= hi)).all()  # inside the range of the others at every time point


def test_validation_errors(outlier_oracle):
    from statdepth_b200 import DepthDegeneracy, FunctionalBoxplot, Outliergram  # noqa: F401
    df = _walks(8, 10, 0)
    for fn in (FunctionalBoxplot, Outliergram):
        with pytest.raises(ValueError):
            fn(df)                                   # not a list
        with pytest.raises(ValueError):
            fn([])
        with pytest.raises(ValueError):
            fn([df.iloc[:2]])                        # J = 2 >= number of time points (the depth's own check)
        with pytest.raises(ValueError):
            fn([df], deep_check=1)
        with pytest.raises(ValueError):
            fn([df.iloc[:, :1]])                     # one curve
        for bad in (-0.5, float('nan'), float('inf'), True, '1.5', None):
            with pytest.raises(ValueError):
                fn([df], factor=bad)
        mv = [_walks(8, 2, k) for k in range(5)]
        with pytest.raises(NotImplementedError):
            fn(mv)
    for bad in (0, 0.0, -0.1, 1.0000001, float('nan'), True, None):
        with pytest.raises(ValueError):
            FunctionalBoxplot([df], central=bad)
    assert outlier_oracle.calls == 0  # every refusal happens before any engine call


# ---------------------------------------------------------------------------------------------------------------
# CPU: two ranks (gloo) shard time rows
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dist_input():
    df = _walks(13, 22, 11)  # 13 rows: uneven split 7 + 6
    df.iloc[2:4, 6] -= 30.0
    return df


def _results(df):
    from statdepth_b200 import FunctionalBoxplot, Outliergram
    box = FunctionalBoxplot([df], factor=1.0)
    og = Outliergram([df])
    return dict(depth=box.depths().values, central=np.array(box.central_region()),
                env=box.envelope().values, fences=box.fences().values, whiskers=box.whiskers().values,
                outside=box.outside_counts().values, mei=og.mei().values, distance=og.distance().values,
                og_depth=og.depths().values)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(OutlierOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results(_dist_input()))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(OutlierOracleEngine(), monkeypatch.setattr)
    exp = _results(_dist_input())
    assert exp['outside'].sum() > 0
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("T,n,slab", [(12, 20_000, 1), (16, 5_000, 0), (6, 200_000, 0)])
def test_rank_sums_equal_band_depth_and_oracle(engine, T, n, slab):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(n)["slab"] == slab
    X = np.random.default_rng(n).standard_normal((T, n)).cumsum(0)
    q, b, a = engine.band_rank_sums(X, want_above=True)
    assert (q == engine.band_depth_counts(X, None, 2, True)).all()
    eq, eb, ea = np_rank_sums(X)
    assert (q == eq).all() and (b == eb).all() and (a == ea).all()


@pytest.mark.gpu
def test_rank_sums_ties_and_layouts(engine):
    rng = np.random.default_rng(5)
    for T, n in ((9, 37), (17, 3001), (5, 20_000)):
        X = np.round(rng.standard_normal((T, n)).cumsum(0))
        X[:, 1] = X[:, 2]
        eq, eb, ea = np_rank_sums(X)
        for M in (X, np.asfortranarray(X)):  # C order: SD_LAYOUT_TN; F order: SD_LAYOUT_NT
            q, b, a = engine.band_rank_sums(M, want_above=True)
            assert (q == eq).all() and (b == eb).all() and (a == ea).all()
        q2, b2 = engine.band_rank_sums(X)
        assert (q2 == eq).all() and (b2 == eb).all()


@pytest.mark.gpu
def test_rank_sums_two_row_blocks(engine):
    """100 000 x 2048: the 1 GB rank workspace holds 1342 rows, so two row blocks; every below is someone's above."""
    import torch
    T, n = 2048, 100_000
    dX = torch.randn((T, n), dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    dX = dX.cumsum(0)
    out = torch.zeros((3, n), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    engine.band_rank_sums_dev(dX.data_ptr(), T, n, n, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr())
    q, b, a = out.cpu().numpy()
    assert b.sum() == a.sum()
    assert b.sum() + a.sum() <= T * n * (n - 1)
    ref = torch.zeros(n, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    engine.band_depth_counts_dev(dX.data_ptr(), T, n, n, ref.data_ptr(), None, n, 2, True)
    assert (ref.cpu().numpy() == q).all()


@pytest.mark.gpu
def test_envelope_equals_numpy(engine):
    rng = np.random.default_rng(9)
    cases = []
    for T, n in ((7, 1001), (1, 333), (3, 40), (2, 300_000), (1, 50_000)):  # the last two split rows into chunks
        X = rng.standard_normal((T, n)).cumsum(0) - 5.0
        X[:, n // 2] = X[:, 3]                   # ties
        cases.append((X, rng.random(n) < 0.4))
        one = np.zeros(n, dtype=bool)
        one[n - 1] = True                        # a single member: the envelope is that curve
        cases.append((X, one))
    Xt = np.round(rng.standard_normal((11, 257)))  # tie-heavy, with -0.0 and 0.0
    Xt[0, :5] = [-0.0, 0.0, -0.0, 1.0, -1.0]
    cases.append((Xt, rng.random(257) < 0.5))
    for X, member in cases:
        for factor in (1.5, 0.0, 0.25):
            lo, hi, out = engine.band_envelope(X, member, factor)
            elo, ehi, eout = np_envelope(X, member, factor)
            assert lo.tolist() == elo.tolist() and hi.tolist() == ehi.tolist()
            assert out.tolist() == eout.tolist(), (X.shape, factor)
            lo2, hi2, none = engine.band_envelope(np.asfortranarray(X), member, factor, want_outside=False)
            assert none is None and lo2.tolist() == elo.tolist() and hi2.tolist() == ehi.tolist()


@pytest.mark.gpu
def test_envelope_device_variant_and_empty_member(engine):
    import torch
    from statdepth_b200 import EngineError
    T, n = 5, 700
    X = np.random.default_rng(2).standard_normal((T, n))
    member = np.zeros(n, dtype=np.uint8)
    member[::3] = 1
    dX = torch.from_numpy(X).cuda()
    dm = torch.from_numpy(member).cuda()
    env = torch.zeros((2, T), dtype=torch.float64, device="cuda")
    out = torch.zeros(n, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    engine.band_envelope_dev(dX.data_ptr(), T, n, n, dm.data_ptr(), 0.5, env[0].data_ptr(), env[1].data_ptr(),
                             out.data_ptr())
    elo, ehi, eout = np_envelope(X, member, 0.5)
    assert env[0].cpu().numpy().tolist() == elo.tolist() and env[1].cpu().numpy().tolist() == ehi.tolist()
    assert out.cpu().numpy().tolist() == eout.tolist()
    with pytest.raises(EngineError) as ei:
        engine.band_envelope(X, np.zeros(n, dtype=np.uint8), 1.5)
    assert ei.value.status == 1
    for bad in (-1.0, float('inf'), float('nan')):
        with pytest.raises(EngineError):
            engine.band_envelope(X, member, bad)
    assert engine.band_envelope(X, member, 1.5)[2].shape == (n,)  # the context stays usable


@pytest.mark.gpu
def test_nonfinite_rejected(engine):
    from statdepth_b200 import EngineError, FunctionalBoxplot, Outliergram
    X = np.random.default_rng(0).standard_normal((16, 90)).cumsum(0)
    member = np.ones(90, dtype=np.uint8)
    for bad in (np.nan, np.inf, -np.inf):
        Y = X.copy()
        Y[7, 33] = bad
        with pytest.raises(EngineError) as ei:
            engine.band_rank_sums(Y)
        assert ei.value.status == 4
        with pytest.raises(EngineError) as ei:
            engine.band_envelope(Y, member, 1.5)
        assert ei.value.status == 4
        for fn in (FunctionalBoxplot, Outliergram):
            with pytest.raises(EngineError) as ei:
                fn([pd.DataFrame(Y)])
            assert ei.value.status == 4
    assert engine.band_rank_sums(X)[0].shape == (90,)


@pytest.mark.gpu
def test_public_objects_full_size(engine):
    """100 000 curves x 1024 points: both public objects equal the numpy oracle exactly."""
    from statdepth_b200 import FunctionalBoxplot, FunctionalDepth, Outliergram
    T, n = 1024, 100_000
    rng = np.random.default_rng(21)
    X = rng.standard_normal((T, n)).cumsum(0)
    top = int(np.argmax(X[-1]))  # far from the central half, unlike a curve of middling level
    X[400:420, top] += 500.0
    df = pd.DataFrame(X)
    box = FunctionalBoxplot([df])
    og = Outliergram([df])
    eb = np_boxplot(X)
    eo = np_outliergram(X)
    fd = FunctionalDepth([df], J=2, relax=True).values
    assert box.depths().values.tolist() == fd.tolist() and og.depths().values.tolist() == fd.tolist()
    assert box.central_region() == eb['central']
    for name in ('envelope', 'fences', 'whiskers'):
        frame = getattr(box, name)()
        assert frame['lower'].tolist() == eb[name][0].tolist() and frame['upper'].tolist() == eb[name][1].tolist()
    assert box.outside_counts().tolist() == eb['outside'].tolist()
    assert top in box.outliers()
    assert og.mei().tolist() == eo['mei'].tolist()
    assert og.distance().tolist() == eo['distance'].tolist()
    assert og.outliers() == list(np.flatnonzero(eo['outlier']))


@pytest.mark.gpu
def test_planted_outliers_on_gpu(engine):
    from statdepth_b200 import FunctionalBoxplot, Outliergram
    df = _planted(seed=3, T=256, n=2000)
    assert 'c7' in FunctionalBoxplot([df]).outliers()
    assert 'c11' not in FunctionalBoxplot([df]).outliers()
    assert 'c11' in Outliergram([df]).outliers()
