"""Extremal depth (ExtremalDepth, FunctionalBoxplot(depth='extremal') and the sd_band_extremity_f64_dev /
sd_extremal_depth_dev entry points).

The contract: b_t(c) / a_t(c) = other curves strictly below / above curve c at row t; m_t(c) = |b - a|; key(c) = the
m_t(c) sorted descending; keys compare lexicographically, larger = more extreme; e(c) = #{h : key(h) >= key(c)} and
ED = e / n.  The CPU part pins the fast numpy rule to the paper's pairwise comparison of depth CDFs and drives the
host layer with an engine of its own answering from numpy; the GPU part pins the CUDA engine to the fast rule."""
import math
import os
import socket
import sys
from fractions import Fraction

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_MAX = 16384  # SD_EXTREMAL_T_MAX


# ---------------------------------------------------------------------------------------------------------------
# numpy oracles
# ---------------------------------------------------------------------------------------------------------------
def np_extremity(X):
    """m int32 [T, n] = |b - a| by searchsorted on each sorted row."""
    X = np.asarray(X, dtype=np.float64)
    T, n = X.shape
    m = np.empty((T, n), dtype=np.int32)
    for t in range(T):
        s = np.sort(X[t])
        b = np.searchsorted(s, X[t], side='left')
        a = n - np.searchsorted(s, X[t], side='right')
        m[t] = np.abs(b - a)
    return m


def np_extremal(m):
    """The fast rule: e int64 [n] from m [T, n] by sorting every curve's extremities descending and ranking the keys
    as big-endian byte strings (bytewise order == lexicographic order of the integers)."""
    m = np.asarray(m)
    T, n = m.shape
    keys = np.ascontiguousarray((-np.sort(-m.astype(np.int64), axis=0)).T).astype('>u4')
    raw = keys.view(np.dtype((np.void, 4 * T))).ravel()
    _, inv, counts = np.unique(raw, return_inverse=True, return_counts=True)
    at_least = np.cumsum(counts[::-1])[::-1]  # curves in this key group or a larger one
    return at_least[inv.ravel()].astype(np.int64)


def paper_extremal(X):
    """The paper's definition, brute force: with the pointwise depths D_t = 1 - m_t / n (kept as the integers
    n - m_t), g is more extreme than h when Phi_g(r) > Phi_h(r) at the smallest depth level r where the two depth
    CDFs differ; e(c) = #{h : c is not more extreme than h}."""
    m = np_extremity(X).astype(np.int64)
    T, n = m.shape
    levels = n - m                              # D * n

    def phi(c, r):
        return int((levels[:, c] <= r).sum())

    def more_extreme(g, h):
        for r in np.unique(np.concatenate([levels[:, g], levels[:, h]])):  # ascending
            if phi(g, r) != phi(h, r):
                return phi(g, r) > phi(h, r)
        return False

    return np.array([sum(not more_extreme(c, h) for h in range(n)) for c in range(n)], dtype=np.int64)


def np_boxplot(X, score, factor=1.5, central=0.5):
    """Central region, envelope, fences and outside counts ranked by the integer score (ties by column)."""
    X = np.asarray(X, dtype=np.float64)
    n = X.shape[1]
    k = max(1, math.ceil(Fraction(central) * n))
    order = sorted(range(n), key=lambda c: (-int(score[c]), c))
    sel = X[:, order[:k]]
    lo, hi = sel.min(axis=1), sel.max(axis=1)
    f = factor * (hi - lo)
    outside = ((X < (lo - f)[:, None]) | (X > (hi + f)[:, None])).sum(axis=0).astype(np.int64)
    return dict(central=order[:k], envelope=(lo, hi), fences=(lo - f, hi + f), outside=outside)


def np_mbd_numerators(X):
    m = np.asarray(X, dtype=np.float64)
    T, n = m.shape
    q = np.zeros(n, dtype=np.int64)
    for t in range(T):
        s = np.sort(m[t])
        b = np.searchsorted(s, m[t], side='left')
        a = n - np.searchsorted(s, m[t], side='right')
        q += (n - 1) * (n - 2) // 2 - b * (b - 1) // 2 - a * (a - 1) // 2
    return q


def _tied(rng, shape):
    """Values on 8 levels, zeros of both signs."""
    X = rng.integers(-4, 4, size=shape).astype(np.float64) * 0.5
    neg = (X == 0) & (rng.random(shape) < 0.5)
    X[neg] = -0.0
    return X


def _spikes(seed):
    """400 noisy curves around one trend; 8 of them get +8.0 on 4 consecutive rows."""
    rng = np.random.default_rng(seed)
    T, n, k = 128, 400, 8
    t = np.linspace(0, 1, T)
    X = np.sin(2 * np.pi * t)[:, None] + rng.normal(0, 1, (1, n)) * 0.5 + rng.normal(0, 0.3, (T, n))
    spikes = rng.choice(n, k, replace=False)
    for c in spikes:
        t0 = rng.integers(0, T - 4)
        X[t0:t0 + 4, c] += 8.0
    return X, spikes


# ---------------------------------------------------------------------------------------------------------------
# CPU test double
# ---------------------------------------------------------------------------------------------------------------
class ExtremalOracleEngine:
    """TEST DOUBLE: the host methods the outlier drivers call, answered by numpy (no `_dev` methods, so the drivers
    take the host path)."""

    def __init__(self):
        self.calls = 0

    def band_depth_counts(self, X, queries=None, j=2, relax=False):
        assert queries is None and j == 2 and relax
        self.calls += 1
        return np_mbd_numerators(X)

    def band_envelope(self, X, member, factor, want_outside=True):
        self.calls += 1
        X = np.asarray(X, dtype=np.float64)
        sel = X[:, np.asarray(member, dtype=bool)]
        lo, hi = sel.min(axis=1), sel.max(axis=1)
        f = factor * (hi - lo)
        out = ((X < (lo - f)[:, None]) | (X > (hi + f)[:, None])).sum(axis=0).astype(np.int64)
        return lo, hi, out if want_outside else None

    def band_extremity(self, X):
        self.calls += 1
        return np_extremity(X)

    def extremal_depth(self, m):
        self.calls += 1
        assert m.dtype == np.int32
        return np_extremal(m)


def _install(fake, setter):
    import statdepth_b200._functional as f
    import statdepth_b200._outliers as o
    setter(o, "get_engine", lambda device=None: fake)
    setter(f, "get_engine", lambda device=None: fake)


@pytest.fixture()
def extremal_oracle(monkeypatch):
    fake = ExtremalOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _walks(T, n, seed, labels=None):
    X = np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)
    return pd.DataFrame(X, columns=labels if labels is not None else range(n))


# ---------------------------------------------------------------------------------------------------------------
# CPU: the two oracles
# ---------------------------------------------------------------------------------------------------------------
def test_fast_rule_equals_papers_definition():
    rng = np.random.default_rng(2016)
    for case in range(320):
        T, n = int(rng.integers(1, 7)), int(rng.integers(1, 9))
        if case % 2:  # tie-heavy: few levels, repeated curves
            X = rng.integers(0, 3, size=(T, n)).astype(np.float64)
            if n > 1:
                X[:, n - 1] = X[:, 0]
        else:
            X = rng.standard_normal((T, n))
        e = np_extremal(np_extremity(X))
        assert e.tolist() == paper_extremal(X).tolist(), (T, n, X)
        assert e.min() >= 1 and e.max() == n


def test_doc_table_known_answer(golden):
    case = golden["doc_table_J2_strict"]
    X = np.array(case["X"], dtype=np.float64)  # 5 time rows x 6 curves f_0 .. f_5
    assert X.shape == (5, 6)
    e = np_extremal(np_extremity(X))
    assert e.tolist() == [2, 5, 3, 6, 1, 4]
    assert paper_extremal(X).tolist() == [2, 5, 3, 6, 1, 4]


# ---------------------------------------------------------------------------------------------------------------
# CPU: host layer on the test double
# ---------------------------------------------------------------------------------------------------------------
def test_extremal_depth_equals_oracle_with_labels(extremal_oracle, golden):
    from statdepth_b200 import ExtremalDepth
    from statdepth_b200.depth import _FunctionalDepthUnivariate
    case = golden["doc_table_J2_strict"]
    df = pd.DataFrame(case["X"], columns=case["columns"])
    d = ExtremalDepth([df])
    assert isinstance(d, _FunctionalDepthUnivariate)
    assert list(d.index) == case["columns"]
    assert d.values.tolist() == (np.array([2, 5, 3, 6, 1, 4]) / 6.0).tolist()
    assert d.deepest().index[0] == 'f_3' and d.outlying().index[0] == 'f_4'
    df = _walks(17, 33, 3, labels=['c%d' % k for k in range(32)] + [('tuple', 1)])
    d = ExtremalDepth([df])
    exp = np_extremal(np_extremity(df.values)).astype(np.float64) / 33
    assert d.values.tolist() == exp.tolist()
    assert list(d.index) == list(df.columns)


def test_tie_rule(extremal_oracle):
    from statdepth_b200 import ExtremalDepth
    rng = np.random.default_rng(4)
    X = rng.standard_normal((9, 12))
    X[:, 5] = X[:, 2]                   # identical curves
    e = np_extremal(np_extremity(X))
    d = ExtremalDepth([pd.DataFrame(X)]).values
    assert d[5] == d[2]
    assert d.tolist() == (e / 12.0).tolist()
    # permuting the time rows of the whole sample permutes every curve's extremities: no depth changes
    assert ExtremalDepth([pd.DataFrame(X[rng.permutation(9)])]).values.tolist() == d.tolist()
    # a curve whose extremities are a permutation of another's (equal at different times) gets the same e
    Z = np.array([[0.0, 1.0, 2.0], [1.0, 2.0, 0.0], [5.0, 5.0, 0.0]])
    m = np_extremity(Z)
    assert m[:, 0].tolist() == [2, 0, 1] and m[:, 1].tolist() == [0, 2, 1]
    dz = ExtremalDepth([pd.DataFrame(Z)]).values
    assert dz.tolist() == [1.0, 1.0, 1 / 3]


def test_boxplot_extremal_equals_oracle_and_mbd_unchanged(extremal_oracle):
    from statdepth_b200 import ExtremalDepth, FunctionalBoxplot, FunctionalDepth
    df = _walks(19, 25, 4, labels=['c%d' % k for k in range(25)])
    df.iloc[3:6, 4] += 40.0
    X = df.values
    cols = list(df.columns)
    e = np_extremal(np_extremity(X))
    for factor, central in ((1.5, 0.5), (0.0, 0.3), (3, 1)):
        res = FunctionalBoxplot([df], factor=factor, central=central, depth='extremal')
        exp = np_boxplot(X, e, float(factor), central)
        assert res.central_region() == [cols[c] for c in exp['central']]
        assert res.median() == cols[exp['central'][0]]
        for name in ('envelope', 'fences'):
            frame = getattr(res, name)()
            assert frame['lower'].tolist() == exp[name][0].tolist()
            assert frame['upper'].tolist() == exp[name][1].tolist()
        assert res.outside_counts().tolist() == exp['outside'].tolist()
        assert res.depths().values.tolist() == ExtremalDepth([df]).values.tolist()
    assert 'c4' in FunctionalBoxplot([df], depth='extremal').outliers()
    # depth='mbd' is the default, and it is the boxplot ranked by the MBD numerator
    q = np_mbd_numerators(X)
    a, b = FunctionalBoxplot([df]), FunctionalBoxplot([df], 1.5, 0.5, False, 'mbd')
    exp = np_boxplot(X, q)
    for res in (a, b):
        assert res.central_region() == [cols[c] for c in exp['central']]
        assert res.outside_counts().tolist() == exp['outside'].tolist()
        assert res.depths().values.tolist() == FunctionalDepth([df], J=2, relax=True).values.tolist()
        assert res.whiskers().equals(a.whiskers()) and res.fences().equals(a.fences())


def test_planted_spikes(extremal_oracle):
    """A short spike leaves MBD high; extremal depth flags exactly the spiked curves."""
    from statdepth_b200 import ExtremalDepth, FunctionalBoxplot
    for seed in range(5):
        X, spikes = _spikes(seed)
        df = pd.DataFrame(X)
        ed = FunctionalBoxplot([df], factor=1.5, central=0.5, depth='extremal')
        mbd = FunctionalBoxplot([df], factor=1.5, central=0.5)
        assert sorted(ed.outliers()) == sorted(spikes.tolist()), seed
        assert not set(spikes.tolist()) <= set(mbd.outliers()), seed
        d = ExtremalDepth([df]).values
        lowest = np.argsort(d, kind='stable')[:int(0.15 * len(d))]
        assert set(spikes.tolist()) <= set(lowest.tolist()), seed


def test_validation_errors(extremal_oracle):
    from statdepth_b200 import ExtremalDepth, FunctionalBoxplot
    df = _walks(8, 10, 0)
    with pytest.raises(ValueError):
        ExtremalDepth(df)                      # not a list
    with pytest.raises(ValueError):
        ExtremalDepth([])
    with pytest.raises(ValueError):
        ExtremalDepth([df.iloc[:2]])           # J = 2 >= number of time points (the depth's own check)
    with pytest.raises(ValueError):
        ExtremalDepth([df], deep_check=1)
    with pytest.raises(ValueError):
        ExtremalDepth([df.iloc[:, :1]])        # one curve
    with pytest.raises(NotImplementedError):
        ExtremalDepth([_walks(8, 2, k) for k in range(5)])
    for bad in ('MBD', 'extreme', None, 1, ['mbd']):
        with pytest.raises(ValueError):
            FunctionalBoxplot([df], depth=bad)
    with pytest.raises(ValueError):
        FunctionalBoxplot([df], factor=-1.0, depth='extremal')
    big = pd.DataFrame(np.zeros((T_MAX + 1, 3)))
    with pytest.raises(NotImplementedError):
        ExtremalDepth([big])
    with pytest.raises(NotImplementedError):
        FunctionalBoxplot([big], depth='extremal')
    assert extremal_oracle.calls == 0  # every refusal happens before any engine call
    ExtremalDepth([pd.DataFrame(np.zeros((T_MAX, 3)))])  # the bound itself is accepted


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


def _results():
    from statdepth_b200 import ExtremalDepth, FunctionalBoxplot
    from statdepth_b200._outliers import _extremal_depth
    df = _dist_input()
    box = FunctionalBoxplot([df], factor=1.0, depth='extremal')
    one_row = np.random.default_rng(3).standard_normal((1, 15))  # T = 1: one rank holds no rows
    return dict(ed=ExtremalDepth([df]).values, central=np.array(box.central_region()),
                env=box.envelope().values, outside=box.outside_counts().values, box_depth=box.depths().values,
                t1=_extremal_depth(one_row))


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(ExtremalOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(ExtremalOracleEngine(), monkeypatch.setattr)
    exp = _results()
    assert exp['t1'].tolist() == np_extremal(np_extremity(np.random.default_rng(3).standard_normal((1, 15)))).tolist()
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the fast rule
# ---------------------------------------------------------------------------------------------------------------
def _dev_extremity(engine, X):
    import torch
    T, n = X.shape
    dX = torch.from_numpy(np.ascontiguousarray(X, dtype=np.float64)).cuda()
    m = torch.full((T, n), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    engine.band_extremity_dev(dX.data_ptr(), T, n, n, m.data_ptr())
    return m.cpu().numpy()


def _dev_extremal(engine, m):
    import torch
    T, n = m.shape
    dm = torch.from_numpy(np.ascontiguousarray(m, dtype=np.int32)).cuda()
    e = torch.zeros(n, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    engine.extremal_depth_dev(dm.data_ptr(), T, n, e.data_ptr())
    return e.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["default", "parts"])
def test_extremity_equals_numpy(engine, monkeypatch, path):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(20_000)["slab"] == 1
    if path == "parts":
        monkeypatch.setenv("SD_MBD_PATH", "parts")
        assert mbd_plan(20_000)["slab"] == 0
    rng = np.random.default_rng(8)
    cases = [rng.standard_normal((12, 20_000)).cumsum(0),   # slab path by default
             rng.standard_normal((16, 5_000)).cumsum(0),
             rng.standard_normal((3, 200_000)).cumsum(0),
             _tied(rng, (9, 30_000)), _tied(rng, (7, 37)),
             rng.standard_normal((1, 3001)), rng.standard_normal((2, 20_000)), rng.standard_normal((1, 2))]
    for X in cases:
        assert _dev_extremity(engine, X).tolist() == np_extremity(X).tolist(), X.shape


def _keys_cases():
    rng = np.random.default_rng(33)
    out = []
    for T in (1, 2, 31, 32, 33, 1024):
        for n in (2, 3, 1000, 100_000):
            if T * n > 40_000_000:
                continue
            m = rng.integers(0, n, size=(T, n), dtype=np.int32)
            out.append(("random", m))
            if n >= 3:
                d = m.copy()
                d[:, 1] = d[:, 0]                          # duplicated curves
                d[:, n - 1] = d[::-1, 0]                   # a time permutation: the same key
                out.append(("dups", d))
            if n >= 1000:
                lp = np.repeat(m[:, :1], n, axis=1)        # every key shares a long prefix
                lp[-1, :] = rng.integers(0, 3, size=n)     # and differs (if at all) only in the smallest values
                out.append(("prefix", lp))
                X = np.round(rng.standard_normal((T, n)) * 2)
                out.append(("rounded", np_extremity(X)))
    for n in (2, 3, 1000):
        out.append(("bound", rng.integers(0, n, size=(T_MAX, n), dtype=np.int32)))
    return out


@pytest.mark.gpu
def test_extremal_depth_equals_fast_rule(engine):
    for name, m in _keys_cases():
        assert _dev_extremal(engine, m).tolist() == np_extremal(m).tolist(), (name, m.shape)


@pytest.mark.gpu
def test_extremal_depth_one_row_million_curves(engine):
    rng = np.random.default_rng(6)
    n = 1_000_000
    m = rng.integers(0, n, size=(1, n), dtype=np.int32)
    m[0, :1000] = m[0, 1000:2000]
    assert _dev_extremal(engine, m).tolist() == np_extremal(m).tolist()


@pytest.mark.gpu
def test_errors(engine):
    from statdepth_b200 import EngineError, ExtremalDepth
    m = np.random.default_rng(0).integers(0, 50, size=(8, 50), dtype=np.int32)
    for bad in (-1, 50, 2 ** 31 - 1):
        mb = m.copy()
        mb[5, 17] = bad
        with pytest.raises(EngineError) as ei:
            _dev_extremal(engine, mb)
        assert ei.value.status == 1
    with pytest.raises(EngineError) as ei:
        _dev_extremal(engine, np.zeros((T_MAX + 1, 4), dtype=np.int32))
    assert ei.value.status == 1
    X = np.random.default_rng(1).standard_normal((16, 90)).cumsum(0)
    for bad in (np.nan, np.inf, -np.inf):
        Y = X.copy()
        Y[7, 33] = bad
        with pytest.raises(EngineError) as ei:
            _dev_extremity(engine, Y)
        assert ei.value.status == 4
        with pytest.raises(EngineError) as ei:
            ExtremalDepth([pd.DataFrame(Y)])
        assert ei.value.status == 4
    assert _dev_extremal(engine, m).tolist() == np_extremal(m).tolist()  # the context stays usable


def cfg2_walks(T, n, seed):
    """The benchmark's random walks (bench.py Ctx.walks): float64 normals from a seeded CUDA generator in blocks of
    128 rows, summed over time."""
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    X = torch.empty((T, n), dtype=torch.float64, device="cuda")
    for r0 in range(0, T, 128):
        X[r0:r0 + 128] = torch.randn((min(128, T - r0), n), dtype=torch.float64, device="cuda", generator=g)
    return X.cumsum(0).cpu().numpy()


@pytest.mark.gpu
def test_full_size(engine):
    """100 000 random walks x 1024 points (cfg2's generator, seed 1): ED and the ED boxplot equal the oracle."""
    from statdepth_b200 import ExtremalDepth, FunctionalBoxplot
    T, n = 1024, 100_000
    X = cfg2_walks(T, n, 1)
    df = pd.DataFrame(X)
    e = np_extremal(np_extremity(X))
    d = ExtremalDepth([df])
    assert d.values.tolist() == (e.astype(np.float64) / n).tolist()
    box = FunctionalBoxplot([df], depth='extremal')
    exp = np_boxplot(X, e)
    assert box.central_region() == exp['central']
    assert box.outside_counts().tolist() == exp['outside'].tolist()
    for name in ('envelope', 'fences'):
        frame = getattr(box, name)()
        assert frame['lower'].tolist() == exp[name][0].tolist() and frame['upper'].tolist() == exp[name][1].tolist()


@pytest.mark.gpu
def test_planted_spikes_on_gpu(engine):
    from statdepth_b200 import FunctionalBoxplot
    for seed in range(5):
        X, spikes = _spikes(seed)
        assert sorted(FunctionalBoxplot([pd.DataFrame(X)], depth='extremal').outliers()) == sorted(spikes.tolist())
