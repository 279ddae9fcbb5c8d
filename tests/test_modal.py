"""h-modal depth (FunctionalModalDepth, FunctionalModalDepthOf, FunctionalReference / DepthClassifier with
depth='modal', sd_modal_*): MD(x) = (1 / n) sum_j phi(||x_j - x|| / h), h = np.quantile of the pair distances.

The CPU part pins a numpy oracle against a per-pair loop and closed forms, the host's bandwidth arithmetic against
np.quantile bit for bit, and drives the host layer with a numpy test double.  The GPU part pins the exact pair
selection to the oracle bit for bit on integer-valued curves (every squared distance exact), on each of its routes,
the depths to the oracle within DESIGN K15's bound, and the bit-identities K15 promises."""
import math
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHI0 = 1.0 / math.sqrt(2.0 * math.pi)
U = 2.0 ** -53


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


def np_pair_d2(A):
    """The n (n - 1) / 2 squared distances of the pairs i < j."""
    A = np.asarray(A, dtype=np.float64)
    iu = np.triu_indices(len(A), k=1)
    return np_d2(A, A)[iu]


def int_pair_d2(A):
    """The same for integer-valued curves, exact through a float64 Gram matrix (every product and sum is an integer
    below 2^53)."""
    A = np.asarray(A, dtype=np.float64)
    G = A @ A.T
    sq = np.diag(G)
    iu = np.triu_indices(len(A), k=1)
    return (sq[iu[0]] + sq[iu[1]]) - 2.0 * G[iu]


def np_bandwidth(A, quantile=0.15):
    return float(np.quantile(np.sqrt(np_pair_d2(A)), quantile))


def np_sums(S, Q, c):
    return np.exp(c * np_d2(S, Q)).sum(axis=1)


def np_modal_depth(A, queries=None, quantile=0.15, bandwidth=None):
    A = np.asarray(A, dtype=np.float64)
    q = np.arange(len(A)) if queries is None else np.asarray(queries)
    h = np_bandwidth(A, quantile) if bandwidth is None else bandwidth
    return np_sums(A, A[q], -0.5 / (h * h)) / len(A) * PHI0


def loop_modal_depth(A, q, h):
    """The definition, one pair at a time."""
    x = A[q]
    s = 0.0
    for j in range(A.shape[0]):
        d = math.sqrt(sum(float(t) * float(t) for t in A[j] - x))
        s += math.exp(-0.5 * (d / h) ** 2) / math.sqrt(2 * math.pi)
    return s / A.shape[0]


def depth_bound(n, F):
    """DESIGN K15: |error| of one depth, kernel or oracle, is at most phi(0) u ((2 F + 8) / e + n + 4)."""
    return PHI0 * U * ((2 * F + 8) / math.e + n + 4)


def assert_depths(got, exp, n, F):
    got, exp = np.asarray(got), np.asarray(exp)
    err = np.abs(got - exp)
    assert (err <= 2 * depth_bound(n, F)).all(), (err.max(), 2 * depth_bound(n, F))


def _frames(F):
    return [pd.DataFrame(F[i]) for i in range(F.shape[0])]


class ModalOracleEngine:
    """TEST DOUBLE: the engine methods the modal drivers call, answered by the numpy oracle, refusing non-finite
    input with SD_ERR_NONFINITE as the engine does (not an Engine, so the reference keeps a host sample).  An
    out-of-sample sum runs over the sample with the query appended, as the in-sample sum of that pooled set does."""

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
        d2 = np.sort(np_pair_d2(X))
        return np.array([d2[k], d2[min(k + 1, len(d2) - 1)]])

    def modal_sums(self, X, c, queries=None):
        self._finite(X)
        X = np.asarray(X, dtype=np.float64)
        q = np.arange(len(X)) if queries is None else np.asarray(queries, dtype=np.int64)
        return np_sums(X, X[q], c)

    def modal_sums_of(self, S, Y, c):
        self._finite(S, Y)
        S = np.asarray(S, dtype=np.float64)
        return np.array([np_sums(np.vstack([S, y[None]]), y[None], c)[0] for y in np.asarray(Y, dtype=np.float64)])


def _install(fake, setter):
    import statdepth_b200._modal as md
    setter(md, "get_engine", lambda device=None: fake)


@pytest.fixture()
def md_oracle(monkeypatch):
    import statdepth_b200._spatial as sp
    fake = ModalOracleEngine()
    _install(fake, monkeypatch.setattr)
    monkeypatch.setattr(sp, "get_engine", lambda device=None: fake)  # a spatial reference holds its sample only
    return fake


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracle and the bandwidth arithmetic
# ---------------------------------------------------------------------------------------------------------------
def test_oracle_equals_pairwise_loop_and_closed_forms():
    rng = np.random.default_rng(0)
    for A in [rng.standard_normal((2, 3)), rng.integers(-1, 2, size=(12, 3)).astype(np.float64),
              rng.standard_normal((9, 1)), rng.standard_normal((15, 7)) * 1e-3 + 5.0]:
        h = np_bandwidth(A)
        got = np_modal_depth(A, bandwidth=h)
        for q in range(len(A)):
            assert abs(got[q] - loop_modal_depth(A, q, h)) <= 1e-14
    assert np_modal_depth(np.ones((1, 3)), bandwidth=0.7).tolist() == [PHI0]           # n = 1: phi(0)
    assert np_modal_depth(np.full((6, 4), 2.5), bandwidth=1.3).tolist() == [PHI0] * 6  # all duplicates
    A = np.array([[0.0, 0.0], [3.0, 4.0]])  # n = 2, d = 5
    for h in (0.5, 5.0, 40.0):
        exp = (PHI0 + math.exp(-0.5 * (5.0 / h) ** 2) * PHI0) / 2
        assert np.allclose(np_modal_depth(A, bandwidth=h), exp, rtol=1e-15, atol=0)
    assert np_bandwidth(A, 0.3) == 5.0


def test_bandwidth_mirror_equals_np_quantile():
    from statdepth_b200._modal import _quantile_bandwidth
    rng = np.random.default_rng(1)
    sizes = [1, 2, 3, 7, 10, 100, 1001, 65536, 10 ** 6]
    qs = [0.0, 0.15, 0.5, 1.0] + rng.random(6).tolist() + [1e-9, 1 - 1e-12, 0.25, 0.75]
    for N in sizes:
        D = np.sort(rng.standard_exponential(N) * 10.0 ** rng.integers(-5, 5))
        if N > 4:
            D[N // 3:N // 2] = D[N // 3]  # runs of ties
        for q in qs:
            got = _quantile_bandwidth(N, q, lambda k: (float(D[k]), float(D[min(k + 1, N - 1)])))
            exp = np.quantile(D, q)
            assert np.float64(got).tobytes() == np.float64(exp).tobytes(), (N, q, got, exp)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the host layer on the test double
# ---------------------------------------------------------------------------------------------------------------
def test_univariate_frames_and_to_compute(md_oracle):
    from statdepth_b200 import FunctionalModalDepth
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(2)
    X = rng.standard_normal((9, 6))
    df = pd.DataFrame(X, columns=list('abcdef'))
    res = FunctionalModalDepth([df])
    assert type(res) is _FunctionalDepthUnivariate and list(res.index) == list('abcdef')
    assert np.allclose(res.values, np_modal_depth(X.T), rtol=1e-14, atol=0)
    sub = FunctionalModalDepth([df], to_compute=['e', 'a'])
    assert list(sub.index) == ['e', 'a'] and sub.values.tolist() == res[['e', 'a']].values.tolist()
    for q in (0.0, 0.5, 1.0):
        assert np.allclose(FunctionalModalDepth([df], quantile=q).values, np_modal_depth(X.T, quantile=q),
                           rtol=1e-14, atol=0)
    assert np.allclose(FunctionalModalDepth([df], bandwidth=0.8).values, np_modal_depth(X.T, bandwidth=0.8),
                       rtol=1e-14, atol=0)
    F = rng.standard_normal((7, 5, 3))
    res = FunctionalModalDepth(_frames(F))
    assert type(res) is _FunctionalDepthSeries and list(res.index) == list(range(7))
    assert np.allclose(res.values, np_modal_depth(F.reshape(7, -1)), rtol=1e-14, atol=0)  # (t, c) order
    sub = FunctionalModalDepth(_frames(F), to_compute=[6, 2])
    assert list(sub.index) == [6, 2] and sub.values.tolist() == res.values[[6, 2]].tolist()
    assert FunctionalModalDepth([df.iloc[:, [0]]], bandwidth=2.0).values.tolist() == [PHI0]  # n = 1


def test_refusals(md_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalModalDepth, FunctionalModalDepthOf, FunctionalReference
    rng = np.random.default_rng(4)
    df = pd.DataFrame(rng.standard_normal((5, 4)), columns=list('wxyz'))
    bad = [
        (ValueError, lambda: FunctionalModalDepth(df)),
        (ValueError, lambda: FunctionalModalDepth([])),
        (ValueError, lambda: FunctionalModalDepth([pd.DataFrame(np.zeros((4, 0)))])),
        (ValueError, lambda: FunctionalModalDepth([pd.DataFrame(np.zeros((4, 2))), pd.DataFrame(np.zeros((5, 2)))])),
        (KeyError, lambda: FunctionalModalDepth([df], to_compute=['q'])),
        (KeyError, lambda: FunctionalModalDepth(_frames(np.zeros((3, 4, 2))), to_compute=[3])),
        (ValueError, lambda: FunctionalModalDepth([df], quantile=-0.1)),
        (ValueError, lambda: FunctionalModalDepth([df], quantile=1.5)),
        (ValueError, lambda: FunctionalModalDepth([df], quantile=float('nan'))),
        (ValueError, lambda: FunctionalModalDepth([df], quantile=0.3, bandwidth=1.0)),
        (ValueError, lambda: FunctionalModalDepth([df], bandwidth=0.0)),
        (ValueError, lambda: FunctionalModalDepth([df], bandwidth=-1.0)),
        (ValueError, lambda: FunctionalModalDepth([df], bandwidth=float('inf'))),
        (ValueError, lambda: FunctionalModalDepth([df], bandwidth=1e-160)),  # h * h is not normal
        (ValueError, lambda: FunctionalModalDepth([df], bandwidth=1e160)),   # h * h overflows
        (ValueError, lambda: FunctionalModalDepth([df.iloc[:, [0]]])),       # n = 1: no pairs
        (ValueError, lambda: FunctionalModalDepthOf([pd.DataFrame(np.zeros((6, 2)))], [df])),
        (ValueError, lambda: FunctionalModalDepthOf([df], [df.iloc[:, [0]]])),
        (ValueError, lambda: FunctionalReference([df], J=3, depth='modal')),
        (ValueError, lambda: FunctionalReference([df], depth='modal', directions=4)),
        (ValueError, lambda: FunctionalReference([df], depth='modal', quantile=2.0)),
        (ValueError, lambda: FunctionalReference([df], depth='spatial', quantile=0.2)),
        (ValueError, lambda: FunctionalReference([df], depth='projection', bandwidth=1.0)),
        (ValueError, lambda: FunctionalReference([df], bandwidth=1.0)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [df]}, depth='modal', directions=4)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [df]}, depth='spatial', bandwidth=1.0)),
        (ValueError, lambda: DepthClassifier({0: [df], 1: [pd.DataFrame(np.zeros((6, 3)))]}, depth='modal')),
    ]
    for exc, fn in bad:
        with pytest.raises(exc):
            fn()
    assert md_oracle.calls == 0
    dup = pd.DataFrame(np.tile(rng.standard_normal((5, 1)), (1, 6)))
    with pytest.raises(ValueError, match='bandwidth='):  # every pair a duplicate: h = 0
        FunctionalModalDepth([dup])
    X = rng.standard_normal((5, 4))
    X[1, 2] = np.nan
    from statdepth_b200 import EngineError
    with pytest.raises(EngineError) as ei:
        FunctionalModalDepth([pd.DataFrame(X)])
    assert ei.value.status == 4


def test_reference_and_classifier_on_the_double(md_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalModalDepth, FunctionalModalDepthOf, FunctionalReference
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(5)
    S = rng.standard_normal((8, 11))
    Y = rng.standard_normal((8, 3))
    Y[:, 1] = S[:, 4]  # a new curve that duplicates a sample curve
    sdf, ydf = pd.DataFrame(S), pd.DataFrame(Y, columns=['p', 'q', 'r'])
    with FunctionalReference([sdf], depth='modal') as ref:
        h = ref.bandwidth
        assert ref.directions is None and h == np_bandwidth(S.T)
        res = ref.depth_of([ydf])
    one = FunctionalModalDepthOf([ydf], [sdf])
    assert type(res) is _FunctionalDepthUnivariate and list(res.index) == ['p', 'q', 'r']
    assert type(one) is _FunctionalDepthUnivariate and res.values.tolist() == one.values.tolist()
    for k in range(3):  # the out-of-sample identity, with the sample's bandwidth given
        pooled = FunctionalModalDepth([pd.concat([sdf, ydf.iloc[:, [k]]], axis=1)], bandwidth=h)
        assert pooled.values[-1] == res.values[k]
        assert FunctionalModalDepthOf([ydf.iloc[:, [k]]], [sdf], bandwidth=h).values[0] == res.values[k]
    with FunctionalReference([sdf], depth='modal', quantile=0.5) as ref:
        assert ref.bandwidth == np_bandwidth(S.T, 0.5)
    with FunctionalReference([sdf], depth='modal', bandwidth=0.25) as ref:
        assert ref.bandwidth == 0.25
    with FunctionalReference([sdf], depth='spatial') as ref:
        assert ref.bandwidth is None
    Fs, Fy = rng.standard_normal((6, 4, 2)), rng.standard_normal((2, 4, 2))
    with FunctionalReference(_frames(Fs), depth='modal') as ref:
        res = ref.depth_of(_frames(Fy))
        one = ref.depth_of(_frames(Fy[1:]))
        h = ref.bandwidth
    assert type(res) is _FunctionalDepthSeries and list(res.index) == [0, 1]
    assert one.values[0] == res.values[1]
    assert FunctionalModalDepth(_frames(np.concatenate([Fs, Fy[:1]])), bandwidth=h).values[-1] == res.values[0]
    # two shifted classes, each with its own bandwidth
    A = rng.standard_normal((30, 16)) * 0.3
    B = A[:15] * 3.0 + np.linspace(0, 3, 16)
    refs = {'a': [pd.DataFrame(A[:15].T)], 'b': [pd.DataFrame(B.T)]}
    with DepthClassifier(refs, depth='modal') as clf:
        assert clf.bandwidths == {'a': np_bandwidth(A[:15]), 'b': np_bandwidth(B)}
        assert clf.bandwidths['a'] != clf.bandwidths['b']
        test = np.vstack([A[15:], A[15:] * 3.0 + np.linspace(0, 3, 16)])
        pred = clf.predict([pd.DataFrame(test.T)])
        d = clf.depths([pd.DataFrame(test.T)])
    assert pred.tolist() == ['a'] * 15 + ['b'] * 15
    exp = FunctionalModalDepthOf([pd.DataFrame(test.T)], refs['b']).values
    assert d['b'].tolist() == exp.tolist()
    with DepthClassifier(refs, depth='modal', bandwidth=0.9) as clf:
        assert clf.bandwidths == {'a': 0.9, 'b': 0.9}
    with DepthClassifier(refs, depth='spatial') as clf:
        assert clf.bandwidths is None


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
    from statdepth_b200 import FunctionalModalDepth, FunctionalModalDepthOf, FunctionalReference
    rng = np.random.default_rng(11)
    uni = pd.DataFrame(rng.integers(-2, 3, size=(6, 13)).astype(np.float64))  # 13 curves: 7 + 6
    F = rng.standard_normal((9, 4, 2))
    new = pd.DataFrame(rng.standard_normal((6, 5)))
    with FunctionalReference([uni], depth='modal') as ref:
        ref_vals = ref.depth_of([new]).values
        one = ref.depth_of([new.iloc[:, [0]]]).values  # one new curve: one rank scores nothing
        h = np.array([ref.bandwidth])
    return dict(uni=FunctionalModalDepth([uni]).values, frames=FunctionalModalDepth(_frames(F)).values,
                tc=FunctionalModalDepth(_frames(F), to_compute=[8, 0, 3]).values,
                of=FunctionalModalDepthOf([new], [uni]).values, ref=ref_vals, one=one, h=h)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(ModalOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(ModalOracleEngine(), monkeypatch.setattr)
    exp = _results()
    for r in range(world):
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: exact pair selection
# ---------------------------------------------------------------------------------------------------------------
QUANTILES = (0.0, 0.15, 0.5, 1.0)


def _check_selection(engine, A, d2, quantiles=QUANTILES):
    """Both order statistics and the bandwidth equal the oracle's bit for bit (d2: the exact pair d2)."""
    from statdepth_b200 import FunctionalReference
    from statdepth_b200._modal import _quantile_bandwidth
    srt = np.sort(d2)
    N = len(srt)
    for q in quantiles:
        ks = []
        _quantile_bandwidth(N, q, lambda k: ks.append(k) or (0.0, 0.0))
        k = ks[0]
        got = engine.modal_pair_select(A, k)
        assert got.tolist() == [srt[k], srt[min(k + 1, N - 1)]], (q, k)
        exp = np.quantile(np.sqrt(d2), q)
        if exp == 0.0:  # at least that share of the pairs are duplicates
            with pytest.raises(ValueError, match='bandwidth='):
                FunctionalReference([pd.DataFrame(A.T)], depth='modal', quantile=q)
            continue
        with FunctionalReference([pd.DataFrame(A.T)], depth='modal', quantile=q) as ref:
            assert ref.bandwidth == exp, q


@pytest.mark.gpu
@pytest.mark.parametrize("F", [1, 7, 1024])
@pytest.mark.parametrize("n", [2, 3, 257, 2000])
def test_exact_selection_integer_curves(engine, n, F):
    A = np.random.default_rng(200 + n + F).integers(-3, 4, size=(n, F)).astype(np.float64)
    _check_selection(engine, A, int_pair_d2(A))


@pytest.mark.gpu
def test_selection_gather_route(engine):
    rng = np.random.default_rng(21)
    A = rng.integers(-8, 9, size=(8000, 256)).astype(np.float64)  # 3.2e7 pairs, d2 up to 256 * 256
    _check_selection(engine, A, int_pair_d2(A), quantiles=(0.15, 0.5, 0.999))


@pytest.mark.gpu
def test_selection_over_budget_and_zero_bandwidth(engine):
    from statdepth_b200 import FunctionalModalDepth, FunctionalReference
    A = np.eye(10)[np.arange(24_000) % 10]  # a regular simplex, 2 400 copies of each vertex: d2 in {0, 2}
    N = 24_000 * 23_999 // 2
    zeros = 10 * (2_400 * 2_399 // 2)
    k = int(0.15 * N)  # 2.6e8 keys equal 2.0: more than the 1 GB candidate buffer holds
    assert engine.modal_pair_select(A, k).tolist() == [2.0, 2.0]
    assert engine.modal_pair_select(A, zeros - 1).tolist() == [0.0, 2.0]
    with FunctionalReference([pd.DataFrame(A.T)], depth='modal') as ref:
        assert ref.bandwidth == math.sqrt(2.0)
    with pytest.raises(ValueError, match='bandwidth='):
        FunctionalReference([pd.DataFrame(A.T)], depth='modal', quantile=0.05)
    with pytest.raises(ValueError, match='bandwidth='):
        FunctionalModalDepth([pd.DataFrame(np.ones((4, 9)))])


# ---------------------------------------------------------------------------------------------------------------
# GPU: depths against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,F", [(2, 1), (3, 7), (257, 1), (257, 1024), (2000, 7), (2000, 256)])
def test_depths_against_oracle(engine, n, F):
    from statdepth_b200 import FunctionalModalDepth
    A = np.random.default_rng(300 + n + F).standard_normal((n, F)).cumsum(axis=1)
    res = FunctionalModalDepth([pd.DataFrame(A.T)]).values
    assert_depths(res, np_modal_depth(A), n, F)
    assert (res >= PHI0 / n * (1 - 1e-15)).all() and (res <= PHI0 * (1 + 1e-15)).all()


@pytest.mark.gpu
def test_multichannel_and_large_univariate(engine):
    from statdepth_b200 import FunctionalModalDepth, FunctionalReference
    rng = np.random.default_rng(7)
    F = rng.standard_normal((5000, 256, 3)).cumsum(axis=1)
    A = F.reshape(5000, -1)
    q = sorted(rng.choice(5000, 40, replace=False).tolist())
    res = FunctionalModalDepth(_frames(F), to_compute=q).values
    h = np_bandwidth(A)
    assert_depths(res, np_modal_depth(A, q, bandwidth=h), 5000, 768)
    X = rng.standard_normal((1024, 20_000)).cumsum(axis=0)  # C order [T, n]: SD_LAYOUT_TN, transposed on the device
    cols = sorted(rng.choice(20_000, 64, replace=False).tolist())
    with FunctionalReference([pd.DataFrame(X[:, :1500])], depth='modal') as ref:
        assert abs(ref.bandwidth - np_bandwidth(X[:, :1500].T)) <= 1e-12 * ref.bandwidth
    res = FunctionalModalDepth([pd.DataFrame(X)], to_compute=cols, bandwidth=30.0).values
    assert_depths(res, np_modal_depth(X.T, cols, bandwidth=30.0), 20_000, 1024)
    full = FunctionalModalDepth([pd.DataFrame(X)], to_compute=cols).values  # the selected bandwidth
    assert np.isfinite(full).all() and (full > 0).all()
    # the F-ordered memory of a column-built DataFrame (SD_LAYOUT_NT) gives the same bits
    c = -0.5 / 30.0 ** 2
    assert engine.modal_sums(np.ascontiguousarray(X.T), c, cols).tolist() == engine.modal_sums(X.T, c, cols).tolist()


# ---------------------------------------------------------------------------------------------------------------
# GPU: bit identities, scaling and errors
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_out_of_sample_and_query_identities(engine):
    from statdepth_b200 import FunctionalModalDepth, FunctionalModalDepthOf, FunctionalReference
    rng = np.random.default_rng(10)
    X = rng.standard_normal((96, 700)).cumsum(axis=0)
    df = pd.DataFrame(X)
    full = FunctionalModalDepth([df]).values
    assert FunctionalModalDepth([df]).values.tolist() == full.tolist()
    tc = [699, 3, 64, 65, 0, 300]
    assert FunctionalModalDepth([df], to_compute=tc).values.tolist() == full[tc].tolist()
    S, new = df.iloc[:, :600], df.iloc[:, 600:]
    with FunctionalReference([S], depth='modal') as ref:
        b = ref.bandwidth
        got = ref.depth_of([new]).values
        single = [ref.depth_of([new.iloc[:, [k]]]).values[0] for k in (0, 57, 99)]
    assert got.tolist() == FunctionalModalDepthOf([new], [S]).values.tolist()
    assert single == got[[0, 57, 99]].tolist()
    for k in (0, 57, 99):
        assert FunctionalModalDepth([pd.concat([S, new.iloc[:, [k]]], axis=1)], bandwidth=b).values[-1] == got[k]
        one = FunctionalModalDepthOf([new.iloc[:, [k]]], [S], bandwidth=2.5).values[0]
        assert FunctionalModalDepth([pd.concat([S, new.iloc[:, [k]]], axis=1)], bandwidth=2.5).values[-1] == one
    F = rng.standard_normal((300, 5, 3))
    Fs, Fn = F[:280], F[280:]
    with FunctionalReference(_frames(Fs), depth='modal') as ref:
        got = ref.depth_of(_frames(Fn)).values
        b = ref.bandwidth
    assert got.tolist() == FunctionalModalDepthOf(_frames(Fn), _frames(Fs)).values.tolist()
    assert FunctionalModalDepth(_frames(np.concatenate([Fs, Fn[:1]])), bandwidth=b).values[-1] == got[0]


@pytest.mark.gpu
def test_scaling_and_errors(engine):
    from statdepth_b200 import EngineError, FunctionalModalDepth, FunctionalReference
    rng = np.random.default_rng(9)
    A = rng.standard_normal((260, 130))
    base = FunctionalModalDepth([pd.DataFrame(A.T)]).values
    with FunctionalReference([pd.DataFrame(A.T)], depth='modal') as ref:
        h = ref.bandwidth
    for k in (-300, -40, 37, 400):
        As = A * 2.0 ** k
        assert FunctionalModalDepth([pd.DataFrame(As.T)]).values.tolist() == base.tolist(), k
        with FunctionalReference([pd.DataFrame(As.T)], depth='modal') as ref:
            assert ref.bandwidth == h * 2.0 ** k, k
    with pytest.raises(EngineError) as ei:
        engine.modal_pair_select(A * 1e160, 5)
    assert ei.value.status == 5
    with pytest.raises(EngineError) as ei:
        engine.modal_sums(A * 1e160, -1.0)
    assert ei.value.status == 5
    A[3, 3] = np.nan
    for call in (lambda: engine.modal_pair_select(A, 0), lambda: engine.modal_sums(A, -1.0),
                 lambda: engine.modal_sums_of(A, A[:2] * 0, -1.0), lambda: engine.modal_sums_of(A * 0, A[:2], -1.0)):
        with pytest.raises(EngineError) as ei:
            call()
        assert ei.value.status == 4


@pytest.mark.gpu
def test_query_set_spanning_several_partial_row_blocks(engine):
    from statdepth_b200 import FunctionalReference
    rng = np.random.default_rng(14)
    S = rng.standard_normal((1, 200_000))
    Y = rng.standard_normal((1, 50_000)) * 1.2  # 1 563 sample tiles: 21 440 queries per 256 MB row block
    with FunctionalReference([pd.DataFrame(S)], depth='modal', bandwidth=0.1) as ref:
        got = ref.depth_of([pd.DataFrame(Y)]).values
        for k in (0, 21_439, 21_440, 42_880, 49_999):
            assert ref.depth_of([pd.DataFrame(Y[:, [k]])]).values[0] == got[k], k
    q = [0, 21_440, 49_999]
    c = -0.5 / 0.1 ** 2
    exp = np.array([np_sums(np.vstack([S.T, Y.T[k][None]]), Y.T[k][None], c)[0] for k in q]) / 200_001 * PHI0
    assert_depths(got[q], exp, 200_001, 1)


@pytest.mark.gpu
def test_reference_of_100000_curves(engine):
    from statdepth_b200 import FunctionalReference
    rng = np.random.default_rng(13)
    S = rng.standard_normal((1024, 100_000))
    Y = rng.standard_normal((1024, 2000)) * 1.1
    with FunctionalReference([pd.DataFrame(S)], depth='modal') as ref:
        h = ref.bandwidth
        got = ref.depth_of([pd.DataFrame(Y)]).values
        one = ref.depth_of([pd.DataFrame(Y[:, [1999]])]).values[0]
    assert one == got[1999]
    d2 = np_d2(S.T[:3000], S.T[:3000])[np.triu_indices(3000, k=1)]  # h of a subsample: the same distribution
    assert abs(h / np.quantile(np.sqrt(d2), 0.15) - 1) < 5e-3
    q = [0, 1, 1999]
    c = -0.5 / (h * h)
    exp = np.array([np_sums(np.vstack([S.T, Y.T[k][None]]), Y.T[k][None], c)[0] for k in q]) / 100_001 * PHI0
    assert_depths(got[q], exp, 100_001, 1024)
