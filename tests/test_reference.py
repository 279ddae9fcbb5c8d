"""Fitted references (FunctionalReference, DepthClassifier) and the sd_band_sort_rows / sd_band_depth_sorted entry
points.

The contract: with b_t / a_t the sample values strictly below / above g(t), b_t = searchsorted(row_t, g(t), 'left') and
a_t = n_S - searchsorted(row_t, g(t), 'right') in the sorted row t; the count of subset size j is
sum_t [C(n_S, j) - C(b_t, j) - C(a_t, j)], the relaxed out-of-sample numerator of FunctionalDepthOf.  The CPU part pins
that formulation to the C oracle on S u {g} and drives the host layer with a numpy test double; the GPU part pins the
CUDA engine to np.sort and to the out-of-sample kernel (sd_band_depth_oos_f64_dev)."""
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------
# numpy oracle
# ---------------------------------------------------------------------------------------------------------------
def _comb(m, j):
    m = np.asarray(m, dtype=np.int64)
    return m * (m - 1) // 2 if j == 2 else m * (m - 1) * (m - 2) // 6


def np_sorted_counts(sorted_rows, Y, J):
    """int64 [J - 1, nY] by searchsorted in the sorted rows."""
    sorted_rows = np.asarray(sorted_rows, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    nS = sorted_rows.shape[1]
    out = np.zeros((J - 1, Y.shape[1]), dtype=np.int64)
    for t in range(sorted_rows.shape[0]):
        b = np.searchsorted(sorted_rows[t], Y[t], side='left')
        a = nS - np.searchsorted(sorted_rows[t], Y[t], side='right')
        for j in range(2, J + 1):
            out[j - 2] += _comb(nS, j) - _comb(b, j) - _comb(a, j)
    return out


class SortedOracleEngine:
    """TEST DOUBLE: the fitted reference answered by np.sort + searchsorted (no `_dev` methods, so the driver takes the
    host path), and FunctionalDepthOf's relaxed counts answered by the C oracle on S u {g}, one g at a time."""

    def __init__(self):
        from oracle import cpu_oracle
        self.o = cpu_oracle
        self.calls = 0

    def band_sort_rows(self, X):
        self.calls += 1
        return np.sort(np.asarray(X, dtype=np.float64), axis=1)

    def band_depth_sorted_counts(self, sorted_rows, Y, J):
        self.calls += 1
        return np_sorted_counts(sorted_rows, Y, J)

    def band_depth_oos_counts(self, S, Y, j=2, relax=False):
        assert relax
        nS = S.shape[1]
        out = np.zeros(Y.shape[1], dtype=np.int64)
        for g in range(Y.shape[1]):
            P = np.ascontiguousarray(np.concatenate([S, Y[:, [g]]], axis=1), dtype=np.float64)
            out[g] = self.o.mbd_counts_all(P, j=j)[nS]
        return out


def _install(fake, setter):
    import statdepth_b200._functional as f
    import statdepth_b200._reference as r
    setter(r, "get_engine", lambda device=None: fake)
    setter(f, "get_engine", lambda device=None: fake)


@pytest.fixture()
def sorted_oracle(monkeypatch):
    fake = SortedOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _walks(T, n, seed, labels=None, shift=0.0):
    X = np.random.default_rng(seed).standard_normal((T, n)).cumsum(0) + shift
    return pd.DataFrame(X, columns=labels if labels is not None else range(n))


def _tied(rng, shape):
    """Values on 8 levels, zeros of both signs."""
    X = rng.integers(-4, 4, size=shape).astype(np.float64) * 0.5
    neg = (X == 0) & (rng.random(shape) < 0.5)
    X[neg] = -0.0
    return X


def _edge_queries(rng, S, nY):
    """New curves tied to sample values, duplicated among themselves, and outside the sample's range."""
    T, nS = S.shape
    Y = rng.standard_normal((T, nY)).cumsum(0)
    Y[:, 0] = S[:, nS // 2]
    if nY > 1:
        Y[:, 1] = S[:, 0]
    if nY > 2:
        Y[:, 2] = Y[:, 1]
    if nY > 4:
        Y[:, 3] = S.min(axis=1) - 1.0
        Y[:, 4] = S.max(axis=1) + 1.0
    Y[0, 0] = S[0].min() - 5.0
    Y[-1, 0] = S[-1].max() + 5.0
    return Y


def _planted_classes(n, T, seed):
    """Two classes of noisy curves around one trend, their levels 2 apart: the midway level is 6.7 standard deviations
    of a curve's level from either class, so no drawn curve sits on the wrong side."""
    rng = np.random.default_rng(seed)
    t = np.arange(T) / T
    trend = np.sin(2 * np.pi * t)

    def draw(m, level):
        return trend[:, None] + level + 0.15 * rng.standard_normal(m)[None, :] + 0.05 * rng.standard_normal((T, m))
    return draw(n, 0.0), draw(n, 2.0), draw(n // 4, 0.0), draw(n // 4, 2.0)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the binary-search formulation and the host layer
# ---------------------------------------------------------------------------------------------------------------
def test_binary_search_formulation_matches_c_oracle(oracle):
    rng = np.random.default_rng(0)
    S_walk = rng.standard_normal((11, 17)).cumsum(0)
    S_tied = _tied(rng, (9, 40))
    Y_tied = _tied(rng, (9, 6))
    Y_tied[:, 0] = S_tied[:, 3]
    Y_tied[:, 1] = -S_tied[:, 5]  # -0.0 against 0.0
    cases = [(S_walk, rng.standard_normal((11, 6)).cumsum(0)),
             (S_walk, _edge_queries(rng, S_walk, 6)),
             (S_tied, Y_tied),
             (rng.standard_normal((7, 1)), rng.standard_normal((7, 4))),
             (rng.standard_normal((7, 2)), rng.standard_normal((7, 4)))]
    cases.append((cases[3][0], np.column_stack([cases[3][0][:, 0], cases[3][0][:, 0] - 1, cases[3][0][:, 0] + 1])))
    cases.append((cases[4][0], np.column_stack([cases[4][0][:, 1], cases[4][0].mean(axis=1)])))
    for S, Y in cases:
        nS = S.shape[1]
        got = np_sorted_counts(np.sort(S, axis=1), Y, 3)
        for j in (2, 3):
            exp = [oracle.mbd_counts_all(np.ascontiguousarray(np.column_stack([S, Y[:, g]])), j=j)[nS]
                   for g in range(Y.shape[1])]
            assert got[j - 2].tolist() == exp, (S.shape, j)


@pytest.mark.parametrize("J", [2, 3])
@pytest.mark.parametrize("order", ["C", "F"])
def test_depth_of_equals_functional_depth_of(sorted_oracle, J, order):
    from statdepth_b200 import FunctionalDepthOf, FunctionalReference
    from statdepth_b200.depth import _FunctionalDepthUnivariate
    rng = np.random.default_rng(3)
    S = rng.standard_normal((10, 14)).cumsum(0)
    S[:, 2] = S[:, 7]
    Y = _edge_queries(rng, S, 6)
    mk = np.asfortranarray if order == "F" else np.ascontiguousarray
    Sdf = pd.DataFrame(mk(S), columns=['s%d' % k for k in range(14)])
    Ydf = pd.DataFrame(mk(Y), columns=['s3', 'n1', 's0', 'n3', 'n3', 'n5'])  # labels repeat sample labels and repeat
    with FunctionalReference([Sdf], J=J) as ref:
        res = ref.depth_of([Ydf])
        assert isinstance(res, _FunctionalDepthUnivariate)
        assert list(res.index) == list(Ydf.columns)
        exp = FunctionalDepthOf([Ydf], [Sdf], J=J, relax=True)
        assert res.values.tolist() == exp.values.tolist()
        again = ref.depth_of([Ydf.iloc[:, 2:]])  # the index answers again
        assert again.values.tolist() == exp.values[2:].tolist()
        empty = ref.depth_of([Ydf.iloc[:, :0]])
        assert len(empty) == 0
    assert sorted_oracle.calls == 1 + 2  # one index, two searches (no call for n_Y = 0)


def test_validation_errors(sorted_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalReference
    S = _walks(8, 10, 0)
    with pytest.raises(ValueError):
        FunctionalReference(S)                          # not a list
    with pytest.raises(NotImplementedError):
        FunctionalReference([_walks(8, 2, k) for k in range(5)])  # multivariate
    with pytest.raises(NotImplementedError):
        FunctionalReference([S], J=4)
    with pytest.raises(ValueError):
        FunctionalReference([S.iloc[:3]], J=3)          # J >= T
    with pytest.raises(ValueError):
        FunctionalReference([S], deep_check=1)
    assert sorted_oracle.calls == 0                      # every refusal happens before any engine call
    ref = FunctionalReference([S])
    Y = _walks(8, 3, 1)
    with pytest.raises(ValueError):
        ref.depth_of(Y)                                  # not a list
    with pytest.raises(NotImplementedError):
        ref.depth_of([Y, Y])
    with pytest.raises(ValueError):
        ref.depth_of([_walks(9, 3, 1)])                  # T differs
    shifted = Y.copy()
    shifted.index = range(1, 9)
    with pytest.raises(ValueError):
        ref.depth_of([shifted], deep_check=True)
    assert len(ref.depth_of([shifted])) == 3            # without deep_check, positions decide
    ref.close()
    ref.close()
    with pytest.raises(ValueError):
        ref.depth_of([Y])
    with pytest.raises(ValueError):
        DepthClassifier({'a': [S]})                      # one class
    with pytest.raises(ValueError):
        DepthClassifier([[S], [S]])                      # not a dict
    calls = sorted_oracle.calls
    with pytest.raises(ValueError):
        DepthClassifier({'a': [S], 'b': [_walks(9, 10, 2)]})  # T differs
    with pytest.raises(NotImplementedError):
        DepthClassifier({'a': [S], 'b': [S]}, J=4)
    assert sorted_oracle.calls == calls
    clf = DepthClassifier({'a': [S], 'b': [S]})
    clf.close()
    with pytest.raises(ValueError):
        clf.predict([Y])


def test_classifier_depths_ties_and_planted_classes(sorted_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalDepthOf
    A, B, YA, YB = _planted_classes(30, 24, 1)
    refs = {'low': [pd.DataFrame(A)], ('high', 1): [pd.DataFrame(B)]}
    Y = pd.DataFrame(np.column_stack([YA, YB]), columns=['y%d' % k for k in range(YA.shape[1] + YB.shape[1])])
    for J in (2, 3):
        with DepthClassifier(refs, J=J) as clf:
            d = clf.depths([Y])
            assert list(d.columns) == ['low', ('high', 1)] and list(d.index) == list(Y.columns)
            for label in refs:
                assert d[label].tolist() == FunctionalDepthOf([Y], refs[label], J=J, relax=True).values.tolist()
            pred = clf.predict([Y])
            assert list(pred.index) == list(Y.columns)
            assert pred.tolist() == ['low'] * YA.shape[1] + [('high', 1)] * YB.shape[1]
    # identical references: every depth ties, every curve goes to the class listed first
    S = pd.DataFrame(A)
    with DepthClassifier({'second': [S], 'first': [S.copy()]}) as clf:
        assert clf.predict([Y]).tolist() == ['second'] * Y.shape[1]


# ---------------------------------------------------------------------------------------------------------------
# CPU: two ranks (gloo) shard time rows
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dist_inputs():
    rng = np.random.default_rng(11)
    S = pd.DataFrame(rng.standard_normal((13, 9)).cumsum(0))  # 13 rows: uneven split 7 + 6
    Y = pd.DataFrame(_edge_queries(rng, S.values, 5))
    S1 = rng.standard_normal((1, 9))                           # one row: the second rank has none
    Y1 = np.column_stack([S1[:, 2], S1[:, 2] + 0.5, rng.standard_normal((1, 3))])
    return S, Y, S1, Y1


def _results():
    from statdepth_b200 import DepthClassifier, FunctionalReference
    from statdepth_b200._reference import _SortedReference
    S, Y, S1, Y1 = _dist_inputs()
    with FunctionalReference([S], J=3) as ref:
        d3 = ref.depth_of([Y]).values
    with DepthClassifier({0: [S], 1: [S + 1.0]}) as clf:
        dd = clf.depths([Y]).values
    one = _SortedReference(S1, 3)
    return dict(d3=d3, dd=dd, t1=one.depths(Y1), t1_counts=one.counts(Y1))


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(SortedOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(SortedOracleEngine(), monkeypatch.setattr)
    exp = _results()
    S, Y, S1, Y1 = _dist_inputs()
    assert exp['t1_counts'].tolist() == np_sorted_counts(np.sort(S1, axis=1), Y1, 3).tolist()
    for r in range(world):  # every rank ends with the full result
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine
# ---------------------------------------------------------------------------------------------------------------
def _dev(A):
    import torch
    return torch.from_numpy(np.ascontiguousarray(A, dtype=np.float64)).cuda()


def _gpu_sorted(engine, X, ld=None):
    """(device index tensor, host copy) of the rows of X [T, nS], stored with leading dimension ld."""
    import torch
    T, nS = X.shape
    ld = nS if ld is None else ld
    buf = np.full((T, ld), 7.0)
    buf[:, :nS] = X
    dX = _dev(buf)
    out = torch.empty((T, nS), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's
    engine.band_sort_rows_dev(dX.data_ptr(), T, nS, ld, out.data_ptr())
    return out, out.cpu().numpy()


def _gpu_counts(engine, index, Y, J):
    import torch
    T, nS = index.shape
    dY = _dev(Y)
    out = torch.full((J - 1, Y.shape[1]), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    engine.band_depth_sorted_counts_dev(index.data_ptr(), T, nS, dY.data_ptr(), Y.shape[1], Y.shape[1], J,
                                        out.data_ptr())
    return out.cpu().numpy()


def _k7_counts(engine, S, Y, j):
    import torch
    T, nS = S.shape
    dS, dY = _dev(S), _dev(Y)
    out = torch.full((Y.shape[1],), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    engine.band_depth_oos_counts_dev(dS.data_ptr(), T, nS, nS, dY.data_ptr(), Y.shape[1], Y.shape[1], out.data_ptr(),
                                     j, True)
    return out.cpu().numpy()


def _sort_cases():
    rng = np.random.default_rng(5)
    return [("slab", rng.standard_normal((12, 20_000)).cumsum(0)),
            ("parts", rng.standard_normal((16, 5_000)).cumsum(0)),
            ("parts_wide", rng.standard_normal((6, 200_000)).cumsum(0)),
            ("tied", _tied(rng, (9, 30_000))),
            ("tied_wide", _tied(rng, (3, 200_000))),
            ("T1", rng.standard_normal((1, 3001))),
            ("nS1", rng.standard_normal((40, 1))),
            ("small", _tied(rng, (5, 37)))]


@pytest.mark.gpu
def test_sorted_rows_equal_numpy(engine):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(20_000)["slab"] == 1 and mbd_plan(5_000)["slab"] == 0 and mbd_plan(200_000)["slab"] == 0
    for name, X in _sort_cases():
        exp = np.sort(X, axis=1)
        _, got = _gpu_sorted(engine, X)
        assert (got == exp).all(), name
        _, got = _gpu_sorted(engine, X, ld=X.shape[1] + 13)  # leading dimension past the sample
        assert (got == exp).all(), name


@pytest.mark.gpu
def test_sorted_counts_equal_out_of_sample_kernel(engine):
    rng = np.random.default_rng(6)
    for name, S in _sort_cases():
        index, _ = _gpu_sorted(engine, S)
        for nY in (1, 7, 50_000):
            Y = _edge_queries(rng, S, nY)
            if name.startswith("tied") and nY > 5:
                Y[:, 5:] = _tied(rng, (S.shape[0], nY - 5))
            c3 = _gpu_counts(engine, index, Y, 3)
            c2 = _gpu_counts(engine, index, Y, 2)
            assert c3.shape == (2, nY) and c2.shape == (1, nY)
            k2, k3 = _k7_counts(engine, S, Y, 2), _k7_counts(engine, S, Y, 3)
            assert (c2[0] == k2).all() and (c3[0] == k2).all() and (c3[1] == k3).all(), (name, nY)
            if nY == 7:
                assert (c3 == np_sorted_counts(np.sort(S, axis=1), Y, 3)).all(), name


@pytest.mark.gpu
def test_full_size_bit_identical_to_functional_depth_of(engine):
    """100 000 curves x 1024 points, three batches of 1 000 new curves; two references alive at once."""
    from statdepth_b200 import FunctionalDepthOf, FunctionalReference
    T, nS = 1024, 100_000
    rng = np.random.default_rng(31)
    S = pd.DataFrame(rng.standard_normal((T, nS)).cumsum(0))
    S2 = pd.DataFrame(rng.standard_normal((T, nS // 2)).cumsum(0) * 2.0 + 1.0)
    ref = FunctionalReference([S])
    ref2 = FunctionalReference([S2], J=3)
    for k in range(3):
        Y = pd.DataFrame(rng.standard_normal((T, 1000)).cumsum(0) * (1.0 + k))
        Y.iloc[:, 0] = S.iloc[:, k].values  # a sample curve again
        got = ref.depth_of([Y])
        assert got.values.tolist() == FunctionalDepthOf([Y], [S], J=2, relax=True).values.tolist(), k
        assert list(got.index) == list(Y.columns)
        if k == 1:
            got2 = ref2.depth_of([Y])
            assert got2.values.tolist() == FunctionalDepthOf([Y], [S2], J=3, relax=True).values.tolist()
    ref.close()
    ref2.close()


@pytest.mark.gpu
def test_nonfinite_rejected_and_reference_stays_usable(engine):
    from statdepth_b200 import EngineError, FunctionalDepthOf, FunctionalReference
    rng = np.random.default_rng(8)
    S = rng.standard_normal((16, 900)).cumsum(0)
    bad = S.copy()
    bad[5, 17] = np.nan
    with pytest.raises(EngineError) as ei:
        FunctionalReference([pd.DataFrame(bad)])
    assert ei.value.status == 4
    ref = FunctionalReference([pd.DataFrame(S)], J=3)
    Y = rng.standard_normal((16, 40)).cumsum(0)
    for v in (np.inf, -np.inf, np.nan):
        Yb = Y.copy()
        Yb[9, 3] = v
        with pytest.raises(EngineError) as ei:
            ref.depth_of([pd.DataFrame(Yb)])
        assert ei.value.status == 4
    got = ref.depth_of([pd.DataFrame(Y)]).values
    assert got.tolist() == FunctionalDepthOf([pd.DataFrame(Y)], [pd.DataFrame(S)], J=3, relax=True).values.tolist()


@pytest.mark.gpu
def test_classifier_on_gpu(engine):
    from statdepth_b200 import DepthClassifier, FunctionalDepthOf
    A, B, YA, YB = _planted_classes(4000, 200, 2)
    refs = {'a': [pd.DataFrame(A)], 'b': [pd.DataFrame(B)]}
    Y = pd.DataFrame(np.column_stack([YA, YB]))
    with DepthClassifier(refs) as clf:
        assert clf.predict([Y]).tolist() == ['a'] * YA.shape[1] + ['b'] * YB.shape[1]
        d = clf.depths([Y])
        for label in refs:
            assert d[label].tolist() == FunctionalDepthOf([Y], refs[label], J=2, relax=True).values.tolist()
