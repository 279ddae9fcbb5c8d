"""Fitted references for projection and random Tukey depth (FunctionalReference / DepthClassifier with
depth='projection' | 'tukey', FunctionalProjectionDepthOf, ProjectionDepthOf and the sd_*_sorted entry points).

The contract: a new observation g gets exactly the depth the in-sample call gives it after g alone is appended to the
reference S, with the same directions U.  Per row (t, k), s the sorted projections of S and y = g's projection:
Tukey h = (n_S + 1) - max(#s < y, #s > y); projection med' / MAD' of s with y inserted at #s < y, selected as
medmad_kernel selects them.  The CPU part pins that selection to np.median and drives the host layer with a numpy
test double; the GPU part pins the CUDA engine to the in-sample kernels on S + [g], bit for bit."""
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp

from test_halfspace import np_band_halfspace
from test_projection import (ProjectionOracleEngine, kernel_medmad, np_medmad, np_outlyingness_rows, np_project)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------
# numpy restatement of the query kernels
# ---------------------------------------------------------------------------------------------------------------
class Inserted:
    """InsertedRow (csrc/sorted_row.cuh): the sorted row s with y inserted at p = #s < y, never materialised."""

    def __init__(self, s, y):
        self.s, self.y = s, y
        self.p = int(np.searchsorted(s, y, 'left'))

    def __len__(self):
        return len(self.s) + 1

    def __getitem__(self, k):
        return self.s[k] if k < self.p else (self.y if k == self.p else self.s[k - 1])


def inserted_medmad(s, y):
    """row_median / row_mad on the virtual row: kernel_medmad (medmad_kernel restated) reading through Inserted."""
    v = Inserted(s, y)
    n = len(v)
    h = n // 2
    med = v[h] if n % 2 else (v[h - 1] + v[h]) / 2.0
    m = 0  # lower bound of med in v, by the kernel's search
    length = n
    while length > 0:
        half = length // 2
        if v[m + half] < med:
            m += half + 1
            length -= half + 1
        else:
            length = half

    def kth(k):
        lo, hi = max(0, k + 1 - (n - m)), min(k + 1, m)
        while lo < hi:
            i = (lo + hi) // 2
            j = k + 1 - i
            if j > 0 and i < m and abs(v[m + j - 1] - med) > abs(v[m - 1 - i] - med):
                lo = i + 1
            else:
                hi = i
        j = k + 1 - lo
        r = abs(v[m - lo] - med) if lo > 0 else None
        if j > 0:
            x = abs(v[m + j - 1] - med)
            if r is None or x > r:
                r = x
        return r

    return med, (kth(h) if n % 2 else (kth(h - 1) + kth(h)) / 2.0)


def _o(y, med, mad):
    return (abs(y - med) / mad) if mad != 0 else (0.0 if y == med else np.inf)


def sorted_tukey(index, Y):
    """index [T, K, nS], projections Y [T, K, nY] -> int64 [nY]."""
    T, K, nS = index.shape
    out = np.zeros(Y.shape[2], dtype=np.int64)
    for t in range(T):
        m = np.full(Y.shape[2], nS + 1, dtype=np.int64)
        for k in range(K):
            b = np.searchsorted(index[t, k], Y[t, k], 'left')
            a = nS - np.searchsorted(index[t, k], Y[t, k], 'right')
            m = np.minimum(m, nS + 1 - np.maximum(b, a))
        out += m
    return out


def sorted_outlyingness(index, Y):
    """index [T, K, nS], projections Y [T, K, nY] -> O [T, nY]."""
    T, K, nY = Y.shape
    O = np.zeros((T, nY))
    for t in range(T):
        for k in range(K):
            for g in range(nY):
                med, mad = inserted_medmad(index[t, k], Y[t, k, g])
                O[t, g] = max(O[t, g], _o(Y[t, k, g], med, mad))
    return O


class ReferenceOracleEngine(ProjectionOracleEngine):
    """TEST DOUBLE: test_projection's numpy engine (the in-sample calls), plus the fitted-reference calls answered by
    np.sort and the restated query kernels (no `_dev` methods, so the driver keeps a host index)."""

    def band_sort_rows(self, X):
        self._finite(X)
        return np.sort(np.asarray(X, dtype=np.float64), axis=1)

    def projection_sort_rows(self, F, U):
        self._finite(F)
        return np.sort(np_project(F, U), axis=2)

    def band_halfspace_sorted_counts(self, index, Y):
        self._finite(Y)
        return sorted_tukey(index[:, None, :], np.asarray(Y, dtype=np.float64)[:, None, :])

    def band_outlyingness_sorted(self, index, Y):
        self._finite(Y)
        return sorted_outlyingness(index[:, None, :], np.asarray(Y, dtype=np.float64)[:, None, :])

    def projection_tukey_sorted_counts(self, index, F, U):
        self._finite(F)
        return sorted_tukey(index, np_project(F, U))

    def projection_outlyingness_sorted(self, index, F, U):
        self._finite(F)
        return sorted_outlyingness(index, np_project(F, U))


def _install(fake, setter):
    import statdepth_b200._halfspace as h
    import statdepth_b200._projection as p
    import statdepth_b200._reference as r
    for mod in (h, p, r):
        setter(mod, "get_engine", lambda device=None: fake)


@pytest.fixture()
def ref_oracle(monkeypatch):
    fake = ReferenceOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _tied(rng, shape, lo=-3, hi=4):
    X = rng.integers(lo, hi, size=shape).astype(np.float64)
    X[(X == 0) & (rng.random(shape) < 0.5)] = -0.0
    return X


def _frames(F):
    return [pd.DataFrame(F[i]) for i in range(F.shape[0])]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the virtual-row selection
# ---------------------------------------------------------------------------------------------------------------
def test_inserted_row_selection_equals_np_median():
    rng = np.random.default_rng(0)
    rows = 0
    for it in range(1800):
        n = [1, 2, 3, 4][it % 4] if it < 400 else int(rng.integers(1, 40))
        kind = it % 3
        s = (rng.standard_normal(n) if kind == 0 else _tied(rng, n) if kind == 1
             else rng.standard_normal(n) * 10.0 ** rng.integers(-300, 300))
        s = np.sort(s)
        ys = [s[0] - 1.0, s[-1] + 1.0, s[n // 2], s[0], s[-1], -0.0, 0.0, float(rng.integers(-3, 4)),
              rng.standard_normal()]
        for y in ys:
            v = np.append(s, y)
            med, mad = inserted_medmad(s, y)
            em = np.median(v)
            assert med == em and mad == np.median(np.abs(v - em)) and not np.signbit(mad), (s, y)
            assert (med, mad) == kernel_medmad(np.sort(v))  # the in-sample selection on the pooled row
            rows += 1
    assert rows >= 1500


# ---------------------------------------------------------------------------------------------------------------
# CPU: the host layer on the test double
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["projection", "tukey"])
def test_curves_equal_pooled_in_sample_call(ref_oracle, kind):
    from statdepth_b200 import FunctionalProjectionDepth, FunctionalProjectionDepthOf, FunctionalReference
    from statdepth_b200.depth import _FunctionalDepthSeries, _FunctionalDepthUnivariate
    rng = np.random.default_rng(1)
    S = _tied(rng, (7, 5, 2))
    Y = _tied(rng, (4, 5, 2))
    Y[0] = S[3]
    with FunctionalReference(_frames(S), depth=kind, directions=6, seed=3) as ref:
        U = ref.directions
        assert U.shape == (6, 2)
        res = ref.depth_of(_frames(Y))
        assert type(res) is _FunctionalDepthSeries and list(res.index) == [0, 1, 2, 3]
        for g in range(4):
            exp = FunctionalProjectionDepth(_frames(np.concatenate([S, Y[g:g + 1]])), kind=kind, directions=U)
            assert np.array_equal(res.values[g], exp.values[7]), g
        one = FunctionalProjectionDepthOf(_frames(Y[2:3]), _frames(S), kind=kind, directions=6, seed=3)
        assert np.array_equal(one.values, res.values[2:3])  # alone equals together
    # univariate: the single direction 1.0; tukey is the integrated halfspace depth
    X = _tied(rng, (6, 9))
    Yu = _tied(rng, (6, 5))
    Yu[:, 0] = X[:, 4]
    Ydf = pd.DataFrame(Yu, columns=['a', 'b', 0, 'a', 7])
    with FunctionalReference([pd.DataFrame(X)], depth=kind) as ref:
        assert ref.directions is None
        res = ref.depth_of([Ydf])
        assert type(res) is _FunctionalDepthUnivariate and list(res.index) == list(Ydf.columns)
        for g in range(5):
            exp = FunctionalProjectionDepth([pd.DataFrame(np.column_stack([X, Yu[:, g]]))], kind=kind)
            assert np.array_equal(res.values[g], exp.values[9]), g


@pytest.mark.parametrize("kind", ["projection", "tukey"])
def test_clouds_equal_pooled_in_sample_call(ref_oracle, kind):
    from statdepth_b200 import ProjectionDepth, ProjectionDepthOf
    from statdepth_b200.depth import _PointwiseDepth
    rng = np.random.default_rng(2)
    S = pd.DataFrame(_tied(rng, (11, 3)), index=['s%d' % i for i in range(11)])
    D = pd.DataFrame(_tied(rng, (5, 3)), index=['q', 's1', 'q', 3, 4])
    D.iloc[1] = S.iloc[1].values
    res = ProjectionDepthOf(D, S, kind=kind, directions=7, seed=5)
    assert isinstance(res, _PointwiseDepth) and list(res.index) == list(D.index)
    for g in range(5):
        pooled = pd.concat([S, D.iloc[g:g + 1]], ignore_index=True)
        exp = ProjectionDepth(pooled, kind=kind, directions=7, seed=5)
        assert np.array_equal(res.values[g], exp.values[11]), g
    assert len(ProjectionDepthOf(D.iloc[:0], S, kind=kind)) == 0


def test_classifier_shares_directions_and_predicts_argmax(ref_oracle):
    from statdepth_b200 import DepthClassifier, FunctionalProjectionDepthOf
    rng = np.random.default_rng(4)
    A = rng.standard_normal((9, 6, 2))
    B = rng.standard_normal((9, 6, 2)) + 1.5
    Y = np.concatenate([rng.standard_normal((3, 6, 2)), rng.standard_normal((3, 6, 2)) + 1.5])
    refs = {'a': _frames(A), ('b', 1): _frames(B)}
    for kind in ('projection', 'tukey'):
        with DepthClassifier(refs, depth=kind, directions=5, seed=8) as clf:
            U = clf.directions
            assert all(np.array_equal(r.directions, U) for r in clf._refs)
            d = clf.depths(_frames(Y))
            assert list(d.columns) == ['a', ('b', 1)] and list(d.index) == list(range(6))
            one = np.column_stack([FunctionalProjectionDepthOf(_frames(Y), refs[k], kind=kind, directions=U).values
                                   for k in refs])
            assert np.array_equal(d.to_numpy(), one)
            labels = list(refs)
            assert clf.predict(_frames(Y)).tolist() == [labels[i] for i in np.argmax(one, axis=1)]


def test_refusals(ref_oracle):
    from statdepth_b200 import DepthClassifier, EngineError, FunctionalReference, ProjectionDepthOf
    rng = np.random.default_rng(5)
    S = _frames(rng.standard_normal((6, 4, 2)))
    X = pd.DataFrame(rng.standard_normal((4, 6)))
    calls = ref_oracle.calls
    with pytest.raises(ValueError):
        FunctionalReference(S, depth='halfspace')
    with pytest.raises(ValueError):
        FunctionalReference(S, J=3, depth='tukey')                  # J applies to mbd only
    with pytest.raises(ValueError):
        FunctionalReference([X], depth='projection', directions=3)  # univariate with directions
    with pytest.raises(ValueError):
        FunctionalReference([X], directions=3)                       # directions with mbd
    with pytest.raises(ValueError):
        FunctionalReference(S[:2] + [pd.DataFrame(np.zeros((4, 3)))], depth='projection')  # d differs
    with pytest.raises(ValueError):
        FunctionalReference(S[:2] + [pd.DataFrame(np.zeros((5, 2)))], depth='projection')  # T differs
    with pytest.raises(ValueError):
        DepthClassifier({'a': S, 'b': _frames(rng.standard_normal((5, 4, 3)))}, depth='projection')  # d differs
    with pytest.raises(ValueError):
        DepthClassifier({'a': S, 'b': _frames(rng.standard_normal((5, 5, 2)))}, depth='projection')  # T differs
    with pytest.raises(ValueError):
        DepthClassifier({'a': S, 'b': [X]}, depth='tukey')           # univariate and multivariate
    with pytest.raises(ValueError):
        ProjectionDepthOf(pd.DataFrame(np.zeros((2, 3))), pd.DataFrame(np.zeros((5, 2))))  # d differs
    assert ref_oracle.calls == calls                                  # refused before any engine call
    ref = FunctionalReference(S, depth='projection', directions=4)
    with pytest.raises(ValueError):
        ref.depth_of(_frames(rng.standard_normal((2, 5, 2))))        # T differs
    with pytest.raises(ValueError):
        ref.depth_of(_frames(rng.standard_normal((2, 4, 3))))        # d differs
    with pytest.raises(ValueError):
        ref.depth_of([X])                                             # univariate against multivariate
    bad = rng.standard_normal((2, 4, 2))
    bad[1, 2, 0] = np.inf
    with pytest.raises(EngineError) as ei:
        ref.depth_of(_frames(bad))
    assert ei.value.status == 4
    assert len(ref.depth_of(_frames(bad[:1]))) == 1                  # still usable
    ref.close()
    with pytest.raises(ValueError):
        ref.depth_of(_frames(bad[:1]))                               # closed
    Sb = rng.standard_normal((6, 4, 2))
    Sb[0, 0, 1] = np.nan
    with pytest.raises(EngineError):
        FunctionalReference(_frames(Sb), depth='tukey')


# ---------------------------------------------------------------------------------------------------------------
# CPU: two ranks (gloo) split time rows of curves and directions of clouds
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _results():
    from statdepth_b200 import FunctionalProjectionDepthOf, ProjectionDepthOf
    rng = np.random.default_rng(9)
    S, Y = _tied(rng, (6, 3, 2)), _tied(rng, (3, 3, 2))  # 3 time rows: uneven split 2 + 1
    X, Yu = _tied(rng, (3, 7)), _tied(rng, (3, 4))
    P, Q = _tied(rng, (9, 2)), _tied(rng, (4, 2))
    out = {}
    for kind in ('projection', 'tukey'):
        out['curves_' + kind] = FunctionalProjectionDepthOf(_frames(Y), _frames(S), kind=kind, directions=5).values
        out['uni_' + kind] = FunctionalProjectionDepthOf([pd.DataFrame(Yu)], [pd.DataFrame(X)], kind=kind).values
        out['cloud_' + kind] = ProjectionDepthOf(pd.DataFrame(Q), pd.DataFrame(P), kind=kind, directions=3).values
        out['cloud1_' + kind] = ProjectionDepthOf(pd.DataFrame(Q), pd.DataFrame(P), kind=kind,  # one direction
                                                  directions=1).values
        out['T1_' + kind] = FunctionalProjectionDepthOf(_frames(Y[:, :1]), _frames(S[:, :1]), kind=kind,  # one row
                                                        directions=4).values
    return out


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import enable_distributed
    _install(ReferenceOracleEngine(), setattr)
    enable_distributed()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_results())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(ReferenceOracleEngine(), monkeypatch.setattr)
    exp = _results()
    for r in range(world):  # every rank ends with the full result
        got = np.load(tmp_path / ("rank%d.npz" % r))
        for k in exp:
            assert np.array_equal(got[k], exp[k]), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the in-sample kernels on S + [g]
# ---------------------------------------------------------------------------------------------------------------
def _dev(A):
    import torch
    return torch.from_numpy(np.ascontiguousarray(A, dtype=np.float64)).cuda()


def _unit(U):
    return np.stack([u / np.linalg.norm(u) for u in U])


def _query(engine, S, U, Fn, sample=None):
    """(counts [nY], O [T, nY]) of the new curves Fn [nY, T, d] against the index of S [nS, T, d], and the in-sample
    (counts, O) of S + [g] for the new curves listed in sample (all when None)."""
    import torch
    nS, T, d = S.shape
    nY, K = Fn.shape[0], U.shape[0]
    dS = _dev(S)
    index = torch.empty((T, K, nS), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.projection_sort_rows_dev(dS.data_ptr(), nS, T, d, U, index.data_ptr())
    del dS
    dY = _dev(Fn)
    cnt = torch.full((nY,), -1, dtype=torch.int64, device="cuda")
    O = torch.full((T, nY), -1.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.projection_tukey_sorted_counts_dev(index.data_ptr(), nS, T, dY.data_ptr(), nY, d, U, cnt.data_ptr())
    engine.projection_outlyingness_sorted_dev(index.data_ptr(), nS, T, dY.data_ptr(), nY, d, U, O.data_ptr())
    cnt, O = cnt.cpu().numpy(), O.cpu().numpy()
    del index
    pool = _dev(np.concatenate([S, Fn[:1]]))
    pc = torch.empty(nS + 1, dtype=torch.int64, device="cuda")
    po = torch.empty((T, nS + 1), dtype=torch.float64, device="cuda")
    exp_c, exp_o = [], []
    for g in (range(nY) if sample is None else sample):
        pool[nS] = torch.from_numpy(np.ascontiguousarray(Fn[g])).cuda()
        torch.cuda.synchronize()
        engine.projection_tukey_counts_dev(pool.data_ptr(), nS + 1, T, d, U, pc.data_ptr())
        engine.projection_outlyingness_dev(pool.data_ptr(), nS + 1, T, d, U, po.data_ptr())
        exp_c.append(int(pc[nS]))
        exp_o.append(po[:, nS].cpu().numpy())
    return cnt, O, np.array(exp_c, dtype=np.int64), np.array(exp_o).T.reshape(T, -1)


def _check(engine, S, U, Fn, sample=None):
    cnt, O, ec, eo = _query(engine, S, U, Fn, sample)
    idx = np.arange(Fn.shape[0]) if sample is None else np.asarray(sample)
    assert np.array_equal(cnt[idx], ec)
    assert np.array_equal(O[:, idx], eo)
    return cnt, O


def _query_uni(engine, X, Y):
    """(counts, O) of the univariate new curves Y [T, nY] against K9's index of X [T, nS]."""
    import torch
    T, nS = X.shape
    nY = Y.shape[1]
    dX = _dev(X)
    index = torch.empty((T, nS), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.band_sort_rows_dev(dX.data_ptr(), T, nS, nS, index.data_ptr())
    del dX
    dY = _dev(Y)
    cnt = torch.full((nY,), -1, dtype=torch.int64, device="cuda")
    O = torch.full((T, nY), -1.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.band_halfspace_sorted_counts_dev(index.data_ptr(), T, nS, dY.data_ptr(), nY, nY, cnt.data_ptr())
    engine.band_outlyingness_sorted_dev(index.data_ptr(), T, nS, dY.data_ptr(), nY, nY, O.data_ptr())
    return cnt.cpu().numpy(), O.cpu().numpy()


def _check_uni(engine, X, Y, sample):
    import torch
    cnt, O = _query_uni(engine, X, Y)
    T, nS = X.shape
    pool = torch.empty((T, nS + 1), dtype=torch.float64, device="cuda")
    pool[:, :nS] = _dev(X)
    pc = torch.empty(nS + 1, dtype=torch.int64, device="cuda")
    po = torch.empty((T, nS + 1), dtype=torch.float64, device="cuda")
    for g in sample:
        pool[:, nS] = _dev(Y[:, g])
        torch.cuda.synchronize()
        engine.band_halfspace_counts_dev(pool.data_ptr(), T, nS + 1, nS + 1, pc.data_ptr())
        engine.band_outlyingness_dev(pool.data_ptr(), T, nS + 1, nS + 1, po.data_ptr())
        assert int(pc[nS]) == cnt[g], g
        assert np.array_equal(po[:, nS].cpu().numpy(), O[:, g]), g
    return cnt, O


@pytest.mark.gpu
@pytest.mark.parametrize("nS", [20_000, 5_000])
def test_both_rank_pipelines(engine, nS):
    from statdepth_b200._engine import mbd_plan
    assert mbd_plan(nS)["slab"] == (1 if nS == 20_000 else 0)
    rng = np.random.default_rng(nS)
    S = rng.standard_normal((nS, 3, 2))
    U = _unit(rng.standard_normal((24, 2)))
    Fn = rng.standard_normal((500, 3, 2)) * 1.5
    Fn[0] = S[7]
    Fn[1] = S[:, :, :].min(axis=0) - 1.0
    _check(engine, S, U, Fn, sample=list(range(12)) + [499])


@pytest.mark.gpu
def test_integer_grids_mad_zero_and_inf(engine):
    rng = np.random.default_rng(11)
    seen = dict(inf=0, S_mad0_pooled_not=0, S_mad_pooled_0=0)
    for nS in (1, 2, 3, 4, 5, 6, 9, 40):
        S = _tied(rng, (nS, 6, 1), -1, 2)
        Fn = _tied(rng, (60, 6, 1), -2, 3)
        U = np.array([[1.0]])
        cnt, O = _check(engine, S, U, Fn)
        Xu = S[:, :, 0].T.copy()
        cu, Ou = _check_uni(engine, Xu, Fn[:, :, 0].T.copy(), range(0, 60, 7))
        assert np.array_equal(cu, cnt) and np.array_equal(Ou, O)  # d = 1 with u = 1 is the univariate path
        seen['inf'] += int(np.isinf(O).sum())
        _, mad = np_medmad(Xu)
        for g in range(60):
            _, madp = np_medmad(np.column_stack([Xu, Fn[g, :, 0]]))
            seen['S_mad0_pooled_not'] += int(((mad == 0) & (madp != 0)).sum())
            seen['S_mad_pooled_0'] += int(((mad != 0) & (madp == 0)).sum())
    assert all(v > 0 for v in seen.values()), seen


@pytest.mark.gpu
def test_edge_shapes(engine):
    rng = np.random.default_rng(12)
    for nS, T, d, K in ((1, 3, 2, 5), (2, 3, 2, 5), (300, 4, 1, 1), (200, 2, 300, 3), (50, 5, 3, 1)):
        S = rng.standard_normal((nS, T, d))
        U = _unit(rng.standard_normal((K, d)))
        Fn = rng.standard_normal((9, T, d))
        Fn[0] = S[0]
        _check(engine, S, U, Fn)


@pytest.mark.gpu
def test_blocked_index_and_direction_blocks(engine):
    rng = np.random.default_rng(13)
    # 200 000 points: 671 rows per block, so K = 1000 directions build in two direction blocks, and T = 4 with
    # K = 200 in two time blocks
    S = rng.standard_normal((200_000, 1, 2))
    U = _unit(rng.standard_normal((1000, 2)))
    _check(engine, S, U, rng.standard_normal((40, 1, 2)) * 2.0, sample=[0, 1, 39])
    S = rng.standard_normal((200_000, 4, 2))
    U = _unit(rng.standard_normal((200, 2)))
    _check(engine, S, U, rng.standard_normal((40, 4, 2)), sample=[0, 39])
    # 200 000 new points: the query runs in two direction blocks
    S = rng.standard_normal((1000, 1, 2))
    U = _unit(rng.standard_normal((1000, 2)))
    Fn = rng.standard_normal((200_000, 1, 2)) * 1.5
    cnt, O = _check(engine, S, U, Fn, sample=[0, 1, 77_777, 199_999])
    one, O1, _, _ = _query(engine, S, U, Fn[77_777:77_778], sample=[])
    assert one[0] == cnt[77_777] and O1[0, 0] == O[0, 77_777]  # scored alone equals scored together


@pytest.mark.gpu
def test_cloud_50000x8_k1000(engine):
    rng = np.random.default_rng(14)
    S = rng.standard_normal((50_000, 1, 8))
    U = _unit(rng.standard_normal((1000, 8)))
    _check(engine, S, U, rng.standard_normal((1000, 1, 8)) * 1.3, sample=[0, 500, 999])


@pytest.mark.gpu
def test_curves_5000x256x3_k200(engine):
    rng = np.random.default_rng(15)
    S = rng.standard_normal((5000, 256, 3)).cumsum(1)
    U = _unit(rng.standard_normal((200, 3)))
    Fn = rng.standard_normal((1000, 256, 3)).cumsum(1)
    Fn[3] = S[10]
    cnt, O = _check(engine, S, U, Fn, sample=[0, 3, 999])
    some = [5, 3, 640]
    c2, O2, _, _ = _query(engine, S, U, Fn[some], sample=[])
    assert np.array_equal(c2, cnt[some]) and np.array_equal(O2, O[:, some])


@pytest.mark.gpu
def test_univariate_100000x1024(engine):
    rng = np.random.default_rng(16)
    X = rng.standard_normal((1024, 100_000)).cumsum(0)
    Y = rng.standard_normal((1024, 1000)).cumsum(0)
    Y[:, 1] = X[:, 5]
    _check_uni(engine, X, Y, [0, 1, 999])


@pytest.mark.gpu
def test_public_calls_equal_pooled_in_sample(engine):
    from statdepth_b200 import (DepthClassifier, FunctionalProjectionDepth, FunctionalProjectionDepthOf,
                                FunctionalReference, ProjectionDepth, ProjectionDepthOf)
    rng = np.random.default_rng(17)
    S = rng.standard_normal((300, 20, 2)).cumsum(1)
    Y = rng.standard_normal((6, 20, 2)).cumsum(1)
    X = rng.standard_normal((20, 400)).cumsum(0)
    Yu = rng.standard_normal((20, 5)).cumsum(0)
    P = pd.DataFrame(rng.standard_normal((700, 4)))
    Q = pd.DataFrame(rng.standard_normal((5, 4)), index=list('abcde'))
    for kind in ('projection', 'tukey'):
        got = FunctionalProjectionDepthOf(_frames(Y), _frames(S), kind=kind, directions=50, seed=2).values
        uni = FunctionalProjectionDepthOf([pd.DataFrame(Yu)], [pd.DataFrame(X)], kind=kind).values
        cl = ProjectionDepthOf(Q, P, kind=kind, directions=64, seed=3).values
        for g in range(5):
            exp = FunctionalProjectionDepth(_frames(np.concatenate([S, Y[g:g + 1]])), kind=kind, directions=50,
                                            seed=2).values[300]
            assert np.array_equal(got[g], exp), (kind, g)
            exp = FunctionalProjectionDepth([pd.DataFrame(np.column_stack([X, Yu[:, g]]))], kind=kind).values[400]
            assert np.array_equal(uni[g], exp), (kind, g)
            exp = ProjectionDepth(pd.concat([P, Q.iloc[g:g + 1]], ignore_index=True), kind=kind, directions=64,
                                  seed=3).values[700]
            assert np.array_equal(cl[g], exp), (kind, g)
        with FunctionalReference(_frames(S), depth=kind, directions=50, seed=2) as ref:
            assert np.array_equal(ref.depth_of(_frames(Y)).values, got)
            assert np.array_equal(ref.depth_of(_frames(Y[4:5])).values, got[4:5])
        refs = {'s': _frames(S), 't': _frames(S[:, ::-1] * 0.5 + 1.0)}
        with DepthClassifier(refs, depth=kind, directions=50, seed=2) as clf:
            one = np.column_stack([FunctionalProjectionDepthOf(_frames(Y), refs[k], kind=kind,
                                                               directions=clf.directions).values for k in refs])
            assert np.array_equal(clf.depths(_frames(Y)).to_numpy(), one)
            assert clf.predict(_frames(Y)).tolist() == [['s', 't'][i] for i in np.argmax(one, axis=1)]


@pytest.mark.gpu
def test_overflowing_projection_raises_as_pooled_call(engine):
    from statdepth_b200 import EngineError, FunctionalProjectionDepth, FunctionalReference
    rng = np.random.default_rng(18)
    S = rng.standard_normal((50, 3, 2))
    U = np.array([[1.0, 1.0], [1.0, -1.0]])
    Y = rng.standard_normal((2, 3, 2))
    Y[1, 1] = 1.5e308  # finite, but its projection on (1, 1) overflows
    for kind in ('projection', 'tukey'):
        with pytest.raises(EngineError) as pooled:
            FunctionalProjectionDepth(_frames(np.concatenate([S, Y[1:]])), kind=kind, directions=U)
        with FunctionalReference(_frames(S), depth=kind, directions=U) as ref:
            with pytest.raises(EngineError) as ei:
                ref.depth_of(_frames(Y))
            assert ei.value.status == pooled.value.status == 4
            assert len(ref.depth_of(_frames(Y[:1]))) == 1  # the reference stays usable
        with pytest.raises(EngineError) as ei:
            FunctionalReference(_frames(np.concatenate([S, Y[1:]])), depth=kind, directions=U)
        assert ei.value.status == 4
