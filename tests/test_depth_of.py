"""Out-of-sample depth (FunctionalDepthOf / PointcloudDepthOf and the sd_*_oos_f64 entry points).

Contract: the value for new observation g is what the in-sample depth returns for g after g alone is appended to
the reference sample S.  The CPU part drives the host layer with an oracle-backed engine of its own (the CPU oracle
on the pooled S u {g}, one g at a time); the GPU part pins the CUDA engine's counts to the same oracle."""
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch.multiprocessing as mp
from scipy.special import binom

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class OosOracleEngine:
    """TEST DOUBLE: the out-of-sample engine methods answered by the CPU oracle on S u {g}, one g at a time, plus
    the in-sample methods the expected values are computed with."""

    def __init__(self):
        from oracle import cpu_oracle
        self.o = cpu_oracle
        self.oos_calls = 0

    # in-sample
    def band_depth_counts(self, X, queries=None, j=2, relax=False):
        X = np.ascontiguousarray(X, dtype=np.float64)
        if relax:
            allc = self.o.mbd_counts_all(X, j=j)
            return allc if queries is None else allc[np.asarray(queries, dtype=np.int64)]
        return self.o.bd_counts(X, queries, j=j)

    def simplicial_counts(self, P, queries=None, tol=1e-7):
        return self.o.simplicial_counts(P, queries, tol)

    def l1_depth(self, P, queries=None):
        return self.o.l1_depth(P, queries)

    # out-of-sample
    def band_depth_oos_counts(self, S, Y, j=2, relax=False):
        self.oos_calls += 1
        nS = S.shape[1]
        out = np.zeros(Y.shape[1], dtype=np.int64)
        for g in range(Y.shape[1]):
            P = np.ascontiguousarray(np.concatenate([S, Y[:, [g]]], axis=1), dtype=np.float64)
            out[g] = self.o.mbd_counts_all(P, j=j)[nS] if relax else self.o.bd_counts(P, [nS], j=j)[0]
        return out

    def simplicial_oos_counts(self, S, Y, tol=1e-7):
        self.oos_calls += 1
        nS = S.shape[0]
        return np.array([self.o.simplicial_counts(np.vstack([S, Y[[g]]]), [nS], tol)[0] for g in range(len(Y))],
                        dtype=np.int64)

    def l1_oos_depth(self, S, Y):
        self.oos_calls += 1
        nS = S.shape[0]
        return np.array([self.o.l1_depth(np.vstack([S, Y[[g]]]), [nS])[0] for g in range(len(Y))])


def _install(fake, setter):
    import statdepth_b200._functional as f
    import statdepth_b200._pointcloud as p
    setter(f, "get_engine", lambda device=None: fake)
    setter(p, "get_engine", lambda device=None: fake)


@pytest.fixture()
def oos_oracle(monkeypatch):
    fake = OosOracleEngine()
    _install(fake, monkeypatch.setattr)
    return fake


def _walks(T, n, seed, labels=None):
    X = np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)
    return pd.DataFrame(X, columns=labels if labels is not None else range(n))


def _appended_functional(S, Y, J, relax):
    """Expected values by the contract: FunctionalDepth on S with the new curve appended (unique label)."""
    from statdepth_b200 import FunctionalDepth
    out = []
    for k in range(Y.shape[1]):
        g = Y.iloc[:, [k]].copy()
        g.columns = ['__new__']
        out.append(FunctionalDepth([pd.concat([S, g], axis=1)], to_compute=['__new__'], J=J, relax=relax).iloc[0])
    return np.array(out)


def _appended_cloud(S, Y, containment):
    from statdepth_b200 import PointcloudDepth
    out = []
    for k in range(Y.shape[0]):
        g = Y.iloc[[k], :].copy()
        g.index = ['__new__']
        out.append(PointcloudDepth(pd.concat([S, g]), to_compute=['__new__'], containment=containment).iloc[0])
    return np.array(out)


# ---------------------------------------------------------------------------------------------------------------
# CPU: host layer on the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("J", [2, 3])
@pytest.mark.parametrize("relax", [True, False])
def test_functional_equals_appended_reference(oos_oracle, J, relax):
    from statdepth_b200 import FunctionalDepthOf
    from statdepth_b200.depth import _FunctionalDepthUnivariate
    S = _walks(9, 12, 0)
    Y = _walks(9, 5, 1, labels=[3, 'b', 0, 'd', 11])  # labels 3, 0 and 11 also name sample curves
    res = FunctionalDepthOf([Y], [S], J=J, relax=relax)
    assert isinstance(res, _FunctionalDepthUnivariate)
    assert list(res.index) == list(Y.columns)
    assert res.values.tolist() == _appended_functional(S, Y, J, relax).tolist()  # same float arithmetic, bit for bit
    assert oos_oracle.oos_calls > 0


def test_functional_denominators_and_ties(oos_oracle, oracle):
    from statdepth_b200 import FunctionalDepthOf
    rng = np.random.default_rng(2)
    S = pd.DataFrame(np.round(rng.standard_normal((7, 10)).cumsum(0)))
    Yv = np.round(rng.standard_normal((7, 4)).cumsum(0))
    Yv[:, 1] = S.values[:, 4]  # equal to a sample curve
    Yv[:, 2] = Yv[:, 3]       # equal to another new curve: new curves never count each other
    Y = pd.DataFrame(Yv)
    T, nS = S.shape
    for relax in (True, False):
        res = FunctionalDepthOf([Y], [S], J=3, relax=relax)
        exp = np.zeros(4)
        for j in (2, 3):
            cnt = np.array([(oracle.mbd_counts_all(np.hstack([S.values, Yv[:, [g]]]), j=j)[nS] if relax else
                             oracle.bd_counts(np.hstack([S.values, Yv[:, [g]]]), [nS], j=j)[0]) for g in range(4)])
            s = cnt.astype(np.float64)
            if relax:
                s = s / float(T)
            exp = exp + s / binom(nS + 1, j)  # C(nS + 1, j): the reference counts the appended curve
        assert res.values.tolist() == exp.tolist()
        assert res.values[2] == res.values[3]


def test_functional_result_type_helpers(oos_oracle):
    from statdepth_b200 import FunctionalDepthOf
    S = _walks(8, 15, 3)
    Y = _walks(8, 6, 4, labels=list('uvwxyz'))
    Y['z'] = S[7].values  # a sample member: deep
    res = FunctionalDepthOf([Y], [S], relax=True)
    assert res.deepest().index[0] == res.ordered().index[0]
    assert list(res.get_deepest_data(n=2).columns) == list(res.ordered().index[:2])
    assert res.get_deepest_data().shape == (8, 1)
    # duplicate labels inside the new data keep their positions
    Yd = Y.copy()
    Yd.columns = ['a', 'a', 'b', 'b', 'c', 'c']
    rd = FunctionalDepthOf([Yd], [S], relax=True)
    assert list(rd.index) == list(Yd.columns) and rd.values.tolist() == res.values.tolist()


def test_functional_empty_new_data(oos_oracle):
    from statdepth_b200 import FunctionalDepthOf
    S = _walks(6, 5, 0)
    res = FunctionalDepthOf([S.iloc[:, :0]], [S], relax=True)
    assert len(res) == 0 and oos_oracle.oos_calls == 0


@pytest.mark.parametrize("d,nS", [(1, 9), (2, 12), (3, 10)])
def test_pointcloud_simplex_equals_appended_reference(oos_oracle, d, nS):
    from statdepth_b200 import PointcloudDepthOf
    from statdepth_b200.depth import _PointwiseDepth
    rng = np.random.default_rng(d)
    S = pd.DataFrame(rng.standard_normal((nS, d)))
    Y = pd.DataFrame(rng.standard_normal((4, d)), index=[0, 'q', 2, 'r'])
    Y.iloc[3] = S.iloc[1].values  # a sample point
    res = PointcloudDepthOf(Y, S, containment='simplex')
    assert isinstance(res, _PointwiseDepth) and list(res.index) == list(Y.index)
    assert res.values.tolist() == _appended_cloud(S, Y, 'simplex').tolist()
    cnt = oos_oracle.simplicial_oos_counts(S.values, Y.values)
    assert res.values.tolist() == (cnt.astype(np.float64) / binom(nS + 1, d + 1)).tolist()


def test_pointcloud_l1_equals_appended_reference(oos_oracle):
    from statdepth_b200 import PointcloudDepthOf
    rng = np.random.default_rng(5)
    S = pd.DataFrame(rng.standard_normal((20, 4)))
    Y = pd.DataFrame(rng.standard_normal((6, 4)), index=list('abcdef'))
    res = PointcloudDepthOf(Y, S, containment='l1')
    assert res.values.tolist() == _appended_cloud(S, Y, 'l1').tolist()
    assert res.deepest().index[0] in list(Y.index)
    Ys = pd.DataFrame(S.values[[3]])  # equal to a sample point: 0 / 0 in the reference
    assert np.isnan(PointcloudDepthOf(Ys, S, containment='l1').iloc[0])


def test_validation_errors(oos_oracle):
    from statdepth_b200 import DepthDegeneracy, FunctionalDepthOf, PointcloudDepthOf
    S = _walks(6, 8, 0)
    Y = _walks(6, 3, 1)
    with pytest.raises(ValueError):
        FunctionalDepthOf(Y, [S])                    # not a list
    with pytest.raises(ValueError):
        FunctionalDepthOf([Y], S)
    with pytest.raises(ValueError):
        FunctionalDepthOf([Y], [S], J=2.0)           # J not an integer
    with pytest.raises(ValueError):
        FunctionalDepthOf([Y], [S], J=1)
    with pytest.raises(ValueError):
        FunctionalDepthOf([Y], [S], J=6)             # J >= number of time points (reference quirk)
    with pytest.raises(ValueError):
        FunctionalDepthOf([Y], [S], relax=1)
    with pytest.raises(ValueError):
        FunctionalDepthOf([Y], [S], containment='bogus')
    with pytest.raises(ValueError):
        FunctionalDepthOf([_walks(7, 3, 1)], [S])    # different number of time points
    Yi = Y.copy()
    Yi.index = range(10, 16)
    FunctionalDepthOf([Yi], [S])                     # indices only matter under deep_check
    with pytest.raises(ValueError):
        FunctionalDepthOf([Yi], [S], deep_check=True)
    with pytest.raises(NotImplementedError):
        FunctionalDepthOf([Y], [S], J=4)
    with pytest.raises(NotImplementedError):
        FunctionalDepthOf([Y], [S], containment='r2_enum')
    with pytest.raises(DepthDegeneracy):
        FunctionalDepthOf([Y], [S], containment='simplex')  # univariate simplex: as FunctionalDepth
    mv = [_walks(6, 2, k) for k in range(5)]
    with pytest.raises(NotImplementedError):
        FunctionalDepthOf(mv, mv, containment='simplex')   # multivariate simplex depth
    P = pd.DataFrame(np.random.default_rng(0).standard_normal((10, 2)))
    with pytest.raises(ValueError):
        PointcloudDepthOf(P.iloc[:2], P.iloc[:, :1])       # different d
    with pytest.raises(ValueError):
        PointcloudDepthOf(P.iloc[:2], P, containment='bogus')
    for c in ('oja', 'mahalanobis'):
        with pytest.raises(NotImplementedError):
            PointcloudDepthOf(P.iloc[:2], P, containment=c)
    P4 = pd.DataFrame(np.random.default_rng(0).standard_normal((10, 4)))
    with pytest.raises(NotImplementedError):
        PointcloudDepthOf(P4.iloc[:2], P4, containment='simplex')
    assert oos_oracle.oos_calls == 1  # the one accepted call: every refusal happens before any engine call


# ---------------------------------------------------------------------------------------------------------------
# CPU: two ranks (gloo) shard rows (relaxed) and new observations (strict, point clouds)
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dist_inputs():
    rng = np.random.default_rng(11)
    S = pd.DataFrame(rng.standard_normal((13, 9)).cumsum(0))      # 13 rows: uneven split 7 + 6
    Y = pd.DataFrame(rng.standard_normal((13, 5)).cumsum(0))      # 5 new curves: 3 + 2
    P = pd.DataFrame(rng.standard_normal((11, 2)))
    Q = pd.DataFrame(rng.standard_normal((5, 2)))
    return S, Y, P, Q


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from statdepth_b200 import FunctionalDepthOf, PointcloudDepthOf, enable_distributed
    fake = OosOracleEngine()
    _install(fake, setattr)
    enable_distributed()
    S, Y, P, Q = _dist_inputs()
    res = dict(relax=FunctionalDepthOf([Y], [S], J=3, relax=True).values,
               strict=FunctionalDepthOf([Y], [S], J=3, relax=False).values,
               simplex=PointcloudDepthOf(Q, P, containment='simplex').values,
               l1=PointcloudDepthOf(Q, P, containment='l1').values)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_matches_single_process(tmp_path, monkeypatch):
    from statdepth_b200 import FunctionalDepthOf, PointcloudDepthOf
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    _install(OosOracleEngine(), monkeypatch.setattr)
    S, Y, P, Q = _dist_inputs()
    exp = dict(relax=FunctionalDepthOf([Y], [S], J=3, relax=True).values,
               strict=FunctionalDepthOf([Y], [S], J=3, relax=False).values,
               simplex=PointcloudDepthOf(Q, P, containment='simplex').values,
               l1=PointcloudDepthOf(Q, P, containment='l1').values)
    for r in range(world):  # every rank ends with the full result
        got = np.load(tmp_path / ("rank%d.npz" % r))
        # row blocks sum the same integers: the relaxed depth is bit-identical too
        for k in exp:
            assert got[k].tolist() == exp[k].tolist(), k


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA engine against the oracle on the pooled matrices
# ---------------------------------------------------------------------------------------------------------------
def _oracle_counts(oracle, S, Y, j, relax):
    nS = S.shape[1]
    out = []
    for g in range(Y.shape[1]):
        P = np.ascontiguousarray(np.hstack([S, Y[:, [g]]]))
        out.append(oracle.mbd_counts_all(P, j=j)[nS] if relax else oracle.bd_counts(P, [nS], j=j)[0])
    return np.array(out, dtype=np.int64)


def _ties(T, n, seed):
    return np.round(np.random.default_rng(seed).standard_normal((T, n)).cumsum(0))


@pytest.mark.gpu
@pytest.mark.parametrize("T,nS,nY,seed", [
    (13, 37, 11, 0),     # part pipeline, small and odd
    (17, 3001, 500, 1),  # part pipeline, odd pooled row
    (9, 5, 40, 2),       # more new curves than sample curves
    (21, 300, 1, 3),     # one new curve: no second rank pass
])
def test_relaxed_counts_equal_oracle(engine, oracle, T, nS, nY, seed):
    from statdepth_b200._engine import mbd_plan
    assert not mbd_plan(nS + nY)["slab"]
    rng = np.random.default_rng(seed)
    for S, Y in ((rng.standard_normal((T, nS)).cumsum(0), rng.standard_normal((T, nY)).cumsum(0)),
                 (_ties(T, nS, seed), _ties(T, nY, seed + 100))):
        if nY > 2:
            Y[:, 0] = S[:, 0]   # new values equal to sample values ...
            Y[:, 1] = Y[:, 2]   # ... and to each other
        for j in (2, 3):
            assert (engine.band_depth_oos_counts(S, Y, j, True) == _oracle_counts(oracle, S, Y, j, True)).all()


@pytest.mark.gpu
def test_relaxed_counts_slab_path(engine, oracle):
    from statdepth_b200._engine import mbd_plan
    T, nS, nY = 64, 20_000, 8
    assert mbd_plan(nS + nY)["slab"] == 1
    rng = np.random.default_rng(7)
    S = rng.standard_normal((T, nS)).cumsum(0)
    Y = rng.standard_normal((T, nY)).cumsum(0)
    Y[:, 3] = S[:, 5]
    for j in (2, 3):
        assert (engine.band_depth_oos_counts(S, Y, j, True) == _oracle_counts(oracle, S, Y, j, True)).all()
    St, Yt = _ties(T, nS, 8), _ties(T, nY, 9)  # tie-heavy rows leave the slab path for the part pipeline
    assert (engine.band_depth_oos_counts(St, Yt, 2, True) == _oracle_counts(oracle, St, Yt, 2, True)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("j", [2, 3])
def test_strict_counts_equal_oracle(engine, oracle, j):
    rng = np.random.default_rng(j)
    for T, nS, nY in ((11, 40, 9), (70, 120, 1), (5, 6, 30)):
        for S, Y in ((rng.standard_normal((T, nS)).cumsum(0), rng.standard_normal((T, nY)).cumsum(0)),
                     (_ties(T, nS, j), _ties(T, nY, j + 1))):
            if nY > 2:
                Y[:, 0] = S[:, 1]
                Y[:, 1] = Y[:, 2]
            assert (engine.band_depth_oos_counts(S, Y, j, False) == _oracle_counts(oracle, S, Y, j, False)).all()


@pytest.mark.gpu
def test_device_pointer_variant(engine, oracle):
    import torch
    T, nS, nY = 33, 2000, 70
    rng = np.random.default_rng(3)
    X = rng.standard_normal((T, nS + nY)).cumsum(0)
    exp = _oracle_counts(oracle, X[:, :nS], X[:, nS:], 2, True)
    dX = torch.from_numpy(X).cuda()
    out = torch.zeros(nY, dtype=torch.int64, device="cuda")
    base, ld = dX.data_ptr(), nS + nY
    torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's
    engine.band_depth_oos_counts_dev(base, T, nS, ld, base + 8 * nS, nY, ld, out.data_ptr(), 2, True)  # in place
    assert (out.cpu().numpy() == exp).all()
    dS, dY = dX[:, :nS].contiguous(), dX[:, nS:].contiguous()  # separate buffers: pooled on the device
    out.zero_()
    torch.cuda.synchronize()
    engine.band_depth_oos_counts_dev(dS.data_ptr(), T, nS, nS, dY.data_ptr(), nY, nY, out.data_ptr(), 2, True)
    assert (out.cpu().numpy() == exp).all()


@pytest.mark.gpu
def test_pointcloud_counts_equal_oracle(engine, oracle):
    import json
    rng = np.random.default_rng(4)
    # d = 2 on both sides of the 64-point switch (nS + 1 <= 64 enumerated, above counted), d = 3 and d = 1 enumerated
    for nS, d in ((40, 2), (63, 2), (64, 2), (300, 2), (25, 3), (30, 1)):
        S = rng.standard_normal((nS, d))
        Y = rng.standard_normal((12, d))
        Y[0] = S[3]
        exp = np.array([oracle.simplicial_counts(np.vstack([S, Y[[g]]]), [nS])[0] for g in range(len(Y))])
        assert (engine.simplicial_oos_counts(S, Y) == exp).all(), (nS, d)
    L = rng.integers(0, 5, size=(90, 2)).astype(np.float64)  # lattice: collinear triples, duplicates
    for nS in (50, 80):
        S, Y = L[:nS], L[nS:]
        exp = np.array([oracle.simplicial_counts(np.vstack([S, Y[[g]]]), [nS])[0] for g in range(len(Y))])
        assert (engine.simplicial_oos_counts(S, Y) == exp).all(), nS
    # the reference's collinear / tolerance-band fixture: a point held out of the 70-point cloud
    with open(os.path.join(ROOT, "tests", "golden", "reference_vectors_large.json")) as fh:
        cases = [c for c in json.load(fh)["cases"] if c["kind"] == "pointcloud" and len(c["P"]) == 70]
    assert cases
    for case in cases:
        P = np.asarray(case["P"], dtype=np.float64)
        q = int(case["to_compute"][0])
        S = np.delete(P, q, axis=0)
        cnt = engine.simplicial_oos_counts(S, P[[q]])
        assert cnt[0] == oracle.simplicial_counts(P, [q])[0], case["name"]
        np.testing.assert_allclose(cnt[0] / binom(70, 3), case["depths"][0], rtol=1e-12)
    for d in (2, 5, 16):
        S = rng.standard_normal((700, d))
        Y = rng.standard_normal((50, d))
        exp = np.array([oracle.l1_depth(np.vstack([S, Y[[g]]]), [len(S)])[0] for g in range(len(Y))])
        np.testing.assert_allclose(engine.l1_oos_depth(S, Y), exp, rtol=1e-12)


@pytest.mark.gpu
def test_nonfinite_new_data_rejected(engine):
    from statdepth_b200 import EngineError
    rng = np.random.default_rng(0)
    S = rng.standard_normal((16, 50)).cumsum(0)
    Y = rng.standard_normal((16, 6)).cumsum(0)
    Y[5, 4] = np.nan
    for j, relax in ((2, True), (3, True), (2, False), (3, False)):
        with pytest.raises(EngineError) as ei:
            engine.band_depth_oos_counts(S, Y, j, relax)
        assert ei.value.status == 4
    P = rng.standard_normal((100, 2))
    Q = rng.standard_normal((3, 2))
    Q[1, 0] = np.inf
    for fn in (engine.simplicial_oos_counts, engine.l1_oos_depth):
        with pytest.raises(EngineError) as ei:
            fn(P, Q)
        assert ei.value.status == 4
        with pytest.raises(EngineError):
            fn(P[:20], Q)  # enumerated side of the switch too
    # the context stays usable
    Y[5, 4] = 0.0
    assert engine.band_depth_oos_counts(S, Y, 2, True).shape == (6,)


@pytest.mark.gpu
def test_public_api_bit_identical_to_batched_path(engine):
    """FunctionalDepthOf against homogeneity._depths_of_each_in (one batched sub-population per new curve)."""
    from statdepth_b200 import FunctionalDepthOf
    from statdepth_b200.homogeneity import _depths_of_each_in
    rng = np.random.default_rng(12)
    T, nF, nG = 256, 20_000, 32
    F = pd.DataFrame(rng.standard_normal((T, nF)).cumsum(0))
    G = pd.DataFrame(rng.standard_normal((T, nG)).cumsum(0), columns=['g%d' % k for k in range(nG)])
    for J, relax in ((2, True), (3, True), (2, False)):
        ours = FunctionalDepthOf([G], [F], J=J, relax=relax).values
        assert ours.tolist() == _depths_of_each_in(F, G, J, relax).tolist(), (J, relax)
    # strict J = 3 enumerates C(nF, 3) triples per new curve: a smaller sample
    Fs, Gs = F.iloc[:64, :300], G.iloc[:64, :8]
    ours = FunctionalDepthOf([Gs], [Fs], J=3, relax=False).values
    assert ours.tolist() == _depths_of_each_in(Fs, Gs, 3, False).tolist()


@pytest.mark.gpu
def test_full_size_relaxed_against_in_sample_path(engine):
    """n_S = 100 000, n_Y = 1 000, T = 1024: 8 new curves equal the in-sample path on [S | g] with query n_S."""
    T, nS, nY = 1024, 100_000, 1000
    rng = np.random.default_rng(13)
    S = rng.standard_normal((T, nS)).cumsum(0)
    Y = rng.standard_normal((T, nY)).cumsum(0)
    got2 = engine.band_depth_oos_counts(S, Y, 2, True)
    got3 = engine.band_depth_oos_counts(S, Y, 3, True)
    P = np.empty((T, nS + 1))
    P[:, :nS] = S
    for g in rng.choice(nY, size=8, replace=False):
        P[:, nS] = Y[:, g]
        assert engine.band_depth_counts(P, [nS], 2, True)[0] == got2[g]
        assert engine.band_depth_counts(P, [nS], 3, True)[0] == got3[g]
