"""The host-buffer and device-pointer entry points of one operation share one body in api.cu: on the same data the
two return the same bits, whatever the host layout.  And the int64 guard of relaxed band depth refuses every input
whose numerators would overflow, on every path that reaches it, leaving the context usable."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

T, N = 40, 3000


def _data(seed=0, T=T, n=N):
    return np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)


def _host(X, order):
    return np.ascontiguousarray(X) if order == "C" else np.asfortranarray(X)


def _dev(A, dtype=None):
    import torch
    A = np.ascontiguousarray(A)
    return torch.from_numpy(A if dtype is None else A.astype(dtype)).cuda()


def _empty(shape, dtype):
    import torch
    return torch.full(shape, -7, dtype=dtype, device="cuda")


def _ready():
    import torch
    torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's


def _same(host, dev):
    dev = dev.cpu().numpy()
    assert host.shape == dev.shape and host.dtype == dev.dtype
    assert host.tobytes() == dev.tobytes()


@pytest.mark.parametrize("order", ["C", "F"])
@pytest.mark.parametrize("j,relax,queries", [(2, True, None), (3, True, [5, 0, 2999, 17]), (2, False, None),
                                             (2, False, [11, 2998, 11])])
def test_band_depth_pair(engine, order, j, relax, queries):
    import torch
    X = _data(1)
    got = engine.band_depth_counts(_host(X, order), queries, j, relax)
    dX = _dev(X)
    dq = None if queries is None else _dev(np.asarray(queries, dtype=np.int64))
    nq = N if queries is None else len(queries)
    out = _empty((nq,), torch.int64)
    _ready()
    engine.band_depth_counts_dev(dX.data_ptr(), T, N, N, out.data_ptr(), None if dq is None else dq.data_ptr(), nq, j,
                                 relax)
    _same(got, out)


@pytest.mark.parametrize("j,relax", [(2, True), (3, True), (2, False)])
def test_band_depth_oos_pair(engine, j, relax):
    import torch
    S, Y = _data(2, n=2000), _data(3, n=37)
    got = engine.band_depth_oos_counts(S, Y, j, relax)
    dS, dY = _dev(S), _dev(Y)
    out = _empty((37,), torch.int64)
    _ready()
    engine.band_depth_oos_counts_dev(dS.data_ptr(), T, 2000, 2000, dY.data_ptr(), 37, 37, out.data_ptr(), j, relax)
    _same(got, out)


@pytest.mark.parametrize("order", ["C", "F"])
def test_rank_sums_pair(engine, order):
    import torch
    X = _data(4)
    q, b, a = engine.band_rank_sums(_host(X, order), want_above=True)
    dX = _dev(X)
    out = _empty((3, N), torch.int64)
    _ready()
    engine.band_rank_sums_dev(dX.data_ptr(), T, N, N, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr())
    for k, host in enumerate((q, b, a)):
        _same(host, out[k])


@pytest.mark.parametrize("order", ["C", "F"])
def test_envelope_pair(engine, order):
    import torch
    X = _data(5)
    member = (np.arange(N) % 3 != 0).astype(np.uint8)
    lo, hi, outside = engine.band_envelope(_host(X, order), member, 1.5)
    dX, dm = _dev(X), _dev(member)
    env = _empty((2, T), torch.float64)
    dout = _empty((N,), torch.int64)
    _ready()
    engine.band_envelope_dev(dX.data_ptr(), T, N, N, dm.data_ptr(), 1.5, env[0].data_ptr(), env[1].data_ptr(),
                             dout.data_ptr())
    _same(lo, env[0])
    _same(hi, env[1])
    _same(outside, dout)


@pytest.mark.parametrize("order", ["C", "F"])
def test_band_halfspace_pair(engine, order):
    import torch
    X = _data(6)
    got = engine.band_halfspace_counts(_host(X, order))
    dX = _dev(X)
    out = _empty((N,), torch.int64)
    _ready()
    engine.band_halfspace_counts_dev(dX.data_ptr(), T, N, N, out.data_ptr())
    _same(got, out)


@pytest.mark.parametrize("order", ["C", "F"])
def test_band_outlyingness_pair(engine, order):
    import torch
    X = _data(7)
    o, med, mad = engine.band_outlyingness(_host(X, order), want_medmad=True)
    dX = _dev(X)
    do = _empty((T, N), torch.float64)
    dmed, dmad = _empty((T,), torch.float64), _empty((T,), torch.float64)
    _ready()
    engine.band_outlyingness_dev(dX.data_ptr(), T, N, N, do.data_ptr(), dmed.data_ptr(), dmad.data_ptr())
    _same(o, do)
    _same(med, dmed)
    _same(mad, dmad)


def test_projection_pairs(engine):
    import torch
    rng = np.random.default_rng(8)
    Nc, Tc, d, K = 2500, 5, 3, 64
    F = rng.standard_normal((Nc, Tc, d))
    U = rng.standard_normal((K, d))
    dF = _dev(F)
    counts = engine.projection_tukey_counts(F, U)
    dc = _empty((Nc,), torch.int64)
    _ready()
    engine.projection_tukey_counts_dev(dF.data_ptr(), Nc, Tc, d, U, dc.data_ptr())
    _same(counts, dc)
    o, med, mad = engine.projection_outlyingness(F, U, want_medmad=True)
    do = _empty((Tc, Nc), torch.float64)
    dmed, dmad = _empty((Tc, K), torch.float64), _empty((Tc, K), torch.float64)
    engine.projection_outlyingness_dev(dF.data_ptr(), Nc, Tc, d, U, do.data_ptr(), dmed.data_ptr(), dmad.data_ptr())
    _same(o, do)
    _same(med, dmed)
    _same(mad, dmad)


# ---------------------------------------------------------------------------------------------------------------
# relaxed J = 3 with 2 700 000 curves: 3 * C(n - 1, 3) >= 9e18, so the numerators cannot be formed in int64
# ---------------------------------------------------------------------------------------------------------------
BIG = 2_700_000


def _overflows(call):
    from statdepth_b200 import EngineError
    with pytest.raises(EngineError) as ei:
        call()
    assert ei.value.status == 5, ei.value
    assert "overflows int64" in str(ei.value)


def _still_usable(engine, oracle):
    X = _data(9, T=8, n=500)
    assert (engine.band_depth_counts(X, None, 2, True) == oracle.mbd_counts_all(X)).all()


def test_overflow_band_depth_host(engine, oracle):
    X1 = np.random.default_rng(10).standard_normal((1, BIG))
    _overflows(lambda: engine.band_depth_counts(X1, None, 3, True))
    _still_usable(engine, oracle)
    X16 = np.random.default_rng(11).standard_normal((16, BIG))  # 346 MB: streamed in row blocks
    _overflows(lambda: engine.band_depth_counts(X16, None, 3, True))
    _still_usable(engine, oracle)


def test_overflow_band_depth_dev(engine, oracle):
    import torch
    dX = _dev(np.random.default_rng(12).standard_normal((1, BIG)))
    out = _empty((BIG,), torch.int64)
    _ready()
    _overflows(lambda: engine.band_depth_counts_dev(dX.data_ptr(), 1, BIG, BIG, out.data_ptr(), None, BIG, 3, True))
    _still_usable(engine, oracle)


def test_overflow_out_of_sample(engine, oracle):
    import torch
    rng = np.random.default_rng(13)
    S, Y = rng.standard_normal((1, BIG)), rng.standard_normal((1, 1))
    _overflows(lambda: engine.band_depth_oos_counts(S, Y, 3, True))
    _still_usable(engine, oracle)
    dS, dY = _dev(S), _dev(Y)
    out = _empty((1,), torch.int64)
    _ready()
    _overflows(lambda: engine.band_depth_oos_counts_dev(dS.data_ptr(), 1, BIG, BIG, dY.data_ptr(), 1, 1,
                                                        out.data_ptr(), 3, True))
    _still_usable(engine, oracle)


def test_overflow_sorted_reference(engine, oracle):
    import torch
    rng = np.random.default_rng(14)
    dS, dY = _dev(rng.standard_normal((1, BIG))), _dev(rng.standard_normal((1, 1)))
    index = _empty((1, BIG), torch.float64)
    out = _empty((2, 1), torch.int64)
    _ready()
    engine.band_sort_rows_dev(dS.data_ptr(), 1, BIG, BIG, index.data_ptr())
    _overflows(lambda: engine.band_depth_sorted_counts_dev(index.data_ptr(), 1, BIG, dY.data_ptr(), 1, 1, 3,
                                                           out.data_ptr()))
    _still_usable(engine, oracle)
