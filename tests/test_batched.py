"""Batched band depth (sd_band_depth_batched_f64): many sub-populations of one matrix in one call.

Equally sized batches take the grouped pass: relaxed depth ranks all batches as one stacked matrix of B*T rows whose
row groups accumulate separately (mbd_all_device with group_rows = T), strict J = 2 depth runs the batched
sign-vector matcher.  Permutation tests, K-sampled FunctionalDepth and functional homogeneity p3 stand on it.

The reference is exact integer arithmetic on the member columns of each batch (np_batched_counts).  Shapes are
chosen so that every route of the grouped pass runs: row blocks of 65 535 rows that split a batch, several parts per
row, the overflow / heavy-class / generic / slab kernels with group offsets, several passes of batches, and the
matcher's chunked launches.  Each case also asserts, from engine.timings(), that it took the route it is about.
"""
import numpy as np
import pandas as pd
import pytest

from statdepth_b200 import _engine as E

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# exact references
# ------------------------------------------------------------------------------------------------
def _comb(x, j):
    """C(x, j) for int64 arrays x >= 0 (0 when x < j)."""
    x = np.asarray(x, dtype=np.int64)
    return x * (x - 1) // 2 if j == 2 else x * (x - 1) * (x - 2) // 6


def _members(membership):
    """Member columns of each batch, in column order, grouped by batch size: {m: (batch ids, cols [nb, m])}."""
    mem = np.asarray(membership) != 0
    sizes = mem.sum(axis=1)
    out = {}
    for m in np.unique(sizes):
        bs = np.flatnonzero(sizes == m)
        out[int(m)] = (bs, np.nonzero(mem[bs])[1].reshape(len(bs), int(m)))
    return out


def np_batched_counts(X, membership, queries, j, relax=True):
    """Relaxed band depth numerators of the queries of every batch, exactly: for each row of a batch's member columns,
    b = members strictly below the query and a = members strictly above it, and the count is
    sum over rows of C(m-1, j) - C(b, j) - C(a, j).  Values are replaced by their rank among the distinct values of X
    (-0.0 == 0.0), and every (row, batch) gets its own key range, so one np.sort + np.searchsorted ranks all batches
    of one size at once."""
    assert relax, "strict depth: use the C oracle's bd_counts on the compacted sub-matrix"
    X = np.asarray(X, dtype=np.float64)
    T, n = X.shape
    qs = np.asarray(queries, dtype=np.int64)
    out = np.zeros(qs.shape, dtype=np.int64)
    codes = np.unique(X, return_inverse=True)[1].reshape(T, n).astype(np.int64)
    span = int(codes.max()) + 1
    for m, (bs, cols) in _members(membership).items():
        nb = len(bs)
        seg = np.arange(T, dtype=np.int64)[:, None] * nb + np.arange(nb, dtype=np.int64)[None, :]  # [T, nb]
        keys = np.sort((codes[:, cols] + (seg * span)[:, :, None]).ravel())
        qk = codes[:, qs[bs]] + (seg * span)[:, :, None]                                           # [T, nb, nq]
        start = (seg * m)[:, :, None]
        below = np.searchsorted(keys, qk, "left") - start
        above = start + m - np.searchsorted(keys, qk, "right")
        out[bs] = (_comb(m - 1, j) - _comb(below, j) - _comb(above, j)).sum(axis=0)
    return out


def np_strict_counts_small(X, membership, queries):
    """Strict J = 2 numerators by brute force over all pairs of other members (small batches only): the pair (u, v)
    counts when min(x_u, x_v) <= x_q <= max(x_u, x_v) at every row."""
    X = np.asarray(X, dtype=np.float64)
    qs = np.asarray(queries, dtype=np.int64)
    out = np.zeros(qs.shape, dtype=np.int64)
    for m, (bs, cols) in _members(membership).items():
        for c0 in range(0, len(bs), 8192):
            b = bs[c0:c0 + 8192]
            Y = X[:, cols[c0:c0 + 8192]].transpose(1, 2, 0)       # [nb, m, T]
            Q = X[:, qs[b]].transpose(1, 2, 0)[:, :, None, :]    # [nb, nq, 1, T]
            le = Y[:, None] <= Q                                  # [nb, nq, m, T]
            ge = Y[:, None] >= Q
            inside = ((le[:, :, :, None] & ge[:, :, None, :]) | (ge[:, :, :, None] & le[:, :, None, :])).all(-1)
            self_ = cols[c0:c0 + 8192][:, None, :] == qs[b][:, :, None]  # [nb, nq, m]: the query itself
            inside &= ~self_[:, :, :, None] & ~self_[:, :, None, :]
            out[b] = np.triu(inside, 1).sum(axis=(2, 3))
    return out


def _local(cols, q):
    """Positions of the global ids q among the sorted member columns cols."""
    pos = np.searchsorted(cols, q)
    assert (cols[pos] == q).all()
    return pos


def engine_per_batch(engine, X, membership, queries, j, relax):
    """Single-matrix engine calls on each batch's compacted sub-matrix."""
    out = np.zeros(np.shape(queries), dtype=np.int64)
    for m, (bs, cols) in _members(membership).items():
        for b, c in zip(bs, cols):
            out[b] = engine.band_depth_counts(np.ascontiguousarray(X[:, c]), _local(c, queries[b]), j, relax)
    return out


def oracle_strict(oracle, X, membership, queries, batches, j=2):
    """The C oracle's strict numerators of the given batches (rows of the result)."""
    mem = np.asarray(membership) != 0
    out = []
    for b in batches:
        c = np.flatnonzero(mem[b])
        out.append(oracle.bd_counts(np.ascontiguousarray(X[:, c]), _local(c, queries[b]), j=j))
    return np.array(out)


def uniform_batches(rng, n, B, m0, nqb=None):
    """B random sub-populations of m0 of the n columns -> (membership [B, n] uint8, members [B, m0] sorted, queries
    [B, nqb]: distinct members in random order, all m0 when nqb is None)."""
    members = np.sort(np.argsort(rng.random((B, n)), axis=1)[:, :m0], axis=1)
    mem = np.zeros((B, n), dtype=np.uint8)
    mem[np.arange(B)[:, None], members] = 1
    k = m0 if nqb is None else nqb
    pick = np.argsort(rng.random((B, m0)), axis=1)[:, :k]
    return mem, members, np.take_along_axis(members, pick, axis=1)


def walks(seed, T, n):
    return np.random.default_rng(seed).standard_normal((T, n)).cumsum(0)


def _slab_rows(rng, kind, T, n):
    """Data kinds of test_gpu_parity's slab tests; `tail_many` makes a quarter of the rows heavy-tailed so that a
    group holds rows ranked by the slab path and rows the part pipeline takes over."""
    if kind == "normal":
        return rng.standard_normal((T, n))
    if kind == "round4":     # moderately tied: the table kernel's sample sees the ties and the part pipeline takes over
        return np.round(rng.standard_normal((T, n)), 4)
    if kind == "tail_many":  # unfit rows (hist kernel validation) among fit ones
        X = rng.standard_normal((T, n))
        X[1::4] = rng.standard_cauchy((len(range(1, T, 4)), n))
        return X
    raise ValueError(kind)


# ------------------------------------------------------------------------------------------------
# CPU: the references themselves
# ------------------------------------------------------------------------------------------------
def _tied_matrix(rng, T, n):
    X = np.round(rng.standard_normal((T, n)).cumsum(0))
    X[:, : n // 4] = np.where(rng.random((T, n // 4)) < 0.5, 0.0, -0.0)  # a +-0.0 class
    X[T // 2] = 3.0                                                        # a constant row
    return X


def test_reference_matches_oracle(oracle):
    rng = np.random.default_rng(3)
    T, n = 11, 40
    X = _tied_matrix(rng, T, n)
    for m0 in (1, 2, 3, 17, 40):
        mem, members, qs = uniform_batches(rng, n, 6, m0)
        for j in (2, 3):
            got = np_batched_counts(X, mem, qs, j)
            for b in range(6):
                sub = np.ascontiguousarray(X[:, members[b]])
                exp = oracle.mbd_counts_all(sub, j=j)[_local(members[b], qs[b])] if m0 > 1 else np.zeros(1, np.int64)
                assert (got[b] == exp).all(), (m0, j, b)
    # ragged batches, repeated and unordered queries, membership bytes other than 1
    mem = (rng.random((9, n)) < 0.5).astype(np.uint8) * rng.integers(1, 256, size=(9, n)).astype(np.uint8)
    mem[:, 0] = 7
    qs = np.stack([rng.choice(np.flatnonzero(mem[b]), 5) for b in range(9)])
    qs[:, -1] = 0
    for j in (2, 3):
        got = np_batched_counts(X, mem, qs, j)
        for b in range(9):
            c = np.flatnonzero(mem[b])
            assert (got[b] == oracle.mbd_counts_all(np.ascontiguousarray(X[:, c]), j=j)[_local(c, qs[b])]).all()


def test_negative_zero_equals_zero():
    X = np.array([[0.0, -0.0, 0.0, 1.0, -1.0]])
    mem = np.ones((1, 5), dtype=np.uint8)
    q = np.arange(5)[None, :]
    # the zeros: 1 below, 1 above, 4 others -> C(4,2) - 0 - 0 = 6; +-1: 4 on one side -> 6 - 6 = 0
    assert np_batched_counts(X, mem, q, 2).tolist() == [[6, 6, 6, 0, 0]]


def test_strict_reference_matches_oracle(oracle):
    rng = np.random.default_rng(4)
    T, n = 6, 30
    for X in (rng.standard_normal((T, n)).cumsum(0), _tied_matrix(rng, T, n)):
        for m0 in (3, 5, 12):
            mem, members, qs = uniform_batches(rng, n, 7, m0, min(m0, 4))
            assert (np_strict_counts_small(X, mem, qs) == oracle_strict(oracle, X, mem, qs, range(7))).all()


def test_permutation_prefix_property(monkeypatch):
    """permutation_test(B=k) draws the first k permutations of permutation_test(B=1000) with the same seed, for the
    batched and the looping evaluation alike: a batched null's prefix can be checked against a short looped run."""
    from statdepth_b200 import homogeneity as H
    drawn = {}

    def fake_batched(pooled, nF, perms, method, relax):
        drawn.setdefault("batched", []).append(perms.copy())
        return np.zeros(len(perms))

    class FakeHomogeneity:
        def __init__(self, F, G, **kw):
            drawn.setdefault("loop", []).append((list(F[0].columns), list(G[0].columns)))

        def homogeneity(self):
            return 0.0

    monkeypatch.setattr(H, "_perm_stats_batched", fake_batched)
    monkeypatch.setattr(H, "FunctionalHomogeneity", FakeHomogeneity)
    F = pd.DataFrame(np.zeros((3, 256)))
    G = pd.DataFrame(np.ones((3, 256)))
    H.permutation_test(F, G, "p1", B=1000, seed=5)
    H.permutation_test(F, G, "p1", B=10, seed=5)
    full, short = drawn["batched"]
    assert full.shape == (1000, 512) and (short == full[:10]).all()
    drawn.clear()
    H.permutation_test(F, G, "p2", B=10, seed=5, relax=False, batched=False)
    loop = drawn["loop"][1:]  # [0] is the observed statistic
    assert [f for f, _ in loop] == [list(p[:256]) for p in full[:10]]
    assert [g for _, g in loop] == [list(p[256:]) for p in full[:10]]


# ------------------------------------------------------------------------------------------------
# GPU: the grouped relaxed pass
# ------------------------------------------------------------------------------------------------
def _check_relaxed(engine, X, mem, qs, sample, per_batch=True, max_launches=None, fallback_rows=0):
    """Batched j = 2, 3 against single-matrix engine calls (every batch) and the exact reference (sampled batches);
    returns the counts and the timings of the batched calls, by j."""
    res, tms = {}, {}
    for j in (2, 3):
        got = engine.band_depth_counts_batched(X, mem, qs, j, True)
        tm = tms[j] = engine.timings()
        if max_launches is not None:
            assert tm["launches"] <= max_launches, tm
        if fallback_rows is not None:
            assert tm["fallback_rows"] == fallback_rows, tm
        sample = np.asarray(sample)
        assert (got[sample] == np_batched_counts(X, mem[sample], qs[sample], j)).all(), j
        if per_batch:
            assert (got == engine_per_batch(engine, X, mem, qs, j, True)).all(), j
        res[j] = got
    return res, tms


@gpu
def test_grouped_cfg5_shape(engine):
    """bench's perm shape: 2 x 256 curves of 256 points, B = 1000 batches of 256 (all queried) -> 256 000 stacked
    rows in 4 row blocks; 65 535 = 255 * 256 + 255, so batch 255 (and 511, 767) straddles two blocks.  Then the
    memF call: 257 members, one query."""
    rng = np.random.default_rng(5)
    T, n, B = 256, 512, 1000
    X = walks(50, T, n)
    mem, members, qs = uniform_batches(rng, n, B, 256)
    _check_relaxed(engine, X, mem, qs, [0, 254, 255, 256, 511, 767, 999], max_launches=60)
    mem1, members1, _ = uniform_batches(rng, n, B, 257)
    q1 = members1[np.arange(B), rng.integers(0, 257, B)][:, None]
    _check_relaxed(engine, X, mem1, q1, [0, 254, 255, 256, 999], max_launches=60)


@gpu
def test_grouped_small_rows_many_batches(engine, monkeypatch):
    """T = 8, B = 9000 batches of 50 -> 72 000 rows; 65 535 = 8 * 8191 + 7: batch 8191 straddles the row blocks.
    Every batch against the exact reference, with both warp rank kernels (sub-bin and sorting network)."""
    rng = np.random.default_rng(6)
    T, n, B = 8, 120, 9000
    X = walks(60, T, n)
    X[:, ::3] = np.round(X[:, ::3], 1)  # some ties
    mem, _, qs = uniform_batches(rng, n, B, 50, 3)
    ref = {j: np_batched_counts(X, mem, qs, j) for j in (2, 3)}
    for rank in ("subbin", "network"):
        if rank == "network":
            monkeypatch.setenv("SD_MBD_RANK", "network")
        for j in (2, 3):
            got = engine.band_depth_counts_batched(X, mem, qs, j, True)
            tm = engine.timings()
            assert tm["launches"] <= 20 and tm["fallback_rows"] == 0, tm
            assert (got == ref[j]).all(), (rank, j, np.flatnonzero((got != ref[j]).any(1))[:10])


@gpu
def test_grouped_several_parts_per_row(engine, monkeypatch):
    """Batches of 2000 curves: 5 parts per row, and 65 535 rows * 5 parts >= 100 000 starts the overflow kernel.
    T = 16, B = 4200: the gathered matrix exceeds 1 GB, so the batches run in passes of 4194 and 6; in the first,
    batch 4095 straddles the row blocks (65 535 = 16 * 4095 + 15).  Two rows of every batch hold a +-0.0 class of
    ~1400 curves, ranked by the heavy-class kernel in both row blocks.  Repeated with the sorting-network rank kernel
    and with every row on the generic kernel."""
    rng = np.random.default_rng(7)
    T, n, B = 16, 2400, 4200
    X = walks(70, T, n)
    for t in (3, 11):
        X[t, rng.random(n) < 0.7] = 0.0
        X[t, rng.random(n) < 0.3] = -0.0
    mem, _, qs = uniform_batches(rng, n, B, 2000, 4)
    sample = [0, 4094, 4095, 4096, 4193, 4194, 4199]
    res, _ = _check_relaxed(engine, X, mem, qs, sample, max_launches=60)
    try:
        engine.set_option(E.OPT_MBD_FORCE_FALLBACK, 1)
        assert (engine.band_depth_counts_batched(X, mem, qs, 2, True) == res[2]).all()
        assert engine.timings()["fallback_rows"] == B * T
    finally:
        engine.set_option(E.OPT_MBD_FORCE_FALLBACK, 0)
    monkeypatch.setenv("SD_MBD_RANK", "network")
    for j in (2, 3):
        assert (engine.band_depth_counts_batched(X, mem, qs, j, True) == res[j]).all(), j


@gpu
@pytest.mark.parametrize("kind", ["normal", "round4", "tail_many"])
def test_grouped_slab_path(engine, monkeypatch, kind):
    """Batches of 16 384 and 20 000 curves take the slab path in groups (slab rows and part-pipeline rows in one
    group for round4 / tail_many); the same with the part pipeline everywhere (SD_MBD_PATH=parts) and with every row
    on the generic kernel (OPT_MBD_FORCE_FALLBACK)."""
    rng = np.random.default_rng(800 + len(kind))
    T, n = 8, 24000
    X = _slab_rows(rng, kind, T, n)
    for m0, B in ((16384, 4), (20000, 3)):
        mem, _, qs = uniform_batches(rng, n, B, m0, 64)
        ref = {j: np_batched_counts(X, mem, qs, j) for j in (2, 3)}
        launches = {}
        for route in ("slab", "parts", "generic"):
            if route == "parts":
                monkeypatch.setenv("SD_MBD_PATH", "parts")
            try:
                if route == "generic":
                    engine.set_option(E.OPT_MBD_FORCE_FALLBACK, 1)
                for j in (2, 3):
                    got = engine.band_depth_counts_batched(X, mem, qs, j, True)
                    tm = engine.timings()
                    assert (got == ref[j]).all(), (route, m0, j)
                    launches[route] = tm["launches"]
                    if route == "generic":
                        assert tm["fallback_rows"] == B * T, tm
                    elif kind == "normal":
                        assert tm["fallback_rows"] == 0, tm
            finally:
                engine.set_option(E.OPT_MBD_FORCE_FALLBACK, 0)
                monkeypatch.delenv("SD_MBD_PATH", raising=False)
        if kind == "normal":  # table + hist + rank (+ finish, compaction, gather) against the 7+ of the part pipeline
            assert launches["slab"] < launches["parts"], launches
        per = engine_per_batch(engine, X, mem, qs, 2, True)
        assert (per == ref[2]).all()


@gpu
def test_grouped_heavy_and_generic_rows(engine):
    """Batches of 200 000 curves, T = 2: with 150 value classes every part overflows and each row is ranked by the
    generic kernel (fallback_rows == B * T); with 70 % of the values in a +-0.0 class the heavy-class kernel ranks
    the zeros and no row falls back."""
    rng = np.random.default_rng(9)
    T, n, B = 2, 230_000, 2
    classes = rng.integers(0, 150, size=(T, n)).astype(np.float64) * 0.5
    zeros = rng.standard_normal((T, n))
    z = rng.random((T, n)) < 0.7
    zeros[z] = np.where(rng.random(int(z.sum())) < 0.5, 0.0, -0.0)
    mem, _, qs = uniform_batches(rng, n, B, 200_000, 256)
    for X, fb in ((classes, B * T), (zeros, 0)):
        _check_relaxed(engine, X, mem, qs, range(B), max_launches=40, fallback_rows=fb)


@gpu
def test_grouped_several_passes(engine, monkeypatch):
    """T = 512, m0 = 20 000: 13 batches fill the 1 GB gather, so B = 30 runs in passes of 13, 13 and 4, each
    accumulating at acc + b0 * m0, and one gather at the end reads all of them.  The rows are ranked by the slab
    path; with 64-curve parts the part lists cap a row block at 2512 rows, so slab row groups straddle row blocks."""
    rng = np.random.default_rng(10)
    T, n, B = 512, 21000, 30
    X = rng.standard_normal((T, n))
    mem, _, qs = uniform_batches(rng, n, B, 20000, 5)
    res, tms = _check_relaxed(engine, X, mem, qs, [12, 13, 29], max_launches=120)
    monkeypatch.setenv("SD_MBD_TARGET_PART", "64")
    for j in (2, 3):
        assert (engine.band_depth_counts_batched(X, mem, qs, j, True) == res[j]).all(), j
        assert engine.timings()["launches"] > tms[j]["launches"] + 6  # at least two more row blocks in each pass


# ------------------------------------------------------------------------------------------------
# GPU: the batched strict matcher
# ------------------------------------------------------------------------------------------------
@gpu
def test_strict_mixed_batches(engine, oracle):
    """Batches of continuous columns (tie-free: answered by the matcher) and of rounded columns (ties: flagged and
    re-enumerated batch by batch) in one call."""
    rng = np.random.default_rng(11)
    T, n, B, m0 = 40, 300, 40, 100
    X = walks(110, T, n)
    X[:, 150:] = np.round(X[:, 150:])
    mem = np.zeros((B, n), dtype=np.uint8)
    members = np.stack([np.sort(rng.choice(150, m0, replace=False) + (150 if b % 3 == 1 else 0)) for b in range(B)])
    mem[np.arange(B)[:, None], members] = 1
    qs = np.stack([rng.permutation(members[b])[:6] for b in range(B)])
    got = engine.band_depth_counts_batched(X, mem, qs, 2, False)
    assert engine.timings()["launches"] < 4 * B
    assert (got == oracle_strict(oracle, X, mem, qs, range(B))).all()


@gpu
def test_strict_chunked_launches(engine, oracle):
    """2000 queries of 2000 curves over 512 points: ~580 MB of sign words per batch, so the signature and match
    kernels take 2 batches per launch: B = 5 runs as 3 launch pairs."""
    rng = np.random.default_rng(12)
    T, n, B = 512, 2200, 5
    X = walks(120, T, n)
    mem, members, qs = uniform_batches(rng, n, B, 2000, 2000)
    got = engine.band_depth_counts_batched(X, mem, qs, 2, False)
    assert engine.timings()["bd_impl_used"] == E.BD_MATCH
    try:
        engine.set_option(E.OPT_BD_IMPL, E.BD_BITS)
        assert (got == engine_per_batch(engine, X, mem, qs, 2, False)).all()
    finally:
        engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)
    sq = qs[:, [0, 1999]]
    assert (got[:, [0, 1999]] == oracle_strict(oracle, X, mem, sq, range(B))).all()


@gpu
def test_strict_more_than_65535_batches(engine):
    """B = 70 000 batches of 12 curves over 4 points: the rank-packing launch takes at most 65 535 batches at a
    time (its batch index is gridDim.y).  Every count against brute force."""
    rng = np.random.default_rng(13)
    T, n, B = 4, 24, 70_000
    X = rng.standard_normal((T, n))
    mem, _, qs = uniform_batches(rng, n, B, 12, 2)
    got = engine.band_depth_counts_batched(X, mem, qs, 2, False)
    assert engine.timings()["bd_impl_used"] == E.BD_MATCH
    assert (got == np_strict_counts_small(X, mem, qs)).all()


@gpu
def test_strict_several_passes(engine, oracle):
    """T = 1024, m0 = 8000: 16 batches fill the 1 GB gather, so B = 20 runs in passes of 16 and 4 whose queries and
    outputs start at b0 * nqb."""
    rng = np.random.default_rng(14)
    T, n, B = 1024, 8200, 20
    X = walks(140, T, n)
    mem, _, qs = uniform_batches(rng, n, B, 8000, 2)
    got = engine.band_depth_counts_batched(X, mem, qs, 2, False)
    assert engine.timings()["bd_impl_used"] == E.BD_MATCH
    assert (got == engine_per_batch(engine, X, mem, qs, 2, False)).all()
    sample = [0, 15, 16, 19]
    assert (got[sample, :1] == oracle_strict(oracle, X, mem, qs[:, :1], sample)).all()


@gpu
def test_strict_matcher_size_limit(engine, oracle):
    """8193 members is the largest batch the matcher takes (8192 other curves); 8194 goes batch by batch to the
    enumerating kernels.  Both give the oracle's counts."""
    rng = np.random.default_rng(15)
    T, n, B = 6, 8400, 2
    X = walks(150, T, n)
    for m0 in (8193, 8194):
        mem, _, qs = uniform_batches(rng, n, B, m0, 3)
        got = engine.band_depth_counts_batched(X, mem, qs, 2, False)
        assert (got == oracle_strict(oracle, X, mem, qs, range(B))).all(), m0


# ------------------------------------------------------------------------------------------------
# GPU: grouped and per-batch paths, small and odd inputs, errors
# ------------------------------------------------------------------------------------------------
@gpu
def test_grouped_and_per_batch_paths_agree(engine, oracle):
    """One batch of another size sends the same batches batch by batch: their counts are bit-identical to the
    grouped call's, for relaxed j = 2, 3, strict j = 2 (also with the bit kernel and the tcgen05 Gram forced) and
    strict j = 3 against the oracle."""
    rng = np.random.default_rng(16)
    T, n, B = 30, 200, 12
    X = walks(160, T, n)
    X[:, 100:] = np.round(X[:, 100:], 1)
    mem, members, qs = uniform_batches(rng, n, B, 80, 5)
    extra = np.zeros((1, n), dtype=np.uint8)
    extra[0, :81] = 1
    mem2 = np.vstack([mem, extra])
    qs2 = np.vstack([qs, np.arange(5)[None, :]])
    for j in (2, 3):
        uni = engine.band_depth_counts_batched(X, mem, qs, j, True)
        assert engine.timings()["launches"] < B
        rag = engine.band_depth_counts_batched(X, mem2, qs2, j, True)
        assert engine.timings()["launches"] > B
        assert (rag[:B] == uni).all() and (uni == np_batched_counts(X, mem, qs, j)).all()
        assert (rag[B:] == np_batched_counts(X, mem2[B:], qs2[B:], j)).all()
    uni = engine.band_depth_counts_batched(X, mem, qs, 2, False)
    assert (uni == oracle_strict(oracle, X, mem, qs, range(B))).all()
    assert (engine.band_depth_counts_batched(X, mem2, qs2, 2, False)[:B] == uni).all()
    for impl in (E.BD_BITS, E.BD_GEMM):
        try:
            engine.set_option(E.OPT_BD_IMPL, impl)
            assert (engine.band_depth_counts_batched(X, mem, qs, 2, False) == uni).all(), impl
            assert (engine.band_depth_counts_batched(X, mem2, qs2, 2, False)[:B] == uni).all(), impl
        finally:
            engine.set_option(E.OPT_BD_IMPL, E.BD_AUTO)
    s3 = engine.band_depth_counts_batched(X, mem, qs, 3, False)
    assert (s3 == oracle_strict(oracle, X, mem, qs, range(B), j=3)).all()
    assert (engine.band_depth_counts_batched(X, mem2, qs2, 3, False)[:B] == s3).all()


@gpu
def test_small_and_odd_batches(engine, oracle):
    rng = np.random.default_rng(17)
    T, n = 9, 60
    X = walks(170, T, n)
    X[:, :20] = np.round(X[:, :20])
    # B = 1 (never grouped), and a batch holding every column: band_depth_counts(X)
    full = np.ones((1, n), dtype=np.uint8)
    q = rng.permutation(n)[None, :]
    for j in (2, 3):
        single = engine.band_depth_counts(X, q[0], j, True)
        assert (engine.band_depth_counts_batched(X, full, q, j, True)[0] == single).all()
    assert (engine.band_depth_counts_batched(X, full, q, 2, False)[0] == oracle.bd_counts(X, q[0])).all()
    both = np.vstack([full, full])
    for j in (2, 3):
        assert (engine.band_depth_counts_batched(X, both, np.vstack([q, q]), j, True) ==
                engine.band_depth_counts(X, None, j, True)[q[0]]).all()
    # m0 = 1, 2, 3: C(m-1, j) is 0 or 1; grouped (B > 1) and single
    for m0 in (1, 2, 3):
        for B in (1, 5):
            mem, _, qs = uniform_batches(rng, n, B, m0)
            for j in (2, 3):
                assert (engine.band_depth_counts_batched(X, mem, qs, j, True) == np_batched_counts(X, mem, qs, j)).all()
            strict = engine.band_depth_counts_batched(X, mem, qs, 2, False)
            assert (strict == np_strict_counts_small(X, mem, qs)).all(), (m0, B)
    # repeated and unordered queries, batches sharing columns, membership bytes other than 1
    B, m0 = 6, 25
    members = np.sort(np.stack([rng.choice(30, m0, replace=False) for _ in range(B)]), axis=1)  # heavily shared
    mem = np.zeros((B, n), dtype=np.uint8)
    mem[np.arange(B)[:, None], members] = rng.integers(1, 256, size=(B, m0)).astype(np.uint8)
    qs = np.stack([members[b][[7, 0, 7, 24, 3, 3]] for b in range(B)])
    for j in (2, 3):
        assert (engine.band_depth_counts_batched(X, mem, qs, j, True) == np_batched_counts(X, mem, qs, j)).all()
    assert (engine.band_depth_counts_batched(X, mem, qs, 2, False) == np_strict_counts_small(X, mem, qs)).all()


def _assert_status(status, fn, *args):
    with pytest.raises(E.EngineError) as ei:
        fn(*args)
    assert ei.value.status == status, str(ei.value)


@gpu
def test_batched_errors_leave_the_context_usable(engine):
    rng = np.random.default_rng(18)
    T, n, B = 10, 80, 6
    X = walks(180, T, n)
    mem, members, qs = uniform_batches(rng, n - 1, B, 30, 4)  # the last column is in no batch
    mem = np.hstack([mem, np.zeros((B, 1), dtype=np.uint8)])
    ragged = mem.copy()
    ragged[0, np.flatnonzero(mem[0] == 0)[0]] = 1
    ref = {j: np_batched_counts(X, mem, qs, j) for j in (2, 3)}

    def still_correct():
        for j in (2, 3):
            assert (engine.band_depth_counts_batched(X, mem, qs, j, True) == ref[j]).all()
        assert (engine.band_depth_counts_batched(X, mem, qs, 2, False) == np_strict_counts_small(X, mem, qs)).all()

    # a query that is not a member
    bad = qs.copy()
    bad[2, 1] = np.flatnonzero(mem[2] == 0)[0]
    for relax in (True, False):
        _assert_status(1, engine.band_depth_counts_batched, X, mem, bad, 2, relax)
        still_correct()
    # NaN in a member column: uniform relaxed, uniform strict, per-batch
    Xn = X.copy()
    Xn[4, members[3, 5]] = np.nan
    for m, relax in ((mem, True), (mem, False), (ragged, True), (ragged, False)):
        _assert_status(4, engine.band_depth_counts_batched, Xn, m, qs, 2, relax)
        still_correct()
    # NaN in a column outside every batch: not read, so the counts are those of the finite matrix
    Xo = X.copy()
    Xo[:, n - 1] = np.nan
    for j in (2, 3):
        assert (engine.band_depth_counts_batched(Xo, mem, qs, j, True) == ref[j]).all()
    # relaxed j = 3 numerators of 2 700 000 curves do not fit int64
    big = 2_700_000
    Xb = rng.standard_normal((1, big + 10))
    memb = np.zeros((2, big + 10), dtype=np.uint8)
    memb[0, :big] = 1
    memb[1, 10:] = 1
    _assert_status(5, engine.band_depth_counts_batched, Xb, memb, np.array([[0], [10]]), 3, True)
    still_correct()


# ------------------------------------------------------------------------------------------------
# GPU: public API
# ------------------------------------------------------------------------------------------------
@gpu
def test_permutation_test_cfg5_prefix():
    """The B = 1000 batched null at bench's perm shape (2 x 256 curves of 256 points) starts with the looped null
    of B = 10 (the same permutations, see test_permutation_prefix_property), exactly."""
    from statdepth_b200.homogeneity import permutation_test
    rng = np.random.default_rng(5)
    F = pd.DataFrame(rng.standard_normal((256, 256)).cumsum(0))
    G = pd.DataFrame(rng.standard_normal((256, 256)).cumsum(0) + 0.5)
    k = 10
    for method, relax in (("p1", True), ("p2", True), ("p3", True), ("p1", False), ("p2", False)):
        full = permutation_test(F, G, method=method, B=1000, seed=5, relax=relax)
        loop = permutation_test(F, G, method=method, B=k, seed=5, relax=relax, batched=False)
        assert full["null"].shape == (1000,)
        assert full["null"][:k].tolist() == loop["null"].tolist(), (method, relax)
        assert full["observed"] == loop["observed"]


@gpu
def test_permutation_test_strict_p3_many_batches():
    """Strict p3 with 300 + 300 curves of 4 points: B = 300 permutations ask for 90 000 sub-populations of 301 curves
    in one batched call (more than 65 535)."""
    from statdepth_b200.homogeneity import permutation_test
    rng = np.random.default_rng(19)
    F = pd.DataFrame(rng.standard_normal((4, 300)))
    G = pd.DataFrame(rng.standard_normal((4, 300)) + 0.3)
    full = permutation_test(F, G, method="p3", B=300, seed=3, relax=False)
    loop = permutation_test(F, G, method="p3", B=3, seed=3, relax=False, batched=False)
    np.testing.assert_allclose(full["null"][:3], loop["null"], rtol=1e-12)
    assert full["observed"] == loop["observed"]


@gpu
@pytest.mark.parametrize("relax,J", [(True, 2), (False, 2), (True, 3)])
def test_k_sampled_depth_blocks(engine, relax, J):
    """K-sampled FunctionalDepth: every block's depth is the single-matrix depth of that block's curves."""
    from scipy.special import binom

    from statdepth_b200 import FunctionalDepth
    from statdepth_b200._functional import _sample_blocks
    T, n, K = 20, 300, 3
    df = pd.DataFrame(walks(190, T, n))
    np.random.seed(7)
    got = FunctionalDepth([df], K=K, J=J, relax=relax)
    np.random.seed(7)
    cols, blocks = _sample_blocks(df, df.columns, K)
    depth = np.zeros(len(blocks))
    for i, (col, members) in enumerate(blocks):
        pos = np.sort(np.asarray(members, dtype=np.int64))
        sub = np.ascontiguousarray(df.to_numpy()[:, pos])
        for j in range(2, J + 1):
            s = float(engine.band_depth_counts(sub, [int(np.searchsorted(pos, col))], j, relax)[0])
            depth[i] += (s / T if relax else s) / binom(len(pos), j)
    exp = depth.reshape(n, K).mean(axis=1)
    np.testing.assert_allclose(got.loc[cols].to_numpy(), exp, rtol=1e-12)
