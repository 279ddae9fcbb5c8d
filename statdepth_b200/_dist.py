"""Multi-GPU sharding of one depth call: one process per GPU, torch.distributed for the plumbing.

* relaxed band depth is additive over time rows  -> every rank ranks a contiguous block of rows
  and the int64 numerators are summed with ONE all-reduce (800 KB at n = 100k);
* strict band depth / simplex / point-cloud depths have independent queries -> every rank takes a
  contiguous block of queries and the results are joined with ONE all-gather;
* homogeneity permutations are independent -> split by permutation, all-gathered.
* random projection depths of point clouds -> split by direction, MIN / MAX all-reduced (exact, order-free).

Sharding is OPT-IN: `statdepth_b200.enable_distributed()` (or STATDEPTH_DISTRIBUTED=1 in the environment) makes
every depth call of this process a COLLECTIVE over the default process group.  Every rank must then make the
same calls with identical data and arguments (a call made by some ranks only, or one that raises on one rank
only, deadlocks the group -- which is why an initialised process group alone does not switch it on); sampled
depths (K=...) draw from each rank's own global numpy RNG, so seed all ranks alike.

With the NCCL backend the relaxed path stays on the device: the rank's rows are uploaded once, the kernels are
only ENQUEUED (SD_OPT_ASYNC_DEVICE), the all-reduce is queued behind them on the engine's stream and one
synchronisation ends the call -- no numpy <-> torch <-> host hops between the kernels and the collective.
The partition / collective / re-assembly logic itself never touches the GPU: the compute callable is injected,
so it is exercised on CPU with the gloo backend (tests/test_distributed.py).
"""
import os

import numpy as np

_ENABLED = None  # None: follow the environment


def enable_distributed(on: bool = True) -> None:
    """Shard every depth call of this process over the default torch.distributed group (see module docstring)."""
    global _ENABLED
    _ENABLED = bool(on)


def enabled() -> bool:
    if _ENABLED is not None:
        return _ENABLED
    return os.environ.get("STATDEPTH_DISTRIBUTED", "0") == "1"


def world():
    """(rank, world_size) of the default process group when sharding is enabled, else (0, 1)."""
    if not enabled():
        return 0, 1
    try:
        import torch.distributed as dist
    except Exception:  # torch missing: single process
        return 0, 1
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


class local_only:
    """Context manager: depth calls inside do not shard (used while an outer loop is itself sharded)."""

    def __enter__(self):
        global _ENABLED
        self.prev = _ENABLED
        _ENABLED = False

    def __exit__(self, *exc):
        global _ENABLED
        _ENABLED = self.prev
        return False


def block(total: int, rank: int, size: int):
    """Balanced contiguous block [lo, hi) of `total` items for `rank` of `size`."""
    base, rem = divmod(int(total), int(size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _nccl() -> bool:
    import torch.distributed as dist
    return dist.get_backend() == "nccl"


def _device_for_collectives():
    import torch
    if _nccl():
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def allreduce(arr: np.ndarray, op: str = "sum") -> np.ndarray:
    """Element-wise reduction of arr over all ranks; op is "sum", "min" or "max"."""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(arr)).to(_device_for_collectives())
    dist.all_reduce(t, op={"sum": dist.ReduceOp.SUM, "min": dist.ReduceOp.MIN, "max": dist.ReduceOp.MAX}[op])
    return t.cpu().numpy()


def allgather_blocks(local: np.ndarray, total: int) -> np.ndarray:
    """Concatenate per-rank blocks (sizes given by block()) along axis 0."""
    import torch
    import torch.distributed as dist
    rank, size = dist.get_rank(), dist.get_world_size()
    dev = _device_for_collectives()
    sizes = [block(total, r, size) for r in range(size)]
    width = max(hi - lo for lo, hi in sizes)
    pad = np.zeros((width,) + local.shape[1:], dtype=local.dtype)
    pad[: local.shape[0]] = local
    mine = torch.from_numpy(pad).to(dev)
    joined = torch.empty((size * width,) + tuple(mine.shape[1:]), dtype=mine.dtype, device=dev)
    dist.all_gather_into_tensor(joined, mine)  # one collective, one D2H
    joined = joined.cpu().numpy().reshape((size, width) + tuple(mine.shape[1:]))
    return np.concatenate([joined[r][: hi - lo] for r, (lo, hi) in enumerate(sizes)], axis=0)


def relaxed_counts_device(eng, X, queries, j):
    """NCCL path of relaxed_counts: rows -> device once, kernels enqueued, all-reduce queued on the engine's
    stream behind them, one synchronisation, one D2H of the summed numerators."""
    import torch
    import torch.distributed as dist

    from ._engine import OPT_ASYNC_DEVICE
    rank, size = world()
    T, n = X.shape
    lo, hi = block(T, rank, size)
    dev = torch.device("cuda", eng.device)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    with torch.cuda.stream(stream):
        out = torch.zeros(n, dtype=torch.int64, device=dev)
        Xl = None
        if hi > lo:
            Xl = torch.from_numpy(np.ascontiguousarray(X[lo:hi], dtype=np.float64)).to(dev)
            eng.set_option(OPT_ASYNC_DEVICE, 1)
            try:
                eng.band_depth_counts_dev(Xl.data_ptr(), hi - lo, n, n, out.data_ptr(), None, n, j, True)
            finally:
                eng.set_option(OPT_ASYNC_DEVICE, 0)
        dist.all_reduce(out)
        eng.sync()  # completes the queued call (raises its error) and the collective behind it
        res = out.cpu().numpy()
    del Xl
    return res if queries is None else res[np.asarray(queries, dtype=np.int64)]


def relaxed_counts(compute, X, queries, j, eng=None):
    """compute(X_rows, queries, j) -> int64[nq]; rows sharded, counts all-reduced."""
    rank, size = world()
    if size == 1:
        return compute(X, queries, j)
    if eng is not None and _nccl() and hasattr(eng, "band_depth_counts_dev") and j in (2, 3) and X.flags.c_contiguous:
        return relaxed_counts_device(eng, X, queries, j)
    T = X.shape[0]
    lo, hi = block(T, rank, size)
    nq = X.shape[1] if queries is None else len(queries)
    local = compute(X[lo:hi], queries, j) if hi > lo else np.zeros(nq, dtype=np.int64)
    return allreduce(np.asarray(local, dtype=np.int64))


def query_sharded(compute, queries, dtype):
    """compute(query_block) -> array[len(block)]; queries sharded, results all-gathered."""
    rank, size = world()
    queries = np.asarray(queries, dtype=np.int64)
    if size == 1:
        return compute(queries)
    lo, hi = block(len(queries), rank, size)
    local = compute(queries[lo:hi]) if hi > lo else np.zeros(0, dtype=dtype)
    return allgather_blocks(np.asarray(local, dtype=dtype), len(queries))
