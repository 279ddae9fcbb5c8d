#!/usr/bin/env python
"""bench.py -- depth-evals/s of the statdepth hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload mbd|bd|perm]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload at every N (strong scaling: the total work is BASELINE's configuration, fixed):
  mbd (default) = BASELINE config 2: modified band depth (relax=True, J=2) of 100 000 curves x 1024
                  time points, float64 random walks.  One step = one depth evaluation of ALL curves.
                  With N ranks every rank ranks a contiguous block of T/N time rows (MBD is additive
                  over rows) and the int64 numerators are all-reduced (NCCL).
  bd            = BASELINE config 3: strict band depth of 8192 curves x 512 points, queries sharded + all-gather.
  perm          = BASELINE config 5: homogeneity permutation test, 2 x 256 curves x 256 points, 1000 permutations
                  sharded over the ranks + all-gather (value = permutations/s through the public API).

One JSON line on rank 0.  `value` = depth-evals/s with the input resident in HBM (device-pointer C ABI);
`e2e` = the same through the host-buffer C ABI call (pinned host input, H2D + kernels + D2H + float depth);
`e2e_api` = the same through the PUBLIC API, FunctionalDepth([DataFrame]) from pageable memory.
The default run also times the other BASELINE configurations briefly and reports them under `secondary`
(cfg3 strict band depth by sign-vector matching and by the tcgen05 Gram, cfg5 permutation test / L1 / simplicial
depth, cfg4 relaxed simplex depth, cfg1 call latency), each sharded over the N ranks like the headline.
`cpu_baseline` (rank 0, N = 1) = the C oracle port of the closed form on all host threads, plus
`reference_python`: the UNMODIFIED reference (oracle/_ref, staged by oracle/make_ref.sh) timed on the same cores
on the configuration it can run (cfg1).  `--impl reference` times the CPU oracle port on the arm's configuration
(the Python reference needs ~25 s per depth-eval at 200 x 100 and ~1e12 s for config 2).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from math import comb

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L2_BYTES = 126 << 20
METRIC = "BD/MBD depth-evals/sec"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mbd", choices=["mbd", "bd", "perm"])
    ap.add_argument("--n", type=int, default=None)
    ap.add_argument("--T", type=int, default=None)
    ap.add_argument("--cpu-sample-rows", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the brief timings of the other BASELINE configs")
    ap.add_argument("--no-reference-python", action="store_true", help="skip timing the staged Python reference (~30 s)")
    ap.add_argument("--bd-impl", default="auto", choices=["auto", "bits", "gemm", "match"])
    ap.add_argument("--nq", type=int, default=None, help="bd workload: number of query curves (default all)")
    ap.add_argument("--ties", action="store_true", help="tie-stress variant: round the random walks to integers")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(float64; inputs are seeded, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU arm's outputs; the reference arm times the CPU oracle on a sample")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Write each array as DIR/<name>.npy in float64 (integer counts below 2**53 are exact).  An array larger than its
    share of DUMP_BYTES is replaced by a fixed, seeded sample of its elements; the sampled positions go to
    DIR/<name>_index.npy, so that two dumps compare element for element."""
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // (2 * len(arrays))  # room for a sample and its index
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // 8, replace=False))
            np.save(os.path.join(dirname, name + "_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(dirname, name + ".npy"), a)


def workload_shape(args):
    if args.workload == "mbd":
        n, T, name = 100_000, 1024, "cfg2: modified band depth (relax=True, J=2), 100k curves x 1024 points"
    elif args.workload == "bd":
        n, T, name = 8192, 512, "cfg3: strict band depth (relax=False, J=2), 8192 curves x 512 points"
    else:
        n, T, name = 512, 256, "cfg5: homogeneity permutation test (p2, relax=True), 2 x 256 curves x 256 points, 1000 permutations"
    if args.n or args.T:
        n, T = args.n or n, args.T or T
        name += " [overridden to n=%d T=%d]" % (n, T)
    if args.ties:
        name += " [tie stress: rounded to integers]"
    return n, T, name


def make_config(args, n, T, name, world):
    """The SAME dictionary in both arms (the driver compares them key by key)."""
    relax = args.workload != "bd"
    if args.workload == "perm":
        shard = "permutations over ranks + all-gather"
    elif relax:
        shard = "time rows over ranks + int64 all-reduce"
    else:
        shard = "query curves over ranks + all-gather"
    return {"workload": name, "curves": n, "time_points": T, "J": 2, "relax": relax,
            "queries": (args.nq or n) if args.workload == "bd" else n, "bd_impl": args.bd_impl,
            "sharding": shard if world > 1 else "single GPU"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes per cfg2 step from the tracked ncu capture of the CURRENT kernels (profiles/traffic_r02.json:
    dram__bytes_read.sum + dram__bytes_write.sum per kernel, with the commit it was taken at)."""
    p = os.path.join(ROOT, "profiles", "traffic_r02.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh)
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm))


# ------------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/)
# ------------------------------------------------------------------------------------------------------
def cpu_baseline(args, n, T, rows=None):
    """Oracle port on all host threads over a bounded sample (a block of time rows / queries / permutations)."""
    from oracle import cpu_oracle
    cpu_oracle.build()
    cores = cpu_oracle.num_threads()
    rng = np.random.default_rng(1)
    if args.workload == "mbd":
        rows = min(T, rows or T)  # default: the whole workload (~1 s wall on 16+ cores)
        X = rng.standard_normal((rows, n)).cumsum(0)
        t0 = time.perf_counter()
        cpu_oracle.mbd_counts_all(X)
        dt = time.perf_counter() - t0
        full = dt * T / rows  # MBD cost is linear in the number of rows
        return dict(value=n / full, unit="depth-evals/s", cores=cores, kind="port",
                    sample="oracle/sd_oracle.c sdo_mbd_counts_all (qsort ranks per row, %d pthreads) on %d of %d time "
                           "rows x %d curves in %.2f s%s" % (cores, rows, T, n, dt,
                                                             "" if rows == T else ", scaled linearly to %d rows" % T),
                    seconds_sample=dt)
    if args.workload == "bd":
        X = rng.standard_normal((T, n)).cumsum(0)
        nq = max(cores, 16)
        q = rng.choice(n, nq, replace=False)
        t0 = time.perf_counter()
        cpu_oracle.bd_counts(X, q)
        dt = time.perf_counter() - t0
        return dict(value=nq / dt, unit="depth-evals/s", cores=cores, kind="port",
                    sample="oracle/sd_oracle.c sdo_bd_counts (bit masks, early exit) on %d of %d query curves in %.2f s"
                           % (nq, n, dt), seconds_sample=dt)
    # perm: p2 statistic of B permutations = three relaxed depth runs per permutation on the oracle
    F, G = perm_inputs()
    X = np.ascontiguousarray(np.concatenate([F.values, G.values], axis=1))
    nF, B = F.shape[1], 16
    t0 = time.perf_counter()
    for b in range(B):
        p = rng.permutation(X.shape[1])
        Fi, Gi = p[:nF], p[nF:]
        dG = cpu_oracle.mbd_counts_all(np.ascontiguousarray(X[:, Gi]))
        g = Gi[int(np.argmax(dG))]
        cpu_oracle.mbd_counts_all(np.ascontiguousarray(X[:, np.append(Fi, g)]))
        cpu_oracle.mbd_counts_all(np.ascontiguousarray(X[:, Fi]))
    dt = time.perf_counter() - t0
    return dict(value=B / dt, unit="permutations/s", cores=cores, kind="port",
                sample="oracle/sd_oracle.c: p2 statistic (three relaxed depth runs) of %d of 1000 permutations in %.2f s"
                       % (B, dt), seconds_sample=dt)


def reference_python(timeout_s=240):
    """The UNMODIFIED reference on this box's host cores (oracle/time_reference.py -> oracle/_ref/statdepth)."""
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "time_reference.py")], capture_output=True,
                             text=True, timeout=timeout_s, cwd=ROOT)
        for line in out.stdout.splitlines()[::-1]:
            if line.startswith("{"):
                return json.loads(line)
        return {"unavailable": "oracle/time_reference.py printed no result: " + out.stderr[-200:]}
    except Exception as e:  # timeout, missing interpreter ...
        return {"unavailable": repr(e)[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, T, name = workload_shape(args)
    world = max(1, args.gpus)
    vals, secs, cb = [], [], None
    for i in range(args.warmup + args.steps):
        cb = cpu_baseline(args, n, T, rows=args.cpu_sample_rows)
        if i >= args.warmup:
            vals.append(cb["value"])
            secs.append(cb["seconds_sample"])
    v = float(np.mean(vals))
    cb.update(value=v)
    cb.pop("seconds_sample", None)
    unit = cb["unit"]
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(args, n, T, name, world),
        "notes": "CPU oracle port of the reference path on all host threads (the reference is pure Python, ~0.04 "
                 "depth-evals/s/core at 200x100, and cannot run at this size); each step is a bounded sample",
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def emit(line: dict):
    """Print THE one JSON line on the real stdout (see _quiet_stdout)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def _quiet_stdout():
    """Libraries (NCCL prints 'NCCL version ...' at init) may write to fd 1: keep fd 1 for the JSON line
    only by pointing it at stderr for the rest of the run."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def perm_inputs():
    import pandas as pd
    rng = np.random.default_rng(5)
    F = pd.DataFrame(rng.standard_normal((256, 256)).cumsum(0))
    G = pd.DataFrame(rng.standard_normal((256, 256)).cumsum(0) + 0.5)
    return F, G


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
class Ctx:
    """What every timed piece needs: the engine, torch plumbing and the rank layout."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from statdepth_b200 import _dist as sdist
        from statdepth_b200 import _engine as E
        self.torch, self.dist, self.sdist, self.E, self.args = torch, dist, sdist, E, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            sdist.enable_distributed(True)  # public-API calls below shard like the headline
        os.environ["STATDEPTH_DEVICE"] = str(self.local)
        self.eng = E.get_engine(self.local)
        self.eng.set_option(E.OPT_PROFILE, 1)
        self.dev = torch.device("cuda", self.local)
        self.stream = torch.cuda.ExternalStream(self.eng.stream(), device=self.dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)

    def walks(self, T, n, seed, ties=False):
        torch = self.torch
        g = torch.Generator(device=self.dev)
        g.manual_seed(seed)
        X = torch.empty((T, n), dtype=torch.float64, device=self.dev)
        for r0 in range(0, T, 128):  # generate in row blocks to bound scratch memory
            X[r0:r0 + 128] = torch.randn((min(128, T - r0), n), dtype=torch.float64, device=self.dev, generator=g)
        X = X.cumsum(0)
        return X.round() if ties else X

    def timed(self, fn, steps, warmup, flush=True):
        """W warm-up steps, then K steps timed with CUDA events on the engine's stream (max over ranks).
        fn() -> (result, timings dict or None)."""
        torch, dist = self.torch, self.dist
        for _ in range(warmup):
            fn()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms, launches, kern_ns, phases, last = 0.0, 0, 0, {}, None
        for _ in range(steps):
            if flush:
                self.flush.fill_(1)
                torch.cuda.synchronize()
                if self.world > 1:
                    dist.barrier()  # ranks leave the (untimed) L2 flush together
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            last, tm = fn()
            torch.cuda.synchronize()  # collectives may run on torch's stream: drain it before the end event
            e1.record(self.stream)
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
            if tm:
                launches += tm["launches"] + (1 if self.world > 1 else 0)
                kern_ns += tm["kernel_ns"]
                for k, v in self.eng.phase_ns().items():
                    phases[k] = phases.get(k, 0) + v
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([total_ms], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, kern_ns, phases, last

    def gather_blocks(self, t, total):
        """all-gather of per-rank query blocks of unequal size (device tensors)."""
        if self.world == 1:
            return t
        torch, dist = self.torch, self.dist
        sizes = [self.sdist.block(total, r, self.world) for r in range(self.world)]
        width = max(hi - lo for lo, hi in sizes)
        mine = torch.zeros(width, dtype=t.dtype, device=self.dev)
        mine[: t.numel()] = t
        joined = torch.empty(width * self.world, dtype=t.dtype, device=self.dev)
        dist.all_gather_into_tensor(joined, mine)
        return torch.cat([joined[r * width: r * width + (hi - lo)] for r, (lo, hi) in enumerate(sizes)])


def bench_band(c: Ctx, n, T, relax, bd_impl, nq_total, steps, warmup, ties=False, seed=1, want_e2e=True):
    """Headline measurement (device-resident `value` + host-buffer `e2e`) of one band-depth configuration."""
    torch, dist, E, eng = c.torch, c.dist, c.E, c.eng
    eng.set_option(E.OPT_BD_IMPL, {"auto": E.BD_AUTO, "bits": E.BD_BITS, "gemm": E.BD_GEMM, "match": E.BD_MATCH}[bd_impl])
    X = c.walks(T, n, seed, ties)
    if relax:   # rows sharded, counts all-reduced
        lo, hi = c.sdist.block(T, c.rank, c.world)
        Xl = X[lo:hi].contiguous()
        nq_local, q_dev = n, None
    else:       # queries sharded, counts all-gathered
        lo, hi = c.sdist.block(nq_total, c.rank, c.world)
        Xl = X
        nq_local = hi - lo
        q_dev = torch.arange(lo, hi, dtype=torch.int64, device=c.dev)
    del X
    Tl = Xl.shape[0]
    out_dev = torch.zeros(max(nq_local, 1), dtype=torch.int64, device=c.dev)
    local_bytes = Xl.numel() * 8
    flush = local_bytes < 2 * L2_BYTES

    def collective(t):
        if c.world == 1:
            return t
        if relax:
            dist.all_reduce(t)
            return t
        return c.gather_blocks(t[:nq_local], nq_total)

    # multi-GPU relaxed depth: the device entry point only enqueues (SD_OPT_ASYNC_DEVICE) and the all-reduce is
    # queued behind the kernels on the engine's stream, so a step has one host synchronisation instead of three
    # (the same path statdepth_b200._dist.relaxed_counts_device gives FunctionalDepth users)
    queued = c.world > 1 and relax
    eng.set_option(E.OPT_ASYNC_DEVICE, 1 if queued else 0)

    def step_resident():
        if nq_local > 0 or relax:
            eng.band_depth_counts_dev(Xl.data_ptr(), Tl, n, n, out_dev.data_ptr(),
                                      None if q_dev is None else q_dev.data_ptr(), nq_local, 2, relax)
        with torch.cuda.stream(c.stream):
            res = collective(out_dev)
        if queued:
            eng.sync()
        return res, eng.timings()

    ms, launches, kern_ns, phases, last = c.timed(step_resident, steps, warmup, flush)
    eng.set_option(E.OPT_ASYNC_DEVICE, 0)
    res = dict(ms=ms, launches=launches, kern_ns=kern_ns, phases=phases, last=last, Tl=Tl, nq_local=nq_local,
               local_bytes=local_bytes, flush=flush)
    if want_e2e:
        host_in = torch.empty(Xl.shape, dtype=torch.float64).pin_memory()
        host_in.copy_(Xl)
        q_host = None if q_dev is None else q_dev.cpu().numpy()

        def step_e2e():
            cnt = eng.band_depth_counts_ptr(host_in.data_ptr(), Tl, n, n, q_host, 2, relax)
            tm = eng.timings()
            if c.world > 1:
                cnt = collective(torch.from_numpy(cnt).to(c.dev)).cpu().numpy()
            s = cnt.astype(np.float64)
            depth = (s / float(T) if relax else s) / float(comb(n, 2))  # the float64 depth the API returns
            return depth, tm

        ms_e2e, _, _, _, depth = c.timed(step_e2e, steps, max(1, warmup), flush)
        res.update(ms_e2e=ms_e2e, depth=depth, host_in=host_in)
    eng.set_option(E.OPT_BD_IMPL, E.BD_AUTO)
    return res


def secondary(c: Ctx):
    """Brief timings of the other BASELINE configurations, sharded over the ranks like the headline."""
    import pandas as pd
    torch, E, eng = c.torch, c.E, c.eng
    out = {}
    peak, _ = peaks()

    # ---- cfg3: strict band depth, 8192 x 512 -------------------------------------------------------
    n, T = 8192, 512
    r = bench_band(c, n, T, False, "auto", n, steps=3, warmup=1, seed=2, want_e2e=False)
    ms = r["ms"] / 3
    # what the matcher moves through HBM per query: sign words (uint2 per word per curve) + signatures, written by
    # the signature kernel and re-read by the match kernel (a LOWER bound: verification re-reads are not counted)
    W, m = T // 32, n - 1
    bytes_q = 2.0 * (W * m * 8 + m * 17)
    nql = r["nq_local"]
    kern_s = r["kern_ns"] / 1e9 / 3
    out["cfg3_strict_bd_match"] = {
        "metric": METRIC, "value": n / (ms / 1e3), "unit": "depth-evals/s", "ms_per_step": ms, "queries": n,
        "n_gpus": c.world, "bd_impl_used": eng.timings()["bd_impl_used"],
        "roofline": {"bound": "hbm", "achieved": bytes_q * nql / kern_s / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": bytes_q * nql / kern_s / 1e9 / peak, "traffic": None,
                     "bytes": "sign words + signatures written by the signature kernel and re-read by the match kernel "
                              "(lower bound of the traffic), per rank",
                     "kernel_ms_per_step": kern_s * 1e3,
                     "phase_ms_per_step": {k: v / 1e6 / 3 for k, v in r["phases"].items()}}}
    nq = 1024
    r = bench_band(c, n, T, False, "gemm", nq, steps=2, warmup=1, seed=2, want_e2e=False)
    ms = r["ms"] / 2
    kern_s = r["kern_ns"] / 1e9 / 2
    ops = 2.0 * (2 * T) * comb(n - 1, 2) * r["nq_local"]
    i8_peak = eng.probe_int8_peak() / 1e12
    out["cfg3_strict_bd_gram"] = {
        "metric": METRIC, "value": nq / (ms / 1e3), "unit": "depth-evals/s", "ms_per_step": ms, "queries": nq,
        "n_gpus": c.world,
        "roofline": {"bound": "tensor", "achieved": ops / kern_s / 1e12, "peak": i8_peak, "unit": "TOP/s (int8)",
                     "frac": ops / kern_s / 1e12 / i8_peak, "traffic": None,
                     "ops": "2*(2T)*C(n-1,2) int8 ops per query, upper triangle only; time INCLUDES operand generation",
                     "peak_source": "measured here: sd_probe_int8_peak (tcgen05.mma kind::i8 issue loop)",
                     "kernel_ms_per_step": kern_s * 1e3}}

    # ---- cfg5: permutation test through the public API, permutations sharded ---------------------------
    from statdepth_b200.homogeneity import permutation_test
    F, G = perm_inputs()
    permutation_test(F, G, method="p2", B=1000, seed=5, relax=True)  # same shape: workspaces grown, untimed
    if c.world > 1:
        c.dist.barrier()
    t0 = time.perf_counter()
    res = permutation_test(F, G, method="p2", B=1000, seed=5, relax=True)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    out["cfg5_permutation_test"] = {"metric": "homogeneity permutations/s (p2, relax=True, 2 x 256 curves x 256 points, "
                                              "B=1000; wall clock through permutation_test, host code included)",
                                    "value": 1000.0 / float(t.item()), "unit": "permutations/s",
                                    "ms_per_step": float(t.item()) * 1e3, "n_gpus": c.world,
                                    "p_value": res["p_value"]}

    # ---- cfg5: L1 and 2-D simplicial depth of 50 000 points, queries sharded ---------------------------------
    from statdepth_b200.testing import generate_noisy_pointcloud
    P = np.ascontiguousarray(generate_noisy_pointcloud(n=50_000, d=2, seed=4).values)
    lo, hi = c.sdist.block(50_000, c.rank, c.world)
    q = np.arange(lo, hi, dtype=np.int64)
    for name, fn in (("cfg5_l1_depth", lambda: eng.l1_depth(P, q)),
                     ("cfg5_simplicial_depth", lambda: eng.simplicial_counts(P, q, 1e-7))):
        fn()
        if c.world > 1:
            c.dist.barrier()
        t0 = time.perf_counter()
        fn()
        tm = eng.timings()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt, tm["kernel_ns"] / 1e9], dtype=torch.float64, device=c.dev)
        if c.world > 1:
            c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
        out[name] = {"metric": "point-cloud depth-evals/s (50 000 points, d = 2; host buffers, wall clock)",
                     "value": 50_000 / float(t[0].item()), "unit": "depth-evals/s", "ms_per_step": float(t[0].item()) * 1e3,
                     "kernel_ms_per_step": float(t[1].item()) * 1e3, "n_gpus": c.world}

    # ---- cfg4: relaxed multivariate simplex depth, 5000 curves x 256 points x 2 channels, 64-query sample ------
    Fm = np.random.default_rng(3).standard_normal((5000, 256, 2)).cumsum(1)
    nq4 = 64 * c.world
    lo, hi = c.sdist.block(nq4, c.rank, c.world)
    q4 = np.arange(lo, hi, dtype=np.int64) * (5000 // nq4)
    eng.simplex_depth_counts(Fm, q4, True, 1e-7)  # same shape: workspaces grown, untimed
    if c.world > 1:
        c.dist.barrier()
    t0 = time.perf_counter()
    eng.simplex_depth_counts(Fm, q4, True, 1e-7)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    out["cfg4_simplex_depth_relaxed_d2"] = {
        "metric": "multivariate simplex depth-evals/s (5000 curves x 256 points x 2 channels, relax=True, tolerance 1e-7; "
                  "%d-query sample, host buffers incl. the 20 MB upload)" % nq4,
        "value": nq4 / float(t.item()), "unit": "depth-evals/s", "ms_per_step": float(t.item()) * 1e3, "n_gpus": c.world}

    # ---- cfg4 strict (pruned enumeration, 2.08e10 triples per query) and Oja depth of the 50 000-point cloud ------------
    nqs = 2 * c.world
    lo, hi = c.sdist.block(nqs, c.rank, c.world)
    qs4 = (np.arange(lo, hi, dtype=np.int64) + 1) * (5000 // (nqs + 1))
    eng.simplex_depth_counts(Fm, qs4[:1], False, 1e-7)
    if c.world > 1:
        c.dist.barrier()
    t0 = time.perf_counter()
    eng.simplex_depth_counts(Fm, qs4, False, 1e-7)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    out["cfg4_simplex_depth_strict_d2"] = {
        "metric": "strict multivariate simplex depth-evals/s (5000 curves x 256 points x 2 channels, relax=False: C(4999,3) = "
                  "2.08e10 triples per query, rows staged in shared memory; %d-query sample)" % nqs,
        "value": nqs / float(t.item()), "unit": "depth-evals/s", "ms_per_step": float(t.item()) * 1e3, "n_gpus": c.world}
    nqo = 2048 * c.world
    lo, hi = c.sdist.block(nqo, c.rank, c.world)
    qo = np.arange(lo, hi, dtype=np.int64) * (50_000 // nqo)
    eng.oja(P, 1.0, qo)
    if c.world > 1:
        c.dist.barrier()
    t0 = time.perf_counter()
    eng.oja(P, 1.0, qo)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    out["cfg5_oja_depth"] = {
        "metric": "Oja depth-evals/s (50 000 points, d = 2: 1.25e9 triangles per query summed by angular prefix sums; "
                  "%d-query sample, host buffers)" % nqo,
        "value": nqo / float(t.item()), "unit": "depth-evals/s", "ms_per_step": float(t.item()) * 1e3, "n_gpus": c.world}

    # ---- cfg1: call latency of the public API at the reference's own size (rank 0 only, unsharded) -------------
    if c.rank == 0:
        from statdepth_b200 import FunctionalDepth
        with c.sdist.local_only():
            df = pd.DataFrame(np.random.default_rng(0).standard_normal((100, 200)).cumsum(0))
            lat = {}
            for relax in (False, True):
                FunctionalDepth([df], relax=relax)
                t0 = time.perf_counter()
                for _ in range(20):
                    FunctionalDepth([df], relax=relax)
                lat["relax" if relax else "strict"] = (time.perf_counter() - t0) / 20 * 1e3
        out["cfg1_public_api_latency"] = {"metric": "ms per FunctionalDepth([df]) call, 200 curves x 100 points (all 200 depths)",
                                          "value": lat["strict"], "unit": "ms", "relaxed_ms": lat["relax"],
                                          "higher_is_better": False, "n_gpus": 1}
    if c.world > 1:
        c.dist.barrier()

    # ---- cfg2 once more through the part pipeline (SD_MBD_PATH=parts): the A/B of the headline's slab path, same box,
    #      same process, same sharding.  Every rank runs it (the step holds a collective); a failure only drops the entry.
    try:
        os.environ["SD_MBD_PATH"] = "parts"
        r = bench_band(c, 100_000, 1024, True, "auto", 100_000, steps=10, warmup=3, seed=1, want_e2e=False)
        ms = r["ms"] / 10
        out["cfg2_part_pipeline"] = {
            "metric": METRIC + " (cfg2 ranked by the part pipeline, SD_MBD_PATH=parts: what the headline's slab path replaces)",
            "value": 100_000 / (ms / 1e3), "unit": "depth-evals/s", "ms_per_step": ms, "n_gpus": c.world,
            "kernel_ms_per_step": r["kern_ns"] / 1e6 / 10,
            "phase_ms_per_step": {k: v / 1e6 / 10 for k, v in r["phases"].items()}}
    except Exception as exc:  # noqa: BLE001
        out["cfg2_part_pipeline"] = {"error": repr(exc)}
    finally:
        os.environ.pop("SD_MBD_PATH", None)
    return out


def main():
    args = parse()
    _quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    c = Ctx(args)
    torch, dist, eng = c.torch, c.dist, c.eng
    world, rank = c.world, c.rank
    n, T, name = workload_shape(args)
    config = make_config(args, n, T, name, world)
    sampler = ClockSampler(c.local)
    if rank == 0:
        sampler.start()

    if args.workload == "perm":
        return main_perm(c, args, n, T, name, config, sampler)

    relax = args.workload == "mbd"
    evals = n if relax else (args.nq or n)
    r = bench_band(c, n, T, relax, args.bd_impl, evals, args.steps, args.warmup, ties=args.ties,
                   seed=1 if relax else 2)
    clocks = sampler.stop() if rank == 0 else None
    ms, ms_e2e, Tl, nq_local = r["ms"], r["ms_e2e"], r["Tl"], r["nq_local"]
    # the counts of the device-resident call and the depths of the host-buffer call, all queries on every rank
    outputs = {"counts": r["last"].cpu().numpy(), "depth": r["depth"]}
    impl_used = {k: v for k, v in eng.timings().items() if k in ("fallback_rows", "bd_impl_used")}

    # ---- sanity inside the bench: tie-free checksum of the relaxed numerators ----------------------
    if relax:
        total = int(r["last"].sum().item())
        expect = T * (n * comb(n - 1, 2) - 2 * comb(n, 3))
        if total != expect and not args.ties:
            raise SystemExit("bench: MBD checksum mismatch %d != %d" % (total, expect))

    # ---- e2e through the PUBLIC API from pageable memory (what a FunctionalDepth user gets) -----------
    e2e_api = None
    if relax and not args.ties:
        import pandas as pd
        from statdepth_b200 import FunctionalDepth
        lo, _ = c.sdist.block(T, rank, world)
        full = np.empty((T, n), dtype=np.float64)  # pageable; every rank holds the whole frame, as a user would
        src = c.walks(T, n, 1)
        full[:] = src.cpu().numpy()
        del src
        df = pd.DataFrame(full, copy=False)
        FunctionalDepth([df], relax=True)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        k_api = args.steps
        for _ in range(k_api):
            d_api = FunctionalDepth([df], relax=True)
        dt = (time.perf_counter() - t0) / k_api
        outputs["depth_api"] = d_api.values
        t = torch.tensor([dt], dtype=torch.float64, device=c.dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_api = {"value": n / float(t.item()), "unit": "depth-evals/s", "ms_per_step": float(t.item()) * 1e3,
                   "api": "FunctionalDepth([pd.DataFrame(X)], relax=True): pageable numpy memory -> pd.Series of %d float64 "
                          "depths, wall clock, %d calls" % (n, k_api),
                   "h2d_bytes_per_step": int(8 * n * Tl), "checksum": float(d_api.values.sum())}
        del df, full

    sec = None
    if not args.no_secondary and not args.ties and not (args.n or args.T):
        sec = secondary(c)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = evals * args.steps / (ms / 1e3)
    e2e_value = evals * args.steps / (ms_e2e / 1e3)
    peak, peak_src = peaks()
    phases, kern_ns = r["phases"], r["kern_ns"]
    kern_s = kern_ns / 1e9 / args.steps
    if relax:
        # roofline of the rank pipeline (all kernels of a step): algorithmic bytes = 8*n*T_local read once + 8*n written
        alg_bytes = 8.0 * n * Tl + 8.0 * n
        achieved = alg_bytes / kern_s / 1e9
        dominant = max(phases, key=phases.get) if phases else None
        tr = measured_traffic() if (n == 100_000 and T == 1024) else None
        traffic = tr["dram_bytes_per_step"] * (Tl / 1024.0) if tr else None
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_source": ("profiles/traffic_r02.json: ncu dram__bytes_read.sum + dram__bytes_write.sum over the "
                                   "kernels of one cfg2 step, captured at commit %s; scaled by this rank's rows"
                                   % tr.get("commit", "?")) if tr else None,
                "peak_source": peak_src,
                "kernel": "all kernels of one step (per-rank); dominant phase: %s" % dominant,
                "algorithmic_bytes_per_step": alg_bytes, "kernel_ms_per_step": kern_s * 1e3,
                "phase_ms_per_step": {k: v / 1e6 / args.steps for k, v in phases.items()}}
        if dominant:  # the same algorithmic bytes over the dominant phase alone
            dom_s = phases[dominant] / 1e9 / args.steps
            roof["dominant_phase"] = {"name": dominant, "ms_per_step": dom_s * 1e3, "achieved": alg_bytes / dom_s / 1e9,
                                      "frac": alg_bytes / dom_s / 1e9 / peak}
    else:
        # strict BD: int8-tensor dense work 2*(2T)*C(n-1,2) ops per depth-eval (SURVEY 8d).  Only --bd-impl gemm does
        # this many operations; for auto / match / bits the honest bound is the bytes the formulation moves (see
        # secondary.cfg3_strict_bd_match in the default run), so the dense-equivalent rate is reported as such.
        ops = 2.0 * (2 * T) * comb(n - 1, 2) * nq_local
        i8_peak = eng.probe_int8_peak() / 1e12
        dense = ops / kern_s / 1e12
        roof = {"bound": "tensor", "achieved": dense if args.bd_impl == "gemm" else None, "peak": i8_peak,
                "unit": "TOP/s (int8)", "frac": dense / i8_peak if args.bd_impl == "gemm" else None, "traffic": None,
                "dense_equivalent_tops": dense,
                "peak_source": "measured here: sd_probe_int8_peak (tcgen05.mma kind::i8 issue loop, operands resident in "
                               "shared memory; nominal dense is 4500)",
                "kernel_ms_per_step": kern_s * 1e3,
                "phase_ms_per_step": {k: v / 1e6 / args.steps for k, v in phases.items()}}

    line = {
        "metric": METRIC, "value": value, "unit": "depth-evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config,
        "notes": {"l2": "flushed between steps (256 MiB write)" if r["flush"] else
                        "per-rank input (%.0f MB) exceeds L2" % (r["local_bytes"] / 1e6),
                  "overhead_ms_per_step": ms / args.steps - kern_s * 1e3},
        "e2e": {"value": e2e_value, "unit": "depth-evals/s", "h2d_bytes_per_step": int(r["local_bytes"]),
                "d2h_bytes_per_step": int(nq_local * 8), "ms_per_step": ms_e2e / args.steps,
                "api": "sd_band_depth_f64 (host buffers, pinned input) + float64 depth on the host"},
        "gpu_launches": int(r["launches"]), "roofline": roof, "clocks": clocks,
        "engine": impl_used,
        "depth_checksum": float(np.sum(r["depth"])),
    }
    if e2e_api:
        line["e2e_api"] = e2e_api
    if sec:
        line["secondary"] = sec
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(args, n, T, rows=args.cpu_sample_rows)
        cb.pop("seconds_sample", None)
        if not args.no_reference_python:
            cb["reference_python"] = reference_python()
        line["cpu_baseline"] = cb
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main_perm(c: Ctx, args, n, T, name, config, sampler):
    """--workload perm: the permutation test of BASELINE config 5 through the public API, permutations sharded."""
    from statdepth_b200.homogeneity import permutation_test
    torch, dist = c.torch, c.dist
    F, G = perm_inputs()
    B = 1000
    for _ in range(max(1, args.warmup)):
        permutation_test(F, G, method="p2", B=B, seed=5, relax=True)
    times, launches = [], 0
    for _ in range(args.steps):
        if c.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = permutation_test(F, G, method="p2", B=B, seed=5, relax=True)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        launches += c.eng.timings()["launches"] * 3
    t = torch.tensor([sum(times)], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if c.rank == 0 else None
    if c.rank != 0:
        dist.destroy_process_group()
        return
    total = float(t.item())
    line = {"metric": METRIC, "value": B * args.steps / total, "unit": "permutations/s", "n_gpus": c.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "notes": {"timing": "wall clock around permutation_test (host code, H2D, batched engine calls, all-gather); "
                                "each permutation = three depth runs of 256-257 curves x 256 points",
                      "p_value": res["p_value"]},
            "e2e": {"value": B * args.steps / total, "unit": "permutations/s",
                    "h2d_bytes_per_step": int(3 * 8 * n * T), "d2h_bytes_per_step": int(8 * B * 256 * 3 // max(1, c.world)),
                    "ms_per_step": total / args.steps * 1e3, "api": "statdepth_b200.homogeneity.permutation_test"},
            "gpu_launches": int(launches), "roofline": None, "clocks": clocks}
    if c.world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(args, n, T)
        cb.pop("seconds_sample", None)
        line["cpu_baseline"] = cb
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"null": res["null"], "observed": [res["observed"]], "p_value": [res["p_value"]]})
    emit(line)
    if c.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
