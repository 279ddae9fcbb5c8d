"""Functional spatial depth (DESIGN K14): time the two passes and the whole call on the GPU, against an FP64 FMA rate
measured in the same run.

    python profiles/spatial_probe.py [--out profiles/spatial_probe.json] [--reps 5]

Cases: in-sample 20 000 x 1024 and 5 000 x 256 x 3; out of sample against a 100 000 x 1024 reference with 1, 1 000 and
10 000 new curves, one-shot (sd_spatial_norms_of_f64 from host buffers, the sample uploaded by every call) and through
the fitted reference (sd_spatial_norms_of_f64_dev, the sample resident).  Device-resident timings are CUDA events on
the engine's stream, median of --reps after one warm-up; the distance / sum split comes from a torch.profiler run of
its own.  Every (pair, feature) term costs two FP64 instructions in each pass (DSUB + DFMA), so the FP64 rate counts
4 n_q n_S F instructions per call, and the share of peak compares it with the rate of a DFMA-only kernel compiled and
timed here (4 independent chains per thread, all SMs).  The numpy oracle is timed on the host at 2 000 x 1024.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FMA_SRC = r"""
#include <cuda_runtime.h>
__global__ void fp64_fma_peak(double *out, int iters) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
    const double b = 0.9999999, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3;
}
extern "C" int launch_fp64_fma_peak(double *out, int iters, int blocks, int threads, void *stream) {
    fp64_fma_peak<<<blocks, threads, 0, (cudaStream_t)stream>>>(out, iters);
    return (int)cudaGetLastError();
}
"""


def fma_rate(eng, torch, stream, dev):
    """Measured DFMA/s of this GPU (each thread: iters * 64 FMAs)."""
    from statdepth_b200.build import _nvcc
    tmp = tempfile.mkdtemp(prefix="sd_fma_")
    src, lib = os.path.join(tmp, "fma.cu"), os.path.join(tmp, "fma.so")
    with open(src, "w") as fh:
        fh.write(FMA_SRC)
    subprocess.check_call([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler",
                           "-fPIC", src, "-o", lib])
    so = ctypes.CDLL(lib)
    sm = eng.info()["sm_count"]
    blocks, threads, iters = sm * 8, 256, 4096
    out = torch.empty(blocks * threads, dtype=torch.float64, device=dev)

    def run():
        assert so.launch_fp64_fma_peak(ctypes.c_void_p(out.data_ptr()), iters, blocks, threads,
                                       ctypes.c_void_p(eng.stream())) == 0
    ms = timed(run, torch, stream, 5)
    return blocks * threads * iters * 64 / (ms * 1e-3)


def timed(fn, torch, stream, reps):
    with torch.cuda.stream(stream):
        fn()
        stream.synchronize()
        t = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            t.append(a.elapsed_time(b))
    return float(np.median(t))


def kernel_split(fn, torch, stream):
    """Device time per spatial kernel (ms) of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with torch.cuda.stream(stream):
        fn()
        stream.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            stream.synchronize()
    split = {}
    for ev in prof.events():
        for key in ("spatial_dist_kernel", "spatial_sum_kernel", "spatial_norm_kernel", "finite_check_kernel"):
            if key in ev.name and ev.device_time_total > 0:
                split[key] = split.get(key, 0.0) + ev.device_time_total / 1e3
    return split


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "spatial_probe.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from statdepth_b200 import get_engine
    from test_spatial import np_spatial_r
    eng = get_engine()
    dev = torch.device("cuda", eng.device)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(device=eng.info()["name"], nvidia_smi=smi[eng.device] if smi else None, cases=[])
    peak = fma_rate(eng, torch, stream, dev)
    res["fp64_fma_per_s_measured"] = peak
    res["fp64_instr_per_s_peak"] = peak  # one DFMA / DSUB issue each
    rng = np.random.default_rng(0)

    def case(name, S, Y, nq, in_sample, one_shot=None):
        nS, F = S.shape
        with torch.cuda.stream(stream):
            dS = torch.from_numpy(S).to(dev)
            dY = dS if in_sample else torch.from_numpy(Y).to(dev)
            r = torch.empty(nq, dtype=torch.float64, device=dev)
        stream.synchronize()

        def run():
            eng.spatial_norms_of_dev(dS.data_ptr(), nS, dY.data_ptr(), nq, F, r.data_ptr())
        ms = timed(run, torch, stream, args.reps)
        split = kernel_split(run, torch, stream)
        instr = 4.0 * nq * nS * F
        row = dict(case=name, n_queries=nq, n_sample=nS, F=F, device_resident_ms=ms, kernel_ms=split,
                   fp64_instr_per_s=instr / (ms * 1e-3), share_of_measured_fp64_peak=instr / (ms * 1e-3) / peak)
        if one_shot is not None:
            t = []
            for k in range(args.reps + 1):
                t0 = time.perf_counter()
                one_shot()
                t.append(time.perf_counter() - t0)
            row["one_shot_host_ms"] = float(np.median(t[1:]) * 1e3)
            row["one_shot_kernel_ms"] = eng.timings()["kernel_ns"] / 1e6
        res["cases"].append(row)
        print(json.dumps(row), flush=True)
        del dS, dY, r

    X = rng.standard_normal((20_000, 1024)).cumsum(axis=1)
    case("in-sample 20000 x 1024", X, None, 20_000, True, lambda: eng.spatial_norms(X))
    X = rng.standard_normal((5_000, 768)).cumsum(axis=1)
    case("in-sample 5000 x 256 x 3", X, None, 5_000, True, lambda: eng.spatial_norms(X))
    S = rng.standard_normal((100_000, 1024))
    for m in (1, 1_000, 10_000):
        Y = rng.standard_normal((m, 1024))
        case("out of sample 100000 x 1024, %d new" % m, S, Y, m, False, lambda: eng.spatial_norms_of(S, Y))
    A = rng.standard_normal((2_000, 1024)).cumsum(axis=1)
    t0 = time.perf_counter()
    np_spatial_r(A, A)
    res["numpy_oracle_2000x1024_s"] = time.perf_counter() - t0
    res["host_cpus"] = os.cpu_count()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
