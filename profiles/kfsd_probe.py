"""Kernelized functional spatial depth (DESIGN K16): time the gram, weight and quad passes on the GPU, against an FP64
FMA rate measured in the same run.

    python profiles/kfsd_probe.py [--out profiles/kfsd_probe.json] [--reps 5]

Cases: in sample 20 000 x 1024 and 5 000 x 256 x 3 (all queries, E built in the call); fitting a reference of
20 000 x 1024 (the pair selection at the 0.15 quantile, then the gram pass into a resident E); 1, 1 000 and 10 000
new curves against 20 000 x 1024 with E resident.  Device-resident calls (sd_kfsd_*_dev, sd_modal_pair_select_f64_dev)
timed with CUDA events on the engine's stream, median of --reps after one warm-up; the per-kernel split comes from a
torch.profiler run of its own.  A (pair, feature) term of the gram or weight pass costs two FP64 instructions (DSUB +
DFMA), so each counts 2 n_q n_S F; the quad pass counts n_q n_S^2 DFMA.  The share of peak compares with the rate of
spatial_probe.py's DFMA-only kernel, compiled and timed here.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from spatial_probe import fma_rate, timed  # noqa: E402

KERNELS = ("kfsd_gram_kernel", "kfsd_weight_kernel", "kfsd_quad_kernel", "kfsd_finish_kernel", "modal_pairs_kernel",
           "modal_cand_hist_kernel", "finite_check")


def kernel_split(fn, torch, stream, peak, instr):
    """(device ms, launches, FP64 instructions / s and share of the measured peak) per kernel of one call, from
    torch.profiler; instr maps a kernel to the FP64 instructions it executes in the call."""
    from torch.profiler import ProfilerActivity, profile
    with torch.cuda.stream(stream):
        fn()
        stream.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            stream.synchronize()
    split = {}
    for ev in prof.events():
        for key in KERNELS:
            if key in ev.name and ev.device_time_total > 0:
                ms, k = split.get(key, (0.0, 0))
                split[key] = (ms + ev.device_time_total / 1e3, k + 1)
    out = {}
    for k, (ms, launches) in split.items():
        out[k] = dict(ms=ms, launches=launches)
        if k in instr:
            out[k]["fp64_instr_per_s"] = instr[k] / (ms * 1e-3)
            out[k]["share_of_measured_fp64_peak"] = instr[k] / (ms * 1e-3) / peak
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kfsd_probe.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from statdepth_b200 import get_engine
    from statdepth_b200._modal import _quantile_bandwidth
    eng = get_engine()
    dev = torch.device("cuda", eng.device)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(device=eng.info()["name"], nvidia_smi=smi[eng.device] if smi else None, cases=[])
    peak = fma_rate(eng, torch, stream, dev)
    res["fp64_fma_per_s_measured"] = peak
    rng = np.random.default_rng(0)

    def rank(n, q=0.15):
        ks = []
        _quantile_bandwidth(n * (n - 1) // 2, q, lambda k: ks.append(k) or (1.0, 1.0))
        return ks[0]

    def upload(A):
        with torch.cuda.stream(stream):
            d = torch.from_numpy(A).to(dev)
        stream.synchronize()
        return d

    def row(name, fn, instr, reps, **kw):
        ms = timed(fn, torch, stream, reps)
        total = sum(instr.values())
        r = dict(case=name, device_resident_ms=ms, kernel_ms=kernel_split(fn, torch, stream, peak, instr),
                 fp64_instr_per_s=total / (ms * 1e-3), share_of_measured_fp64_peak=total / (ms * 1e-3) / peak, **kw)
        res["cases"].append(r)
        print(json.dumps(r), flush=True)
        return r

    def sigma_c(dX, n, F):
        d2 = eng.modal_pair_select_dev(dX.data_ptr(), n, F, rank(n))
        h = float(np.sqrt(d2[0]))
        return h, -1.0 / (h * h)

    def in_sample(name, X, reps):
        n, F = X.shape
        dX = upload(X)
        h, c = sigma_c(dX, n, F)
        out = torch.empty(n, dtype=torch.float64, device=dev)
        row(name, lambda: eng.kfsd_norms_dev(dX.data_ptr(), n, F, c, None, out.data_ptr()),
            dict(kfsd_gram_kernel=2.0 * n * n * F, kfsd_weight_kernel=2.0 * n * n * F,
                 kfsd_quad_kernel=float(n) ** 3), reps, n=n, F=F, bandwidth=h)
        del dX, out

    X = rng.standard_normal((20_000, 1024)).cumsum(axis=1)
    in_sample("in-sample 20000 x 1024", X, args.reps)
    X = rng.standard_normal((5_000, 768)).cumsum(axis=1)
    in_sample("in-sample 5000 x 256 x 3", X, args.reps)
    nS, F = 20_000, 1024
    dS = upload(rng.standard_normal((nS, F)))
    h, c = sigma_c(dS, nS, F)
    E = torch.empty((nS, nS), dtype=torch.float64, device=dev)

    def fit():
        d2 = eng.modal_pair_select_dev(dS.data_ptr(), nS, F, rank(nS))
        hh = float(np.sqrt(d2[0]))
        eng.kfsd_gram_dev(dS.data_ptr(), nS, F, -1.0 / (hh * hh), E.data_ptr())

    row("fit reference 20000 x 1024: selection + gram", fit, dict(kfsd_gram_kernel=2.0 * nS * nS * F), args.reps,
        n=nS, F=F, bandwidth=h)
    eng.kfsd_gram_dev(dS.data_ptr(), nS, F, c, E.data_ptr())
    for m in (1, 1_000, 10_000):
        dY = upload(rng.standard_normal((m, F)))
        out = torch.empty(m, dtype=torch.float64, device=dev)
        row("out of sample 20000 x 1024, %d new" % m,
            lambda: eng.kfsd_norms_of_dev(dS.data_ptr(), nS, E.data_ptr(), dY.data_ptr(), m, F, c, out.data_ptr()),
            dict(kfsd_weight_kernel=2.0 * m * nS * F, kfsd_quad_kernel=float(m) * nS * nS), args.reps,
            n_sample=nS, n_queries=m, F=F, blocks_per_pass=((nS + 127) // 128) * ((m + 63) // 64))
        del dY, out
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
