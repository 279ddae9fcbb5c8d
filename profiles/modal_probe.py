"""h-modal depth (DESIGN K15): time the pair selection and the sum pass on the GPU, against an FP64 FMA rate measured
in the same run.

    python profiles/modal_probe.py [--out profiles/modal_probe.json] [--reps 5]

Cases: in sample 20 000 x 1024 and 5 000 x 256 x 3 (selection at the 0.15 quantile and the all-queries sum pass timed
separately); fitting a reference of 100 000 x 1024 (selection only); 1, 1 000 and 10 000 new curves against
100 000 x 1024 (the out-of-sample sum pass, the sample resident).  Device-resident calls (sd_modal_*_dev) timed with
CUDA events on the engine's stream, median of --reps after one warm-up; the per-kernel split comes from a
torch.profiler run of its own.  Every (pair, feature) term of a pass costs two FP64 instructions (DSUB + DFMA): the sum
pass counts 2 n_q n_col F of them, a selection pass over the pairs 2 (pairs in the launched tiles) F.  The share of
peak compares with the rate of spatial_probe.py's DFMA-only kernel, compiled and timed here.
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

KERNELS = ("modal_pairs_kernel", "modal_cand_hist_kernel", "modal_sum_kernel", "modal_finish_kernel",
           "finite_check")


def kernel_split(fn, torch, stream):
    """(device ms, launches) per modal kernel of one call, from torch.profiler."""
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
    return {k: dict(ms=v[0], launches=v[1]) for k, v in split.items()}


def tile_pairs(n):
    """Pairs the selection's launched tiles (64 x 128, those holding some i < j) compute."""
    bq, bs = 64, 128
    tot = 0
    for by in range((n + bq - 1) // bq):
        q0 = by * bq
        for bx in range((n + bs - 1) // bs):
            if bx * bs + bs - 1 > q0:
                tot += min(bq, n - q0) * min(bs, n - bx * bs)
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "modal_probe.json"))
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
        r = dict(case=name, device_resident_ms=ms, kernel_ms=kernel_split(fn, torch, stream),
                 fp64_instr_per_s=instr / (ms * 1e-3), share_of_measured_fp64_peak=instr / (ms * 1e-3) / peak, **kw)
        res["cases"].append(r)
        print(json.dumps(r), flush=True)
        return r

    def in_sample(name, X, reps):
        n, F = X.shape
        dX = upload(X)
        k = rank(n)
        sel = row(name + ": selection", lambda: eng.modal_pair_select_dev(dX.data_ptr(), n, F, k), 0.0, reps,
                  n=n, F=F, k=k)
        d2 = eng.modal_pair_select_dev(dX.data_ptr(), n, F, k)
        h = float(np.sqrt(d2[0]))
        launches = sel["kernel_ms"].get("modal_pairs_kernel", {}).get("launches", 0)
        sel["pair_passes"] = launches
        sel["fp64_instr_per_s"] = 2.0 * tile_pairs(n) * F * launches / (sel["device_resident_ms"] * 1e-3)
        sel["share_of_measured_fp64_peak"] = sel["fp64_instr_per_s"] / peak
        out = torch.empty(n, dtype=torch.float64, device=dev)
        c = -0.5 / (h * h)
        row(name + ": sums", lambda: eng.modal_sums_dev(dX.data_ptr(), n, F, c, None, out.data_ptr()),
            2.0 * n * n * F, reps, n=n, F=F)
        del dX, out

    X = rng.standard_normal((20_000, 1024)).cumsum(axis=1)
    in_sample("in-sample 20000 x 1024", X, args.reps)
    X = rng.standard_normal((5_000, 768)).cumsum(axis=1)
    in_sample("in-sample 5000 x 256 x 3", X, args.reps)
    S = rng.standard_normal((100_000, 1024))
    dS = upload(S)
    k = rank(100_000)
    r = row("fit reference 100000 x 1024: selection", lambda: eng.modal_pair_select_dev(dS.data_ptr(), 100_000, 1024,
                                                                                        k), 0.0, 3, n=100_000, F=1024, k=k)
    launches = r["kernel_ms"].get("modal_pairs_kernel", {}).get("launches", 0)
    r["pair_passes"] = launches
    r["fp64_instr_per_s"] = 2.0 * tile_pairs(100_000) * 1024 * launches / (r["device_resident_ms"] * 1e-3)
    r["share_of_measured_fp64_peak"] = r["fp64_instr_per_s"] / peak
    h = float(np.sqrt(eng.modal_pair_select_dev(dS.data_ptr(), 100_000, 1024, k)[0]))
    c = -0.5 / (h * h)
    for m in (1, 1_000, 10_000):
        dY = upload(rng.standard_normal((m, 1024)))
        out = torch.empty(m, dtype=torch.float64, device=dev)
        row("out of sample 100000 x 1024, %d new" % m,
            lambda: eng.modal_sums_of_dev(dS.data_ptr(), 100_000, dY.data_ptr(), m, 1024, c, out.data_ptr()),
            2.0 * m * 100_001 * 1024, args.reps, n_sample=100_000, n_queries=m, F=1024,
            blocks=((100_001 + 127) // 128) * ((m + 63) // 64))
        del dY, out
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
