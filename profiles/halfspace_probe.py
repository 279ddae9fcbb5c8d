"""Halfspace (Tukey) depth on the B200: each call beside the call that runs the same rank passes, and the public
classes end to end.

    python profiles/halfspace_probe.py OUT_DIR [--reps 10] [--warmup 2] [--e2e-reps 3]

Cases (seeded):
  * cloud: 50 000 standard normal points, all queries: sd_pointcloud_halfspace_f64 beside
    sd_pointcloud_simplicial_f64 at tol 0 and at tol 1e-7 (both run the same two rank passes of the angular keys).
  * bivariate curves: 5 000 random walks x 256 points x 2 channels, 64 queries and all 5 000:
    sd_functional_halfspace_f64.
  * univariate curves: 100 000 random walks x 1024 points (bench.py's generator, seed 1), resident on the device:
    sd_band_halfspace_f64_dev beside sd_band_rank_sums_f64_dev (the same rank-only passes).
The cloud and bivariate entry points take host buffers (0.8 MB and 20 MB, uploaded inside the call): CUDA events on
the engine's stream around the call, and the engine's own device time between its upload and its download
(kernel_ns), each the median of --reps after --warmup.  End to end: HalfspaceDepth and FunctionalHalfspaceDepth from
pageable DataFrames, host clock, median of --e2e-reps after one warm-up call.  Writes OUT_DIR/halfspace_probe.json
with the device name, power limit and max SM clock read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--e2e-reps", type=int, default=3)
    args = ap.parse_args()
    import pandas as pd
    import torch

    from depth_of_probe import device_info, event_times
    from statdepth_b200 import FunctionalHalfspaceDepth, HalfspaceDepth
    from statdepth_b200._engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("halfspace_probe needs a GPU")
    os.makedirs(args.out_dir, exist_ok=True)
    eng = get_engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", 0))
    res = {"device": device_info(), "engine": eng.info(), "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events on the engine's stream around each call (median); host-buffer calls also report "
                     "the engine's device time between upload and download (kernel_ns, median)",
           "cases": {}, "end_to_end": {}}

    def timed(case, name, fn, host_call):
        kernel = []

        def call():
            fn()
            if host_call:
                kernel.append(eng.timings()["kernel_ns"] * 1e-9)

        ts = event_times(call, args.reps, args.warmup, stream)
        r = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts))}
        if host_call:
            r["kernel_median_s"] = float(np.median(kernel[args.warmup:]))
        case[name] = r
        print(name, json.dumps(r), flush=True)

    rng = np.random.default_rng(0)
    P = rng.standard_normal((50_000, 2))
    case = {"n": 50_000, "queries": 50_000}
    timed(case, "pointcloud_halfspace_f64", lambda: eng.halfspace_counts(P), True)
    timed(case, "pointcloud_simplicial_f64_tol0", lambda: eng.simplicial_counts(P, None, 0.0), True)
    timed(case, "pointcloud_simplicial_f64_tol1e-7", lambda: eng.simplicial_counts(P, None, 1e-7), True)
    h = eng.halfspace_counts(P)
    case["h_range"] = [int(h.min()), int(h.max())]
    res["cases"]["cloud_50000"] = case

    F = rng.standard_normal((5000, 256, 2)).cumsum(1)
    for nq in (64, 5000):
        q = None if nq == 5000 else rng.choice(5000, nq, replace=False)
        case = {"N": 5000, "T": 256, "queries": nq}
        timed(case, "functional_halfspace_f64", lambda: eng.functional_halfspace_counts(F, q), True)
        res["cases"]["bivariate_5000x256_q%d" % nq] = case

    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    T, n = 1024, 100_000
    X = torch.empty((T, n), dtype=torch.float64, device="cuda")
    for r0 in range(0, T, 128):
        X[r0:r0 + 128] = torch.randn((min(128, T - r0), n), dtype=torch.float64, device="cuda", generator=g)
    X = X.cumsum(0)
    out = torch.empty((3, n), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's
    p = X.data_ptr()
    case = {"T": T, "n": n}
    timed(case, "band_halfspace_f64_dev", lambda: eng.band_halfspace_counts_dev(p, T, n, n, out[0].data_ptr()), False)
    timed(case, "band_rank_sums_f64_dev",
          lambda: eng.band_rank_sums_dev(p, T, n, n, out[1].data_ptr(), out[2].data_ptr()), False)
    res["cases"]["univariate_100000x1024"] = case

    df = pd.DataFrame(X.cpu().numpy())  # pageable host memory, as a user's frame
    del X
    torch.cuda.empty_cache()
    cloud = pd.DataFrame(P, columns=["x", "y"])
    curves = [pd.DataFrame(F[i], columns=["x", "y"]) for i in range(F.shape[0])]
    for name, fn in (("HalfspaceDepth_50000", lambda: HalfspaceDepth(cloud)),
                     ("FunctionalHalfspaceDepth_univariate_100000x1024", lambda: FunctionalHalfspaceDepth([df])),
                     ("FunctionalHalfspaceDepth_bivariate_5000x256", lambda: FunctionalHalfspaceDepth(curves))):
        fn()
        ts = []
        for _ in range(args.e2e_reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        res["end_to_end"][name] = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts)),
                                   "reps": args.e2e_reps, "timing": "host clock around the public call"}
        print(name, json.dumps(res["end_to_end"][name]), flush=True)
    with open(os.path.join(args.out_dir, "halfspace_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"device": res["device"]}))


if __name__ == "__main__":
    main()
