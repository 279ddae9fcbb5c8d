"""Fitted reference on the device: build time of the sorted index (sd_band_sort_rows_f64_dev) and query time
(sd_band_depth_sorted_f64_dev) against the out-of-sample kernel it can replace (sd_band_depth_oos_f64_dev), then the
public objects end to end.

    python profiles/reference_probe.py OUT_DIR [--reps 20] [--warmup 3] [--nY 1,100,1000,10000,100000]

Reference: n_S = 100 000 random-walk curves x T = 1024 points, new curves from the same process.  Device part: the
pooled [S | Y] matrix is resident on the device; the out-of-sample kernel ranks it in place, the query reads Y from
the same memory (leading dimension n_S + n_Y); every repetition is timed with CUDA events on the engine's stream, median
of --reps after --warmup.  The index (819 MB) and the sample are far larger than the 126 MB L2.  The counts of both
paths are asserted equal.  End to end: pageable DataFrames, host clock, median of 5.  Writes OUT_DIR/reference_probe.json
with the device name and power limit read in the same run.
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


def host_times(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append(time.perf_counter() - t0)
    return out


def summary(ts):
    return {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nS", type=int, default=100_000)
    ap.add_argument("--T", type=int, default=1024)
    ap.add_argument("--nY", default="1,100,1000,10000,100000")
    ap.add_argument("--e2e-nY", type=int, default=1000)
    args = ap.parse_args()
    import pandas as pd
    import torch

    from depth_of_probe import device_info, event_times
    from statdepth_b200 import DepthClassifier, FunctionalDepthOf, FunctionalReference
    from statdepth_b200._engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("reference_probe needs a GPU")
    eng = get_engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", 0))
    T, nS = args.T, args.nS
    nYs = [int(v) for v in args.nY.split(",") if v]
    res = {"device": device_info(), "engine": eng.info(), "nS": nS, "T": T, "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events on the engine's stream around each call, inputs resident on the device",
           "build": None, "query": [], "e2e": None}

    gen = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn((T, nS + max(nYs)), dtype=torch.float64, device="cuda", generator=gen).cumsum_(0)
    S = X[:, :nS].contiguous()
    index = torch.empty((T, nS), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's

    def build():
        eng.band_sort_rows_dev(S.data_ptr(), T, nS, nS, index.data_ptr())

    ts = event_times(build, args.reps, args.warmup, stream)
    res["build"] = dict(summary(ts), bytes_sorted=8 * T * nS)
    print(json.dumps({"build": res["build"]}), flush=True)
    del S
    torch.cuda.empty_cache()

    for nY, J in [(n, 2) for n in nYs] + [(args.e2e_nY, 3)]:
        Xp = X[:, :nS + nY].contiguous()
        ld = nS + nY
        base = Xp.data_ptr()
        out = torch.zeros((J - 1, nY), dtype=torch.int64, device="cuda")
        k7 = torch.zeros((J - 1, nY), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()

        def query():
            eng.band_depth_sorted_counts_dev(index.data_ptr(), T, nS, base + 8 * nS, nY, ld, J, out.data_ptr())

        def oos():
            for j in range(2, J + 1):
                eng.band_depth_oos_counts_dev(base, T, nS, ld, base + 8 * nS, nY, ld, k7[j - 2].data_ptr(), j, True)

        tq = event_times(query, args.reps, args.warmup, stream)
        tk = event_times(oos, args.reps, args.warmup, stream)
        equal = bool((out.cpu() == k7.cpu()).all())
        assert equal, "sorted-reference counts differ from the out-of-sample kernel at nY=%d J=%d" % (nY, J)
        q, k = summary(tq), summary(tk)
        row = {"nY": nY, "J": J, "query": q, "oos_kernel": k, "counts_equal": equal,
               "speedup_query_vs_oos": k["median_s"] / q["median_s"],
               "build_plus_query_s": res["build"]["median_s"] + q["median_s"],
               "build_plus_query_vs_oos": (res["build"]["median_s"] + q["median_s"]) / k["median_s"],
               "searches_per_s": 2 * nY * T / q["median_s"]}
        res["query"].append(row)
        print(json.dumps(row), flush=True)
        del Xp, out, k7
        torch.cuda.empty_cache()
    del X, index
    torch.cuda.empty_cache()

    # end to end from pageable DataFrames (host clock; every call ends in a device synchronisation)
    rng = np.random.default_rng(1)
    ref_df = pd.DataFrame(rng.standard_normal((T, nS)).cumsum(0))
    other_df = pd.DataFrame(rng.standard_normal((T, nS)).cumsum(0) + 2.0)
    new_df = pd.DataFrame(rng.standard_normal((T, args.e2e_nY)).cumsum(0))
    t_fit = host_times(lambda: FunctionalReference([ref_df]).close(), 5)
    ref = FunctionalReference([ref_df])
    t_ref = host_times(lambda: ref.depth_of([new_df]), 5)
    t_oos = host_times(lambda: FunctionalDepthOf([new_df], [ref_df], relax=True), 5)
    assert ref.depth_of([new_df]).values.tolist() == FunctionalDepthOf([new_df], [ref_df], relax=True).values.tolist()
    ref.close()
    clf = DepthClassifier({"a": [ref_df], "b": [other_df]})
    t_clf = host_times(lambda: clf.predict([new_df]), 5)
    clf.close()
    res["e2e"] = {"timing": "host clock, median of 5 after one warm-up, pageable DataFrames", "nY": args.e2e_nY,
                  "fit_FunctionalReference": summary(t_fit), "depth_of": summary(t_ref),
                  "FunctionalDepthOf": summary(t_oos), "DepthClassifier_predict_2_classes": summary(t_clf),
                  "upload_bytes_depth_of": 8 * T * args.e2e_nY,
                  "upload_bytes_FunctionalDepthOf": 8 * T * (nS + args.e2e_nY)}
    print(json.dumps(res["e2e"]), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "reference_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"device": res["device"]}))


if __name__ == "__main__":
    main()
