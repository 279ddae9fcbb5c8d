"""Extremal depth on the device: the extremity pass (stage 1), the per-curve key sort (stage 2a) and the ordering
(stage 2b) beside the rank-sums call that runs the same rank-only passes, and the public objects end to end.

    python profiles/extremal_probe.py OUT_DIR [--reps 20] [--warmup 3] [--e2e-reps 5]

Inputs, resident on the device: 100 000 random walks x 1024 points (bench.py's generator, seed 1), the same rounded
(np.round: a tie-stress variant) and 10^6 curves x 1 point.  CUDA events on the engine's stream around each call,
median of --reps after --warmup: sd_band_extremity_f64_dev (stage 1), sd_extremal_depth_dev (stages 2a + 2b), both
back to back (total), and sd_band_rank_sums_f64_dev (the like-for-like rank-pass reference).  Stages 2a and 2b run
inside one call, so their split comes from a torch.profiler pass of its own after the event timings: per call, the
summed device time of extremal_keys_kernel (2a) and of every other kernel of the call (2b: ids, merge sort, group
starts, scan, scatter).  End to end: ExtremalDepth and FunctionalBoxplot with both depths from a pageable DataFrame,
host clock, median of --e2e-reps after one warm-up call.  Writes OUT_DIR/extremal_probe.json with the device name,
power limit and max SM clock read in the same run.
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


def stage_split(fn, reps, out_dir, tag):
    """(2a, 2b) median device seconds per call from a torch.profiler trace of reps calls."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(out_dir, "extremal_trace_%s.json" % tag))
    keys, other = 0.0, 0.0
    for ev in prof.key_averages():
        dev_us = getattr(ev, "device_time_total", None)
        if dev_us is None:
            dev_us = ev.cuda_time_total
        if "extremal_keys_kernel" in ev.key:
            keys += dev_us
        elif ev.device_type.name == "CUDA" and "Memset" not in ev.key and "Memcpy" not in ev.key:
            other += dev_us
    return keys * 1e-6 / reps, other * 1e-6 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-reps", type=int, default=5)
    args = ap.parse_args()
    import pandas as pd
    import torch

    from depth_of_probe import device_info, event_times
    from statdepth_b200 import ExtremalDepth, FunctionalBoxplot
    from statdepth_b200._engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("extremal_probe needs a GPU")
    os.makedirs(args.out_dir, exist_ok=True)
    eng = get_engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", 0))
    res = {"device": device_info(), "engine": eng.info(), "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events on the engine's stream around each call, input resident on the device; "
                     "stage 2a / 2b split: torch.profiler kernel times in a separate pass",
           "cases": {}, "end_to_end": {}}

    def walks(T, n, seed):
        g = torch.Generator(device="cuda")
        g.manual_seed(seed)
        X = torch.empty((T, n), dtype=torch.float64, device="cuda")
        for r0 in range(0, T, 128):
            X[r0:r0 + 128] = torch.randn((min(128, T - r0), n), dtype=torch.float64, device="cuda", generator=g)
        return X.cumsum(0)

    def run_case(tag, X):
        T, n = X.shape
        p = X.data_ptr()
        m = torch.empty((T, n), dtype=torch.int32, device="cuda")
        e = torch.empty(n, dtype=torch.int64, device="cuda")
        qb = torch.empty((2, n), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's

        def stage1():
            eng.band_extremity_dev(p, T, n, n, m.data_ptr())

        def stage2():
            eng.extremal_depth_dev(m.data_ptr(), T, n, e.data_ptr())

        def total():
            stage1()
            stage2()

        calls = {"stage1_band_extremity_f64_dev": stage1, "stage2_extremal_depth_dev": stage2, "total": total,
                 "band_rank_sums_f64_dev": lambda: eng.band_rank_sums_dev(p, T, n, n, qb[0].data_ptr(),
                                                                          qb[1].data_ptr())}
        r = {"T": T, "n": n}
        for name, fn in calls.items():
            ts = event_times(fn, args.reps, args.warmup, stream)
            r[name] = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts))}
            print(tag, name, json.dumps(r[name]), flush=True)
        try:
            keys_s, order_s = stage_split(stage2, args.reps, args.out_dir, tag)
            r["stage2a_keys_profiler_s"] = keys_s
            r["stage2b_order_profiler_s"] = order_s
        except Exception as exc:  # the event timings above stand without the split
            keys_s = order_s = None
            r["stage_split_error"] = repr(exc)
        r["e_range"] = [int(e.min()), int(e.max())]
        print(tag, "2a", keys_s, "2b", order_s, flush=True)
        res["cases"][tag] = r

    X = walks(1024, 100_000, 1)
    run_case("walks_100000x1024", X)
    run_case("walks_rounded_100000x1024", X.round())
    g = torch.Generator(device="cuda")
    g.manual_seed(2)
    run_case("T1_n1000000", torch.randn((1, 1_000_000), dtype=torch.float64, device="cuda", generator=g))

    df = pd.DataFrame(X.cpu().numpy())  # pageable host memory, as a user's frame
    del X
    torch.cuda.empty_cache()
    for name, fn in (("ExtremalDepth", lambda: ExtremalDepth([df])),
                     ("FunctionalBoxplot_extremal", lambda: FunctionalBoxplot([df], depth='extremal')),
                     ("FunctionalBoxplot_mbd", lambda: FunctionalBoxplot([df]))):
        fn()
        ts = []
        for _ in range(args.e2e_reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        res["end_to_end"][name] = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts)),
                                   "reps": args.e2e_reps, "timing": "host clock around the public call"}
        print(name, json.dumps(res["end_to_end"][name]), flush=True)
    with open(os.path.join(args.out_dir, "extremal_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"device": res["device"]}))


if __name__ == "__main__":
    main()
