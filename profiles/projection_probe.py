"""Random projection depths on the B200: device-resident calls beside the exact calls they approximate or share rank
passes with, a per-phase split, and the public classes end to end.

    python profiles/projection_probe.py OUT_DIR [--reps 10] [--warmup 2] [--e2e-reps 3]

Cases (seeded; K random unit directions from np.random.default_rng(0)):
  * cloud 50 000 x 2, K = 1 000: sd_projection_tukey_f64_dev beside sd_pointcloud_halfspace_f64 (exact, host buffer,
    same run), with the approximation gap RT - HD of the numerators (max and mean);
  * clouds 50 000 x d, d in {3, 8, 64}, K = 1 000: sd_projection_tukey_f64_dev and sd_projection_outlyingness_f64_dev;
  * curves 5 000 x 256 x 3 (random walks), K = 200: the same two calls;
  * univariate 100 000 x 1024 random walks: sd_band_outlyingness_f64_dev beside sd_band_rank_sums_f64_dev.
Device calls: CUDA events on the engine's stream, median of --reps after --warmup.  Phase split: a torch.profiler
pass of its own (2 calls per case), the summed device time per call of projection_kernel (projection), of the rank
pipeline's and the row sort's kernels (ranking / sorting) and of rt_min_kernel, medmad_kernel and pd_max_kernel
(reduction).  End to end: ProjectionDepth / FunctionalProjectionDepth from pageable DataFrames, host clock, median
of --e2e-reps after one warm-up call.  Writes OUT_DIR/projection_probe.json with the device name, power limit and
max SM clock read in the same run.
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

REDUCTION = ("rt_min_kernel", "medmad_kernel", "pd_max_kernel")


def phase_split(fn, reps=2):
    """Mean device seconds per call by phase from a torch.profiler pass."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {"projection_s": 0.0, "ranking_or_sorting_s": 0.0, "reduction_s": 0.0, "other_s": 0.0}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = getattr(ev, "cuda_time_total", 0.0)
        name = ev.key
        if "Memcpy" in name or "Memset" in name:
            key = "other_s"
        elif "projection_kernel" in name:
            key = "projection_s"
        elif any(k in name for k in REDUCTION):
            key = "reduction_s"
        elif "mbd_" in name or "sort_" in name:
            key = "ranking_or_sorting_s"
        else:
            key = "other_s"
        out[key] += us * 1e-6 / reps
    return out


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
    from statdepth_b200 import FunctionalProjectionDepth, ProjectionDepth
    from statdepth_b200._engine import get_engine
    from statdepth_b200._projection import draw_directions
    if not torch.cuda.is_available():
        raise SystemExit("projection_probe needs a GPU")
    os.makedirs(args.out_dir, exist_ok=True)
    eng = get_engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", 0))
    res = {"device": device_info(), "engine": eng.info(), "reps": args.reps, "warmup": args.warmup,
           "timing": "CUDA events on the engine's stream around each call (median); the exact halfspace call takes "
                     "host buffers and also reports the engine's device time between upload and download "
                     "(kernel_ns, median); phases from a separate torch.profiler pass",
           "cases": {}, "end_to_end": {}}

    def timed(case, name, fn, host_call=False, split=True):
        kernel = []

        def call():
            fn()
            if host_call:
                kernel.append(eng.timings()["kernel_ns"] * 1e-9)

        ts = event_times(call, args.reps, args.warmup, stream)
        r = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts))}
        if host_call:
            r["kernel_median_s"] = float(np.median(kernel[args.warmup:]))
        if split:
            try:
                r["phases"] = phase_split(fn)
            except Exception as exc:  # the event timings stand without the split
                r["phase_split_error"] = repr(exc)
        case[name] = r
        print(name, json.dumps(r), flush=True)

    def dev(A):
        t = torch.from_numpy(np.ascontiguousarray(A)).cuda()
        torch.cuda.synchronize()
        return t

    rng = np.random.default_rng(0)
    for d in (2, 3, 8, 64):
        N, K = 50_000, 1000
        P = rng.standard_normal((N, d))
        U = draw_directions(d, K, seed=0)
        dP = dev(P)
        cnt = torch.empty(N, dtype=torch.int64, device="cuda")
        o = torch.empty(N, dtype=torch.float64, device="cuda")
        case = {"N": N, "d": d, "K": K}
        timed(case, "projection_tukey_f64_dev",
              lambda: eng.projection_tukey_counts_dev(dP.data_ptr(), N, 1, d, U, cnt.data_ptr()))
        if d == 2:
            timed(case, "pointcloud_halfspace_f64_exact", lambda: eng.halfspace_counts(P), True, False)
            gap = eng.projection_tukey_counts(P[:, None, :], U) - eng.halfspace_counts(P)
            case["rt_minus_hd"] = {"max": int(gap.max()), "mean": float(gap.mean()), "min": int(gap.min())}
        else:
            timed(case, "projection_outlyingness_f64_dev",
                  lambda: eng.projection_outlyingness_dev(dP.data_ptr(), N, 1, d, U, o.data_ptr()))
        res["cases"]["cloud_50000x%d_k%d" % (d, K)] = case
        del dP

    N, T, d, K = 5000, 256, 3, 200
    F = rng.standard_normal((N, T, d)).cumsum(1)
    U = draw_directions(d, K, seed=0)
    dF = dev(F)
    cnt = torch.empty(N, dtype=torch.int64, device="cuda")
    o = torch.empty((T, N), dtype=torch.float64, device="cuda")
    case = {"N": N, "T": T, "d": d, "K": K}
    timed(case, "projection_tukey_f64_dev",
          lambda: eng.projection_tukey_counts_dev(dF.data_ptr(), N, T, d, U, cnt.data_ptr()))
    timed(case, "projection_outlyingness_f64_dev",
          lambda: eng.projection_outlyingness_dev(dF.data_ptr(), N, T, d, U, o.data_ptr()))
    res["cases"]["curves_5000x256x3_k200"] = case
    del dF, o

    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    T, n = 1024, 100_000
    X = torch.empty((T, n), dtype=torch.float64, device="cuda")
    for r0 in range(0, T, 128):
        X[r0:r0 + 128] = torch.randn((min(128, T - r0), n), dtype=torch.float64, device="cuda", generator=g)
    X = X.cumsum(0)
    o = torch.empty((T, n), dtype=torch.float64, device="cuda")
    out = torch.empty((2, n), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    p = X.data_ptr()
    case = {"T": T, "n": n}
    timed(case, "band_outlyingness_f64_dev", lambda: eng.band_outlyingness_dev(p, T, n, n, o.data_ptr()))
    timed(case, "band_rank_sums_f64_dev",
          lambda: eng.band_rank_sums_dev(p, T, n, n, out[0].data_ptr(), out[1].data_ptr()), split=False)
    res["cases"]["univariate_100000x1024"] = case

    df = pd.DataFrame(X.cpu().numpy())  # pageable host memory, as a user's frame
    del X, o
    torch.cuda.empty_cache()
    cloud8 = pd.DataFrame(rng.standard_normal((50_000, 8)))
    curves = [pd.DataFrame(F[i]) for i in range(F.shape[0])]
    for name, fn in (("ProjectionDepth_50000x8_projection", lambda: ProjectionDepth(cloud8)),
                     ("ProjectionDepth_50000x8_tukey", lambda: ProjectionDepth(cloud8, kind='tukey')),
                     ("FunctionalProjectionDepth_univariate_100000x1024", lambda: FunctionalProjectionDepth([df])),
                     ("FunctionalProjectionDepth_5000x256x3_k200_projection",
                      lambda: FunctionalProjectionDepth(curves, directions=200)),
                     ("FunctionalProjectionDepth_5000x256x3_k200_tukey",
                      lambda: FunctionalProjectionDepth(curves, kind='tukey', directions=200))):
        fn()
        ts = []
        for _ in range(args.e2e_reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        res["end_to_end"][name] = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts)),
                                   "reps": args.e2e_reps, "timing": "host clock around the public call"}
        print(name, json.dumps(res["end_to_end"][name]), flush=True)
    with open(os.path.join(args.out_dir, "projection_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"device": res["device"]}))


if __name__ == "__main__":
    main()
