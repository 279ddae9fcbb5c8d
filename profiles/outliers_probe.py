"""Functional outlier detection on the device: the rank-sums call and the envelope call against the MBD call they sit
next to, and the two public objects end to end against FunctionalDepth.

    python profiles/outliers_probe.py OUT_DIR [--reps 20] [--warmup 3] [--n 100000] [--T 1024]

Input: n random-walk curves x T points, resident on the device for the entry-point timings (CUDA events on the
engine's stream around each call, median of --reps after --warmup).  The envelope call takes the central half by
MBD as members, with and without outside counts; its algorithmic bytes are X once per pass (8 T n each; the count
pass is a second) plus the member mask, over the median time, against the HBM copy rate bench.py uses.  End to end:
FunctionalBoxplot, Outliergram and FunctionalDepth([df], relax=True) from the same pageable DataFrame, host clock,
median of --e2e-reps after one warm-up call.  Writes OUT_DIR/outliers_probe.json with the device name, power limit
and max SM clock read in the same run.
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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-reps", type=int, default=5)
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--T", type=int, default=1024)
    args = ap.parse_args()
    import pandas as pd
    import torch

    import bench
    from depth_of_probe import device_info, event_times
    from statdepth_b200 import FunctionalBoxplot, FunctionalDepth, Outliergram
    from statdepth_b200._engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("outliers_probe needs a GPU")
    eng = get_engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", 0))
    peak_gbs, peak_src = bench.peaks()
    T, n = args.T, args.n
    res = {"device": device_info(), "engine": eng.info(), "n": n, "T": T, "reps": args.reps, "warmup": args.warmup,
           "hbm_copy_gbs": peak_gbs, "hbm_copy_source": peak_src,
           "timing": "CUDA events on the engine's stream around each call, input resident on the device",
           "calls": {}, "end_to_end": {}}
    gen = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn((T, n), dtype=torch.float64, device="cuda", generator=gen).cumsum_(0)
    q = torch.zeros(n, dtype=torch.int64, device="cuda")
    qb = torch.zeros((2, n), dtype=torch.int64, device="cuda")
    env = torch.zeros((2, T), dtype=torch.float64, device="cuda")
    out = torch.zeros(n, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's
    p = X.data_ptr()
    eng.band_depth_counts_dev(p, T, n, n, q.data_ptr(), None, n, 2, True)
    member = torch.zeros(n, dtype=torch.uint8, device="cuda")
    member[torch.argsort(-q.cpu(), stable=True)[: (n + 1) // 2].cuda()] = 1
    torch.cuda.synchronize()
    x_bytes = 8 * T * n
    calls = {
        "band_depth_f64_dev": (lambda: eng.band_depth_counts_dev(p, T, n, n, q.data_ptr(), None, n, 2, True), None),
        "band_rank_sums_f64_dev": (lambda: eng.band_rank_sums_dev(p, T, n, n, qb[0].data_ptr(), qb[1].data_ptr()),
                                   None),
        "band_envelope_f64_dev_with_outside": (
            lambda: eng.band_envelope_dev(p, T, n, n, member.data_ptr(), 1.5, env[0].data_ptr(), env[1].data_ptr(),
                                          out.data_ptr()), 2 * x_bytes + n),
        "band_envelope_f64_dev": (
            lambda: eng.band_envelope_dev(p, T, n, n, member.data_ptr(), 1.5, env[0].data_ptr(), env[1].data_ptr()),
            x_bytes + n),
    }
    for name, (fn, nbytes) in calls.items():
        ts = event_times(fn, args.reps, args.warmup, stream)
        med = float(np.median(ts))
        r = {"median_s": med, "min_s": float(min(ts)), "max_s": float(max(ts)),
             "launches": eng.timings()["launches"]}
        if nbytes is not None:
            r.update(algorithmic_bytes=nbytes, achieved_gbs=nbytes / med / 1e9,
                     frac_of_hbm_copy=nbytes / med / 1e9 / peak_gbs)
        res["calls"][name] = r
        print(name, json.dumps(r), flush=True)
    res["rank_sums_q_equals_mbd"] = bool((qb[0].cpu() == q.cpu()).all())

    df = pd.DataFrame(X.cpu().numpy())  # pageable host memory, as a user's frame
    del X, qb, env, out, member
    torch.cuda.empty_cache()
    for name, fn in (("FunctionalDepth_relax", lambda: FunctionalDepth([df], relax=True)),
                     ("FunctionalBoxplot", lambda: FunctionalBoxplot([df])),
                     ("Outliergram", lambda: Outliergram([df]))):
        fn()
        ts = []
        for _ in range(args.e2e_reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        res["end_to_end"][name] = {"median_s": float(np.median(ts)), "min_s": float(min(ts)), "max_s": float(max(ts)),
                                   "reps": args.e2e_reps, "timing": "host clock around the public call"}
        print(name, json.dumps(res["end_to_end"][name]), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "outliers_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"device": res["device"]}))


if __name__ == "__main__":
    main()
