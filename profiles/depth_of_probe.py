"""Out-of-sample relaxed band depth on the device: kernel time of sd_band_depth_oos_f64_dev against the per-curve
batched path it replaces (sd_band_depth_batched_f64 with one sub-population S u {g} per new curve).

    python profiles/depth_of_probe.py OUT_DIR [--reps 20] [--warmup 3] [--nY 1000,10000,100000]

Sample: n_S = 100 000 random-walk curves x T = 1024 points, new curves from the same process.  The pooled [S | Y]
matrix is resident on the device (the call uses it in place); every repetition is timed with CUDA events on the
engine's stream, after warm-up.  Algorithmic bytes per call: the pooled matrix once, 8 T (n_S + n_Y), over kernel time,
against the HBM copy rate bench.py uses.  Writes OUT_DIR/depth_of_probe.json with the device name and power limit
read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as exc:  # the number is still reported, without the setting it was taken at
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % exc
    return info


def event_times(fn, reps, warmup, stream):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        out.append(a.elapsed_time(b) * 1e-3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nS", type=int, default=100_000)
    ap.add_argument("--T", type=int, default=1024)
    ap.add_argument("--nY", default="1000,10000,100000")
    ap.add_argument("--batched-nY", type=int, default=16)
    args = ap.parse_args()
    import torch

    import bench
    from statdepth_b200._engine import get_engine, mbd_plan
    if not torch.cuda.is_available():
        raise SystemExit("depth_of_probe needs a GPU")
    eng = get_engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", 0))
    peak_gbs, peak_src = bench.peaks()
    T, nS = args.T, args.nS
    res = {"device": device_info(), "engine": eng.info(), "nS": nS, "T": T, "reps": args.reps,
           "warmup": args.warmup, "hbm_copy_gbs": peak_gbs, "hbm_copy_source": peak_src,
           "timing": "CUDA events on the engine's stream around each call, pooled input resident on the device",
           "oos": [], "batched": None}
    nYs = [int(v) for v in args.nY.split(",") if v]
    gen = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn((T, nS + max(nYs)), dtype=torch.float64, device="cuda", generator=gen).cumsum_(0)
    for nY in nYs:
        # [S | Y] as one matrix of ld = nS + nY: the call ranks it in place
        Xp = X[:, :nS + nY].contiguous()
        out = torch.zeros(nY, dtype=torch.int64, device="cuda")
        base, ld = Xp.data_ptr(), nS + nY
        torch.cuda.synchronize()  # the engine's stream does not order itself behind torch's

        def call():
            eng.band_depth_oos_counts_dev(base, T, nS, ld, base + 8 * nS, nY, ld, out.data_ptr(), 2, True)

        ts = event_times(call, args.reps, args.warmup, stream)
        med = float(np.median(ts))
        nbytes = 8 * T * (nS + nY)
        res["oos"].append({"nY": nY, "pooled_row_slab_path": bool(mbd_plan(nS + nY)["slab"]),
                           "Y_row_slab_path": bool(mbd_plan(nY, ld)["slab"]) if nY > 1 else None,
                           "median_s": med, "min_s": float(min(ts)), "max_s": float(max(ts)),
                           "depth_evals_per_s": nY / med, "per_new_curve_s": med / nY,
                           "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / med / 1e9,
                           "frac_of_hbm_copy": nbytes / med / 1e9 / peak_gbs,
                           "kernel_ns_engine": eng.timings()["kernel_ns"]})
        print(json.dumps(res["oos"][-1]), flush=True)
        del Xp, out
        torch.cuda.empty_cache()

    # the path it replaces: one sub-population S u {g} per new curve (homogeneity._depths_of_each_in)
    nG = args.batched_nY
    Xh = X[:, :nS + nG].cpu().numpy()
    mem = np.zeros((nG, nS + nG), dtype=np.uint8)
    mem[:, :nS] = 1
    mem[np.arange(nG), nS + np.arange(nG)] = 1
    q = (nS + np.arange(nG, dtype=np.int64))[:, None]
    for _ in range(max(1, args.warmup // 2)):
        eng.band_depth_counts_batched(Xh, mem, q, 2, True)
    kern, wall = [], []
    for _ in range(3):
        t0 = time.perf_counter()
        eng.band_depth_counts_batched(Xh, mem, q, 2, True)
        wall.append(time.perf_counter() - t0)
        kern.append(eng.timings()["kernel_ns"] * 1e-9)
    kmed = float(np.median(kern))
    res["batched"] = {"nY": nG, "reps": 3, "timing": "engine kernel_ns (CUDA events around the call's kernels)",
                      "median_kernel_s": kmed, "per_new_curve_s": kmed / nG, "depth_evals_per_s": nG / kmed,
                      "median_wall_s_with_h2d": float(np.median(wall))}
    print(json.dumps(res["batched"]), flush=True)
    # same answer on the 16 curves
    outd = torch.zeros(nG, dtype=torch.int64, device="cuda")
    Xg = X[:, :nS + nG].contiguous()
    torch.cuda.synchronize()
    eng.band_depth_oos_counts_dev(Xg.data_ptr(), T, nS, nS + nG, Xg.data_ptr() + 8 * nS, nG, nS + nG,
                                  outd.data_ptr(), 2, True)
    res["batched"]["counts_equal_oos"] = bool((outd.cpu().numpy() ==
                                               eng.band_depth_counts_batched(Xh, mem, q, 2, True)[:, 0]).all())
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "depth_of_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"device": res["device"], "batched_equal": res["batched"]["counts_equal_oos"]}))


if __name__ == "__main__":
    main()
