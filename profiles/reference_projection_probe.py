"""Fitted references for projection and random Tukey depth (K13): build time of the projected index and query time of
new observations, beside the in-sample call on S + [g] that scores one new observation without a reference.

    python profiles/reference_projection_probe.py [OUT_DIR] [--reps 10] [--warmup 2]

Three sizes, everything resident on the device, times from CUDA events on the engine's stream (median of --reps after
--warmup):
  univariate   S = 100 000 random-walk curves x 1024 points (K9's index), n_Y = 1, 1 000, 10 000;
  curves       S = 5 000 curves x 256 points x 3 channels, K = 200, n_Y = 1, 100, 1 000;
  cloud        S = 50 000 points x 8, K = 1 000, n_Y = 1 000.
Per size: the build (sd_band_sort_rows / sd_projection_sort_rows), each query (Tukey and outlyingness), and the
in-sample Tukey and outlyingness calls on the pooled S + [g] (device input; what scoring ONE new observation costs
today).  The index and the samples are larger than the 126 MB L2 except the cloud's sample.  Writes
OUT_DIR/reference_projection_probe.json (default profiles/) with the card name, power limit and max SM clock read in
the same run.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))


def summary(ts):
    return {"median_ms": float(np.median(ts)) * 1e3, "min_ms": float(min(ts)) * 1e3, "max_ms": float(max(ts)) * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir", nargs="?", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch

    from depth_of_probe import device_info, event_times
    from statdepth_b200._engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("reference_projection_probe needs a GPU")
    eng = get_engine(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    rng = np.random.default_rng(0)

    def times(fn):
        return summary(event_times(fn, args.reps, args.warmup, stream))

    def on_dev(A):
        t = torch.from_numpy(np.ascontiguousarray(A, dtype=np.float64)).to(dev)
        torch.cuda.synchronize()
        return t

    out = {"device": device_info(), "reps": args.reps, "warmup": args.warmup}

    # univariate: K9's sorted rows
    T, nS = 1024, 100_000
    X = rng.standard_normal((T, nS)).cumsum(0)
    dX = on_dev(X)
    index = torch.empty((T, nS), dtype=torch.float64, device=dev)
    res = {"shape": "%d curves x %d points" % (nS, T),
           "build_ms": times(lambda: eng.band_sort_rows_dev(dX.data_ptr(), T, nS, nS, index.data_ptr()))}
    pool = torch.empty((T, nS + 1), dtype=torch.float64, device=dev)
    pool[:, :nS] = dX
    del dX
    pc = torch.empty(nS + 1, dtype=torch.int64, device=dev)
    po = torch.empty((T, nS + 1), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    res["in_sample_one_new_curve"] = {
        "tukey_ms": times(lambda: eng.band_halfspace_counts_dev(pool.data_ptr(), T, nS + 1, nS + 1, pc.data_ptr())),
        "outlyingness_ms": times(lambda: eng.band_outlyingness_dev(pool.data_ptr(), T, nS + 1, nS + 1,
                                                                   po.data_ptr()))}
    del pool, po
    for nY in (1, 1000, 10_000):
        dY = on_dev(rng.standard_normal((T, nY)).cumsum(0))
        c = torch.empty(nY, dtype=torch.int64, device=dev)
        o = torch.empty((T, nY), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        res["query_nY_%d" % nY] = {
            "tukey_ms": times(lambda: eng.band_halfspace_sorted_counts_dev(index.data_ptr(), T, nS, dY.data_ptr(),
                                                                           nY, nY, c.data_ptr())),
            "outlyingness_ms": times(lambda: eng.band_outlyingness_sorted_dev(index.data_ptr(), T, nS, dY.data_ptr(),
                                                                              nY, nY, o.data_ptr()))}
    out["univariate"] = res
    del index
    torch.cuda.empty_cache()

    def projected(name, nS, T, d, K, nYs, walk):
        S = rng.standard_normal((nS, T, d))
        if walk:
            S = S.cumsum(1)
        U = rng.standard_normal((K, d))
        U /= np.linalg.norm(U, axis=1, keepdims=True)
        dS = on_dev(S)
        index = torch.empty((T, K, nS), dtype=torch.float64, device=dev)
        res = {"shape": "%d x %d x %d, K = %d" % (nS, T, d, K), "index_GB": T * K * nS * 8 / 1e9,
               "build_ms": times(lambda: eng.projection_sort_rows_dev(dS.data_ptr(), nS, T, d, U,
                                                                      index.data_ptr()))}
        pool = torch.empty((nS + 1, T, d), dtype=torch.float64, device=dev)
        pool[:nS] = dS
        del dS
        pc = torch.empty(nS + 1, dtype=torch.int64, device=dev)
        po = torch.empty((T, nS + 1), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        res["in_sample_one_new_curve"] = {
            "tukey_ms": times(lambda: eng.projection_tukey_counts_dev(pool.data_ptr(), nS + 1, T, d, U,
                                                                      pc.data_ptr())),
            "outlyingness_ms": times(lambda: eng.projection_outlyingness_dev(pool.data_ptr(), nS + 1, T, d, U,
                                                                             po.data_ptr()))}
        del pool, po
        for nY in nYs:
            Fn = rng.standard_normal((nY, T, d))
            dY = on_dev(Fn.cumsum(1) if walk else Fn)
            c = torch.empty(nY, dtype=torch.int64, device=dev)
            o = torch.empty((T, nY), dtype=torch.float64, device=dev)
            torch.cuda.synchronize()
            res["query_nY_%d" % nY] = {
                "tukey_ms": times(lambda: eng.projection_tukey_sorted_counts_dev(index.data_ptr(), nS, T,
                                                                                 dY.data_ptr(), nY, d, U,
                                                                                 c.data_ptr())),
                "outlyingness_ms": times(lambda: eng.projection_outlyingness_sorted_dev(index.data_ptr(), nS, T,
                                                                                        dY.data_ptr(), nY, d, U,
                                                                                        o.data_ptr()))}
        del index
        torch.cuda.empty_cache()
        out[name] = res

    projected("curves", 5000, 256, 3, 200, (1, 100, 1000), True)
    projected("cloud", 50_000, 1, 8, 1000, (1000,), False)
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "reference_projection_probe.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
