"""cfg2 step (100k curves x 1024 rows, HBM-resident) under several settings of the K1 rank path, one process:
    python profiles/slab_probe.py [config ...]     config = name:ENV=VAL,ENV=VAL
Prints ms per step (CUDA events on the engine's stream, L2 flushed between steps), the per-phase device times and
whether the counts equal the part pipeline's.
    PROBE_TRACE=out.json python profiles/slab_probe.py
instead traces PROBE_STEPS default steps with torch.profiler (phase events off) and writes, per step, every device
activity on the engine's stream in order with its duration and the idle gap before it, plus their medians."""
import os, sys, json, statistics
sys.path.insert(0, '.')
import torch
from statdepth_b200 import _engine as E

n, T = 100_000, int(os.environ.get("PROBE_T", "1024"))
steps = int(os.environ.get("PROBE_STEPS", "10"))
eng = E.get_engine(0)
eng.set_option(E.OPT_PROFILE, 1)
dev = torch.device("cuda", 0)
stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
g = torch.Generator(device=dev); g.manual_seed(1)
X = torch.empty((T, n), dtype=torch.float64, device=dev)
for r0 in range(0, T, 128):
    X[r0:r0 + 128] = torch.randn((min(128, T - r0), n), dtype=torch.float64, device=dev, generator=g)
X = X.cumsum(0)
if os.environ.get("PROBE_TIES"):
    X = X.round()
out = torch.zeros(n, dtype=torch.int64, device=dev)


def trace(path):
    """Per-step device activities of the engine's stream (kernels, memsets, copies) from a torch.profiler trace."""
    from torch.profiler import profile, ProfilerActivity
    eng.set_option(E.OPT_PROFILE, 0)
    for _ in range(3):
        eng.band_depth_counts_dev(X.data_ptr(), T, n, n, out.data_ptr(), None, n, 2, True)
    torch.cuda.synchronize()
    raw = path + ".chrome.json"
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            flush.fill_(1)  # on torch's stream: marks the step boundary in the trace
            torch.cuda.synchronize()
            eng.band_depth_counts_dev(X.data_ptr(), T, n, n, out.data_ptr(), None, n, 2, True)
            torch.cuda.synchronize()
    prof.export_chrome_trace(raw)
    with open(raw) as f:
        evs = json.load(f)["traceEvents"]
    os.remove(raw)
    dev_ev = sorted((e for e in evs if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")),
                    key=lambda e: e["ts"])
    step_list, cur = [], None
    for e in dev_ev:
        if "fill" in e["name"].lower() or "Fill" in e["name"]:
            cur = []
            step_list.append(cur)
            continue
        if cur is not None:
            cur.append(e)
    rows = []
    for acts in step_list:
        if not acts:
            continue
        row, prev_end = [], None
        for e in acts:
            row.append({"name": e["name"][:60], "cat": e["cat"], "us": e["dur"],
                        "gap_before_us": None if prev_end is None else e["ts"] - prev_end})
            prev_end = e["ts"] + e["dur"]
        rows.append({"span_us": prev_end - acts[0]["ts"], "busy_us": sum(e["dur"] for e in acts), "acts": row})
    med = {"span_us": statistics.median(r["span_us"] for r in rows),
           "busy_us": statistics.median(r["busy_us"] for r in rows),
           "acts": [{"name": a["name"], "us": statistics.median(r["acts"][i]["us"] for r in rows),
                     "gap_before_us": None if i == 0 else statistics.median(r["acts"][i]["gap_before_us"] for r in rows)}
                    for i, a in enumerate(rows[0]["acts"]) if all(len(r["acts"]) == len(rows[0]["acts"]) for r in rows)]}
    res = {"T": T, "n": n, "steps": len(rows), "gpu": torch.cuda.get_device_name(0), "median": med, "per_step": rows}
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"trace": path, "median": med}), flush=True)


if os.environ.get("PROBE_TRACE"):
    trace(os.environ["PROBE_TRACE"])
    sys.exit(0)
configs = sys.argv[1:] or ["parts:SD_MBD_PATH=parts", "slab:"]
ref = None
KEYS = ("SD_MBD_PATH", "SD_MBD_SLAB_G", "SD_MBD_SLAB_THREADS", "SD_MBD_SLAB_MIN", "SD_MBD_SLAB_HIST_THREADS")
for cfg in configs:
    name, _, envs = cfg.partition(":")
    for k in KEYS:
        os.environ.pop(k, None)
    for kv in filter(None, envs.split(",")):
        k, v = kv.split("=")
        os.environ[k] = v
    for _ in range(3):
        eng.band_depth_counts_dev(X.data_ptr(), T, n, n, out.data_ptr(), None, n, 2, True)
    torch.cuda.synchronize()
    ms, phases, launches = 0.0, {}, 0
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.band_depth_counts_dev(X.data_ptr(), T, n, n, out.data_ptr(), None, n, 2, True)
        e1.record(stream)
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        tm = eng.timings()
        launches = tm["launches"]
        for k, v in eng.phase_ns().items():
            phases[k] = phases.get(k, 0) + v
    res = out.clone()
    same = None if ref is None else bool((res == ref).all().item())
    if ref is None:
        ref = res
    print(json.dumps({"config": name, "env": envs, "ms_per_step": ms / steps, "Mdepth_evals_per_s": n / (ms / steps) / 1e3,
                      "phases_ms": {k: v / steps / 1e6 for k, v in phases.items() if v}, "launches": launches,
                      "fallback_rows": tm["fallback_rows"], "equals_first_config": same,
                      "checksum": int(res.sum().item())}), flush=True)
