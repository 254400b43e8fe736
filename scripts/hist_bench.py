#!/usr/bin/env python
"""Value distributions on the device (Engine.histograms / Engine.value_ranges, include/spgg.h: spgg_histograms /
spgg_value_ranges) against the host path they replace (get_state, then np.histogram per channel and class).

    python scripts/hist_bench.py [--L 1000 4096 16384 32768] [--out profiles/hist_bench.json]

For each L, on one handle (fp32 Q, int8 R) in two states, "contended" (fresh from spgg_init_random: R = 0 on every
site, so all sites share one R bin) and "spread" (after 200 iterations), and for each case: the R histograms, the
R and Q histograms, the same with the greedy-policy counts, at 20 and 1024 bins, and the value_ranges call:
  call_ms      CUDA events on the default stream around one call with explicit ranges (kernels, the copies of
               edges and counts, the host checks), median of the repetitions after a warm-up
  kernel_ms    the device time of the k_hist* kernels of one call, from torch.profiler in a separate pass
  bytes        the byte model: L^2 / 8 for the bit plane + L^2 elem_R + nq L^2 elem_Q for the planes read
  GBps, hbm_share   bytes over kernel_ms, and that rate over the 6547.5 GB/s the project measured for HBM
  host_s       L <= 4096: get_state + np.histogram of every channel and class, wall clock, one core
The working set of L <= 4096 (<= 285 MB) is partly served from the 126 MB L2 after the warm-up; at L >= 16384 it is
4.6 GB and more, read from HBM.  The device's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import spgg_b200  # noqa: E402
from bench import C4  # noqa: E402

HBM_GBPS = 6547.5
RANGES = {"R": (-10.0, 10.0), "Q": (-1.0, 1.0)}
# name -> (method, fields, policy)
CASES = {"R": ("histograms", ("R",), False), "RQ": ("histograms", ("R", "Q"), False),
         "RQ+policy": ("histograms", ("R", "Q"), True), "ranges": ("value_ranges", ("R", "Q"), False)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def call_ms(fn, reps):
    fn()                                   # warm-up (the first call also allocates the scratch)
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def kernel_ms(fn, reps):
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if "k_hist" in e.name:
            key = e.name.split("<")[0].split("(")[0].replace("void ", "")
            per[key] = per.get(key, 0.0) + e.device_time / 1000.0 / reps
    return sum(per.values()), per


def byte_model(L, fields, nq=4, elem_r=1, elem_q=4):
    return L * L * (1 / 8 + (elem_r if "R" in fields else 0) + (nq * elem_q if "Q" in fields else 0))


def host_path(eng, bins, fields):
    t0 = time.perf_counter()
    S, R, Q = eng.get_state(want_q="Q" in fields)
    coop = (S == 0).ravel()
    chans = ([R.ravel()] if "R" in fields else []) + ([Q.reshape(-1, 4)[:, z] for z in range(4)] if "Q" in fields else [])
    out = []
    for x, f in zip(chans, (["R"] if "R" in fields else []) + ["Q"] * 4):
        out.append([np.histogram(x, bins, RANGES[f])[0], np.histogram(x[coop], bins, RANGES[f])[0]])
    return time.perf_counter() - t0, np.array(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, nargs="+", default=[1000, 4096, 16384, 32768])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hist_bench.json"))
    args = ap.parse_args()
    res = {"device": gpu_info(),
           "method": "call_ms: CUDA events around one Engine call with explicit ranges (median after a warm-up); "
                     "kernel_ms: torch.profiler device time of the k_hist* kernels per call; bytes from the byte "
                     f"model; hbm_share = GB/s over the measured {HBM_GBPS} GB/s; host: get_state + np.histogram",
           "results": {}}
    for L in args.L:
        eng = spgg_b200.Engine(dict(C4, L=L), seeds=1, precision="fp32")
        eng.init_random(7)
        rl = {}
        for state in ("contended", "spread"):
            if state == "spread":
                eng.step(200)
                eng.status()
            for name, (method, fields, pol) in CASES.items():
                for bins in ((20, 1024) if method == "histograms" else (None,)):
                    if method == "histograms":
                        def fn():
                            return eng.histograms(bins, fields=fields, ranges=RANGES, policy=pol)
                    else:
                        def fn():
                            return eng.value_ranges(fields=fields)
                    reps = args.reps if L <= 16384 else max(3, args.reps // 2)
                    med, mn = call_ms(fn, reps)
                    kms, per = kernel_ms(fn, reps)
                    nbytes = byte_model(L, fields)
                    r = {"call_ms": med, "call_ms_min": mn, "kernel_ms": kms, "kernels_ms": per, "bytes": nbytes,
                         "GBps": nbytes / kms / 1e6 if kms else None,
                         "hbm_share": nbytes / kms / 1e6 / HBM_GBPS if kms else None}
                    if L <= 4096 and method == "histograms":
                        hs, want = host_path(eng, bins, fields)
                        got = fn()
                        packed = ([got["R"][None]] if "R" in fields else []) + \
                                 ([np.moveaxis(got["Q"].reshape(2, 4, bins), 0, 1)] if "Q" in fields else [])
                        assert np.array_equal(np.concatenate(packed), want), (L, state, name, bins)
                        r["host_s"] = hs
                    else:
                        r["host_s"] = "not measured"
                    key = f"{state},{name}" + (f",bins={bins}" if bins else "")
                    rl[key] = r
                    print(L, key, json.dumps({k: v for k, v in r.items() if k != "kernels_ms"}), flush=True)
        eng.close()
        res["results"][str(L)] = rl
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
