#!/usr/bin/env python
"""State overlaps on the device (Engine.snapshot / Engine.overlap, include/spgg.h: spgg_snapshot / spgg_overlap)
against the host path they replace (two get_state calls and a NumPy diff).

    python scripts/overlap_bench.py [--L 1000 4096 16384 32768] [--out profiles/overlap_bench.json]

For each L, on one handle (fp32 Q, int8 R): a snapshot of the fresh state (spgg_init_random), then 200 iterations,
then:
  snapshot     call_ms of one snapshot of S, R and Q (CUDA events, median after a warm-up) and GB/s over its byte
               model: the planes read once and written once, 2 x (L^2 / 8 + L^2 elem_R + nq L^2 elem_Q)
  S, S+R, S+R+Q   the overlap call with those fields:
    call_ms      CUDA events on the default stream around one call (kernels, the result copy), median
    kernel_ms    the device time of the k_overlap* kernels of one call, from torch.profiler in a separate pass
    bytes        the byte model: two copies of the planes read, 2 x (L^2 / 8 [+ L^2 elem_R] [+ nq L^2 elem_Q])
    GBps, hbm_share   bytes over kernel_ms, and that rate over the 6547.5 GB/s the project measured for HBM
  host_s       L <= 4096: two get_state calls + the NumPy counts, changed counts, max and sums, one core
The working set of L <= 4096 (<= 575 MB with R and Q) is partly served from the 126 MB L2 after the warm-up; at L >=
16384 it is 9.2 GB and more, read from HBM.  The device's name and power limit are read in the same run.
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
CASES = {"S": (), "S+R": ("R",), "S+R+Q": ("R", "Q")}


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
        if "k_overlap" in e.name:
            key = e.name.split("<")[0].split("(")[0].replace("void ", "")
            per[key] = per.get(key, 0.0) + e.device_time / 1000.0 / reps
    return sum(per.values()), per


def plane_bytes(L, fields, nq=4, elem_r=1, elem_q=4):
    return L * L * (1 / 8 + (elem_r if "R" in fields else 0) + (nq * elem_q if "Q" in fields else 0))


def host_path(eng, fields):
    """two get_state calls (the state at the snapshot and now; the same handle serves both here) + NumPy"""
    t0 = time.perf_counter()
    then = eng.get_state(want_q="Q" in fields)
    now = eng.get_state(want_q="Q" in fields)
    S0, S1 = then[0].ravel(), now[0].ravel()
    counts = [[np.count_nonzero((S0 == a) & (S1 == b)) for b in (0, 1)] for a in (0, 1)]
    chans = ([(now[1].ravel(), then[1].ravel())] if "R" in fields else []) + \
            ([(now[2].reshape(-1, 4)[:, z], then[2].reshape(-1, 4)[:, z]) for z in range(4)] if "Q" in fields else [])
    out = []
    for a, b in chans:
        d = a - b
        ad = np.abs(d)
        out.append((np.count_nonzero(a != b), ad.max(), ad.sum(), (d * d).sum()))
    return time.perf_counter() - t0, counts, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, nargs="+", default=[1000, 4096, 16384, 32768])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "overlap_bench.json"))
    args = ap.parse_args()
    res = {"device": gpu_info(),
           "method": "call_ms: CUDA events around one Engine call (median after a warm-up); kernel_ms: "
                     "torch.profiler device time of the k_overlap* kernels per call; bytes from the byte model; "
                     f"hbm_share = GB/s over the measured {HBM_GBPS} GB/s; host: two get_state calls + NumPy",
           "results": {}}
    for L in args.L:
        eng = spgg_b200.Engine(dict(C4, L=L), seeds=1, precision="fp32")
        eng.init_random(7)
        reps = args.reps if L <= 16384 else max(3, args.reps // 2)
        rl = {}
        nb = 2 * plane_bytes(L, ("R", "Q"))
        med, mn = call_ms(lambda: eng.snapshot(1), reps)
        rl["snapshot"] = {"call_ms": med, "call_ms_min": mn, "bytes": nb, "GBps": nb / med / 1e6,
                          "hbm_share": nb / med / 1e6 / HBM_GBPS}
        print(L, "snapshot", json.dumps(rl["snapshot"]), flush=True)
        eng.drop_snapshot(1)
        eng.snapshot(0)
        eng.step(200)
        eng.status()
        for name, fields in CASES.items():
            def fn():
                return eng.overlap(0, fields=fields)
            med, mn = call_ms(fn, reps)
            kms, per = kernel_ms(fn, reps)
            nbytes = 2 * plane_bytes(L, fields)
            r = {"call_ms": med, "call_ms_min": mn, "kernel_ms": kms, "kernels_ms": per, "bytes": nbytes,
                 "GBps": nbytes / kms / 1e6 if kms else None,
                 "hbm_share": nbytes / kms / 1e6 / HBM_GBPS if kms else None}
            if L <= 4096:
                hs, _, _ = host_path(eng, fields)
                r["host_s"] = hs
            else:
                r["host_s"] = "not measured"
            rl[name] = r
            print(L, name, json.dumps({k: v for k, v in r.items() if k != "kernels_ms"}), flush=True)
        eng.close()
        res["results"][str(L)] = rl
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
