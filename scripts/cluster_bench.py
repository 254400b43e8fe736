#!/usr/bin/env python
"""Cluster labelling on the device (Engine.cluster_sizes / cluster_labels, include/spgg.h: spgg_clusters)
against the host path it replaces (get_state, then scipy.ndimage.label and np.bincount).

    python scripts/cluster_bench.py [--L 1000 4096 ...] [--out profiles/cluster_bench.json]

For each L, on one handle: a random lattice with cooperators at density 0.5 (spgg_init_random; at every L)
and 0.6 (percolating; uploaded with set_state, only for L <= 8192, where the host arrays stay below 3 GB),
and the state after 1000 iterations of the C4 physics of bench.py.  Per state:
  device_us_sizes    CUDA events around cluster_sizes(): the five labelling launches and the copy of n
                     and of the sizes (median of the repetitions, after one warm-up call)
  device_us_labels   the same around cluster_labels(): labelling, label kernel, copy of L*L int32
  host_s             L <= 8192: get_state(want_q=False) + label(S == 0) + bincount, wall clock
The labels of both paths are compared on every state with L <= 8192.  The device's name and power limit are
recorded beside the numbers.
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
from scipy.ndimage import label  # noqa: E402

import spgg_b200  # noqa: E402
from bench import C4  # noqa: E402


def device_us(fn, reps):
    fn()                                   # warm-up (first call also allocates the scratch)
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e3)
    return float(np.median(times)), float(np.min(times))


def measure(eng, L, reps, host):
    r = {}
    sizes = None
    r["device_us_sizes"], r["device_us_sizes_min"] = device_us(lambda: eng.cluster_sizes(), reps)
    r["device_us_labels"], r["device_us_labels_min"] = device_us(lambda: eng.cluster_labels(), max(3, reps // 4))
    sizes = eng.cluster_sizes()
    r["n_clusters"] = int(len(sizes))
    r["largest"] = int(sizes.max()) if len(sizes) else 0
    r["cooperators"] = int(sizes.sum())
    if host:
        t0 = time.perf_counter()
        S = eng.get_state(want_q=False)[0]
        t1 = time.perf_counter()
        lab, n = label(S == 0)
        hs = np.bincount(lab.ravel(), minlength=n + 1)[1:]
        t2 = time.perf_counter()
        r["host_s"] = t2 - t0
        r["host_get_state_s"] = t1 - t0
        r["host_label_bincount_s"] = t2 - t1
        r["speedup_sizes_vs_host"] = r["host_s"] / (r["device_us_sizes"] * 1e-6)
        dl, dn = eng.cluster_labels()
        r["equal_to_scipy"] = bool(n == dn and np.array_equal(hs, sizes) and np.array_equal(lab, dl))
    print(L, json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, nargs="+", default=[1000, 4096, 8192, 16384, 32768])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--iterations", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cluster_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cluster_bench.py measures the device: no CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"device": gpu[0] if gpu else torch.cuda.get_device_name(0),
           "method": "CUDA events on the default stream around one Engine call, median of --reps calls after a "
                     "warm-up call; host path: wall clock of get_state(want_q=False) + scipy.ndimage.label + "
                     "np.bincount on one core",
           "results": {}}
    for L in args.L:
        res = {}
        host = L <= 8192
        try:
            eng = spgg_b200.Engine(dict(C4, L=L), seeds=1, precision="fp32")
        except (RuntimeError, ValueError) as e:
            out["results"][str(L)] = {"error": str(e)}
            continue
        try:
            eng.init_random(7)
            res["random_p0.5"] = measure(eng, L, args.reps, host)
            if L <= 8192:
                rs = np.random.RandomState(L)
                S = (rs.rand(L, L) >= 0.6).astype(np.uint8)
                eng.set_state(S, np.zeros((L, L)), np.zeros((L, L, 2, 2)))
                del S
                res["random_p0.6"] = measure(eng, L, args.reps, host)
            eng.init_random(7)
            eng.step(args.iterations)
            res[f"c4_after_{args.iterations}"] = measure(eng, L, args.reps, host)
        except (RuntimeError, ValueError) as e:
            res["error"] = str(e)
        finally:
            eng.close()
        out["results"][str(L)] = res
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
