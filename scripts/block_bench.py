#!/usr/bin/env python
"""Block fields on the device (Engine.block_fields, include/spgg.h: spgg_block_fields) against the host path it
replaces (get_state, then a NumPy reshape-sum per block).

    python scripts/block_bench.py [--L 1000 4096 16384 32768] [--out profiles/block_bench.json]

For each L, on one handle holding a random lattice (spgg_init_random, fp32 Q, int8 R), each b in {8, 32, 256, L}
and each field set (counts only, + R, + R + Q):
  call_ms      CUDA events on the default stream around one block_fields call (kernels, the copy of the result
               to pageable host memory and the host's fill-in of n), median of the repetitions after a warm-up
  kernel_ms    the device time of the k_block_* kernels of one call, from torch.profiler in a separate pass
  bytes        the byte model: L^2 / 8 for the bit plane, + L^2 for int8 R, + 16 L^2 for fp32 Q
  GBps, hbm_share   bytes over kernel_ms, and that rate over the 6547.5 GB/s the project measured for HBM
  host_s       L <= 4096: get_state of what the field set needs + the NumPy reshape-sum, wall clock, one core
The working set of L <= 4096 (<= 288 MB with Q) is partly served from the 126 MB L2 after the warm-up; at
L >= 16384 it is 4.6 GB and more, read from HBM.  The device's name and power limit are read in the same run.
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
FIELD_SETS = {"counts": (), "R": ("R",), "RQ": ("R", "Q")}


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
        if e.name.startswith("void spgg::k_block") or e.name.startswith("spgg::k_block") or "k_block_" in e.name:
            key = e.name.split("<")[0].split("(")[0].replace("void ", "")
            per[key] = per.get(key, 0.0) + e.device_time / 1000.0 / reps
    return sum(per.values()), per


def byte_model(L, fields):
    return L * L * (1 / 8 + (1 if "R" in fields else 0) + (16 if "Q" in fields else 0))


def host_path(eng, L, b, fields):
    t0 = time.perf_counter()
    S, R, Q = eng.get_state(want_q="Q" in fields)
    B = -(-L // b)
    pad = B * b - L

    def bsum(x):
        x = np.pad(x, ((0, pad), (0, pad)) + ((0, 0),) * (x.ndim - 2))
        return x.reshape((B, b, B, b) + x.shape[2:]).sum(axis=(1, 3))

    c = (S == 0)
    out = {"n_C": bsum(c.astype(np.int64))}
    if "R" in fields:
        out["R"] = np.stack([bsum(R), bsum(np.where(c, R, 0.0))], 2)
    if "Q" in fields:
        out["Q"] = np.stack([bsum(Q), bsum(np.where(c[..., None, None], Q, 0.0))], 2)
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, nargs="+", default=[1000, 4096, 16384, 32768])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "block_bench.json"))
    args = ap.parse_args()
    res = {"device": gpu_info(),
           "method": "call_ms: CUDA events around one Engine.block_fields call (median after a warm-up); kernel_ms: "
                     "torch.profiler device time of the k_block_* kernels per call; bytes from the byte model; "
                     f"hbm_share = GB/s over the measured {HBM_GBPS} GB/s; host: get_state + NumPy reshape-sum",
           "results": {}}
    for L in args.L:
        eng = spgg_b200.Engine(dict(C4, L=L), seeds=1, precision="fp32")
        eng.init_random(7)
        rl = {}
        for b in sorted({8, 32, 256, L}):
            if (-(-L // b)) ** 2 > 1 << 24:
                continue
            for name, fields in FIELD_SETS.items():
                reps = args.reps if L <= 16384 else max(3, args.reps // 2)
                med, mn = call_ms(lambda: eng.block_fields(b, fields=fields), reps)
                kms, per = kernel_ms(lambda: eng.block_fields(b, fields=fields), reps)
                nbytes = byte_model(L, fields)
                r = {"call_ms": med, "call_ms_min": mn, "kernel_ms": kms, "kernels_ms": per, "bytes": nbytes,
                     "GBps": nbytes / kms / 1e6 if kms else None,
                     "hbm_share": nbytes / kms / 1e6 / HBM_GBPS if kms else None}
                if L <= 4096:
                    hs, want = host_path(eng, L, b, fields)
                    got = eng.block_fields(b, fields=fields)
                    assert np.array_equal(got["n_C"], want["n_C"]), (L, b, name)
                    if "R" in fields:
                        assert np.array_equal(got["R"], want["R"]), (L, b, name)
                    if "Q" in fields:
                        assert np.allclose(got["Q"], want["Q"], rtol=1e-9, atol=1e-12), (L, b, name)
                    r["host_s"] = hs
                else:
                    r["host_s"] = "not measured"
                rl[f"b={b},{name}"] = r
                print(L, b, name, json.dumps({k: v for k, v in r.items() if k != "kernels_ms"}), flush=True)
        eng.close()
        res["results"][str(L)] = rl
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
