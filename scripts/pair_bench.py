#!/usr/bin/env python
"""Strategy pair counts on the device (Engine.pair_counts, include/spgg.h: spgg_pair_counts) against the host
path it replaces (get_state, then one np.roll + compare + count per offset and axis).

    python scripts/pair_bench.py [--L 1000 4096 16384 32768] [--out profiles/pair_bench.json]

For each L, on one handle holding a random lattice (spgg_init_random, cooperators at density 0.5) and each
max_d in {1, 64, L/2}:
  device_ms       CUDA events on the default stream around one pair_counts(max_d) call (both axes, every
                  offset 0..max_d, the copy of the counts), median of the repetitions after a warm-up call
  word_ops_per_s  2 axes x L^2/32 words x (max_d + 1) offsets over device_ms: evaluated 32-site word pairs
  host_s          L <= 4096 and max_d <= 64 (and L/2 at L = 1000): get_state of S alone + the NumPy loop on
                  one core, wall clock; larger host runs take minutes and are "not measured"
The device counts are compared with the host counts wherever both are measured.  With two or more GPUs the
script also runs itself under torchrun (--strips) and times StripEngine.pair_counts with one strip per GPU.
The device's name and power limit are read in the same run and recorded beside the numbers.
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


def device_ms(fn, reps):
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


def host_counts(S, max_d):
    """the NumPy path a user has without the device counts (same layout as pair_counts)"""
    c = S == 0
    out = np.zeros((2, max_d + 1, 2), np.int64)
    for ax in (0, 1):
        out[ax, 0, 0] = np.count_nonzero(c)
        for d in range(1, max_d + 1):
            p = np.roll(c, -d, axis=ax)
            out[ax, d] = (np.count_nonzero(c & p), np.count_nonzero(c != p))
    return out


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def single(args):
    out = {"device": gpu_info(),
           "method": "CUDA events on the default stream around one Engine.pair_counts call, median of the "
                     "repetitions after a warm-up call; host path: wall clock of spgg_get_state (S only) + "
                     "np.roll / compare / count_nonzero per offset and axis on one core",
           "results": {}}
    for L in args.L:
        res = {}
        eng = spgg_b200.Engine(dict(C4, L=L), seeds=1, precision="fp32")
        try:
            eng.init_random(7)
            S = None
            for md in sorted({1, 64, L // 2}):
                reps = args.reps if L * L * md < 2 ** 36 else 3
                med, mn = device_ms(lambda: eng.pair_counts(md), reps)
                r = {"device_ms": med, "device_ms_min": mn, "reps": reps,
                     "word_ops_per_s": 2 * L * L / 32 * (md + 1) / (med * 1e-3)}
                if L <= 4096 and (md <= 64 or L <= 1000):
                    t0 = time.perf_counter()
                    S = np.empty(L * L, np.uint8)
                    spgg_b200.load().spgg_get_state(eng._h, 0, S.ctypes.data, None, None)
                    S = S.reshape(L, L)
                    t1 = time.perf_counter()
                    want = host_counts(S, md)
                    t2 = time.perf_counter()
                    r.update(host_s=t2 - t0, host_get_state_s=t1 - t0, host_numpy_s=t2 - t1,
                             speedup_vs_host=(t2 - t0) / (med * 1e-3),
                             equal_to_numpy=bool(np.array_equal(want, eng.pair_counts(md))))
                else:
                    r["host_s"] = "not measured"
                res[f"max_d={md}"] = r
                print(L, md, json.dumps(r), flush=True)
        finally:
            eng.close()
        out["results"][str(L)] = res
        torch.cuda.empty_cache()
    n = torch.cuda.device_count()
    if n >= 2 and not args.no_strips:
        tmp = os.path.join(os.path.dirname(os.path.abspath(args.out)), "pair_bench_strips.json")
        subprocess.run([sys.executable, "-m", "torch.distributed.run", f"--nproc_per_node={n}", os.path.abspath(__file__),
                        "--strips", "--L", str(max(args.L)), "--reps", str(args.reps), "--out", tmp], check=True)
        with open(tmp) as f:
            out["strips"] = json.load(f)
        os.remove(tmp)
    else:
        out["strips"] = f"not measured ({n} GPU)"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


def strips_main(args):
    """under torchrun, one strip per GPU: StripEngine.pair_counts (record, NCCL all-gather, counts, all-reduce)"""
    import torch.distributed as dist
    from spgg_b200 import strips
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl")
    L = args.L[0]
    se = strips.StripEngine(dict(C4, L=L), seed=1, precision="fp32")
    se.init_random(7)
    res = {"world": world, "L": L, "device": gpu_info()}
    for md in (1, 64, L // 2):
        dist.barrier()
        t = []
        for i in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            se.pair_counts(md)
            torch.cuda.synchronize()
            if i:
                t.append((time.perf_counter() - t0) * 1e3)
        res[f"max_d={md}"] = {"call_ms_median": float(np.median(t)), "method": "host clock around the call "
                              "(it ends in a synchronising copy), median of 3 after a warm-up call"}
    se.close()
    if rank == 0:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, nargs="+", default=[1000, 4096, 16384, 32768])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--strips", action="store_true", help="(internal) the torchrun worker")
    ap.add_argument("--no-strips", action="store_true", help="skip the strip run on a multi-GPU box")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pair_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pair_bench.py measures the device: no CUDA device")
    if args.strips:
        strips_main(args)
    else:
        single(args)


if __name__ == "__main__":
    main()
