#!/usr/bin/env python
"""Cluster labelling of a lattice split into row strips (StripEngine.cluster_sizes, include/spgg.h:
spgg_strip_clusters), one rank per GPU:

    torchrun --nproc_per_node N scripts/strip_cluster_bench.py [--L 32768] [--out profiles/strip_cluster_bench.json]

With fewer GPUs than ranks the ranks share the GPUs and the records travel through gloo (host-staged);
such a run measures the labelling's overheads, not multi-GPU scaling, and says so in "transport".
States: a random lattice with cooperators at density 0.5 (init_random) and the state after --iterations
iterations of the C4 physics of bench.py.  Per state, CUDA events on every rank around each phase of one
cluster_sizes() call (the calls are synchronous), median over --reps calls after a warm-up call, then the
maximum over the ranks:
  local_ms      spgg_strip_clusters: strip-local labelling + the boundary record
  gather_ms     the all-gather of the records
  resolve_ms    spgg_strip_clusters_resolve: seams, global numbering, this strip's owned sizes
  sizes_ms      the owned sizes to the host and their all-gather (every rank gets the whole array)
  total_ms      the whole call
Rank 0 writes the JSON with the device's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from bench import C4  # noqa: E402
from spgg_b200 import strips  # noqa: E402

PHASES = ("local_ms", "gather_ms", "resolve_ms", "sizes_ms", "total_ms")


def timed_call(se):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ev[0].record()
    rec = se._label_strip("C", False)
    ev[1].record()
    rec = se._gather_records(rec)
    ev[2].record()
    n = se._resolve_records(rec)
    ev[3].record()
    sizes = se._gather_sizes(se._owned_sizes(n))
    ev[4].record()
    ev[4].synchronize()
    t = [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
    return t + [ev[0].elapsed_time(ev[4])], sizes


def measure(se, reps):
    timed_call(se)                                   # warm-up: allocates the scratch
    rows = []
    for _ in range(reps):
        dist.barrier()
        t, sizes = timed_call(se)
        rows.append(t)
    med = torch.tensor(np.median(np.array(rows), axis=0), dtype=torch.float64)
    if not se.host_staged:
        med = med.to(se.dev)
    dist.all_reduce(med, op=dist.ReduceOp.MAX)
    r = dict(zip(PHASES, med.cpu().tolist()))
    r.update(n_clusters=int(len(sizes)), largest=int(sizes.max()) if len(sizes) else 0,
             cooperators=int(sizes.sum()))
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--iterations", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "strip_cluster_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("strip_cluster_bench.py measures the device: no CUDA device")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    ngpu = torch.cuda.device_count()
    local = int(os.environ.get("LOCAL_RANK", rank)) % ngpu
    torch.cuda.set_device(local)
    backend = "nccl" if world <= ngpu else "gloo"
    dist.init_process_group(backend, rank=rank, world_size=world)
    se = strips.StripEngine(dict(C4, L=args.L), seed=2024, precision="fp32", device=local)
    res = {}
    se.init_random(7)
    res["random_p0.5"] = measure(se, args.reps)
    se.init_random(7)
    left = args.iterations
    while left > 0:
        se.step(min(100, left))
        left -= 100
    res[f"c4_after_{args.iterations}"] = measure(se, args.reps)
    se.close()
    if rank == 0:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()
        out = {"device": gpu[0] if gpu else torch.cuda.get_device_name(0), "gpus_visible": ngpu,
               "L": args.L, "ranks": world, "strip_rows": se.rows,
               "transport": (f"NCCL, one GPU per rank" if backend == "nccl" else
                             f"gloo through pinned host memory, {world} ranks sharing {ngpu} GPU(s): "
                             "overheads of the labelling, not a multi-GPU scaling figure"),
               "method": "CUDA events around each phase of StripEngine.cluster_sizes(of='C'), median of --reps "
                         "calls after a warm-up call, maximum over the ranks",
               "results": res}
        print(json.dumps(out), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
