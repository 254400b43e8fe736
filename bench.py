#!/usr/bin/env python
"""Benchmark of the SPGG lattice step (BASELINE.json metric: site-updates/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A bench "step" is one chunk of ``--inner`` lattice iterations (default 100) of the whole
L x L lattice through ``spgg_step`` (statistics on).  N=1 runs BASELINE config 4
(L=4096, reputation state, M=1, r=3, kappa=1, w_P=0.95, fp32 throughput mode).
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_SITE_FP32 = 34.25   # BASELINE.md section 3: Q 16r+16w, R int8 1r+1w, S bit 1/8r+1/8w
C4 = dict(r=3.0, c=1, cost=1, alpha=0.8, gamma=0.9, epsilon=0.5, epsilon_decay=0.99,
          epsilon_min=0.01, influence_factor=1.0, use_second_order=False, lambda_epsilon=0.01,
          delta_R_C=1, delta_R_D=1, R_min=-10, R_max=10, reward_weight_payoff=0.95,
          rep_gain_C=1.0, state_representation="reputation")


def ncu_traffic(L):
    """DRAM bytes per k_step launch from the committed `ncu --set full` capture
    (profiles/k_step_traffic.json, written by scripts/make_profile_summary.py), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "k_step_traffic.json")) as f:
            d = json.load(f)
        return float(d["traffic_bytes_per_launch"]) if int(d.get("L", 0)) == int(L) else None
    except Exception:
        return None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def c4_config(L, inner):
    """`config` of the N=1 line (both arms print the same one)."""
    return {"workload": f"C4: single lattice L={L}, reputation state, M=1, r=3, kappa=1, "
                        f"w_P=0.95, Q-learning; {inner} iterations per bench step, "
                        "statistics on, Philox draws",
            "L": L, "iterations_per_step": inner, "precision": "fp32 Q (float4) + int8 R + bit S",
            "l2": f"state {state_bytes_dev(L) / 1e6:.0f} MB per pass > 126 MB L2 (no flush needed)",
            "e2e_def": "SPGG C-ABI with host buffers: ONE set_state (H2D of uint8 S, f64 R, f64 Q) + "
                       "K chunks with the stat rows read back each chunk + ONE get_state (D2H), all "
                       "inside the timed region; the simulation is device-resident, so the state "
                       "transfers are amortised over the K x iterations_per_step iterations of the run"}


def c5_config(L, world, inner):
    """`config` of the N > 1 line (both arms print the same one)."""
    return {"workload": f"C5: one L={L} lattice in {world} row strips, reputation state, M=1, r=3, kappa=1, "
                        f"w_P=0.95, Q-learning; {inner} iterations per bench step, per iteration the two boundary "
                        "rows of every strip reach its neighbours' ghost rows and the strips' 4-float reports (global "
                        "reward-difference maximum, uniform-lattice test) are max-combined - through peer-mapped memory "
                        "over NVLink where the planes can be mapped, NCCL send/recv + all-reduce otherwise "
                        "(extras.transport of the native line says which); statistics on, Philox draws",
            "L": L, "iterations_per_step": inner, "n_strips": world,
            "precision": "fp32 Q (float4) + int8 R + bit S",
            "l2": "per-GPU state far larger than the 126 MB L2 (no flush needed)",
            "scaling_note": "strong scaling over N>=2 at fixed L; N=1 runs config 4 (L=4096) and reports the "
                            "one-GPU L=32768 iteration under extras.scaling_anchor"}


def reference_root():
    """The unmodified reference: /root/reference in the build container, oracle/_ref (shipped by
    oracle/fetch_ref.py) on the GPU box, else None."""
    from oracle import fetch_ref
    return fetch_ref.reference_root()


def cpu_reference(L, n_warm, n_timed):
    """The UNMODIFIED reference (`SPGG.run`, NumPy, one process: its ops are single-threaded)
    timed on this host; h5py / matplotlib stubbed (absent from the image), `label` neutralised
    for L > 1000 (BASELINE.md section 4).  Returns (site-updates/s, seconds per iteration)."""
    from oracle import ref_harness
    sec, _iv = ref_harness.time_reference(n_warm, n_timed, seed=0, L=L, **C4)
    return L * L / sec, sec


def cpu_port(L, iters, seed=0):
    """Fallback when no copy of the reference is present: its NumPy path restated
    (oracle/spgg_numpy.py, pinned bit-exact to the reference).  Returns (site-updates/s, s)."""
    from oracle import spgg_numpy
    p = dict(C4, L=L, iterations=iters)
    rs = np.random.RandomState(seed)
    Q = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
    S = rs.randint(0, 2, (L, L)).astype(np.int64)
    R = np.zeros((L, L))
    eps = p["epsilon"]
    t0 = time.perf_counter()
    for _ in range(iters):
        u = rs.rand(L, L)
        b = rs.randint(0, 2, (L, L))
        S, R, Q, _st = spgg_numpy.qlearning_step(S, R, Q, eps, u, b, p)
        eps = max(eps * p["epsilon_decay"], p["epsilon_min"])
    dt = time.perf_counter() - t0
    return L * L * iters / dt, dt / iters


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host
    cores - the UNMODIFIED reference tree (oracle/_ref, shipped by oracle/fetch_ref.py) run
    through its public `SPGG(**params).run(h5)`; when no copy is present, its NumPy restatement
    (oracle port).  One process: the reference's per-lattice loop is single-threaded NumPy (its
    only parallelism is one process per parameter tuple, runner.py:142, and C4 is one lattice).
    A bench step here is ONE iteration of a bounded sample lattice of the C4 physics, sized so
    that the K + W iterations end within a few minutes (the full L=4096 lattice when they fit:
    about 27 s per iteration)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    L_full = args.L or (4096 if args.gpus <= 1 else 32768)
    budget_s, rate = 150.0, 0.7e6           # ~0.6-1.2 M site-updates/s measured in the survey
    Ls = int(min(L_full, (budget_s * rate / max(1, steps + warm)) ** 0.5))
    Ls = max(128, Ls - Ls % 32)
    root = reference_root()
    if root is not None:
        value, sec = cpu_reference(Ls, warm, steps)
        kind = "reference"
        how = f"unmodified reference ({'oracle/_ref' if 'oracle' in root else root}), SPGG.run"
    else:
        value, sec = cpu_port(Ls, warm + steps)
        kind = "port"
        how = "NumPy restatement of the reference loop (oracle/spgg_numpy.py)"
    sample = (f"{steps} timed iterations of an L={Ls} lattice with the C4 physics "
              f"({'the full workload lattice' if Ls == L_full else f'bounded sample of the L={L_full} workload'}), "
              f"{how}, 1 process")
    line = {
        "impl": "reference", "metric": "site-updates/s", "value": value, "unit": "site-updates/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": c4_config(L_full, args.inner) if args.gpus <= 1 else c5_config(args.L or 32768, args.gpus, args.inner),
        "cpu_baseline": {"value": value, "unit": "site-updates/s", "cores": 1, "kind": kind,
                         "sample": sample, "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": "site-updates/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--inner", type=int, default=100, help="lattice iterations per bench step")
    ap.add_argument("--L", type=int, default=None)
    ap.add_argument("--impl", default="native")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip extras.scaling_anchor / extras.variants")
    ap.add_argument("--only-variants", action="store_true", help="print extras.variants only (kernel tuning)")
    ap.add_argument("--cpu-L", type=int, default=4096)
    ap.add_argument("--workload", default="c4", choices=["c4", "sweep", "c1", "c2"],
                    help="c4: the headline L=4096 lattice (default); sweep: BASELINE config 3, the "
                         "r x kappa x M grid as 60 batched L=200 replicas; c1 / c2: the single small "
                         "lattices of configs 0-2 (none of these is a driver bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                         "(see dump_outputs); c4 workload on one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.workload != "c4" or args.only_variants
                              or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs covers the native c4 workload on one GPU")

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import spgg_b200
    from spgg_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        from spgg_b200 import strips
        return strips.bench_main(args, rank, local_rank, world)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    if args.only_variants:
        v = measure_extras(args.L or 4096, measured_peak_gbs()[0], anchor=False)["variants"]
        for k_, d in v.items():
            print(f"{k_:38s} {d.get('us_per_iteration', float('nan')):9.1f} us  frac {d.get('roofline_frac', float('nan')):.3f}  {d.get('path', d.get('error', ''))[:60]}")
        return
    if args.workload != "c4":
        return bench_sweep(args)
    dev = 0
    torch.cuda.set_device(dev)
    L = args.L or 4096
    K, W, inner = args.steps, args.warmup, args.inner
    p = dict(C4, L=L)
    n_sites = L * L
    peak, peak_src = measured_peak_gbs()

    # host state in pinned memory (reference layouts: uint8 S, f64 R, f64 Q)
    rs = np.random.RandomState(0)
    S_h = torch.empty((L, L), dtype=torch.uint8).pin_memory()
    R_h = torch.zeros((L, L), dtype=torch.float64).pin_memory()
    Q_h = torch.empty((L, L, 2, 2), dtype=torch.float64).pin_memory()
    S_h.numpy()[...] = rs.randint(0, 2, (L, L))
    Q_h.numpy()[...] = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
    S_out = torch.empty_like(S_h).pin_memory()
    R_out = torch.empty_like(R_h).pin_memory()
    Q_out = torch.empty_like(Q_h).pin_memory()

    eng = spgg_b200.Engine(p, seeds=2024, precision="fp32", device=dev)
    lib, h = eng.lib, eng._h
    stream = torch.cuda.current_stream().cuda_stream

    def upload():
        _lib.check(lib.spgg_set_state(h, 0, S_h.data_ptr(), R_h.data_ptr(), Q_h.data_ptr()))

    # ---------------- warm-up
    upload()
    for _ in range(W):
        eng.step(inner, stream)
    eng.sync()

    # ---------------- device-resident timed region (value)
    upload()
    l0 = eng.status().kernel_launches
    sampler = ClockSampler(dev)
    sampler.start()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        _lib.check(lib.spgg_step(h, inner, stream))
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    eng.sync()
    launches = eng.status().kernel_launches - l0
    if eng.status().iteration != K * inner:
        raise SystemExit(f"the timed steps ran {eng.status().iteration} iterations, not {K} x {inner}")
    value = n_sites * inner * K / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, inner)

    # ---------------- end to end through the public API with host buffers
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    upload()
    d2h_stats = 0
    for _ in range(K):
        eng.step(inner, stream)
        rows = eng.stats()
        d2h_stats += rows.nbytes
    _lib.check(lib.spgg_get_state(h, 0, S_out.data_ptr(), R_out.data_ptr(), Q_out.data_ptr()))
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    state_bytes = S_h.numel() + R_h.numel() * 8 + Q_h.numel() * 8
    e2e_value = n_sites * inner * K / t_e2e

    # ---------------- per-kernel timing (roofline of the dominant kernel, k_step)
    # one event pair per iteration around spgg_phase_iteration: a single k_step_fast launch when the
    # handle speculates on the global maximum (the default), k_gmax + k_step otherwise
    n_probe = min(200, inner * K)
    st0 = eng.status()
    _lib.check(lib.spgg_begin_steps(h, n_probe, stream))
    _lib.check(lib.spgg_phase_kernel(h, 0, 1, stream))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_probe + 1)]
    evs[0].record()
    for s in range(1, n_probe + 1):
        _lib.check(lib.spgg_phase_iteration(h, 1 if s < n_probe else 0, stream))
        evs[s].record()
    _lib.check(lib.spgg_end_steps(h, stream))
    torch.cuda.synchronize()
    eng.sync()
    st1 = eng.status()
    speculative = (st1.speculative_launches - st0.speculative_launches) >= n_probe - 1
    t_iter = float(np.mean([evs[s].elapsed_time(evs[s + 1]) for s in range(1, n_probe - 1)])) * 1e-3
    # the exact pair, launch by launch (what a handle without speculation runs): k_gmax, then k_step
    _lib.check(lib.spgg_begin_steps(h, n_probe, stream))
    _lib.check(lib.spgg_phase_kernel(h, 0, 1, stream))
    ev2 = []
    for s in range(1, n_probe + 1):
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        _lib.check(lib.spgg_phase_gmax(h, stream))
        b.record()
        _lib.check(lib.spgg_phase_kernel(h, 1, 1 if s < n_probe else 0, stream))
        c.record()
        ev2.append((a, b, c))
    _lib.check(lib.spgg_end_steps(h, stream))
    torch.cuda.synchronize()
    eng.sync()
    t_gmax = float(np.mean([a.elapsed_time(b) for a, b, c in ev2[:-1]])) * 1e-3
    t_step_exact = float(np.mean([b.elapsed_time(c) for a, b, c in ev2[:-1]])) * 1e-3
    t_step = t_iter if speculative else t_step_exact
    achieved = BYTES_PER_SITE_FP32 * n_sites / t_step / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu_traffic(L),
                "kernel": "k_step_fast<M=1, reputation, update+select> (fused SPGG iteration"
                          + (", speculative global maximum: the only launch of an iteration)" if speculative else ")"),
                "algorithmic_bytes_per_launch": BYTES_PER_SITE_FP32 * n_sites,
                "kernel_us": t_step * 1e6,
                "exact_pair_us": {"k_gmax": t_gmax * 1e6, "k_step": t_step_exact * 1e6},
                "gmax_kernel_us": None if speculative else t_gmax * 1e6,
                "speculation": {"launches": int(st1.speculative_launches), "failures": int(st1.speculation_failures)},
                "algorithmic_bytes_per_site": BYTES_PER_SITE_FP32, "peak_source": peak_src,
                "whole_step_frac": BYTES_PER_SITE_FP32 * value / 1e9 / peak}

    # ---------------- CPU baseline beside it (bounded sample)
    cpu = None
    if not args.no_cpu_baseline:
        if reference_root() is not None:
            v, dt = cpu_reference(args.cpu_L, 1, 1)
            cpu = {"value": v, "unit": "site-updates/s", "cores": 1, "kind": "reference",
                   "sample": f"1 timed iteration (after 1 warm-up iteration) of the L={args.cpu_L} lattice, C4 "
                             f"physics, with the unmodified reference's SPGG.run ({dt:.1f} s per iteration)",
                   "host_cpus": os.cpu_count()}
        else:
            v, dt = cpu_port(args.cpu_L, 1)
            cpu = {"value": v, "unit": "site-updates/s", "cores": 1, "kind": "port",
                   "sample": f"1 iteration of the L={args.cpu_L} lattice with the NumPy restatement of the "
                             f"reference path ({dt:.1f} s); no copy of the reference on this box",
                   "host_cpus": os.cpu_count()}

    eng.close()
    del eng
    extras = {}
    if not args.no_extras:
        extras = measure_extras(L, peak)

    line = {
        "metric": "site-updates/s", "value": value, "unit": "site-updates/s", "n_gpus": 1,
        "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": c4_config(L, inner),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "site-updates/s",
                "h2d_bytes_per_step": state_bytes / K, "d2h_bytes_per_step": (state_bytes + d2h_stats) / K,
                "seconds": t_e2e},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "extras": extras,
    }
    print(json.dumps(line), flush=True)


DUMP_SITES = 1 << 18    # sites sampled for the state dump
DUMP_ROWS = 4096        # statistics rows of the dump: the last ones of the step


def dump_outputs(out_dir, eng, inner):
    """What the timed path computed in its last step, as a caller of spgg_step receives it:
    ``stats`` the statistics rows of that step's last min(inner, DUMP_ROWS) iterations, and ``S``,
    ``R``, ``Q`` the state it left (float64 R and Q in the reference's layout, S as float32 0 = C /
    1 = D) at a fixed seeded sample of DUMP_SITES sites, whose flat indices are ``sites`` (the whole
    state of the L=4096 lattice is 700 MB).  At most 15 MB for any arguments.  The inputs are fixed
    by the arguments, so two builds can be compared file by file; the float statistics sums may
    differ in the last bits between runs."""
    os.makedirs(out_dir, exist_ok=True)
    S, R, Q = eng.get_state()
    n = S.size
    sites = np.sort(np.random.RandomState(0).choice(n, min(DUMP_SITES, n), replace=False))
    rows = min(inner, DUMP_ROWS)
    out = {"stats": eng.stats(first=1 + inner - rows, n=rows),
           "sites": sites.astype(np.float64),
           "S": S.reshape(-1)[sites].astype(np.float32),
           "R": R.reshape(-1)[sites],
           "Q": Q.reshape(n, -1)[sites]}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


BYTES_PER_SITE = {"fp32": 34.25, "fp32_rfloat": 40.25, "fp64": 80.25}   # BASELINE.md section 3


def measure_iteration(params, precision="fp32", n_warm=3, n_iter=10, seed=2024):
    """us per iteration of one device-resident lattice (init on the device, CUDA events)."""
    import torch
    import spgg_b200
    eng = spgg_b200.Engine(params, seeds=seed, precision=precision, device=0)
    try:
        eng.init_random(seed)
        stream = torch.cuda.current_stream().cuda_stream
        eng.step(n_warm, stream)
        eng.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.step(n_iter, stream)
        e1.record()
        torch.cuda.synchronize()
        eng.sync()
        return 1e3 * e0.elapsed_time(e1) / n_iter, eng.describe()
    finally:
        eng.close()


def measure_extras(L, peak, anchor=True):
    """Beside the headline (VERDICT r1): the one-GPU iteration of the L=32768 lattice the strip runs
    split (so that N-GPU numbers can be read against the same lattice), and the paths next to the
    headline kernel - reference precision, second-order neighbourhood, action state, a lattice side
    that is not a multiple of 128."""
    out = {}
    try:
        if not anchor:
            raise RuntimeError("skipped")
        L5 = 32768
        us, desc = measure_iteration(dict(C4, L=L5), n_warm=2, n_iter=6)
        out["scaling_anchor"] = {"L": L5, "n_gpus": 1, "us_per_iteration": us,
                                 "value": L5 * L5 / (us * 1e-6), "unit": "site-updates/s",
                                 "roofline_frac": 34.25 * L5 * L5 / (us * 1e-6) / 1e9 / peak, "path": desc}
    except Exception as e:
        out["scaling_anchor"] = {"error": str(e)[:200]}
    variants = {}
    cases = {
        "fp64_reference_precision": (dict(C4, L=L), "fp64", BYTES_PER_SITE["fp64"]),
        "second_order_M2": (dict(C4, L=L, use_second_order=True), "fp32", BYTES_PER_SITE["fp32"]),
        "action_state": (dict(C4, L=L, state_representation="action"), "fp32", BYTES_PER_SITE["fp32"]),
        "action_state_M2": (dict(C4, L=L, state_representation="action", use_second_order=True, r=4.0,
                                 reward_weight_payoff=1.0), "fp32", BYTES_PER_SITE["fp32"]),
        "L4000_not_128_aligned": (dict(C4, L=4000), "fp32", BYTES_PER_SITE["fp32"]),
        "fractional_reputation_steps_fp32_R": (dict(C4, L=L, rep_gain_C=0.3, delta_R_D=0.7), "fp32",
                                               BYTES_PER_SITE["fp32_rfloat"]),
    }
    for name, (p, prec, bps) in cases.items():
        try:
            us, desc = measure_iteration(p, prec, n_warm=3, n_iter=24)   # one chunk: its select-only first launch is 1/24 of it
            n = p["L"] * p["L"]
            variants[name] = {"L": p["L"], "us_per_iteration": us, "site_updates_per_s": n / (us * 1e-6),
                              "bytes_per_site": bps, "roofline_frac": bps * n / (us * 1e-6) / 1e9 / peak,
                              "path": desc}
        except Exception as e:
            variants[name] = {"error": str(e)[:200]}
    out["variants"] = variants
    return out


def bench_sweep(args):
    """Small-lattice workloads on one GPU (not the driver's bench line; BASELINE configs 0-3):
      sweep  C3: r in {1,2,3,3.6,4,5} x kappa in {0,.5,1,1.5,2} x M in {1,2}, w_P=1, L=200 (the
             reference's figure_2_3_4 set is a subset) as two batched handles of 30 replicas;
      c1     the default_config.yaml run: one L=100 lattice, reputation state, M=1, r=3;
      c2     one L=200 lattice, action state, M=2, r=4.
    These lattices live in shared memory for a whole chunk (csrc/spgg_resident.cuh: one
    thread-block cluster per replica); SPGG_NO_RESIDENT=1 times the per-iteration kernels."""
    import torch
    import spgg_b200
    inner = args.inner
    if args.workload == "sweep":
        L = args.L or 200
        plist = [dict(C4, L=L, r=r, influence_factor=k, use_second_order=m, reward_weight_payoff=1.0)
                 for m in (False, True) for r in (1, 2, 3, 3.6, 4, 5) for k in (0, 0.5, 1, 1.5, 2)]
        what = f"C3: {len(plist)} replicas L={L} (r x kappa x M grid), two batched handles"
    elif args.workload == "c1":
        L = args.L or 100
        plist = [dict(C4, L=L)]
        what = f"C1: one lattice L={L}, reputation state, M=1, r=3, kappa=1, w_P=0.95"
    else:
        L = args.L or 200
        plist = [dict(C4, L=L, r=4.0, use_second_order=True, reward_weight_payoff=1.0,
                      state_representation="action")]
        what = f"C2: one lattice L={L}, action state, M=2, r=4, kappa=1"
    engines = []
    for m in (False, True):
        ps = [p for p in plist if p["use_second_order"] == m]
        if not ps:
            continue
        eng = spgg_b200.Engine(ps, seeds=list(range(len(ps))), precision="fp32")
        for r in range(len(ps)):
            eng.init_random(100 + r, replica=r)
        engines.append(eng)
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(args.warmup):
        for eng in engines:
            eng.step(inner, stream)
    torch.cuda.synchronize()
    l0 = sum(eng.status().kernel_launches for eng in engines)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        for eng in engines:
            eng.step(inner, stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    for eng in engines:
        eng.sync()
    launches = sum(eng.status().kernel_launches for eng in engines) - l0
    value = len(plist) * L * L * inner * args.steps / (ms * 1e-3)
    resident = launches <= 2 * len(engines) * args.steps
    peak, peak_src = measured_peak_gbs()
    print(json.dumps({"metric": "site-updates/s", "value": value, "unit": "site-updates/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                      "data": "synthetic", "gpu_launches": int(launches),
                      "us_per_iteration": 1e3 * ms / (args.steps * inner),
                      "config": {"workload": f"{what}, {inner} iterations per bench step, "
                                             + ("lattice-resident cluster kernel (state in shared memory, no HBM "
                                                "traffic inside a chunk: latency/issue-bound, not HBM-bound)"
                                                if resident else "per-iteration kernels (L2-resident, launch-bound)")},
                      "roofline": {"bound": "hbm", "achieved": BYTES_PER_SITE_FP32 * value / 1e9, "peak": peak,
                                   "unit": "GB/s", "frac": BYTES_PER_SITE_FP32 * value / 1e9 / peak,
                                   "traffic": None, "peak_source": peak_src,
                                   "note": "same 34.25 B/site formula as C4 for comparison only; the state never "
                                           "leaves the chip between iterations"}}),
          flush=True)
    for eng in engines:
        eng.close()


def state_bytes_dev(L):
    return L * L * (16 + 1 + 1 + 0.125)


if __name__ == "__main__":
    main()
