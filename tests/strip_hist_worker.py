"""Worker processes of tests/test_gpu_strip_hist.py (one rank each, RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT in
the environment): value distributions of a lattice split into row strips (StripEngine.histograms, include/spgg.h:
spgg_value_ranges / spgg_histograms on strip handles) against one handle holding the whole lattice and NumPy."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FIELD_SETS = ((), ("R",), ("Q",), ("R", "Q"))


def _same(got, whole, what):
    assert set(got) == set(whole), what
    for k in got:
        if k != "replica":
            assert np.array_equal(got[k], whole[k]), (what, k)


def _check(se, eng, state, bins, ranges, what):
    """the strips' result == one whole-lattice handle's == NumPy, every field set"""
    from test_gpu_hist import _packed
    from test_hist_host import default_edges, numpy_histograms
    S, R, Q = state
    for fields in FIELD_SETS:
        got = se.histograms(bins, fields=fields, ranges=ranges)
        _same(got, eng.histograms(bins, fields=fields, ranges=ranges), (what, fields))
        flags = (1 if "R" in fields else 0) | (2 if "Q" in fields else 0)
        if flags and ranges is None:
            counts, pol = numpy_histograms(S, R, Q, default_edges(S, R, Q, bins, flags), "qlearning", flags)
            assert np.array_equal(_packed(got, 4), counts) and np.array_equal(got["policy"], pol), (what, fields)


def _state(L, rs, p_coop):
    S = (rs.rand(L, L) >= p_coop).astype(np.uint8)
    R = rs.randint(-10, 11, (L, L)).astype(np.float64)
    Q = rs.uniform(-0.5, 0.5, (L, L, 2, 2)).astype(np.float32).astype(np.float64)
    return S, R, Q


def geometries(rank, world, L):
    import torch
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    p = full_params(dict(C1, L=L))
    se = strips.StripEngine(p, seed=5, precision="fp32", device=dev)
    eng = spgg_b200.Engine(p, seeds=5, precision="fp32", device=dev)
    rs = np.random.RandomState(L)
    for p_coop in (0.1, 0.9):
        st = _state(L, rs, p_coop)
        se.set_state_global(*st)
        eng.set_state(*st)
        for bins in (1, 20, 1024):
            _check(se, eng, st, bins, None, (L, world, p_coop, bins))
        _check(se, eng, st, 7, {"R": (-3, 4), "Q": (-0.25, 0.25)}, (L, world, p_coop, "ranges"))
    se.close()
    eng.close()


def dynamics(rank, world, which_case):
    """A state from the dynamics (same seed on the strips and on one handle): equal results, and the strip run's
    digests do not change when histograms are taken between its chunks."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, C2, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    physics, L, precision = {"fast": (C1, 256, "fp32"), "general": (C2, 100, "fp32"),
                             "fp64": (C1, 64, "fp64")}[which_case]
    p = full_params(dict(physics, L=L))
    chunks = (7, 13)
    out = {}
    for taken in (True, False):
        se = strips.StripEngine(p, seed=31, precision=precision, device=dev)
        se.init_random(9)
        got = []
        for c in chunks:
            se.step(c)
            if taken:
                got.append(se.histograms(20))
        out[taken] = se.digest()
        if taken:
            eng = spgg_b200.Engine(p, seeds=31, precision=precision, device=dev)
            eng.init_random(9)
            for c, g in zip(chunks, got):
                eng.step(c)
                _same(g, eng.histograms(20), (which_case, c))
            eng.close()
        se.close()
        dist.barrier()
    assert out[True] == out[False], "histograms between chunks changed the run"


def main():
    import torch.distributed as dist
    mode = sys.argv[1]
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group(sys.argv[2], rank=rank, world_size=world)
    try:
        if mode == "geometries":
            geometries(rank, world, int(sys.argv[3]))
        elif mode == "dynamics":
            dynamics(rank, world, sys.argv[3])
        else:
            raise SystemExit(f"unknown mode {mode}")
    finally:
        dist.destroy_process_group()
    print(f"rank {rank} ok")


if __name__ == "__main__":
    main()
