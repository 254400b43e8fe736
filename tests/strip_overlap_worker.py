"""Worker processes of tests/test_gpu_strip_overlap.py (one rank each, RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT in
the environment): state overlaps of a lattice split into row strips (StripEngine.snapshot / StripEngine.overlap,
include/spgg.h: spgg_snapshot / spgg_overlap on strip handles) against one handle holding the whole lattice and
NumPy."""
import os
import pickle
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FIELD_SETS = ((), ("R",), ("Q",), ("R", "Q"))


def _same_everywhere(got, what):
    """every rank holds the same dict, bit for bit"""
    import torch.distributed as dist
    mine = pickle.dumps({k: np.asarray(v).tobytes() for k, v in got.items()})
    everyone = [None] * dist.get_world_size()
    dist.all_gather_object(everyone, mine)
    assert all(e == mine for e in everyone), what


def _check(se, eng, then, L, what):
    """the strips' result == one whole-lattice handle's (sums within the bound) == NumPy, every field subset"""
    from test_gpu_overlap import _compare, _packed
    from test_overlap_host import numpy_overlap, sum_bound
    now = eng.get_state()
    for fields in FIELD_SETS:
        got = se.overlap(0, fields=fields)
        whole = eng.overlap(0, fields=fields)
        assert set(got) == set(whole), (what, fields)
        g, w = _packed(got), _packed(whole)
        assert np.array_equal(g[0], w[0]) and np.array_equal(g[1], w[1]) and np.array_equal(g[2][:, 0], w[2][:, 0]), \
            (what, fields)
        assert (np.abs(g[2][:, 1:] - w[2][:, 1:]) <= sum_bound(L * L, w[2])).all(), (what, fields)
        assert got["t0"] == whole["t0"] and got["t"] == whole["t"], (what, fields)
        _compare(g, numpy_overlap(then, now, fields), L * L, True, fields, (what, fields))
        _same_everywhere(got, (what, fields))


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
    a, b = _state(L, rs, 0.2), _state(L, rs, 0.7)
    se.set_state_global(*a)
    eng.set_state(*a)
    se.snapshot(0)
    eng.snapshot(0)
    _check(se, eng, a, L, (L, world, "identity"))
    se.set_state_global(*b)
    eng.set_state(*b)
    _check(se, eng, a, L, (L, world, "uploads"))
    se.close()
    eng.close()


def dynamics(rank, world, which_case):
    """A state from the dynamics (same seed on the strips and on one handle): equal results, and the strip run's
    digests do not change when snapshots and overlaps are taken between its chunks."""
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
        if taken:
            eng = spgg_b200.Engine(p, seeds=31, precision=precision, device=dev)
            eng.init_random(9)
            se.snapshot(0)
            eng.snapshot(0)
            then = eng.get_state()
        for c in chunks:
            se.step(c)
            if taken:
                eng.step(c)
                _check(se, eng, then, L, (which_case, c))
        out[taken] = se.digest()
        if taken:
            eng.close()
        se.close()
        dist.barrier()
    assert out[True] == out[False], "overlaps between chunks changed the run"


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
