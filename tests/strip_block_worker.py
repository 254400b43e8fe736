"""Worker processes of tests/test_gpu_strip_blocks.py (one rank each, RANK / WORLD_SIZE / MASTER_ADDR /
MASTER_PORT in the environment): block fields of a lattice split into row strips (StripEngine.block_fields,
include/spgg.h: spgg_block_fields) against one handle holding the whole lattice and the NumPy restatement."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

U = 2.0 ** -53


def _packed(got, nq):
    from test_gpu_blocks import _packed as p
    return p(got, nq)


def _check(got, whole, want, nq, world, exact_r, what):
    """got: the strips' dict; whole: one handle's dict; want: numpy_block_fields(flags=3) of the lattice"""
    from test_blocks_host import sum_bound
    c, s, a = want
    gc, gs = _packed(got, nq)
    wc, ws = _packed(whole, nq)
    assert np.array_equal(gc, c) and np.array_equal(gc, wc), (what, "counts")
    sel = ([0] if "R" in got else []) + (list(range(1, 1 + nq)) if "Q" in got else [])
    s, a = s[..., sel], a[..., sel]
    assert gs.shape == s.shape == ws.shape, what
    if "R" in got and exact_r:
        assert np.array_equal(gs[..., 0], s[..., 0]) and np.array_equal(ws[..., 0], s[..., 0]), (what, "int8 R")
    # each side within (n-1) 2^-53 sum|x| of the exact sums; the strips add up to `world` partials on top
    bound = sum_bound(c, a) + world * U * a
    assert (np.abs(gs - ws) <= bound).all(), (what, float(np.abs(gs - ws).max()))
    assert (np.abs(gs - s) <= bound).all(), (what, float(np.abs(gs - s).max()))


def _state(L, rs, p_coop, nq=4):
    S = (rs.rand(L, L) >= p_coop).astype(np.uint8)
    R = rs.randint(-10, 11, (L, L)).astype(np.float64)
    Q = rs.uniform(-0.5, 0.5, (L, L) + (2,) * (2 if nq == 4 else 3)).astype(np.float32).astype(np.float64)
    return S, R, Q


def geometries(rank, world, L, bs):
    """Uploaded random states: the strips' result == one whole-lattice handle's == NumPy, every field set."""
    import torch
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    from test_blocks_host import numpy_block_fields
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    p = full_params(dict(C1, L=L))
    se = strips.StripEngine(p, seed=5, precision="fp32", device=dev)
    eng = spgg_b200.Engine(p, seeds=5, precision="fp32", device=dev)
    rs = np.random.RandomState(L)
    for p_coop in (0.1, 0.5, 0.9):
        S, R, Q = _state(L, rs, p_coop)
        se.set_state_global(S, R, Q)
        eng.set_state(S, R, Q)
        for b in bs:
            want = numpy_block_fields(S, R, Q, b, 3)
            for fields in ((), ("R",), ("Q",), ("R", "Q")):
                _check(se.block_fields(b, fields), eng.block_fields(b, fields=fields), want, 4, world, True,
                       (L, world, b, fields, p_coop))
    se.close()
    eng.close()


def dynamics(rank, world, which_case):
    """A state from the dynamics (same seed on the strips and on one handle): equal results, and the strip run's
    digests do not change when block fields are taken between its chunks."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, C2, full_params
    from test_blocks_host import numpy_block_fields
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
                got.append([se.block_fields(b) for b in (5, 32, L)])
        out[taken] = se.digest()
        if taken:
            S, R, Q = se.gather_state()
            exact = precision == "fp32"
            eng = spgg_b200.Engine(p, seeds=31, precision=precision, device=dev)
            eng.init_random(9)
            for c, g in zip(chunks, got):
                eng.step(c)
                for b, gb in zip((5, 32, L), g):
                    wb = eng.block_fields(b)
                    if c == chunks[-1]:
                        _check(gb, wb, numpy_block_fields(S, R, Q, b, 3), 4, world, exact, (which_case, b))
                    else:
                        assert np.array_equal(gb["n_C"], wb["n_C"]), (which_case, c, b)
            eng.close()
        se.close()
        dist.barrier()
    assert out[True] == out[False], "block fields between chunks changed the run"


def large(rank, world, L):
    """Counts only at L = 16384 over the ranks, against one handle created after the strips are closed."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    p = full_params(dict(C1, L=L))
    bs = (8, 32, 1000, L)
    se = strips.StripEngine(p, seed=4, precision="fp32", device=dev)
    se.init_random(12)
    se.step(3)
    got = [se.block_fields(b, ()) for b in bs]
    se.close()
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        eng = spgg_b200.Engine(p, seeds=4, precision="fp32", device=dev)
        eng.init_random(12)
        eng.step(3)
        for g, b in zip(got, bs):
            w = eng.block_fields(b, fields=())
            assert np.array_equal(w["n"], g["n"]) and np.array_equal(w["n_C"], g["n_C"]), b
        eng.close()
    dist.barrier()


def world_one(rank, world):
    """A StripEngine of world 1 is a whole-lattice handle: bit-identical results."""
    import torch
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    assert world == 1
    torch.cuda.set_device(0)
    for L in (64, 100, 256):
        p = full_params(dict(C1, L=L))
        se = strips.StripEngine(p, seed=2, precision="fp32", device=0)
        eng = spgg_b200.Engine(p, seeds=2, precision="fp32", device=0)
        S, R, Q = _state(L, np.random.RandomState(L), 0.5)
        se.set_state_global(S, R, Q)
        eng.set_state(S, R, Q)
        for b in (1, 7, 32, L):
            g, w = se.block_fields(b), eng.block_fields(b)
            for k in w:
                assert g[k].tobytes() == w[k].tobytes(), (L, b, k)
        se.close()
        eng.close()


def main():
    import torch.distributed as dist
    mode = sys.argv[1]
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group(sys.argv[2], rank=rank, world_size=world)
    try:
        if mode == "geometries":
            geometries(rank, world, int(sys.argv[3]), [int(x) for x in sys.argv[4].split(",")])
        elif mode == "dynamics":
            dynamics(rank, world, sys.argv[3])
        elif mode == "large":
            large(rank, world, int(sys.argv[3]))
        elif mode == "world1":
            world_one(rank, world)
        else:
            raise SystemExit(f"unknown mode {mode}")
    finally:
        dist.destroy_process_group()
    print(f"rank {rank} ok")


if __name__ == "__main__":
    main()
