"""Worker processes of tests/test_gpu_strip_pairs.py (one rank each, RANK / WORLD_SIZE / MASTER_ADDR /
MASTER_PORT in the environment): strategy pair counts of a lattice split into row strips
(StripEngine.pair_counts, include/spgg.h: spgg_strip_pair_counts) against NumPy and one handle holding the
whole lattice."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _path(L, precision="fp32"):
    return "fast" if precision == "fp32" and L % 32 == 0 and L >= 128 else "general"


def _state(L):
    return np.zeros((L, L)), np.zeros((L, L, 2, 2))


def _want(S, max_d):
    from test_pairs_host import numpy_pair_counts
    L = S.shape[0]
    ds = None if L <= 1024 else sorted({d for d in (1, 2, 31, 32, 33, 1000, max_d) if d <= max_d})
    return numpy_pair_counts(S, max_d, ds)


def _check(got, want, what):
    sel = want >= 0
    assert got.dtype == np.int64 and got.shape == want.shape, what
    assert np.array_equal(got[sel], want[sel]), (what, np.argwhere((got != want) & sel)[:8])
    nC = got[0, 0, 0]
    assert np.array_equal(2 * (nC - got[:, :, 0]), got[:, :, 1]), what


def patterns(L):
    ii, jj = np.indices((L, L))
    yield "checkerboard", ((ii + jj) % 2).astype(np.uint8)
    yield "horizontal stripes 33", ((ii // 33) % 2).astype(np.uint8)
    yield "vertical stripes 31", ((jj // 31) % 2).astype(np.uint8)
    rs = np.random.RandomState(L)
    for p in (0.1, 0.5, 0.9):
        yield f"random {p}", (rs.rand(L, L) >= p).astype(np.uint8)


def geometries(rank, world, L, max_ds):
    """Uploaded patterns: the counts summed over the strips == NumPy == one whole-lattice handle."""
    import torch
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    p = full_params(dict(C1, L=L))
    se = strips.StripEngine(p, seed=5, precision="fp32", device=dev)
    assert se.eng.describe().startswith(_path(L)), se.eng.describe()
    eng = spgg_b200.Engine(p, seeds=5, precision="fp32", device=dev) if rank == 0 else None
    R0, Q0 = _state(L)
    for name, S in patterns(L):
        se.set_state_global(S, R0, Q0)
        if eng is not None:
            eng.set_state(S, R0, Q0)
        for md in max_ds:
            got = se.pair_counts(md)
            _check(got, _want(S, md), (name, L, md, world))
            if eng is not None:
                assert np.array_equal(eng.pair_counts(md), got), (name, L, md)
    se.close()
    if eng is not None:
        eng.close()


def dynamics(rank, world, which_case):
    """States from the dynamics, stepped in chunks: after each chunk the strips' counts == the single handle's
    (same seed); counting between chunks leaves the strip run's digests unchanged."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, C2, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    physics, L, precision = {"fast": (C1, 256, "fp32"), "fast_c2": (C2, 256, "fp32"),
                             "general": (C2, 100, "fp32"), "fp64": (C1, 64, "fp64")}[which_case]
    p = full_params(dict(physics, L=L))
    chunks = (7, 13, 20)
    out = {}
    for counted in (True, False):
        se = strips.StripEngine(p, seed=31, precision=precision, device=dev)
        assert se.eng.describe().startswith(_path(L, precision)), se.eng.describe()
        se.init_random(9)
        got = []
        for c in chunks:
            se.step(c)
            if counted:
                got.append(se.pair_counts(L // 2))
        out[counted] = se.digest()
        if counted:
            if os.environ.get("SPGG_SPEC_TEST_POISON") and se.spec_mode:
                assert se.reruns > 0, "the spoiled guesses were not re-run"
            S = se.gather_state(want_q=False)[0]
            _check(got[-1], _want(S, L // 2), which_case)
        se.close()
        if counted and rank == 0:
            eng = spgg_b200.Engine(p, seeds=31, precision=precision, device=dev)
            eng.init_random(9)
            for c, g in zip(chunks, got):
                eng.step(c)
                assert np.array_equal(eng.pair_counts(L // 2), g), (which_case, c)
            eng.close()
        dist.barrier()
    assert out[True] == out[False], "counting between chunks changed the run"


def large(rank, world, L, n_steps):
    """A large lattice from init_random + a few steps; the whole-lattice handle on rank 0 is created after the
    strips are closed."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    p = full_params(dict(C1, L=L))
    se = strips.StripEngine(p, seed=4, precision="fp32", device=dev)
    assert se.eng.describe().startswith(_path(L)), se.eng.describe()
    se.init_random(12)
    se.step(n_steps)
    got = [se.pair_counts(md) for md in (1, 100, L // 2)]
    se.close()
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        eng = spgg_b200.Engine(p, seeds=4, precision="fp32", device=dev)
        eng.init_random(12)
        eng.step(n_steps)
        for g, md in zip(got, (1, 100, L // 2)):
            assert np.array_equal(eng.pair_counts(md), g), md
        S = np.empty(L * L, np.uint8)
        assert eng.lib.spgg_get_state(eng._h, 0, S.ctypes.data, None, None) == 0
        eng.close()
        _check(got[-1], _want(S.reshape(L, L), L // 2), "large")
    dist.barrier()


def world_one(rank, world):
    """A StripEngine of world 1 (a whole-lattice handle through the strip entry points) == spgg_pair_counts."""
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
        R0, Q0 = _state(L)
        for name, S in patterns(L):
            se.set_state_global(S, R0, Q0)
            eng.set_state(S, R0, Q0)
            for md in sorted({1, min(33, L // 2), L // 2}):
                got = se.pair_counts(md)
                _check(got, _want(S, md), (name, L, md))
                assert np.array_equal(eng.pair_counts(md), got)
        se.close()
        eng.close()


def errors(rank, world):
    """The counts take records that describe one lattice, with the max_d and max_rows of the call."""
    import torch
    import torch.distributed as dist
    from spgg_b200 import strips, _lib
    from helpers import C1, full_params
    assert world == 2
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    L, md, mr = 64, 8, 8
    se = strips.StripEngine(full_params(dict(C1, L=L)), seed=1, precision="fp32", device=dev)
    lib, h = se.lib, se.h
    se.init_random(3)
    nb = int(lib.spgg_strip_pair_record_bytes(h, md, mr))
    assert nb == 4 * (8 + mr * 2)
    rec = torch.zeros(3 * nb, dtype=torch.uint8, device=dev)
    out = np.zeros((2, md + 1, 2), np.int64)

    def gather(max_d, max_rows):
        mine = rec[rank * nb:(rank + 1) * nb]
        assert lib.spgg_strip_pair_record(h, max_d, max_rows, mine.data_ptr()) == 0
        torch.cuda.synchronize()
        host = mine.cpu()
        parts = [torch.empty_like(host) for _ in range(world)]
        dist.all_gather(parts, host)
        rec[:2 * nb].copy_(torch.cat(parts).to(dev))
        torch.cuda.synchronize()

    def counts(w=2, r=rank, buf=None, max_d=md, max_rows=mr):
        return lib.spgg_strip_pair_counts(h, w, r, (rec if buf is None else buf).data_ptr(), max_d, max_rows,
                                          out.ctypes.data)

    gather(md, mr)
    assert counts() == 0
    t = torch.from_numpy(out.copy())
    dist.all_reduce(t)
    assert np.array_equal(t.numpy(), se.pair_counts(md))
    other_d = rec.clone()
    other_d.view(torch.int32)[nb // 4 + 4] = md + 8           # record 1 was written for another max_d
    assert counts(buf=other_d) == _lib.E_INVALID
    assert counts(max_d=md - 1, max_rows=md - 1) == _lib.E_INVALID   # not the max_d / max_rows of the records
    assert counts(w=1, r=0) == _lib.E_INVALID                # one record does not cover the lattice
    assert counts(w=3) == _lib.E_INVALID                     # the third record is not a record
    assert counts(w=2, r=2) == _lib.E_INVALID
    assert counts(w=2, r=1 - rank) == _lib.E_INVALID         # another strip's record
    assert counts(buf=torch.cat([rec[nb:2 * nb], rec[:nb]])) == _lib.E_INVALID   # rows out of rank order
    bad_L = rec.clone()
    bad_L.view(torch.int32)[1] = L + 1
    assert counts(buf=bad_L) == _lib.E_INVALID               # records of another lattice
    bad_magic = rec.clone()
    bad_magic.view(torch.int32)[0] = 0
    assert counts(buf=bad_magic) == _lib.E_INVALID
    assert counts() == 0
    for max_d, max_rows in ((0, 0), (L // 2 + 1, 8), (8, 9), (40, 31), (-1, 1)):
        assert lib.spgg_strip_pair_record_bytes(h, max_d, max_rows) == _lib.E_INVALID, (max_d, max_rows)
        assert lib.spgg_strip_pair_record(h, max_d, max_rows, rec.data_ptr()) == _lib.E_INVALID
        assert counts(max_d=max_d, max_rows=max_rows) == _lib.E_INVALID
    assert lib.spgg_strip_pair_record(h, md, mr, None) == _lib.E_INVALID
    assert lib.spgg_strip_pair_counts(h, 2, rank, None, md, mr, out.ctypes.data) == _lib.E_INVALID
    assert lib.spgg_strip_pair_counts(h, 2, rank, rec.data_ptr(), md, mr, None) == _lib.E_INVALID
    se.close()
    dist.barrier()


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
            large(rank, world, int(sys.argv[3]), int(sys.argv[4]))
        elif mode == "world1":
            world_one(rank, world)
        elif mode == "errors":
            errors(rank, world)
        else:
            raise SystemExit(f"unknown mode {mode}")
    finally:
        dist.destroy_process_group()
    print(f"rank {rank} ok")


if __name__ == "__main__":
    main()
