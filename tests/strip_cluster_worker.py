"""Worker processes of tests/test_gpu_strip_clusters.py (one rank each, RANK / WORLD_SIZE /
MASTER_ADDR / MASTER_PORT in the environment): cluster labelling of a lattice split into row strips
(StripEngine.cluster_sizes / cluster_labels, include/spgg.h: spgg_strip_clusters) against scipy, the
torus oracle and one handle holding the whole lattice."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

COMBOS = (("C", False), ("D", False), ("C", True), ("D", True))


def _expected(S, of, periodic):
    from scipy.ndimage import label
    from test_clusters_host import periodic_label
    m = np.asarray(S) == (0 if of == "C" else 1)
    if periodic:
        return periodic_label(m)
    lab, n = label(m)
    return lab.astype(np.int32), n


def _path(L, precision="fp32"):
    return "fast" if precision == "fp32" and L % 32 == 0 and L >= 128 else "general"


def _serpentine(L):
    S = np.ones((L, L), np.uint8)
    S[::2, :] = 0
    for i in range(1, L, 2):
        S[i, L - 1 if (i // 2) % 2 == 0 else 0] = 0
    return S


def patterns(L, row0s, rows):
    """(name, S) with S == 0 the cooperators; row0s / rows: the strips of the partition."""
    ii, jj = np.indices((L, L))
    yield "all C", np.zeros((L, L), np.uint8)
    yield "all D", np.ones((L, L), np.uint8)
    yield "checkerboard", ((ii + jj) % 2).astype(np.uint8)
    yield "vertical stripes", (jj % 2).astype(np.uint8)
    yield "horizontal stripes", (ii % 2).astype(np.uint8)
    yield "serpentine", _serpentine(L)
    comb = np.ones((L, L), np.uint8)
    comb[0, :] = 0
    comb[:, ::2] = 0
    yield "comb", comb
    ring = np.ones((L, L), np.uint8)
    ring[:, L // 3] = 0                                  # a vertical ring: one cluster on the torus and off it
    ring[: L // 4, 2 * L // 3] = 0                       # two pieces that join only across row L-1 | 0
    ring[L - L // 4:, 2 * L // 3] = 0
    yield "vertical ring", ring
    rs = np.random.RandomState(L)
    for k in range(len(row0s)):                          # one strip with every row selected, noise elsewhere
        S = (rs.rand(L, L) < 0.5).astype(np.uint8)
        S[row0s[k]:row0s[k] + rows[k]] = 0
        yield f"strip {k} all C", S
    for p in (0.3, 0.5, 0.593, 0.7):
        yield f"random {p}", (rs.rand(L, L) >= p).astype(np.uint8)


def _state(L, nq=4):
    return np.zeros((L, L)), np.zeros((L, L) + ((2, 2) if nq == 4 else (2, 2, 2)))


def _check_strip(se, S, rank, eng=None, combos=COMBOS, labels=True, name=""):
    a, b = se.row0, se.row0 + se.rows
    for of, periodic in combos:
        want, n = _expected(S, of, periodic)
        sizes = se.cluster_sizes(of=of, periodic=periodic)
        what = f"{name} L={se.L} of={of} periodic={periodic}"
        assert sizes.dtype == np.int64 and len(sizes) == n, (what, len(sizes), n)
        assert np.array_equal(sizes, np.bincount(want.ravel(), minlength=n + 1)[1:]), what
        if labels:
            got, ng = se.cluster_labels(of=of, periodic=periodic)
            assert ng == n and got.dtype == np.int32 and got.shape == (se.rows, se.L), what
            assert np.array_equal(got, want[a:b]), (what, int((got != want[a:b]).sum()))
        if eng is not None and rank == 0:
            assert np.array_equal(eng.cluster_sizes(of=of, periodic=periodic), sizes), what
            if labels:
                assert np.array_equal(eng.cluster_labels(of=of, periodic=periodic)[0], want), what


def geometries(rank, world, Ls):
    """Uploaded patterns: gathered labels and sizes == scipy / the torus oracle == one whole-lattice handle."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    for L in Ls:
        p = full_params(dict(C1, L=L))
        se = strips.StripEngine(p, seed=5, precision="fp32", device=dev)
        assert se.eng.describe().startswith(_path(L)), se.eng.describe()
        parts = [None] * world
        dist.all_gather_object(parts, (se.row0, se.rows))
        eng = spgg_b200.Engine(p, seeds=5, precision="fp32", device=dev) if rank == 0 else None
        R0, Q0 = _state(L)
        big = L >= 2048
        for name, S in patterns(L, [q[0] for q in parts], [q[1] for q in parts]):
            if big and not name.startswith(("random", "serpentine", "vertical ring")):
                continue
            se.set_state_global(S, R0, Q0)
            if eng is not None:
                eng.set_state(S, R0, Q0)
            _check_strip(se, S, rank, eng, name=name)
        se.close()
        if eng is not None:
            eng.close()
        dist.barrier()


def dynamics(rank, world, which_case):
    """States from the dynamics, stepped in chunks: after each chunk the strips' sizes == the single
    handle's (same seed); labelling between chunks leaves the strip run's digests unchanged."""
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
    for labelled in (True, False):
        se = strips.StripEngine(p, seed=31, precision=precision, device=dev)
        assert se.eng.describe().startswith(_path(L, precision)), se.eng.describe()
        se.init_random(9)
        got = []
        for c in chunks:
            se.step(c)
            if labelled:
                got.append([se.cluster_sizes(of=of, periodic=per) for of, per in COMBOS])
                lab, n = se.cluster_labels(of="D", periodic=True)
                assert n == len(got[-1][3])
        out[labelled] = se.digest()
        if labelled:
            if os.environ.get("SPGG_SPEC_TEST_POISON") and se.spec_mode:
                assert se.reruns > 0, "the spoiled guesses were not re-run"
            S = se.gather_state(want_q=False)[0]
        se.close()
        if labelled and rank == 0:
            eng = spgg_b200.Engine(p, seeds=31, precision=precision, device=dev)
            eng.init_random(9)
            for c, sizes in zip(chunks, got):
                eng.step(c)
                for (of, per), s in zip(COMBOS, sizes):
                    assert np.array_equal(eng.cluster_sizes(of=of, periodic=per), s), (which_case, c, of, per)
            assert np.array_equal(eng.get_state(want_q=False)[0], S)
            eng.close()
        dist.barrier()
    assert out[True] == out[False], "labelling between chunks changed the run"


def large(rank, world, L, n_steps):
    """A large lattice from init_random + a few steps; the whole-lattice handle on rank 0 is created after
    the strips are closed."""
    import torch
    import torch.distributed as dist
    import spgg_b200
    from spgg_b200 import strips
    from helpers import C1, full_params
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    p = full_params(dict(C1, L=L))
    combos = (("C", False), ("D", True))
    se = strips.StripEngine(p, seed=4, precision="fp32", device=dev)
    assert se.eng.describe().startswith(_path(L)), se.eng.describe()
    se.init_random(12)
    se.step(n_steps)
    got = [se.cluster_sizes(of=of, periodic=per) for of, per in combos]
    lab, n = se.cluster_labels()
    assert n == len(got[0]) and lab.max() <= n and lab.min() >= 0
    se.close()
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        eng = spgg_b200.Engine(p, seeds=4, precision="fp32", device=dev)
        eng.init_random(12)
        eng.step(n_steps)
        for (of, per), s in zip(combos, got):
            want = eng.cluster_sizes(of=of, periodic=per)
            assert np.array_equal(want, s), (of, per, len(want), len(s))
        eng.close()
    dist.barrier()


def world_one(rank, world):
    """A StripEngine of world 1 (whole-lattice handle through the strip entry points) == spgg_clusters."""
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
        for name, S in patterns(L, [0], [L]):
            se.set_state_global(S, R0, Q0)
            eng.set_state(S, R0, Q0)
            _check_strip(se, S, 0, eng, name=name)
        se.init_random(3)
        se.step(5)
        eng.set_state(*se.gather_state())
        _check_strip(se, se.gather_state(want_q=False)[0], 0, eng, name="after steps")
        se.close()
        eng.close()


def errors(rank, world):
    """Getters need a resolved pass of the current state; the resolution rejects records that do not
    describe one labelling of one lattice."""
    import torch
    import torch.distributed as dist
    from spgg_b200 import strips, _lib
    from helpers import C1, full_params
    assert world == 2
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    L = 64
    se = strips.StripEngine(full_params(dict(C1, L=L)), seed=1, precision="fp32", device=dev)
    lib, h = se.lib, se.h
    sizes = np.zeros(L * L, np.int64)
    labels = np.zeros(L * L, np.int32)
    nb = int(lib.spgg_strip_cluster_record_bytes(h))
    assert nb > 0
    rec = torch.zeros(3 * nb, dtype=torch.uint8, device=dev)
    n, first, tot = C.c_int64(), C.c_int64(), C.c_int64()

    def getters_fail():
        assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, 0) == _lib.E_STATE
        assert lib.spgg_cluster_labels(h, labels.ctypes.data) == _lib.E_STATE

    def gather(which, flags):
        """This strip's record into slot `rank` of rec, then the records of both ranks everywhere."""
        mine = rec[rank * nb:(rank + 1) * nb]
        assert lib.spgg_strip_clusters(h, which, flags, mine.data_ptr()) == 0
        torch.cuda.synchronize()
        host = mine.cpu()
        parts = [torch.empty_like(host) for _ in range(world)]
        dist.all_gather(parts, host)
        rec[:2 * nb].copy_(torch.cat(parts).to(dev))
        torch.cuda.synchronize()

    def resolve(w=2, r=rank, buf=None):
        return lib.spgg_strip_clusters_resolve(h, w, r, (rec if buf is None else buf).data_ptr(),
                                               C.byref(n), C.byref(first), C.byref(tot))

    getters_fail()
    se.init_random(3)
    getters_fail()
    gather(0, 0)
    getters_fail()                                           # a pass that is not resolved yet
    assert resolve() == 0
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value) == 0
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value + 1) == _lib.E_INVALID
    assert lib.spgg_cluster_labels(h, labels.ctypes.data) == 0
    assert resolve() == _lib.E_STATE                         # the pass was consumed
    se.step(2)
    getters_fail()
    gather(0, 0)
    assert resolve() == 0
    S, R, Q = se.get_state_local()
    se.set_state_local(S, R, Q)
    getters_fail()
    gather(0, 0)
    assert resolve() == 0
    gather(1, 0)                                             # a new pass discards the resolved result
    getters_fail()
    # records that do not describe one labelling of the lattice
    gather(rank, 0)                                          # which differs between the ranks
    assert resolve() == _lib.E_INVALID
    getters_fail()
    gather(0, rank)                                          # flags differ
    assert resolve() == _lib.E_INVALID
    gather(0, 0)
    assert resolve(w=1, r=0) == _lib.E_INVALID               # one record does not cover the lattice
    assert resolve(w=3) == _lib.E_INVALID                    # the third record is not a record
    assert resolve(w=2, r=2) == _lib.E_INVALID
    swapped = torch.cat([rec[nb:2 * nb], rec[:nb]])
    assert resolve(buf=swapped) == _lib.E_INVALID            # rows out of rank order
    assert resolve() == 0                                    # the pass survives rejected resolutions
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value) == 0
    assert lib.spgg_strip_clusters(h, 2, 0, rec.data_ptr()) == _lib.E_INVALID
    assert lib.spgg_strip_clusters(h, 0, 2, rec.data_ptr()) == _lib.E_INVALID
    assert lib.spgg_strip_clusters(h, 0, 0, None) == _lib.E_INVALID
    se.close()
    # a re-run from a wrong guess of the global maximum (spgg_strip_rewind) leaves no result behind
    os.environ["SPGG_SPEC_TEST_POISON"] = "3"
    try:
        se = strips.StripEngine(full_params(dict(C1, L=256)), seed=1, precision="fp32", device=dev)
    finally:
        del os.environ["SPGG_SPEC_TEST_POISON"]
    assert se.eng.describe().startswith("fast")
    se.init_random(3)
    se.cluster_sizes()
    se.step(12)
    se.sync()
    assert se.reruns > 0
    assert se.lib.spgg_cluster_sizes(se.h, sizes.ctypes.data, 0) == _lib.E_STATE
    se.close()
    dist.barrier()


def main():
    import torch.distributed as dist
    mode = sys.argv[1]
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group(sys.argv[2], rank=rank, world_size=world)
    try:
        if mode == "geometries":
            geometries(rank, world, [int(x) for x in sys.argv[3].split(",")])
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
