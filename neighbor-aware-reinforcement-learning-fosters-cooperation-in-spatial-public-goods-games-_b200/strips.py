"""Row-strip decomposition of one large lattice over the GPUs of a node
(BASELINE config 5: L=32768 at 2/4/8 B200), one process per GPU.

The reference has no distributed mode (its only parallelism is one process per parameter
tuple, ``src/experiments/runner.py:117-156``); what the strips must reproduce is the
single-lattice loop body ``src/model/spgg.py:368-592``.  Only two things cross a strip
boundary in that loop:

* the stencils read neighbours' R (radius M, ``spgg.py:292-307``), strategy bits (radius 2,
  ``spgg.py:373-377``) and reward codes (radius M, ``spgg.py:478-486``)  ->  one halo
  exchange per iteration: ``GH`` boundary rows of the three planes, packed into one
  contiguous buffer per direction (``spgg_halo_pack`` / ``spgg_halo_unpack``);
* ``global_max = np.max(np.abs(diffs))`` (``spgg.py:488``) is lattice-global  ->  one scalar
  all-reduce(MAX) per iteration between the light k_gmax kernel and the fused k_step.

Q is strictly site-local and never moves.  The Philox counters are keyed on the *global*
row and column, so an N-strip run is bit-identical (S, R, Q, integer statistics) to the
single-GPU run of the same seed (tests/test_gpu_strips.py).

``torch.distributed`` (NCCL over NVLink on the GPU box, gloo in the CPU tests) is the
transport; the kernels come from the C ABI.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import time
from typing import Sequence

import numpy as np

from . import _lib as L_

# stat columns that are not plain sums over sites
_MAX_COLS = (L_.ST_GMAX,)


# ------------------------------------------------------------------ partition (pure host logic)
def strip_rows(L: int, world: int, rank: int, align: int = 16) -> tuple[int, int]:
    """(row0, rows) of strip ``rank``: contiguous blocks of rows, multiples of ``align``
    (the fast kernel's tile height) while the lattice allows it; remainders go to the first strips."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    unit = align if (L % align == 0 and L // align >= world) else 1
    blocks = L // unit
    if blocks < world:
        raise ValueError(f"L={L} cannot be split into {world} strips")
    base, extra = divmod(blocks, world)
    nb = base + (1 if rank < extra else 0)
    b0 = rank * base + min(rank, extra)
    rows, row0 = nb * unit, b0 * unit
    if rows < 4:
        raise ValueError(f"strips of {rows} rows are thinner than the two ghost-row halos")
    return row0, rows


def assemble_block_fields(L: int, b: int, world: int, parts) -> tuple[np.ndarray, np.ndarray]:
    """The whole lattice's block fields from the strips' (``StripEngine.block_fields``): ``parts[k]`` is rank
    k's (counts, sums), counts int64 (nI, B, 2) and sums float64 (nI, B, 2, m) over the block rows holding
    its rows (``engine.block_rows``), possibly padded past nI.  The strips are added in rank order into
    (B, B, 2) and (B, B, 2, m): integer channels exactly, float channels in an order fixed by the partition."""
    from .engine import block_rows
    B = -(-L // b)
    m = parts[0][1].shape[-1]
    counts = np.zeros((B, B, 2), np.int64)
    sums = np.zeros((B, B, 2, m))
    for k in range(world):
        row0, rows = strip_rows(L, world, k)
        I0, nI = block_rows(L, b, row0, rows)
        counts[I0:I0 + nI] += parts[k][0][:nI]
        sums[I0:I0 + nI] += parts[k][1][:nI]
    return counts, sums


def neighbours(world: int, rank: int) -> tuple[int, int]:
    """(up, down): ranks owning the rows just above (row0-1) and just below; periodic."""
    return (rank - 1) % world, (rank + 1) % world


def exchange_halos(dist, to_up, to_down, from_up, from_down, rank: int, world: int, group=None):
    """One halo exchange: my top rows go to ``up`` (they become its bottom ghosts), my
    bottom rows to ``down``.  Sends are posted [up, down], receives [down, up]: with two
    ranks both neighbours are the same peer and messages between a pair match in order."""
    up, down = neighbours(world, rank)
    if world == 1:
        from_down.copy_(to_up)       # my own top rows are the ghosts below my last row
        from_up.copy_(to_down)
        return
    ops = [dist.P2POp(dist.isend, to_up, up, group), dist.P2POp(dist.isend, to_down, down, group),
           dist.P2POp(dist.irecv, from_down, down, group), dist.P2POp(dist.irecv, from_up, up, group)]
    for w in dist.batch_isend_irecv(ops):
        w.wait()


def reduce_stat_rows(dist, rows, world: int, device=None, group=None):
    """Per-strip statistic rows (sums over the strip's sites) -> whole-lattice rows on every
    rank.  Counts are exact integers in doubles, so their sum is exact; ST_GMAX is a max."""
    import torch
    rows = np.ascontiguousarray(rows, dtype=np.float64)
    if world == 1:
        return rows
    t = torch.from_numpy(rows.copy())
    if device is not None and dist.get_backend(group) != "gloo":
        t = t.to(device)
    mx = t[:, list(_MAX_COLS)].clone()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    t[:, list(_MAX_COLS)] = mx
    return t.cpu().numpy()


class _DevArray:
    """Zero-copy view of device memory owned by the C library as a torch tensor."""

    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


# ------------------------------------------------------------------ the strip engine
class StripEngine:
    """One strip of an ``L x L`` lattice on this process's GPU.  ``params`` uses the
    reference ctor's argument names (spgg.py:50-56).

    Per iteration (TMA fast path): ONE fused launch that guesses the lattice-global maximum
    (spgg.py:488) and reports the strip's own; beside the halo exchange of the rows it just wrote, a
    second stream max-reduces the 4-float report over the ranks (its own communicator) and a
    one-thread kernel compares it with the guess, keeps it as the next guess and raises the
    uniform-lattice stop flag of spgg.py:405.  A wrong guess is re-run (``_settle``); every rank
    sees the same reduced values, so every rank takes the same decision without talking.
    Strips that cannot use the fast path (fp64, unaligned L, other TD rules) run the exact pair
    k_gmax -> all-reduce(MAX) -> k_step per iteration."""

    def __init__(self, params: dict, seed: int = 0, precision: str = "fp32", device: int | None = None,
                 group=None):
        import torch
        import torch.distributed as dist
        from .engine import Engine
        self.torch, self.dist, self.group = torch, dist, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.L = int(params.get("L", 50))
        self.row0, self.rows = strip_rows(self.L, self.world, self.rank)
        self.device = int(torch.cuda.current_device() if device is None else device)
        self.precision = precision
        # every strip uses the same Philox key: counters carry the global row
        self.eng = Engine(params, seeds=seed, precision=precision, device=self.device,
                          rows=self.rows, row0=self.row0)
        self.lib, self.h = self.eng.lib, self.eng._h
        nb = int(self.lib.spgg_halo_bytes(self.h))
        dev = torch.device("cuda", self.device)
        self.dev = dev
        self.buf = {k: torch.empty(nb, dtype=torch.uint8, device=dev)
                    for k in ("to_up", "to_down", "from_up", "from_down")}
        self._gtype = "<f8" if precision == "fp64" else "<f4"
        # gloo (CPU tests, or several ranks sharing one GPU) moves the halos through the host
        self.host_staged = dist.is_initialized() and dist.get_backend(group) == "gloo"
        if self.host_staged:
            self.hbuf = {k: torch.empty(nb, dtype=torch.uint8).pin_memory() for k in self.buf}
        # the report reduce runs beside the halo exchange: its own stream and its own communicator
        self.side = torch.cuda.Stream(device=dev)
        self.group2 = None
        if self.world > 1 and not self.host_staged:
            ranks = dist.get_process_group_ranks(group) if group is not None else list(range(self.world))
            self.group2 = dist.new_group(ranks=ranks)
        # peer-mapped halos: with NCCL (one GPU per rank, NVLink) the neighbours map each other's planes and
        # the boundary tiles store their rows straight into the neighbour's ghost rows
        self.p2p = False
        self.ring = False
        if self.world > 1 and not self.host_staged and os.environ.get("SPGG_NO_P2P_HALO") is None:
            self.p2p = self._attach_neighbours()
        self.iteration = 0
        self._last_n = 0
        self._open = 0          # iterations of the chunk still to be settled (0: none)
        self._side_ev = None
        self.spec_mode = False
        self.reruns = 0
        self._uniform_start = False

    def _attach_neighbours(self) -> bool:
        """Exchange the IPC handles of the planes with the two neighbours (all ranks take part).  False -
        on every rank - if any rank could not map its neighbours: the NCCL halo exchange stays."""
        dist, lib, h = self.dist, self.lib, self.h
        mine = (C.c_ubyte * 384)()
        ok = lib.spgg_ipc_export(h, mine) == 0
        everyone: list = [None] * self.world
        dist.all_gather_object(everyone, (bytes(mine) if ok else None, self.rows), group=self.group)
        up, down = neighbours(self.world, self.rank)
        if ok and all(e[0] is not None for e in everyone):
            for which, peer in ((0, up), (1, down)):
                same = 1 if (which == 1 and down == up) else 0
                buf = (C.c_ubyte * 384).from_buffer_copy(everyone[peer][0])
                if lib.spgg_ipc_attach(h, which, buf, int(everyone[peer][1]), same) != 0:
                    ok = False
                    break
        else:
            ok = False
        flags: list = [None] * self.world
        dist.all_gather_object(flags, bool(ok), group=self.group)
        if not all(flags):
            return False
        # the ring of report slots: every rank maps every rank's
        self.ring = False
        if os.environ.get("SPGG_NO_RING") is None and self.world <= 16:
            one = (C.c_ubyte * 64)()
            ok = lib.spgg_ring_export(h, one) == 0
            rings: list = [None] * self.world
            dist.all_gather_object(rings, bytes(one) if ok else None, group=self.group)
            if all(r is not None for r in rings):
                allh = (C.c_ubyte * (64 * self.world)).from_buffer_copy(b"".join(rings))
                ok = lib.spgg_ring_attach(h, self.world, self.rank, allh) == 0
            else:
                ok = False
            dist.all_gather_object(flags, bool(ok), group=self.group)
            self.ring = all(flags)
            if not self.ring and ok:
                raise RuntimeError("some rank could not map the report rings; set SPGG_NO_RING=1")
        return True

    # -- state
    def set_state_global(self, S, R, Q):
        """Every rank passes the whole lattice (or anything indexable by global row, e.g. a
        memory-mapped array); each uploads only its own rows."""
        a, b = self.row0, self.row0 + self.rows
        self.set_state_local(np.asarray(S[a:b]), np.asarray(R[a:b]), np.asarray(Q[a:b]))

    def set_state_local(self, S, R, Q):
        """This rank's own rows only: arrays of ``rows`` x L sites (global rows row0 .. row0+rows)."""
        self._settle()
        self.eng.set_state(S, R, Q)
        self.iteration = 0
        # a lattice that is uniform from the start never acts (spgg.py:405 breaks in iteration 1)
        S = np.asarray(S)
        flags = np.array([float((S != 0).any()), float((S == 0).any())])    # holds a D / holds a C
        if self.world > 1:
            t = self.torch.from_numpy(flags)
            if not self.host_staged:
                t = t.to(self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
            flags = t.cpu().numpy()
        self._uniform_start = bool(flags[0] == 0.0 or flags[1] == 0.0)

    def init_random(self, seed: int):
        self._settle()
        self.eng.init_random(seed)
        self.iteration = 0
        self._uniform_start = False
        if self.ring:
            self.dist.barrier(group=self.group)   # a new run empties the rings: nobody pushes before all did

    def get_state_local(self, want_q=True):
        self._settle()
        return self.eng.get_state(want_q=want_q)

    def gather_state(self, want_q=True):
        """Whole lattice on every rank (test / small-lattice helper)."""
        self._settle()
        S, R, Q = self.eng.get_state(want_q=want_q)
        if self.world == 1:
            return S, R, Q
        parts: list = [None] * self.world
        self.dist.all_gather_object(parts, (S, R, Q), group=self.group)
        cat = lambda i: np.concatenate([p[i] for p in parts], axis=0)
        return cat(0), cat(1), (cat(2) if want_q else None)

    def digest(self):
        """(S, R, Q) digests of the WHOLE lattice: the strips' digests add up modulo 2^64
        (include/spgg.h: spgg_state_digest)."""
        self._settle()
        d = np.array(self.eng.digest(), dtype=np.uint64)
        if self.world == 1:
            return tuple(int(x) for x in d)
        parts: list = [None] * self.world
        self.dist.all_gather_object(parts, [int(x) for x in d], group=self.group)
        return tuple(sum(p[i] for p in parts) % 2 ** 64 for i in range(3))

    # -- clusters (include/spgg.h: spgg_strip_clusters)
    def _clusters(self, of, periodic) -> int:
        """Label the whole lattice: strip-local pass, one all-gather of the boundary records, resolution
        on every rank.  Returns the number of clusters this strip owns; ``_n_total``: those of the lattice."""
        return self._resolve_records(self._gather_records(self._label_strip(of, periodic)))

    def _label_strip(self, of, periodic):
        """Strip-local labelling; returns the device buffer of all ranks' records with this rank's filled in."""
        from .engine import cluster_which
        lib, h = self.lib, self.h
        which = cluster_which(of)
        self._settle()
        nb = int(lib.spgg_strip_cluster_record_bytes(h))
        L_.check(min(nb, 0))
        rec = self.torch.empty(self.world * nb, dtype=self.torch.uint8, device=self.dev)
        mine = rec[self.rank * nb:(self.rank + 1) * nb]
        L_.check(lib.spgg_strip_clusters(h, which, L_.CLUSTER_PERIODIC if periodic else 0, mine.data_ptr()))
        return rec

    def _gather_records(self, rec):
        """The one collective of the labelling: every rank's record into every rank's buffer, in rank order."""
        torch = self.torch
        if self.world == 1:
            return rec
        nb = rec.numel() // self.world
        mine = rec[self.rank * nb:(self.rank + 1) * nb]
        if self.host_staged:
            hrec = torch.empty(rec.numel(), dtype=torch.uint8).pin_memory()
            hmine = torch.empty(nb, dtype=torch.uint8).pin_memory()
            hmine.copy_(mine)
            self.dist.all_gather(list(hrec.split(nb)), hmine, group=self.group)
            rec.copy_(hrec)
        else:
            self.dist.all_gather_into_tensor(rec, mine.clone(), group=self.group)
        torch.cuda.current_stream().synchronize()
        return rec

    def _resolve_records(self, rec) -> int:
        n, first, total = C.c_int64(), C.c_int64(), C.c_int64()
        L_.check(self.lib.spgg_strip_clusters_resolve(self.h, self.world, self.rank, rec.data_ptr(), C.byref(n),
                                                      C.byref(first), C.byref(total)))
        self._n_total = int(total.value)
        return int(n.value)

    def _owned_sizes(self, n: int) -> np.ndarray:
        sizes = np.empty(n, np.int64)
        L_.check(self.lib.spgg_cluster_sizes(self.h, sizes.ctypes.data, n))
        return sizes

    def _gather_sizes(self, sizes: np.ndarray) -> np.ndarray:
        """Every rank's owned sizes, concatenated in rank order (= label order), on every rank."""
        torch = self.torch
        if self.world == 1:
            return sizes
        counts = [None] * self.world
        self.dist.all_gather_object(counts, len(sizes), group=self.group)
        pad = max(max(counts), 1)
        t = torch.zeros(pad, dtype=torch.int64)
        t[:len(sizes)] = torch.from_numpy(sizes)
        if self.host_staged:
            parts = [torch.empty_like(t) for _ in range(self.world)]
            self.dist.all_gather(parts, t, group=self.group)
            out = torch.cat([p[:c] for p, c in zip(parts, counts)])
        else:
            td = t.to(self.dev)
            allp = torch.empty(self.world * pad, dtype=torch.int64, device=self.dev)
            self.dist.all_gather_into_tensor(allp, td, group=self.group)
            out = torch.cat([p[:c] for p, c in zip(allp.split(pad), counts)]).cpu()
        return out.numpy()

    def cluster_sizes(self, of="C", periodic: bool = False) -> np.ndarray:
        """``Engine.cluster_sizes`` of the WHOLE lattice (all ranks call this; every rank gets the same
        int64 array): sizes of the 4-connected clusters of cooperators (``of="C"``) or defectors (``"D"``)
        in the order of each cluster's first site in raster order, ``periodic=True`` joining clusters
        across the edges of the torus."""
        return self._gather_sizes(self._owned_sizes(self._clusters(of, periodic)))

    def cluster_labels(self, of="C", periodic: bool = False):
        """This rank's rows of ``scipy.ndimage.label(S == of)`` over the whole lattice (all ranks call
        this): (labels int32 (rows, L), n) with n the number of clusters of the lattice."""
        self._clusters(of, periodic)
        labels = np.empty((self.rows, self.L), np.int32)
        L_.check(self.lib.spgg_cluster_labels(self.h, labels.ctypes.data))
        return labels, self._n_total

    # -- strategy pair counts (include/spgg.h: spgg_strip_pair_counts)
    def pair_counts(self, max_d: int) -> np.ndarray:
        """``Engine.pair_counts`` of the WHOLE lattice (all ranks call this; every rank gets the same int64
        array of shape (2, max_d+1, 2)): each strip counts the pairs whose first site it owns, from its own
        rows and the first rows of the strips below it (one all-gather of fixed-size records); the counts
        are summed over the ranks."""
        lib, h, torch = self.lib, self.h, self.torch
        max_d = int(max_d)
        self._settle()
        # the padding every rank agrees on: no strip holds more rows than the largest
        max_rows = min(max_d, max(strip_rows(self.L, self.world, r)[1] for r in range(self.world)))
        nb = int(lib.spgg_strip_pair_record_bytes(h, max_d, max_rows))
        L_.check(min(nb, 0))
        rec = torch.empty(self.world * nb, dtype=torch.uint8, device=self.dev)
        L_.check(lib.spgg_strip_pair_record(h, max_d, max_rows, rec[self.rank * nb:(self.rank + 1) * nb].data_ptr()))
        rec = self._gather_records(rec)
        out = np.zeros((2, max_d + 1, 2), np.int64)
        L_.check(lib.spgg_strip_pair_counts(h, self.world, self.rank, rec.data_ptr(), max_d, max_rows, out.ctypes.data))
        if self.world == 1:
            return out
        t = torch.from_numpy(out)
        if not self.host_staged:
            t = t.to(self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t.cpu().numpy()

    # -- block fields (include/spgg.h: spgg_block_fields)
    def block_fields(self, b: int, fields=("R", "Q")) -> dict:
        """``Engine.block_fields`` of the WHOLE lattice (all ranks call this; every rank gets the same dict of
        (B, B) arrays): each strip sums its own rows over the block rows they touch, the partials are
        all-gathered (padded to the largest block-row count) and added in rank order
        (``assemble_block_fields``)."""
        from .engine import block_flags, block_result, block_rows
        torch = self.torch
        flags = block_flags(fields)
        b = int(b)
        self._settle()
        part = self.eng.block_fields(b, fields=fields)
        nq = self.eng.nq
        m = (1 if flags & L_.BLOCK_R else 0) + (nq if flags & L_.BLOCK_Q else 0)
        nI = part["n"].shape[0]
        counts = np.stack([part["n"], part["n_C"]], axis=-1)
        sums = np.zeros(counts.shape[:2] + (2, m))
        if flags & L_.BLOCK_R:
            sums[..., 0] = part["R"]
        if flags & L_.BLOCK_Q:
            sums[..., m - nq:] = part["Q"].reshape(sums.shape[:3] + (nq,))
        if self.world > 1:
            pad = max(block_rows(self.L, b, *strip_rows(self.L, self.world, r))[1] for r in range(self.world))
            B, w = counts.shape[1], counts.shape[1] * 2 * (1 + m)
            # counts and the bytes of the sums travel as one int64 tensor per rank
            t = torch.zeros((pad, w), dtype=torch.int64)
            t[:nI] = torch.from_numpy(np.concatenate([counts.reshape(nI, -1), sums.reshape(nI, -1).view(np.int64)], 1))
            if self.host_staged:
                got = [torch.empty_like(t) for _ in range(self.world)]
                self.dist.all_gather(got, t, group=self.group)
            else:
                allp = torch.empty((self.world * pad, w), dtype=torch.int64, device=self.dev)
                self.dist.all_gather_into_tensor(allp, t.to(self.dev), group=self.group)
                got = list(allp.cpu().split(pad))
            parts = []
            for g in got:
                a = g.numpy()
                parts.append((a[:, :B * 2].reshape(pad, B, 2), a[:, B * 2:].copy().view(np.float64).reshape(pad, B, 2, m)))
            counts, sums = assemble_block_fields(self.L, b, self.world, parts)
        return block_result(counts, sums, flags, (2, 2) if nq == 4 else (2, 2, 2))

    # -- stepping
    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def _exchange(self, st):
        b = self.buf
        L_.check(self.lib.spgg_halo_pack(self.h, b["to_up"].data_ptr(), b["to_down"].data_ptr(), st))
        if self.host_staged:
            hb = self.hbuf
            hb["to_up"].copy_(b["to_up"]); hb["to_down"].copy_(b["to_down"])
            self.torch.cuda.current_stream().synchronize()
            exchange_halos(self.dist, hb["to_up"], hb["to_down"], hb["from_up"], hb["from_down"],
                           self.rank, self.world, self.group)
            b["from_up"].copy_(hb["from_up"]); b["from_down"].copy_(hb["from_down"])
        else:
            exchange_halos(self.dist, b["to_up"], b["to_down"], b["from_up"], b["from_down"],
                           self.rank, self.world, self.group)
        L_.check(self.lib.spgg_halo_unpack(self.h, b["from_up"].data_ptr(), b["from_down"].data_ptr(), st))

    def _reduce_max(self, t, group):
        if self.world == 1:
            return
        if self.host_staged:
            th = t.cpu()
            self.dist.all_reduce(th, op=self.dist.ReduceOp.MAX, group=group)
            t.copy_(th)
        else:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=group)

    def _report_and_verify(self):
        """After a launch: max-reduce its report over the ranks and let the device act on it
        (guess check, next guess, stop flag) - on the side stream, beside the halo exchange."""
        torch = self.torch
        ptr = self.lib.spgg_strip_report_ptr(self.h)
        rep = torch.as_tensor(_DevArray(ptr, 4, "<f4"), device=self.dev)
        main = torch.cuda.current_stream()
        if self.ring:
            # the ranks combined their reports themselves (system-scope atomics into every rank's ring);
            # one thread waits on the device until all are in and takes the verdict
            L_.check(self.lib.spgg_strip_verify(self.h, self._stream()))
            self._side_ev = None
            return
        if self.world == 1 or self.host_staged:
            self._reduce_max(rep, self.group)
            L_.check(self.lib.spgg_strip_verify(self.h, self._stream()))
            self._side_ev = None
            return
        ev = torch.cuda.Event()
        ev.record(main)
        self.side.wait_event(ev)
        with torch.cuda.stream(self.side):
            self.dist.all_reduce(rep, op=self.dist.ReduceOp.MAX, group=self.group2)
            L_.check(self.lib.spgg_strip_verify(self.h, C.c_void_p(self.side.cuda_stream)))
            self._side_ev = torch.cuda.Event()
            self._side_ev.record(self.side)

    def _join_side(self):
        if self._side_ev is not None:
            self.torch.cuda.current_stream().wait_event(self._side_ev)
            self._side_ev = None

    def _iteration(self, s: int, n: int, gtab):
        """Finish iteration s of the chunk (and choose the action of s+1 unless it is the last)."""
        lib, h = self.lib, self.h
        st = self._stream()
        sel = 1 if s < n else 0
        if not (self.p2p and self.spec_mode):
            self._exchange(st)                               # codes / R / strategies just written
        if self.spec_mode:
            # the verdict on the previous launch; with peer-mapped halos this reduce is also what orders
            # the neighbours' stores into my ghost rows before my next launch reads them
            self._join_side()
            if lib.spgg_strip_can_speculate(h, sel):
                L_.check(lib.spgg_strip_iteration(h, sel, st))
            else:                                            # no guess yet: the exact pair
                L_.check(lib.spgg_phase_gmax(h, st))
                self._reduce_max(gtab[s:s + 1], self.group)
                L_.check(lib.spgg_phase_kernel(h, 1, sel, st))
            self._report_and_verify()
            return
        L_.check(lib.spgg_phase_gmax(h, st))                 # strip-local max |reward difference|
        self._reduce_max(gtab[s:s + 1], self.group)          # spgg.py:488 is lattice-global
        L_.check(lib.spgg_phase_kernel(h, 1, sel, st))

    def step(self, n: int):
        """n iterations of spgg.py:368-592 over the whole lattice (all ranks call this)."""
        self._settle()
        if self._uniform_start:
            self._last_n = 0
            return
        lib, h = self.lib, self.h
        st = self._stream()
        L_.check(lib.spgg_begin_steps(h, int(n), st))
        # device table of the per-iteration maxima of this call: entry s belongs to iteration s
        self._gtab = self.torch.as_tensor(_DevArray(lib.spgg_gmax_device_ptr(h), n + 1, self._gtype),
                                          device=self.dev)
        self._exchange(st)                                   # ghosts of the starting state
        L_.check(lib.spgg_phase_kernel(h, 0, 1, st))         # action of the first iteration
        self.spec_mode = bool(lib.spgg_strip_report_ptr(h))
        if self.spec_mode:
            self._report_and_verify()                        # a uniform lattice stops here (spgg.py:405)
        for s in range(1, n + 1):
            self._iteration(s, n, self._gtab)
        L_.check(lib.spgg_end_steps(h, st))
        self._last_n = int(n)
        self._open = int(n)

    def _settle(self):
        """Close the chunk: wait for both streams, re-run from the first wrong guess (if any; the
        same launch on every rank), then let the library finish its bookkeeping."""
        if not self._open:
            return
        n = self._open
        while True:
            self._join_side()
            self.torch.cuda.current_stream().synchronize()
            bad = int(self.lib.spgg_strip_failed(self.h)) if self.spec_mode else 0
            if bad <= 0:
                break
            self.reruns += 1
            L_.check(self.lib.spgg_strip_rewind(self.h, bad))
            if self.ring:
                self.dist.barrier(group=self.group)   # every ring is empty before anyone pushes again
            for s in range(bad, n + 1):
                self._iteration(s, n, self._gtab)
        self._open = 0
        self.eng.sync()
        st = self.eng.status()
        self.iteration = int(st.iteration)

    def sync(self):
        self._settle()

    def stats_local(self):
        self._settle()
        self.eng._last_n = self._last_n
        return self.eng.stats()

    def stats(self):
        """Whole-lattice statistic rows of the last ``step`` call (row 0 = starting state)."""
        return reduce_stat_rows(self.dist, self.stats_local(), self.world,
                                device=self.dev, group=self.group)

    def stopped_at(self) -> int:
        """-1, or the t whose S_t is uniform over the WHOLE lattice (iteration t+1 breaks, spgg.py:405)."""
        self._settle()
        return 0 if self._uniform_start else int(self.eng.status().stopped_at)

    def kernel_launches(self) -> int:
        self._settle()
        return int(self.eng.status().kernel_launches)

    def close(self):
        try:
            self._settle()
            if self.p2p:   # the neighbours store into this strip's planes and ring: free them only when all are done
                self.torch.cuda.synchronize(self.dev)
                self.dist.barrier(group=self.group)
        finally:
            self.eng.close()


# ------------------------------------------------------------------ bench leg for N > 1
def bench_main(args, rank: int, local_rank: int, world: int):
    """``bench.py --gpus N`` under torchrun: BASELINE config 5, one L x L lattice (default
    L=32768) split into N row strips; barrier + synchronize on both sides of exactly K timed
    steps, device-side timing, max over ranks; rank 0 prints the JSON line.  Outside the timed
    region: a parity check of the N-strip run against ONE handle holding the whole lattice on
    rank 0 (position-keyed digests of S, R, Q + the integer statistics), and BASELINE config 3
    (the r x kappa sweep as batched replicas dealt to the ranks) under ``extras.c3_sweep``."""
    import torch
    import torch.distributed as dist
    from bench import C4, BYTES_PER_SITE_FP32, ClockSampler, measured_peak_gbs, c5_config

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    L = args.L or 32768
    K, W, inner = args.steps, args.warmup, args.inner
    p = dict(C4, L=L)
    se = StripEngine(p, seed=2024, precision="fp32", device=local_rank)
    se.init_random(2024)
    for _ in range(W):
        se.step(inner)
    se.sync()
    l0 = se.kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        se.step(inner)
    se._join_side()
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clocks = sampler.stop() if rank == 0 else None
    se.sync()
    launches = se.kernel_launches() - l0
    reruns_timed = se.reruns
    transport = {"halo": "peer-mapped planes (stores over NVLink)" if se.p2p else "NCCL send/recv",
                 "reports": "peer-mapped rings (system-scope atomics)" if se.ring else "NCCL all-reduce(MAX)"}
    spec = se.eng.status()
    n_sites = L * L
    value = n_sites * inner * K / (ms * 1e-3)

    # the same strip without its neighbours (no halo exchange, no reduce): what the GPU alone needs per
    # iteration under the clocks of this very run - the difference to us_per_iteration is the
    # communication that is not hidden
    n_solo = max(10, min(50, inner))
    L_.check(se.lib.spgg_begin_steps(se.h, n_solo, se._stream()))
    L_.check(se.lib.spgg_phase_kernel(se.h, 0, 1, se._stream()))
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    L_.check(se.lib.spgg_phase_iteration(se.h, 1, se._stream()))
    s0.record()
    for s_ in range(2, n_solo + 1):
        L_.check(se.lib.spgg_phase_iteration(se.h, 1 if s_ < n_solo else 0, se._stream()))
    s1.record()
    L_.check(se.lib.spgg_end_steps(se.h, se._stream()))
    torch.cuda.synchronize()
    se.eng.sync()
    solo = torch.tensor([1e3 * s0.elapsed_time(s1) / (n_solo - 1)], device=dev, dtype=torch.float64)
    dist.all_reduce(solo, op=dist.ReduceOp.MAX)
    solo_us = float(solo.item())

    # end to end: host state in (pinned), K steps with the whole-lattice stat rows read back
    # each step, final strategies/reputations out; every rank moves its own strip
    S_h = torch.empty((se.rows, L), dtype=torch.uint8).pin_memory()
    R_h = torch.zeros((se.rows, L), dtype=torch.float64).pin_memory()
    Q_h = torch.empty((se.rows, L, 2, 2), dtype=torch.float64).pin_memory()
    rs = np.random.RandomState(100 + rank)
    S_h.numpy()[...] = rs.randint(0, 2, (se.rows, L))
    Q_h.numpy()[...] = rs.uniform(-0.01, 0.01, (se.rows, L, 2, 2))
    S_o, R_o = torch.empty_like(S_h).pin_memory(), torch.empty_like(R_h).pin_memory()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    L_.check(se.lib.spgg_set_state(se.h, 0, S_h.data_ptr(), R_h.data_ptr(), Q_h.data_ptr()))
    dist.barrier()      # a new run empties the report rings: nobody steps before every rank has uploaded
    d2h = 0
    for _ in range(K):
        se.step(inner)
        d2h += se.stats().nbytes
    L_.check(se.lib.spgg_get_state(se.h, 0, S_o.data_ptr(), R_o.data_ptr(), None))
    torch.cuda.synchronize()
    dist.barrier()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    t_e2e = float(t_e2e.item())
    h2d_bytes = world * (S_h.numel() + 8 * R_h.numel() + 8 * Q_h.numel())
    d2h_bytes = world * (S_o.numel() + 8 * R_o.numel() + d2h)
    strip_rows_n = se.rows
    se.close()
    del S_h, R_h, Q_h, S_o, R_o

    # ---- parity at the benchmarked geometry (VERDICT r1): N strips == one handle, same seed
    n_chk = 6
    ints = [0, 1, 2, 3, 11, 12, 13, 14, 15, 16, 31, 32, 33]
    se2 = StripEngine(p, seed=2024, precision="fp32", device=local_rank)
    se2.init_random(77)
    se2.step(n_chk)
    dig_n = se2.digest()
    rows_n = se2.stats()[1:, ints]
    se2.close()
    parity = None
    if rank == 0:
        from .engine import Engine
        try:
            eng = Engine(p, seeds=2024, precision="fp32", device=local_rank)
            eng.init_random(77)
            eng.step(n_chk)
            dig_1 = eng.digest()
            rows_1 = eng.stats()[1:, ints]
            eng.close()
            parity = {"ok": bool(tuple(dig_1) == tuple(dig_n) and np.array_equal(rows_1, rows_n)),
                      "iterations": n_chk, "digests_equal": bool(tuple(dig_1) == tuple(dig_n)),
                      "integer_statistics_equal": bool(np.array_equal(rows_1, rows_n)),
                      "what": f"{world} strips vs one handle holding the whole L={L} lattice on rank 0: "
                              "position-keyed 64-bit digests of S, R, Q (spgg_state_digest) and the integer "
                              "columns + the exact global maximum of every statistics row"}
        except Exception as e:   # e.g. the whole lattice does not fit next to another tenant
            parity = {"ok": None, "error": str(e)[:200]}
    dist.barrier()

    # ---- BASELINE config 3 on N GPUs (VERDICT r1): batched replicas, no data-path collective
    c3 = None
    try:
        c3 = bench_c3(rank, world, local_rank)
    except Exception as e:
        c3 = {"error": str(e)[:200]}
    dist.barrier()

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        achieved = BYTES_PER_SITE_FP32 * value / 1e9 / world
        line = {
            "metric": "site-updates/s", "value": value, "unit": "site-updates/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": c5_config(L, world, inner),
            "clocks": clocks,
            "e2e": {"value": n_sites * inner * K / t_e2e, "unit": "site-updates/s",
                    "h2d_bytes_per_step": h2d_bytes / K, "d2h_bytes_per_step": d2h_bytes / K,
                    "seconds": t_e2e},
            "gpu_launches": int(launches) * world,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None,
                         "kernel": "whole iteration per GPU: one k_step_fast launch (speculative global maximum) + "
                                   "halo exchange, the report all-reduce runs beside it",
                         "algorithmic_bytes_per_site": BYTES_PER_SITE_FP32, "peak_source": peak_src},
            "cpu_baseline": None,
            "parity_check": parity,
            "extras": {"strip_rows": strip_rows_n, "us_per_iteration": 1e3 * ms / (K * inner),
                       "transport": transport,
                       "compute_only_us_per_iteration": solo_us,
                       "communication_not_hidden_frac": 1.0 - solo_us / (1e3 * ms / (K * inner)),
                       "speculation": {"launches": int(spec.speculative_launches), "reruns_in_timed_region": int(reruns_timed)},
                       "c3_sweep": c3},
        }
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def bench_c3(rank: int, world: int, local_rank: int):
    """BASELINE config 3 over the ranks of this job: (a) the r x kappa x M grid as 60 batched L=200
    replicas (``sweep.run_sweep``), (b) the reference's own ``figure_2_3_4`` set - 10 tuples, L=100,
    100 001 iterations, HDF5 files written - through ``runner.run_experiments`` (the reference's
    ``runner.py:117-156`` signature).  Wall clock between barriers (host work included)."""
    import shutil
    import tempfile
    import torch
    import torch.distributed as dist
    from bench import C4
    from . import sweep, runner
    torch.cuda.set_device(local_rank)
    L, its = 200, 2000
    plist = [dict(C4, L=L, r=r, influence_factor=k, use_second_order=m, reward_weight_payoff=1.0)
             for m in (False, True) for r in (1, 2, 3, 3.6, 4, 5) for k in (0, 0.5, 1, 1.5, 2)]
    seeds = list(range(500, 500 + len(plist)))
    sweep.run_sweep(plist[:world], seeds[:world], iterations=50)          # warm the kernels up
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = sweep.run_sweep(plist, seeds, iterations=its)
    torch.cuda.synchronize()
    dist.barrier()
    t_a = time.perf_counter() - t0
    done = sum(o["iterations"] for o in res)
    combos = [(3.6, k, m, 0.8, 1.0, 1.0, "reputation") for k in (0.0, 0.5, 1.0, 1.5, 2.0) for m in (False, True)]
    tmp = tempfile.mkdtemp(prefix=f"spgg_c3_{rank}_")
    try:
        dist.barrier()
        t0 = time.perf_counter()
        out = runner.run_experiments(combos, use_progress_bar=False, base_dir=tmp, seed=11)
        torch.cuda.synchronize()
        dist.barrier()
        t_b = time.perf_counter() - t0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return {"replica_grid": {"replicas": len(plist), "L": L, "iterations_each": its, "seconds": t_a,
                             "site_updates_per_s": done * L * L / t_a, "n_gpus": world},
            "figure_2_3_4": {"tuples": len(combos), "L": 100, "iterations_each": 100001, "seconds": t_b,
                             "site_updates_per_s": len(combos) * 100 * 100 * 100001 / t_b,
                             "hdf5_files_written": len(out), "n_gpus": world}}
