"""Cluster labelling of a lattice split into row strips (StripEngine.cluster_sizes / cluster_labels,
include/spgg.h: spgg_strip_clusters): every rank gets the sizes of the whole lattice and the labels of
its own rows, equal to scipy.ndimage.label, to the torus oracle of test_clusters_host.py and to one
handle holding the whole lattice.  On a one-GPU box the ranks share cuda:0 and gather the boundary
records through gloo; with >= 2 GPUs the NCCL path is tested as well."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from helpers import C1, full_params

pytestmark = pytest.mark.gpu
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "strip_cluster_worker.py")


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _ranks(argv, world, timeout=900, extra_env=None):
    """Run ``world`` copies of strip_cluster_worker.py (rendezvous on 127.0.0.1); every one must pass."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = []
    for rank in range(world):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), **(extra_env or {}))
        procs.append(subprocess.Popen([sys.executable, WORKER] + [str(a) for a in argv], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        try:
            out, _ = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            p.kill()
            out = p.communicate()[0] + "\n[timeout]"
        assert p.returncode == 0, out


@pytest.mark.parametrize("Ls,world", [
    ("64,96,160", 2),      # 32-row strips; 48 rows: a partial CCL tile row; a partial 256-column tile (fast path)
    ("64,1000", 4),        # 16-row strips, shorter than a CCL tile; 250-row strips on the general path
    ("100", 3),            # ragged 34 / 33 / 33 rows, general path
    ("4096", 2),           # several tile rows and columns per strip (fast path)
    ("4096", 4),
])
def test_geometries_gloo(Ls, world):
    _ranks(["geometries", "gloo", Ls], world)


def test_geometries_nccl():
    n = _ngpu()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    _ranks(["geometries", "nccl", "160,1000"], min(n, 4))


@pytest.mark.parametrize("case,world,env", [
    ("fast", 2, None),
    ("fast_c2", 4, {"SPGG_SPEC_TEST_POISON": "5"}),   # labelling meets a pending re-run of a wrong guess
    ("general", 3, None),
    ("fp64", 2, None),
])
def test_states_from_the_dynamics(case, world, env):
    _ranks(["dynamics", "gloo", case], world, extra_env=env)


def test_large_lattice():
    _ranks(["large", "gloo", 16384, 3], 4, timeout=1800)


def test_world_of_one_equals_the_whole_lattice_handle():
    _ranks(["world1", "gloo"], 1)


def test_errors_and_invalidation():
    _ranks(["errors", "gloo"], 2)


def test_lattices_beyond_int32_site_indices_are_refused():
    """L * L >= 2^31: refused before the labelling allocates anything; so are batched strips."""
    import spgg_b200
    from spgg_b200 import _lib
    L = 46341
    eng = spgg_b200.Engine(full_params(dict(C1, L=L)), rows=16, row0=0, precision="fp32")
    lib, h = eng.lib, eng._h
    assert lib.spgg_strip_cluster_record_bytes(h) == _lib.E_UNSUPPORTED
    buf = np.zeros(64, np.uint8)
    assert lib.spgg_strip_clusters(h, 0, 0, buf.ctypes.data) == _lib.E_UNSUPPORTED
    assert b"2^31" in lib.spgg_last_error()
    eng.close()
    batch = spgg_b200.Engine([full_params(dict(C1, L=64))] * 2, rows=32, row0=0, precision="fp32")
    assert batch.lib.spgg_strip_cluster_record_bytes(batch._h) == _lib.E_UNSUPPORTED
    assert batch.lib.spgg_strip_clusters(batch._h, 0, 0, buf.ctypes.data) == _lib.E_UNSUPPORTED
    batch.close()
