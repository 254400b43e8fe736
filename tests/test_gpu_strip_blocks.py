"""Block fields of a lattice split into row strips (StripEngine.block_fields, include/spgg.h: spgg_block_fields
on strip handles): the partials of the strips, gathered and added in rank order, equal one handle holding the
whole lattice and NumPy, on every field set.  On a one-GPU box the ranks share cuda:0 and gather through gloo;
with >= 2 GPUs the NCCL path is tested as well."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "strip_block_worker.py")


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _ranks(argv, world, timeout=900, extra_env=None):
    """Run ``world`` copies of strip_block_worker.py (rendezvous on 127.0.0.1); every one must pass."""
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


@pytest.mark.parametrize("L,world,bs", [
    (64, 4, "1,5,16,17,40,64"),       # 16-row strips: b = 17 and 40 straddle strips, b = 40 and 64 span several
    (100, 3, "1,7,33,34,51,100"),     # ragged 34 / 33 / 33 rows, general path
    (1000, 4, "8,32,300,1000"),
    (4096, 2, "32,100,2049,4096"),    # fast path
])
def test_geometries_gloo(L, world, bs):
    _ranks(["geometries", "gloo", L, bs], world)


def test_geometries_nccl():
    n = _ngpu()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    _ranks(["geometries", "nccl", 1000, "8,32,300,1000"], min(n, 4))


@pytest.mark.parametrize("case,world", [("fast", 2), ("general", 3), ("fp64", 2)])
def test_states_from_the_dynamics(case, world):
    _ranks(["dynamics", "gloo", case], world)


def test_large_lattice_counts():
    _ranks(["large", "gloo", 16384], 4, timeout=1800)


def test_world_of_one_equals_the_whole_lattice_handle():
    _ranks(["world1", "gloo"], 1)
