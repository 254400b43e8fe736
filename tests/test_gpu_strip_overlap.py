"""State overlaps of a lattice split into row strips (StripEngine.snapshot / StripEngine.overlap, include/spgg.h:
spgg_snapshot / spgg_overlap on strip handles): the strips' counts summed, maxima maxed and fp64 sums added in rank
order equal one handle holding the whole lattice (the sums within the bound) and NumPy, and every rank gets the same
dict.  On a one-GPU box the ranks share cuda:0 and reduce through gloo; with >= 2 GPUs the NCCL path is tested as
well."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "strip_overlap_worker.py")


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _ranks(argv, world, timeout=900):
    """Run ``world`` copies of strip_overlap_worker.py (rendezvous on 127.0.0.1); every one must pass."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = []
    for rank in range(world):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, WORKER] + [str(a) for a in argv], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        try:
            out, _ = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            p.kill()
            out = p.communicate()[0] + "\n[timeout]"
        assert p.returncode == 0, out


@pytest.mark.parametrize("L,world", [
    (64, 2),       # 32-row strips
    (100, 3),      # ragged 34 / 33 / 33 rows, general path
    (4096, 2),     # fast path
])
def test_geometries_gloo(L, world):
    _ranks(["geometries", "gloo", L], world)


def test_geometries_nccl():
    n = _ngpu()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    _ranks(["geometries", "nccl", 1000], min(n, 3))


@pytest.mark.parametrize("case,world", [("fast", 2), ("general", 3), ("fp64", 2)])
def test_states_from_the_dynamics(case, world):
    _ranks(["dynamics", "gloo", case], world)
