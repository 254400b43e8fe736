"""Strategy pair counts of a lattice split into row strips (StripEngine.pair_counts, include/spgg.h:
spgg_strip_pair_counts): the counts summed over the strips equal NumPy and one handle holding the whole
lattice, on every rank.  On a one-GPU box the ranks share cuda:0 and gather the records through gloo; with
>= 2 GPUs the NCCL path is tested as well."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "strip_pair_worker.py")


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _ranks(argv, world, timeout=900, extra_env=None):
    """Run ``world`` copies of strip_pair_worker.py (rendezvous on 127.0.0.1); every one must pass."""
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


@pytest.mark.parametrize("L,world,max_ds", [
    (64, 4, "1,16,17,32"),        # 16-row strips: max_d = 32 takes rows from the two strips below
    (100, 3, "1,33,34,50"),       # ragged 34 / 33 / 33 rows, general path
    (1000, 4, "1,64,500"),        # 250-row strips on the general path
    (4096, 2, "1,64,2048"),       # fast path
    (4096, 4, "1,64,2048"),
])
def test_geometries_gloo(L, world, max_ds):
    _ranks(["geometries", "gloo", L, max_ds], world)


def test_geometries_nccl():
    n = _ngpu()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    _ranks(["geometries", "nccl", 1000, "1,64,500"], min(n, 4))


@pytest.mark.parametrize("case,world,env", [
    ("fast", 2, None),
    ("fast_c2", 4, {"SPGG_SPEC_TEST_POISON": "5"}),   # counting meets a pending re-run of a wrong guess
    ("general", 3, None),
    ("fp64", 2, None),
])
def test_states_from_the_dynamics(case, world, env):
    _ranks(["dynamics", "gloo", case], world, extra_env=env)


def test_large_lattice():
    _ranks(["large", "gloo", 16384, 3], 4, timeout=1800)


def test_world_of_one_equals_the_whole_lattice_handle():
    _ranks(["world1", "gloo"], 1)


def test_records_that_disagree_and_bad_arguments():
    _ranks(["errors", "gloo"], 2)
