"""Row strips with the real kernels: an N-strip run equals the single-handle run bit for
bit (S, R, Q, integer statistics; float sums to tolerance - the summation order differs).
On a one-GPU box the ranks share cuda:0 and exchange through gloo (host-staged halos);
with >= 2 GPUs the NCCL path (device buffers, NVLink) is tested as well."""
import pytest

from helpers import launch_ranks

pytestmark = pytest.mark.gpu


def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("precision,second,state,L,world", [
    ("fp32", 0, "reputation", 256, 2),      # fast path (TMA) strips
    ("fp32", 1, "action", 256, 4),
    ("fp32", 1, "reputation", 100, 3),      # general path, ragged strips
    ("fp64", 0, "reputation", 64, 2),
    ("fp32", 0, "reputation", 160, 2),      # fast path with a partial last tile column, 80-row strips
    # the benchmarked tile geometry: n_tx = 32 tile columns, 2048-row strips, every persistent CTA
    # walks several tiles and the strip's own top / bottom tiles take the ghost-row path
    ("fp32", 0, "reputation", 4096, 2),
])
def test_strips_equal_single_lattice_gloo(precision, second, state, L, world):
    res = launch_ranks(["gpu", "gloo", precision, second, state, L, 12], world, timeout=900)
    for rc, out in res:
        assert rc == 0, out


@pytest.mark.parametrize("precision,second,state,L", [
    ("fp32", 0, "reputation", 512),
    ("fp32", 1, "reputation", 384),
    ("fp32", 0, "reputation", 4096),
])
def test_strips_equal_single_lattice_nccl(precision, second, state, L):
    n = _ngpu()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(n, 4)
    res = launch_ranks(["gpu", "nccl", precision, second, state, L, 12], world, timeout=600)
    for rc, out in res:
        assert rc == 0, out


def test_strips_rerun_a_wrong_guess_of_the_global_maximum():
    """The one-launch iteration over strips with every 5th guess spoiled on purpose: the verdict comes
    from the max-reduced report, every rank re-runs from the same launch, results unchanged."""
    res = launch_ranks(["gpu", "gloo", "fp32", 0, "reputation", 256, 24], 2, timeout=600,
                       extra_env={"SPGG_SPEC_TEST_POISON": "5"})
    for rc, out in res:
        assert rc == 0, out
    if _ngpu() >= 2:     # peer-mapped halos + report ring: the re-run empties the rings behind a barrier
        res = launch_ranks(["gpu", "nccl", "fp32", 0, "reputation", 512, 24], 2, timeout=600,
                           extra_env={"SPGG_SPEC_TEST_POISON": "5"})
        for rc, out in res:
            assert rc == 0, out


def test_strips_stop_on_a_uniform_lattice_like_the_reference():
    """VERDICT r1: early exit (spgg.py:405) in strip mode - the uniform-lattice test is global."""
    res = launch_ranks(["exit", "gloo", 256], 2, timeout=600)
    for rc, out in res:
        assert rc == 0, out
    if _ngpu() >= 2:
        res = launch_ranks(["exit", "nccl", 256], 2, timeout=600)
        for rc, out in res:
            assert rc == 0, out


@pytest.mark.parametrize("world", [1, 2])
def test_replica_sweep_sharded_over_ranks(world):
    """BASELINE config 3: the r x kappa grid as batched replicas dealt to the ranks; each replica
    must equal its stand-alone run bit for bit (S, R, integer series)."""
    res = launch_ranks(["sweep", "gloo"], world, timeout=600)
    for rc, out in res:
        assert rc == 0, out
