"""BASELINE config 1: 2-layer MLP on MNIST-shaped synthetic data, world_size 2, CPU plumbing.

Every mode is checked against a single-process oracle (sum of all ranks' coded gradients →
``torch.optim``), and all ranks must end bit-identical.
"""
import pytest

from pytorch_ps_mpi_b200.launch import spawn
from tests import _mp


SYNC_CASES = {          # (mode, optim, coding, coalesce)
    "shm": [("ps", "sgd", "identity", False), ("ps", "adam", "cast", False), ("allgather", "sgd", "identity", False),
            ("allgather", "sgd", "topk", False),
            ("ps", "sgd", "svd", False),          # a host-path-only (user-style) coding through the generic wire format
            ("ps", "sgd", "cast", True), ("allgather", "sgd", "cast", True)],     # one framed message per step (coalesce=True)
    "gloo": [("ps", "sgd", "topk", False), ("allgather", "adam", "scale", False)],
}


@pytest.mark.parametrize("transport", ["shm", "gloo"])
def test_mlp_sync(transport):
    """Every scenario of a transport runs in one pair of processes (see ``_mp.mlp_train_many``)."""
    spawn(_mp.mlp_train_many, 2, (transport, SYNC_CASES[transport]), env=_mp.CPU_ONLY, timeout=300)


@pytest.mark.parametrize("transport", ["shm", "gloo"])
def test_three_ranks_sync_average_groups_async(transport):
    """3 ranks: sync PS vs the oracle (shm), ``average=True`` + several param groups, AsySG-InCon with quota 1 (both transports)."""
    spawn(_mp.three_rank_suite, 3, (transport,), env=_mp.CPU_ONLY, timeout=300)


def test_shm_transport_detects_dead_peer():
    from pytorch_ps_mpi_b200.launch import spawn as _spawn
    import multiprocessing
    # rank 1 exits with os._exit(0) on purpose; rank 0 must notice instead of hanging
    _spawn(_mp.shm_dead_peer, 2, env=_mp.CPU_ONLY, timeout=90)


def test_async_consistent_reads():
    spawn(_mp.mlp_async_consistent, 3, env=_mp.CPU_ONLY)


@pytest.mark.parametrize("n", [2, 3])
def test_reference_equivalent_comparator(n):
    """The comparator bench.py runs in the same invocation as the product arm: right numerics, no hang, on gloo."""
    spawn(_mp.comparator_host, n, env=dict(_mp.CPU_ONLY, PSB200_TRANSPORT="gloo"), timeout=180)
