"""Re-creation of the reference's comm tests against the new façade.

``/root/reference/test_comms.py:9-26`` (gather / bcast of Python objects),
``/root/reference/test_mpi.py:34-96`` (variable-size gathers) and
``/root/reference/test_iallgather.py:37-54`` (size exchange + all-gather-v), run as 2- and
3-rank SPMD jobs with plain pytest (the reference needed ``mpirun -n 2 py.test``).
"""
import pytest

from pytorch_ps_mpi_b200.launch import spawn
from tests import _mp

TRANSPORTS = ["shm", "gloo"]


@pytest.mark.parametrize("transport", TRANSPORTS)
@pytest.mark.parametrize("n", [2, 3])
def test_gather_bcast_iallgather_any_source(transport, n):
    """The reference's three test files re-created (``test_comms.py:9-26``, ``test_iallgather.py:37-54``, ``test_mpi.py:34-96``)
    + any-source point-to-point, at 2 and 3 ranks over both transports — one set of processes per (transport, n)."""
    names = ["gather_objects", "bcast_objects"] + (["iallgather_objects", "p2p_any_source"] if n == 3 else [])
    spawn(_mp.comm_suite, n, (transport, names), env=_mp.CPU_ONLY, timeout=240)


def test_single_process_world():
    import pytorch_ps_mpi_b200 as ps
    comms = ps.comms
    obj = {"a": [1, 2, 3]}
    recv, req, t = comms.igather(obj, name="solo")
    assert comms.irecv(recv, req, name="solo") == [obj]
    assert comms.irecv1(*comms.ibroadcast(obj)) == obj
    ia = comms.Iallgather()
    m, meta = comms.format_for_send(obj)
    assert meta["packaged_bytes"] == len(m) and meta["msg_bytes"] + 16 == len(m)
    (req, count), = ia.prepare([len(m)])
    req.Wait()
    assert ia.recv(*ia.send(m, count)) == [obj]


def test_shm_transport_stress():
    """Native ShmComm under load: 4 ranks, 64 KB rings, up to 300 KB messages, 30 rounds of all-to-all."""
    spawn(_mp.shm_stress, 4, env=_mp.CPU_ONLY, timeout=240)
