"""GPU test: a handle and a comm object release every device buffer, pinned buffer, stream and event they own.  The measure
is the library's own count of what its resource owners hold (cmdb_debug_live_resources), not the device's free memory,
which other processes on the GPU change at any time."""
import ctypes
import gc
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

D, FM = 768, 28
P = FM * FM
ROWS, OFFSET = 3000, 1000


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import Bank, Comm, synth
    from cmdiad_b200 import _lib as L
    from cmdiad_b200.fusion import LateFusion
    assert torch.cuda.is_available()
    return dict(Bank=Bank, Comm=Comm, LateFusion=LateFusion, L=L, lib=L.load(), synth=synth, cent=synth.centroids(D, 128))


def _live(lib):
    """(device bytes, pinned host bytes, streams, events) held by the library in this process"""
    gc.collect()   # handles of earlier tests that only the cyclic collector frees must not go away mid-test
    out = np.zeros(4, np.int64)
    assert lib.cmdb_debug_live_resources(out.ctypes.data_as(ctypes.c_void_p)) == 0
    return tuple(int(v) for v in out)


def _cycle(env):
    """one lifecycle of every resource a handle can own; returns the count before the handles are destroyed"""
    Bank, L, lib, sy = env["Bank"], env["L"], env["lib"], env["synth"]
    rows = sy.patches(ROWS, D, seed=5, cent=env["cent"])
    q = np.stack([sy.patches(P, D, seed=50 + i, anomalous_frac=0.01, cent=env["cent"]) for i in range(3)])
    b = Bank(D, ROWS)
    b.append(rows)
    b.coreset_select(100, None)
    b.finalize()
    b.build_knn()
    keys = b.read_knn(0, ROWS).clone()
    L.check(lib.cmdb_bank_set_option(b._h, L.OPT_TIMING, 1))
    b.score_batch(q, (FM, FM), 224)
    b.score_batch(torch.from_numpy(q).cuda(), (FM, FM), 112)   # another out_hw: the scratch is freed and rebuilt
    b.score_batch(q, (FM, FM), 224)
    rebuilt = _live(lib)
    b.score_batch(torch.from_numpy(q).cuda(), (FM, FM), 112)
    b.score_batch(q, (FM, FM), 224)
    assert _live(lib) == rebuilt, "a rebuild of the scratch with the same sizes changed what the handle holds"

    other = Bank(D, ROWS)
    other.append(rows)
    other.finalize()
    fusion = env["LateFusion"]([b, other], [1.0, 0.5], [1.0, 2.0], [0.3, -0.2], 0.1, [0.5, 0.25], -0.05)
    fusion.eval_reserve(4, 224)
    fusion.score_batch([q, q], [(FM, FM), (FM, FM)], 224, keep_on_device=True)
    b.finalize()   # drops the neighbour table and the scratch

    shard = Bank(D, ROWS - OFFSET, row_offset=OFFSET)
    shard.append(rows[OFFSET:])
    shard.finalize()
    shard.set_knn_table(keys, ROWS)
    comm = env["Comm"](0)
    shard.attach_comm(comm)
    shard.attach_comm(None)
    held = _live(lib)
    comm.close()
    for h in (shard, other, b):
        h.close()
    return held


def test_handles_release_what_they_own(env):
    import torch.distributed as dist
    lib = env["lib"]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        start = _live(lib)
        held = []
        for cycle in range(3):
            held.append(_cycle(env))
            assert _live(lib) == start, f"cycle {cycle}: not everything was released"
            assert held[-1] == held[0], f"cycle {cycle}: the handles hold more than in the first cycle"
        assert held[0][0] > start[0] and held[0][1] > start[1] and held[0][2] > start[2] and held[0][3] > start[3]
    finally:
        dist.destroy_process_group()
