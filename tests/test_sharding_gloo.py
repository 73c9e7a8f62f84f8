"""CPU suite, part 3: the N > 1 path.  The row-sharded scoring protocol (include/cmdiad_b200.h) is run over gloo with
world_size 2: local work is float32 squared distances on each rank's shard, the collectives and the key / ownership
encodings are the ones the GPU path uses (cmdiad_b200/sharding.py), and the result must equal the un-sharded argmin of
d2 (lowest row on ties) exactly."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cmdiad_b200 import sharding, synth


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _d2(a, b):
    """float32 squared distances [len(a), len(b)] (float64 sums, rounded once): the arithmetic of every rank and of the
    un-sharded reference"""
    a64, b64 = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return ((a64[:, None, :] - b64[None, :, :]) ** 2).sum(-1).astype(np.float32)


def _near_tie_query(x, y, seed):
    """a query q whose float32 d2 to y is below that to x while float32 sqrt makes the two distances equal"""
    g = np.random.Generator(np.random.PCG64(seed))
    for _ in range(100_000):
        q = (x + 0.2 * g.standard_normal(x.shape[0])).astype(np.float32)
        dx, dy = _d2(q[None], np.stack([x, y]))[0]
        if dy < dx and np.sqrt(dy) == np.sqrt(dx):
            return q
    raise AssertionError("no near-tie query found")


def _case(R, P, D):
    """bank and queries of the table protocol test: clustered rows, an exact duplicate across the two shards (the lower
    global row must win), and a near-duplicate across them (row TIE_J is 2 ulps away from row TIE_I in two coordinates)
    with a query for which TIE_J is strictly nearer in float32 d2 while the float32 distances are equal"""
    cent = synth.centroids(D, 64)
    lib = synth.patches(R, D, seed=3, cent=cent)
    lib[R // 2 + 3] = lib[5]
    ti, tj = TIE_I, R // 2 + TIE_J_OFF
    lib[tj] = lib[ti]
    lib[tj, :2] = np.nextafter(np.nextafter(lib[ti, :2], np.float32(np.inf)), np.float32(np.inf))
    patch = synth.patches(P, D, seed=4, anomalous_frac=0.02, cent=cent)
    patch[7] = lib[5] + 1e-3
    patch[TIE_Q] = _near_tie_query(lib[ti], lib[tj], 11)
    return lib, patch


TIE_I, TIE_J_OFF, TIE_Q = 17, 40, 9


def _table_worker(rank, world, port, R, P, D, ret):
    """three-phase protocol with the replicated neighbour table: MIN over packed (d2, row) keys, lookup, SUM of squared
    distances"""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    lib, patch = _case(R, P, D)
    lo, hi = sharding.shard_range(R, rank, world)
    mine = lib[lo:hi]
    # the replicated table: every rank computes the entries of ITS rows against the whole bank, slices are all-gathered
    # (uneven shards are padded to the largest one and cut again, as Bank.build_knn_sharded does)
    wd = _d2(mine, lib)
    part = torch.full(((R + world - 1) // world, 3), -1, dtype=torch.int64)
    for i in range(mine.shape[0]):
        order = np.lexsort((np.arange(R), wd[i]))[:3]
        part[i] = torch.from_numpy(sharding.pack_keys(wd[i][order], order))
    gathered = torch.empty((world * part.shape[0], 3), dtype=torch.int64)
    dist.all_gather_into_tensor(gathered, part)
    counts = [sharding.shard_range(R, r, world) for r in range(world)]
    table = torch.cat([gathered[r * part.shape[0]:r * part.shape[0] + (b - a)] for r, (a, b) in enumerate(counts)]).numpy()
    # phase 1: local argmin d2 (lowest row on ties), keys of (d2, global row), MIN, then min_val = sqrt(d2)
    d2 = _d2(patch, mine)
    mi = np.lexsort((np.broadcast_to(np.arange(hi - lo), d2.shape), d2), axis=1)[:, 0]
    keys = torch.from_numpy(sharding.pack_keys(d2[np.arange(P), mi], mi + lo))
    # the same keys packed with the distance instead of d2 (the exchange this protocol replaced)
    keys_dist = torch.from_numpy(sharding.pack_keys(np.sqrt(d2[np.arange(P), mi]), mi + lo))
    dist.all_reduce(keys, op=dist.ReduceOp.MIN)
    dist.all_reduce(keys_dist, op=dist.ReduceOp.MIN)
    min_d2, min_idx = sharding.unpack_keys(keys.numpy())
    min_val = np.sqrt(min_d2)
    # phase 2: lookup (no bank access for m_star: its global row indexes the table) + owned squared distances
    s_idx = int(np.argmax(min_val))
    _, nn = sharding.unpack_keys(table[min_idx[s_idx]])
    knn = torch.from_numpy(sharding.knn_d2_contribution(mine, lo, patch[s_idx], nn[1:]))
    dist.all_reduce(knn, op=dist.ReduceOp.SUM)
    if rank == 0:
        ret.put(dict(min_val=min_val.copy(), min_idx=min_idx.copy(), s_idx=s_idx, nn=nn.copy(), d2=knn.numpy().copy(),
                     owner=sharding.owner_of(min_idx, R, world), min_idx_dist=sharding.unpack_keys(keys_dist.numpy())[1]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_three_phase_table_protocol_over_gloo():
    R, P, D, world = 1203, 64, 64, 2
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_table_worker, args=(r, world, port, R, P, D, ret)) for r in range(world)]
    for p in procs:
        p.start()
    got = ret.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    lib, patch = _case(R, P, D)
    # un-sharded reference: argmin float32 d2 over the whole bank, lowest row on ties; min_val = float32 sqrt(d2)
    d2 = _d2(patch, lib)
    mi = np.lexsort((np.broadcast_to(np.arange(R), d2.shape), d2), axis=1)[:, 0]
    mv = np.sqrt(d2[np.arange(P), mi])
    s_idx = int(np.argmax(mv))
    assert (got["min_idx"] == mi).all() and (got["min_val"] == mv).all() and got["s_idx"] == s_idx
    assert got["min_idx"][7] == 5  # duplicate rows 5 and R//2+3 live on different shards: lowest global row wins
    # the near-tie across the shards: equal float32 distances, the higher row strictly nearer in d2 -- it must win, as in
    # one bank, where a MIN over (distance, row) keys returns the lower row
    ti, tj = TIE_I, R // 2 + TIE_J_OFF
    assert sharding.shard_range(R, 0, world)[1] <= tj and ti < sharding.shard_range(R, 0, world)[1]
    assert d2[TIE_Q, tj] < d2[TIE_Q, ti] and np.sqrt(d2[TIE_Q, tj]) == np.sqrt(d2[TIE_Q, ti])
    assert mi[TIE_Q] == tj and got["min_idx"][TIE_Q] == tj
    assert got["min_idx_dist"][TIE_Q] == ti
    wd = _d2(lib[mi[s_idx]][None], lib)[0]
    ref_nn = np.lexsort((np.arange(R), wd))[:3]
    assert (got["nn"] == ref_nn).all()
    want = sharding.knn_d2_contribution(lib, 0, patch[s_idx], ref_nn[1:])
    assert (got["d2"] == want).all()  # x + 0 == x: the SUM all-reduce returns the owner's value exactly
    lo1, _ = sharding.shard_range(R, 1, world)
    assert (got["owner"] == (got["min_idx"] >= lo1)).all()


def test_key_packing_properties():
    g = np.random.Generator(np.random.PCG64(0))
    d = np.abs(g.standard_normal(1000)).astype(np.float32)
    d[:10] = d[10:20]  # ties
    rows = g.permutation(1000).astype(np.int64)
    k = sharding.pack_keys(d, rows)
    assert (k >= 0).all()
    order = np.argsort(k, kind="stable")
    ref = np.lexsort((rows, d))
    assert (order == ref).all()
    d2, r2 = sharding.unpack_keys(k)
    assert (d2 == d).all() and (r2 == rows).all()
    for n, w in ((10, 3), (200000, 8), (7, 8)):
        for r in range(w):
            lo, hi = sharding.shard_range(n, r, w)
            if hi > lo:
                assert (sharding.owner_of(np.arange(lo, hi), n, w) == r).all()


def _stage_worker(rank, world, port, B, P, D, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    # host logic of Bank._stage_sharded (the device copy itself is a torch copy): slice, pad, all-gather, cut
    x = torch.from_numpy(np.stack([synth.patches(P, D, seed=40 + i, dist="G") for i in range(B)]))
    rows = B * P
    per, lo, hi = sharding.stage_slice(rows, world, rank)
    part = torch.zeros(per, D)
    part[:hi - lo] = x.reshape(rows, D)[lo:hi]
    gathered = torch.empty(per * world, D)
    dist.all_gather_into_tensor(gathered, part)
    full = gathered[:rows].view(B, P, D)
    ok = bool((full == x).all()) and tuple(full.shape) == (B, P, D)
    ret.put((rank, ok))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("B,P", [(4, 96), (3, 49)])   # 384 rows split evenly, 147 rows with a padded last slice
def test_cooperative_query_staging_over_gloo(B, P):
    """Bank._stage_sharded: every rank contributes 1/world of the query rows, the all-gather must reproduce the batch on
    every rank (row counts that do not divide by the world size are padded and cut again)."""
    world, D = 2, 64
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_stage_worker, args=(r, world, port, B, P, D, ret)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(ret.get(timeout=240) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got == {0: True, 1: True}
