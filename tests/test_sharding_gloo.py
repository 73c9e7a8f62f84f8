"""CPU suite, part 3: the N > 1 path.  The row-sharded scoring protocol (include/cmdiad_b200.h) is run over gloo with
world_size 2: local work is done by the CPU oracle on each rank's shard, the collectives and the key / ownership
encodings are the ones the GPU path uses (cmdiad_b200/sharding.py), and the result must equal the unsharded oracle
exactly."""
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


def _table_worker(rank, world, port, R, P, D, ret):
    """three-phase protocol with the replicated neighbour table: MIN over packed keys, lookup, SUM of squared distances"""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    cent = synth.centroids(D, 64)
    lib = synth.patches(R, D, seed=3, cent=cent)
    lib[R // 2 + 3] = lib[5]  # an exact duplicate across the two shards: the lower global row must win
    patch = synth.patches(P, D, seed=4, anomalous_frac=0.02, cent=cent)
    patch[7] = lib[5] + 1e-3
    lo, hi = sharding.shard_range(R, rank, world)
    mine = lib[lo:hi]
    # the replicated table: every rank computes the entries of ITS rows against the whole bank, slices are all-gathered
    # (uneven shards are padded to the largest one and cut again, as Bank.build_knn_sharded does)
    wd = torch.cdist(torch.from_numpy(mine), torch.from_numpy(lib), compute_mode="donot_use_mm_for_euclid_dist") ** 2
    part = torch.full(((R + world - 1) // world, 3), -1, dtype=torch.int64)
    for i in range(mine.shape[0]):
        order = np.lexsort((np.arange(R), wd[i].numpy()))[:3]
        part[i] = torch.from_numpy(sharding.pack_keys(wd[i].numpy()[order], order))
    gathered = torch.empty((world * part.shape[0], 3), dtype=torch.int64)
    dist.all_gather_into_tensor(gathered, part)
    counts = [sharding.shard_range(R, r, world) for r in range(world)]
    table = torch.cat([gathered[r * part.shape[0]:r * part.shape[0] + (b - a)] for r, (a, b) in enumerate(counts)]).numpy()
    # phase 1
    d = torch.cdist(torch.from_numpy(patch), torch.from_numpy(mine), compute_mode="donot_use_mm_for_euclid_dist")
    mv, mi = torch.min(d, dim=1)
    keys = torch.from_numpy(sharding.pack_keys(mv.numpy(), mi.numpy() + lo))
    dist.all_reduce(keys, op=dist.ReduceOp.MIN)
    min_val, min_idx = sharding.unpack_keys(keys.numpy())
    # phase 2: lookup (no bank access for m_star: its global row indexes the table) + owned squared distances
    s_idx = int(np.argmax(min_val))
    _, nn = sharding.unpack_keys(table[min_idx[s_idx]])
    d2 = torch.from_numpy(sharding.knn_d2_contribution(mine, lo, patch[s_idx], nn[1:]))
    dist.all_reduce(d2, op=dist.ReduceOp.SUM)
    if rank == 0:
        ret.put(dict(min_val=min_val.copy(), min_idx=min_idx.copy(), s_idx=s_idx, nn=nn.copy(), d2=d2.numpy().copy(),
                     owner=sharding.owner_of(min_idx, R, world)))
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
    cent = synth.centroids(D, 64)
    lib = synth.patches(R, D, seed=3, cent=cent)
    lib[R // 2 + 3] = lib[5]
    patch = synth.patches(P, D, seed=4, anomalous_frac=0.02, cent=cent)
    patch[7] = lib[5] + 1e-3
    d = torch.cdist(torch.from_numpy(patch), torch.from_numpy(lib), compute_mode="donot_use_mm_for_euclid_dist")
    mv, mi = torch.min(d, dim=1)
    s_idx = int(torch.argmax(mv))
    assert (got["min_idx"] == mi.numpy()).all() and (got["min_val"] == mv.numpy()).all() and got["s_idx"] == s_idx
    assert got["min_idx"][7] == 5  # duplicate rows 5 and R//2+3 live on different shards: lowest global row wins
    wd = torch.cdist(torch.from_numpy(lib[mi[s_idx]:mi[s_idx] + 1]), torch.from_numpy(lib),
                     compute_mode="donot_use_mm_for_euclid_dist")[0] ** 2
    ref_nn = np.lexsort((np.arange(R), wd.numpy()))[:3]
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
