"""torchrun --nproc-per-node N scripts/shard_check.py : row-sharded scoring == single-GPU scoring, bit for bit.

Covers both transports of the sharded round with the replicated neighbour table (NCCL collectives; exchanges over
peer-mapped memory), the table itself, replicated and distributed finishing, host and device queries, several rounds per
call, pipelined rounds, and a witness bank: near-duplicate rows on ranks 0 and N - 1 whose distances to a query are equal
in float32 while their squared distances are not (the exchange keys must carry d^2 to pick the same row as one bank).
Prints one line per check and a final SHARD CHECK OK / FAILED (rank 0); exit code 1 on failure."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cmdiad_b200 import Bank, synth  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
R, D, P = 30_011, 768, 784
cent = synth.centroids(D)
lib = synth.patches(R, D, seed=1, cent=cent)
lo, hi = R * rank // world, R * (rank + 1) // world
shard = Bank(D, hi - lo, device=local, row_offset=lo)
shard.append(lib[lo:hi])
shard.finalize()
full = Bank(D, R, device=local)
full.append(lib)
full.finalize()
full.build_knn()
NAMES = ("min_idx", "min_val", "s", "s_star", "s_idx", "nn_idx", "m_star_knn", "w", "s_map")
bad = 0


def same(a, b, names=NAMES):
    return all((getattr(a, n) == getattr(b, n)).all() for n in names)


def report(what, ok):
    global bad
    bad += int(not ok)
    if rank == 0:
        print(f"{what}: sharded == single-GPU: {ok}", flush=True)


n_img = 70  # three rounds of <= 32 images
pb = np.stack([synth.patches(P, D, seed=80 + t, anomalous_frac=0.01, cent=cent) for t in range(n_img)])
bb = full.score_batch(pb, (28, 28), 224, full=True)
from cmdiad_b200 import Comm  # noqa: E402
comm = Comm(local)
for mode in ("table/nccl", "table/peer-memory"):
    if mode == "table/nccl":
        shard.build_knn_sharded()
        keys_sh = shard.read_knn(0, R).numpy()
        keys_1 = full.read_knn(0, R).numpy()
        report("replicated neighbour table == single-GPU table", bool((keys_sh == keys_1).all()))
    if mode == "table/peer-memory":
        shard.attach_comm(comm)   # exchanges fused into the kernels over peer-mapped memory: no NCCL in the scoring path
    tag = mode
    for src_name, src in (("host", pb), ("device", torch.from_numpy(pb).cuda())):
        ab = shard.score_sharded_batch(src, (28, 28), 224, full=True)
        report(f"[{tag}] {n_img} images, {src_name} queries, replicated finish", all(same(ab[t], bb[t]) for t in range(n_img)))
    dd = shard.score_sharded_batch(pb, (28, 28), 224, full=True, distribute=True)
    ok = True
    for t in range(n_img):
        mine = t % world == rank
        ok &= (dd[t] is not None) == mine and (not mine or same(dd[t], bb[t]))
    report(f"[{tag}] distributed finish (rank r returns images r, r+{world}, ...)", ok)
    # scalars of the images finished elsewhere are replicated
    arr = shard.score_sharded_batch(pb[:5], (28, 28), 224, distribute=True)
    ok = all(float(arr[0].s[0]) == float(bb[0].s[0]) for _ in range(1)) if rank == 0 else True
    report(f"[{tag}] scalars available on every rank", ok)
    for t in range(2):
        a = shard.score_sharded(pb[t], (28, 28), 224, full=True)
        report(f"[{tag}] single image {t}", same(a, bb[t]))
    # three rounds outstanding (three result slots on two compute lanes), 8 rounds of 8 images
    for src_name, src in (("host", torch.from_numpy(pb).pin_memory()), ("device", torch.from_numpy(pb).cuda())):
        pending, got = [], []
        for k in range(8):
            pending.append(shard.score_sharded_async(src[8 * k:8 * k + 8], (28, 28), 224, full=True))
            if len(pending) == 3:
                got.extend(pending.pop(0).wait())
        while pending:
            got.extend(pending.pop(0).wait())
        report(f"[{tag}] 8 rounds, three outstanding, {src_name} queries", all(same(got[t], bb[t]) for t in range(64)))

# Witness bank: rows J[t] on the last rank are copies of rows I[t] on rank 0 nudged by 2 ulps in two coordinates.  For a
# query near such a pair the float32 d^2 differ by about an ulp while sqrtf makes the distances equal ("witnesses"): a
# single bank returns the nearer row J[t], and so must the exchange of (d^2, row) keys on both transports.
g = np.random.Generator(np.random.PCG64(77))
Rw, Dw, n_pairs = 4099, 64, 24
libw = g.standard_normal((Rw, Dw), dtype=np.float32)
I = 100 + np.arange(n_pairs)
J = Rw * (world - 1) // world + 300 + np.arange(n_pairs)
for i, j in zip(I, J):
    libw[j] = libw[i]
    for c in g.choice(Dw, 2, replace=False):
        step = np.float32(np.inf) if g.random() < 0.5 else np.float32(-np.inf)
        libw[j, c] = np.nextafter(np.nextafter(libw[j, c], step), step)
qw = np.concatenate([libw[i] + 0.2 * g.standard_normal((128, Dw), dtype=np.float32) for i in I]).astype(np.float32)
pair = np.repeat(np.arange(n_pairs), 128)
fullw = Bank(Dw, Rw, device=local)
fullw.append(libw)
fullw.finalize()
fullw.build_knn()


def exact_min(b, q):
    v, i = np.empty(q.shape[0], np.float32), np.empty(q.shape[0], np.int64)
    assert b._lib.cmdb_debug_exact_min(b._h, q.ctypes.data, q.shape[0], v.ctypes.data, i.ctypes.data) == 0
    return v, i


pairs_i, pairs_j = Bank(Dw, n_pairs, device=local), Bank(Dw, n_pairs, device=local)
pairs_i.append(libw[I])
pairs_j.append(libw[J])
pairs_i.finalize()
pairs_j.finalize()
vi, _ = exact_min(pairs_i, qw)
vj, _ = exact_min(pairs_j, qw)
_, jf = exact_min(fullw, qw)
n_wit = int(((vi == vj) & (jf == J[pair])).sum())
pairs_i.close()
pairs_j.close()
xw = qw.reshape(12, 256, Dw)
bw = fullw.score_batch(xw, (16, 16), 64, full=True)
lo_w, hi_w = Rw * rank // world, Rw * (rank + 1) // world
shardw = Bank(Dw, hi_w - lo_w, device=local, row_offset=lo_w)
shardw.append(libw[lo_w:hi_w])
shardw.finalize()
shardw.build_knn_sharded()
for tag in ("nccl", "peer-memory"):
    if tag == "peer-memory":
        shardw.attach_comm(comm)
    aw = shardw.score_sharded_batch(xw, (16, 16), 64, full=True)
    report(f"[witness bank/{tag}] {n_wit} near-tie witnesses across ranks 0 and {world - 1}",
           all(same(aw[t], bw[t]) for t in range(12)))
shardw.attach_comm(None)
shardw.close()
fullw.close()
t = torch.tensor([bad], device="cuda")
dist.all_reduce(t)
if rank == 0:
    print("SHARD CHECK", "OK" if int(t) == 0 else f"FAILED on {int(t)} rank-checks", f"(world {world})", flush=True)
shard.close()
full.close()
comm.close()
dist.destroy_process_group()
sys.exit(0 if int(t) == 0 else 1)
