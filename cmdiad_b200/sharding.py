"""Host-side helpers of the row-sharded protocol (SURVEY 8e): shard ranges, packed (value,row) keys, ownership.

The device produces and consumes exactly these encodings (csrc/api.cu pack_keys_kernel / unpack_keys_kernel,
csrc/score_tail.cu pack_min_key); they are restated here so that the protocol can be exercised without a GPU
(tests/test_sharding_gloo.py runs it over gloo with world_size 2) and so that callers can plan shards."""
import numpy as np


def shard_range(n_rows, rank, world):
    """contiguous block of global rows owned by `rank` (same split as bench.py / Bank row_offset)"""
    return n_rows * rank // world, n_rows * (rank + 1) // world


def owner_of(row, n_rows, world):
    """rank owning a global row under shard_range"""
    row = np.asarray(row, dtype=np.int64)
    r = (row * world + world - 1) // n_rows  # upper bound, then fix up
    r = np.minimum(r, world - 1)
    lo = n_rows * r // world
    r = np.where(row < lo, r - 1, r)
    return r


def pack_keys(dist_f32, global_rows):
    """key = float_bits(d) << 32 | row.  d >= 0, so signed int64 order == (d, row) lexicographic order: an integer MIN
    all-reduce is argmin with lowest-global-row tie-break."""
    bits = np.ascontiguousarray(dist_f32, dtype=np.float32).view(np.uint32).astype(np.int64)
    return (bits << 32) | np.asarray(global_rows, dtype=np.int64)


def unpack_keys(keys):
    keys = np.asarray(keys, dtype=np.int64)
    d = (keys >> 32).astype(np.uint32).view(np.float32)
    return d, keys & 0xFFFFFFFF


def stage_slice(n_rows, world, rank):
    """cooperative staging of a round's host queries (Bank._stage_sharded): rank r copies rows [lo, hi) over PCIe into
    a `per`-row block (zero padded), the blocks are all-gathered and cut back to n_rows.  Returns (per, lo, hi)."""
    per = (n_rows + world - 1) // world
    return per, min(n_rows, rank * per), min(n_rows, (rank + 1) * per)


def knn_d2_contribution(rows_local, row_offset, m_test, nn_global_rows):
    """three-phase protocol with the replicated neighbour table (cmdb_score_shard_lookup): this shard's contribution to
    ||m_test - bank[nn_k]||^2 -- the float32 squared distance for the neighbour rows it owns, 0 for the others.  A float
    SUM all-reduce then yields the owner's value exactly (x + 0 + ... + 0)."""
    nn = np.asarray(nn_global_rows, dtype=np.int64)
    out = np.zeros(len(nn), dtype=np.float32)
    loc = nn - row_offset
    for k, l in enumerate(loc):
        if 0 <= l < rows_local.shape[0]:
            d = (np.asarray(m_test, np.float32) - rows_local[l]).astype(np.float32)
            out[k] = np.float32(np.sum(d.astype(np.float64) ** 2))
    return out
