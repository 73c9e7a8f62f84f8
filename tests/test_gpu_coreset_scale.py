"""GPU suite: the projection and the greedy coreset loop at the bank sizes they run at, compared exactly (int64 indices,
bit patterns of float16 / float64 min-distances, float64 projections) with the C oracle (canonical order), and on the
small FP16 cases also with the reference loop's own torch-CUDA restatement (coreset_torch_literal).

Covers what the small-bank tests in test_gpu_coreset.py cannot reach: the min-distance vector in global memory
(tests/test_coreset_plan.py has the placement rule), more than 65 536 FP16 picks (the grid all-gather's flag carries
pick & 0xffff), the all-tie tail of n_select == N, +inf FP16 distances, the projection's persistent tile loop over
hundreds of tiles per CTA and over row ranges off the tile grid, and handles with a row offset."""
import ctypes

import numpy as np
import pytest
import torch

from tests import cases
from tests.test_coreset_plan import restated_plan

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import Bank
    from cmdiad_b200 import _lib as L
    from oracle import restate as O
    assert torch.cuda.is_available()
    return dict(Bank=Bank, L=L, O=O, sms=torch.cuda.get_device_properties(0).multi_processor_count)


def identity_csr(d):
    """explicit CSR of the identity on the first d columns: z = x[:, :d] in float64, any (odd) width d"""
    return (np.arange(d + 1, dtype=np.int32), np.arange(d, dtype=np.int32), np.ones(d), d)


def device_normal(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda", dtype=torch.float32) * scale


def bank_of(env, x):
    b = env["Bank"](x.shape[1], x.shape[0])
    b.append(x)
    return b


def plan(env, N, d, dtype_mode):
    from cmdiad_b200 import _lib as L
    rpc, in_smem = ctypes.c_int64(), ctypes.c_int()
    L.check(L.load().cmdb_debug_coreset_plan(env["sms"], N, d, dtype_mode, ctypes.byref(rpc), ctypes.byref(in_smem)))
    assert (rpc.value, bool(in_smem.value)) == restated_plan(env["sms"], N, d, dtype_mode)[:2]
    return rpc.value, bool(in_smem.value)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape
    u = np.uint16 if a.dtype == np.float16 else np.uint64
    return bool((a.view(u) == b.view(u)).all())


def first_diff(a, b):
    d = np.nonzero(np.asarray(a) != np.asarray(b))[0]
    return f"first divergence at pick {d[:1]} of {len(a)}"


# ---- min-distance vector in global memory ----------------------------------------------------------------------------

def test_global_placement_natural_size_fp64(env):
    """1.3 M rows x d' = 301 in float64 mode: past the shared-memory limit on a B200, so the kernel reads and writes
    the min-distances through L2 -- free-running against the oracle, then teacher-forced onto the first and last rows
    of CTA ranges and of their 4-warp groups (min_d[sel] zeroed by another CTA than the one that found it)"""
    O, L = env["O"], env["L"]
    N, D, dp = 1_300_000, 320, 301
    rpc, in_smem = plan(env, N, dp, L.CORESET_FP64)
    assert not in_smem, "this shape must use global placement"
    x = device_normal((N, D), 20261021)
    b = bank_of(env, x)
    z = x[:, :dp].double().cpu().numpy()
    del x
    torch.cuda.empty_cache()
    csr = identity_csr(dp)

    n = 200
    idx, mn = b.coreset_select(n, csr, L.CORESET_FP64, return_min=True)
    ref, st = O.coreset_restated(z, n, "TF32", return_state=True)
    assert (idx == ref).all(), first_diff(idx, ref)
    assert same_bits(mn, st["min_last"])

    rows = []
    for c in sorted({0, 1, env["sms"] // 2, env["sms"] - 1}):
        r0, r1 = c * rpc, min(N, (c + 1) * rpc)
        rpg = -(-(r1 - r0) // 4)
        for g in range(4):
            g0, g1 = r0 + g * rpg, min(r1, r0 + (g + 1) * rpg)
            rows += [g0, g0 + 1, g1 - 2, g1 - 1]
    rows = list(dict.fromkeys(rows))
    force = np.array([0] + rows, dtype=np.int64)
    got, mn = b.coreset_select(len(force), csr, L.CORESET_FP64, force_idx=force, return_min=True)
    ref, st = O.coreset_restated(z, len(force), "TF32", force_idx=force, return_state=True)
    assert (got == ref).all(), first_diff(got, ref)
    assert same_bits(mn, st["min_last"])
    assert (mn[force] == 0).all()
    b.close()


SMALL_SHAPES = [(1001, 100, 64), (5000, 128, 200), (2500, 130, 100), (4097, 131, 150), (148 * 16 * 4 + 3, 301, 60),
                (300, 267, 300), (50, 64, 1)]


def small_case(N, d):
    """the banks of test_gpu_coreset.test_coreset_shapes_no_projection"""
    g = np.random.Generator(np.random.PCG64(N * 7 + d))
    if d % 64 != 0:
        D = (d + 63) // 64 * 64
        x = g.standard_normal((N, D), dtype=np.float32)
        return x, identity_csr(d), x[:, :d].astype(np.float64)
    x = g.standard_normal((N, d), dtype=np.float32)
    return x, None, x.astype(np.float64)


def check_forced_global(env, b, z, n, csr):
    O, L = env["O"], env["L"]
    for mode, name in ((L.CORESET_FP16, "FP16"), (L.CORESET_FP64, "TF32")):
        i_s, m_s = b.coreset_select(n, csr, mode, return_min=True)
        i_g, m_g = b.coreset_select(n, csr, mode, return_min=True, _mind_global=True)
        ref, st = O.coreset_restated(z, n, name, return_state=True)
        assert (i_g == i_s).all(), (name, first_diff(i_g, i_s))
        assert (i_g == ref).all(), (name, first_diff(i_g, ref))
        assert same_bits(m_g, m_s) and same_bits(m_g, st["min_last"]), name


@pytest.mark.parametrize("N,d,n", SMALL_SHAPES)
def test_forced_global_placement_shapes(env, N, d, n):
    """the global-memory branch (natural for FP16 only above ~10 M rows) == the shared-memory branch == the oracle"""
    x, csr, z = small_case(N, d)
    assert plan(env, N, d, env["L"].CORESET_FP16)[1] and plan(env, N, d, env["L"].CORESET_FP64)[1]
    b = bank_of(env, x)
    check_forced_global(env, b, z, n, csr)
    b.close()


def test_forced_global_placement_golden(env, golden):
    O, L = env["O"], env["L"]
    lib = cases.rgb_normalised_lib(golden)
    csr = O.sparse_components(lib.shape[0], lib.shape[1], 0.9, 0)
    n = int(0.1 * lib.shape[0])
    b = bank_of(env, lib)
    check_forced_global(env, b, O.project_restated(lib, *csr), n, csr)
    idx = b.coreset_select(n, csr, L.CORESET_FP64, _mind_global=True)
    assert (idx == golden["rgb_case"]["coreset_idx_TF32"]).all()
    b.close()


# ---- long selections and the tie tail --------------------------------------------------------------------------------

def test_fp16_selection_beyond_65536_picks(env):
    """66 500 picks from 70 000 rows at d' = 131: the all-gather's 16-bit pick flag wraps once, and the late picks run
    where most keys tie -- free-running against the oracle, final min-distances included.

    The oracle, not coreset_torch_literal: on this bank torch-CUDA's half norm leaves the canonical order the kernel and
    the oracle share (torch 2.11 on a B200: the literal departs from both at pick 13 898 with identical initial
    distances, while kernel and oracle agree on every pick and on the final min-distance bits)."""
    O, L = env["O"], env["L"]
    N, D, dp, n = 70_000, 192, 131, 66_500
    x = device_normal((N, D), 7)
    b = bank_of(env, x)
    z = x[:, :dp].double().cpu().numpy()
    idx, mn = b.coreset_select(n, identity_csr(dp), L.CORESET_FP16, return_min=True)
    ref, st = O.coreset_restated(z, n, "FP16", return_state=True)
    assert (idx == ref).all(), first_diff(idx, ref)
    assert same_bits(mn, st["min_last"])
    assert len(np.unique(idx)) == n
    b.close()


def test_select_every_row_all_tie_tail(env):
    """n_select == N on a bank of duplicated rows: once every distinct row is picked all min-distances are 0 and every
    later argmax is row 0, exactly as torch.argmax"""
    O, L = env["O"], env["L"]
    g = np.random.Generator(np.random.PCG64(31))
    base = g.standard_normal((1200, 192), dtype=np.float32)
    x = np.concatenate([base, base, base[:600]], 0)
    N, dp = x.shape[0], 131
    csr = identity_csr(dp)
    z = x[:, :dp].astype(np.float64)
    b = bank_of(env, x)
    for mode, name in ((L.CORESET_FP16, "FP16"), (L.CORESET_FP64, "TF32")):
        idx, mn = b.coreset_select(N, csr, mode, return_min=True)
        ref, st = O.coreset_restated(z, N, name, return_state=True)
        assert (idx == ref).all(), (name, first_diff(idx, ref))
        assert same_bits(mn, st["min_last"]) and (mn == 0).all()
        assert len(np.unique(idx[:1200])) == 1200 and (idx[1200:] == 0).all(), name
    lit = O.coreset_torch_literal(torch.from_numpy(z), N, "FP16", device="cuda").numpy()
    assert (b.coreset_select(N, csr, L.CORESET_FP16) == lit).all()
    b.close()


def test_fp16_infinite_distances(env):
    """|z| < 65 504 everywhere, but many FP16 distances round to +inf: the argmax over +inf keys takes the lowest row"""
    O, L = env["O"], env["L"]
    N, D, dp, n = 4000, 192, 131, 400
    g = np.random.Generator(np.random.PCG64(65504))
    scale = np.exp(g.uniform(np.log(300.0), np.log(7000.0), size=(N, 1))).astype(np.float32)
    x = (g.standard_normal((N, D), dtype=np.float32) * scale).astype(np.float32)
    z = x[:, :dp].astype(np.float64)
    assert np.abs(z).max() < 65504
    b = bank_of(env, x)
    idx, mn = b.coreset_select(n, identity_csr(dp), L.CORESET_FP16, return_min=True)
    ref, st = O.coreset_restated(z, n, "FP16", return_state=True)
    n_inf0 = int(np.isinf(st["min0"]).sum())
    assert 10 < n_inf0 < N - 10, n_inf0
    # rows of the largest scales are +inf away from every other row: the first picks walk them in row order
    assert (np.diff(idx[1:11]) > 0).all(), idx[:11]
    lit =O.coreset_torch_literal(torch.from_numpy(z), n, "FP16", device="cuda").numpy()
    assert (idx == lit).all(), first_diff(idx, lit)
    assert (idx == ref).all(), first_diff(idx, ref)
    assert same_bits(mn, st["min_last"])
    b.close()


# ---- projection at scale ---------------------------------------------------------------------------------------------

def _projection_rows(D, d_proj, nnz):
    """rows per tile project_rows picks (shared-memory budget of 220 KB)"""
    csr_bytes = 4 * (d_proj + 1) + 2 * nnz + 16
    rt = 32
    while rt > 8 and 4 * rt * (D + 1) + csr_bytes > 220 * 1024:
        rt >>= 1
    return rt


@pytest.mark.parametrize("D,rt", [(768, 32), (1920, 16)])
def test_projection_at_scale(env, D, rt):
    """300 007 rows: every CTA walks ~60-130 tiles; sub-ranges that start and end off the tile grid equal the same slice
    of the whole-bank projection"""
    O = env["O"]
    N = 300_007
    xd = device_normal((N, D), 1000 + D)
    b = bank_of(env, xd)
    x = xd.cpu().numpy()
    del xd
    csr = O.sparse_components(N, D, 0.9, 0)
    assert _projection_rows(D, csr[3], int(csr[0][-1])) == rt
    assert N / rt / env["sms"] > 60
    z = b.project(csr)
    ref = O.project_restated(x, *csr)
    assert (z == ref).all()
    for row0, n in ((12_345, 77_777), (1, N - 2), (N - 50_001, 50_001), (rt * 1000 + rt - 1, rt * 300 + 1)):
        assert (b.project(csr, row0, n) == ref[row0:row0 + n]).all(), (row0, n)
    b.close()


def test_projection_generic_csr_at_scale(env):
    """non-uniform magnitudes (float64 data + int32 indices through L1) over 300 007 rows"""
    O = env["O"]
    N, D, d_proj = 300_007, 768, 211
    g = np.random.Generator(np.random.PCG64(17))
    per = g.integers(5, 40, size=d_proj)
    indices = np.concatenate([g.choice(D, k, replace=False) for k in per]).astype(np.int32)
    indptr = np.concatenate([[0], np.cumsum(per)]).astype(np.int32)
    data = g.standard_normal(int(indptr[-1]))
    csr = (indptr, indices, data, d_proj)
    xd = device_normal((N, D), 5)
    b = bank_of(env, xd)
    x = xd.cpu().numpy()
    del xd
    ref = O.project_restated(x, *csr)
    assert (b.project(csr) == ref).all()
    assert (b.project(csr, 12_345, 77_777) == ref[12_345:12_345 + 77_777]).all()
    b.close()


# ---- handles with a row offset ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("dp", [131, 301])
def test_row_offset_handle_selects_like_offset_zero(env, dp):
    """coreset_select on a handle with row_offset k (a loaded shard, for example) returns the local rows an offset-0
    handle holding the same rows returns; (k * d') & 3 takes the values 1, 2 and 3"""
    O, L = env["O"], env["L"]
    N, n = 3001, 150
    D = (dp + 63) // 64 * 64
    g = np.random.Generator(np.random.PCG64(dp))
    x = g.standard_normal((N, D), dtype=np.float32)
    csr = identity_csr(dp)
    z = x[:, :dp].astype(np.float64)
    base = bank_of(env, x)
    want = {}
    for mode, name in ((L.CORESET_FP16, "FP16"), (L.CORESET_FP64, "TF32")):
        want[mode] = base.coreset_select(n, csr, mode, return_min=True)
        assert (want[mode][0] == O.coreset_restated(z, n, name)).all()
    base.close()
    assert {(k * dp) & 3 for k in (1, 2, 3, 5)} == {1, 2, 3}
    for k in (1, 2, 3, 5):
        b = env["Bank"](D, N, row_offset=k)
        b.append(x)
        for mode in (L.CORESET_FP16, L.CORESET_FP64):
            idx, mn = b.coreset_select(n, csr, mode, return_min=True)
            assert (idx == want[mode][0]).all(), (k, mode, first_diff(idx, want[mode][0]))
            assert same_bits(mn, want[mode][1]), (k, mode)
            assert (b.coreset_select(n, csr, mode) == idx).all()
        b.close()


# ---- device state --------------------------------------------------------------------------------------------------

def test_persisting_l2_limit_restored(env):
    """the coreset call may enlarge the process-wide persisting-L2 carve-out while it runs and hands it back as found"""
    L = env["L"]
    rt = ctypes.CDLL("libcudart.so.12")
    cuda_limit_persisting_l2 = 0x06   # cudaLimitPersistingL2CacheSize
    x, csr, _ = small_case(5000, 128)
    b = bank_of(env, x)

    def limit():
        v = ctypes.c_size_t()
        assert rt.cudaDeviceGetLimit(ctypes.byref(v), cuda_limit_persisting_l2) == 0
        return v.value

    before = limit()
    b.coreset_select(200, csr, L.CORESET_FP16)
    assert limit() == before
    b.coreset_select(200, csr, L.CORESET_FP64)
    assert limit() == before
    b.close()
