"""CPU suite: where the greedy coreset kernel keeps its running min-distance vector, restated on the host from the kernel's
shared-memory layout and checked against the rule the library applies (cmdb_debug_coreset_plan, the function
launch_coreset calls).

One persistent CTA per SM; CTA c owns rows [c * rows_per_cta, min(N, (c + 1) * rows_per_cta)) with
rows_per_cta = ceil(N / num_sms).  Dynamic shared memory of coreset_kernel (csrc/coreset.cu):

    tile  [kCsWarps = 16][32][33] acc_t     (float in FP16 mode, double in float64 mode)
    last  [d'] storage type                 (half / double)
    <= 16 bytes to the next 16-byte boundary
    red   64 x 8 bytes                      (per-warp argmax value / row)
    mind  [rows_per_cta] storage type       (only while the whole block is <= 200 KB)

Above 200 KB the min-distances stay in global memory and every access goes through L2.  On a B200 (148 SMs) that
happens from these bank sizes on (N is the first size that uses global memory):

    d'    float64 ('TF32') mode            FP16 mode
    131   8 507 rows/CTA, N = 1 259 037   68 213 rows/CTA, N = 10 095 525
    221   8 417 rows/CTA, N = 1 245 717   68 123 rows/CTA, N = 10 082 205
    301   8 337 rows/CTA, N = 1 233 877   68 043 rows/CTA, N = 10 070 365
    375   8 263 rows/CTA, N = 1 222 925   67 969 rows/CTA, N = 10 059 413

So the benchmark's 200 000-row and 1 000 000-row banks keep the vector in shared memory in both modes;
tests/test_gpu_coreset_scale.py runs the global branch at a natural size (float64, 1.3 M rows) and forced.
"""
import ctypes

import pytest

K_CS_WARPS = 16           # kCsThreads / 32
SMEM_LIMIT = 200 * 1024   # launch_coreset's budget for the whole block
FP16, FP64 = 0, 1         # CMDB_CORESET_FP16 / CMDB_CORESET_FP64
DIMS = [32, 64, 127, 128, 131, 301, 341, 375, 1024]
SMS = [148, 132, 1]


def sizes(dtype_mode):
    """(storage bytes, accumulator bytes) per element"""
    return (2, 4) if dtype_mode == FP16 else (8, 8)


def kernel_layout_bytes(d, dtype_mode, rows_in_smem):
    """bytes coreset_kernel's pointer arithmetic actually touches: tile | last | align 16 | red | mind"""
    elem, acc = sizes(dtype_mode)
    tile = K_CS_WARPS * 32 * 33 * acc
    red = (tile + elem * d + 15) // 16 * 16
    return red + 64 * 8 + elem * rows_in_smem


def restated_plan(num_sms, N, d, dtype_mode):
    """(rows_per_cta, mind in shared memory, dynamic shared memory of the launch)"""
    elem, acc = sizes(dtype_mode)
    fixed = K_CS_WARPS * 32 * 33 * acc + elem * d + 16 + 64 * 8   # the alignment gap reserved at its maximum
    rows_per_cta = -(-N // num_sms)
    smem = fixed + elem * rows_per_cta
    in_smem = smem <= SMEM_LIMIT
    return rows_per_cta, in_smem, smem if in_smem else fixed


def flip_point(num_sms, d, dtype_mode):
    """largest N whose min-distances still fit shared memory"""
    elem, acc = sizes(dtype_mode)
    fixed = K_CS_WARPS * 32 * 33 * acc + elem * d + 16 + 64 * 8
    return (SMEM_LIMIT - fixed) // elem * num_sms


@pytest.fixture(scope="module")
def hook(built):
    from cmdiad_b200 import _lib as L
    lib = L.load()

    def plan(num_sms, N, d, dtype_mode):
        rpc, in_smem = ctypes.c_int64(-1), ctypes.c_int(-1)
        L.check(lib.cmdb_debug_coreset_plan(num_sms, N, d, dtype_mode, ctypes.byref(rpc), ctypes.byref(in_smem)))
        assert in_smem.value in (0, 1)
        return rpc.value, bool(in_smem.value)
    return plan


@pytest.mark.parametrize("dtype_mode", [FP16, FP64], ids=["FP16", "FP64"])
@pytest.mark.parametrize("num_sms", SMS)
@pytest.mark.parametrize("d", DIMS)
def test_plan_matches_restatement(hook, d, num_sms, dtype_mode):
    flip = flip_point(num_sms, d, dtype_mode)
    assert flip > 0
    Ns = {1, 2, 3, num_sms - 1, num_sms, num_sms + 1, 4 * num_sms + 3, 200_000, 1_000_000, 1_300_000, 10_100_000,
          flip // 2, flip - 1, flip, flip + 1, 2 * flip, (1 << 32) - 2}
    for N in sorted(n for n in Ns if n >= 1):
        rpc, in_smem, smem = restated_plan(num_sms, N, d, dtype_mode)
        assert hook(num_sms, N, d, dtype_mode) == (rpc, in_smem), (N, d, num_sms, dtype_mode)
        # the host's reservation covers what the kernel addresses, in both placements
        assert kernel_layout_bytes(d, dtype_mode, rpc if in_smem else 0) <= smem <= SMEM_LIMIT
    # the switch sits exactly at the flip point: N - 1 and N in shared memory, N + 1 in global memory
    assert hook(num_sms, flip - 1, d, dtype_mode)[1]
    assert hook(num_sms, flip, d, dtype_mode)[1]
    assert not hook(num_sms, flip + 1, d, dtype_mode)[1]
    assert hook(num_sms, flip + 1, d, dtype_mode)[0] == flip // num_sms + 1


@pytest.mark.parametrize("num_sms", SMS)
def test_cta_ranges_cover_every_row_once(hook, num_sms):
    """the kernel's CTA ranges [c * rows_per_cta, min(N, (c + 1) * rows_per_cta)) tile [0, N); when N < num_sms (and
    for some N above it) trailing CTAs own no rows and still take part in every pick's all-gather"""
    for N in (1, 2, 5, 50, 147, 148, 149, 296, 297, 1001, 4 * 148 + 3, 148 * 16 * 4 + 3, 1_233_877):
        rpc, _ = hook(num_sms, N, 301, FP64)
        assert num_sms * rpc >= N and (rpc - 1) * num_sms < N
        covered, empty = 0, 0
        for c in range(num_sms):
            r0 = c * rpc
            r1 = min(N, r0 + rpc)
            n = max(0, r1 - r0)
            if n:
                assert r0 == covered   # contiguous, in CTA order, no overlap
            covered += n
            empty += n == 0
        assert covered == N
        assert empty == num_sms - (-(-N // rpc))
        if N < num_sms:
            assert rpc == 1 and empty == num_sms - N > 0


def test_b200_thresholds_in_docstring(hook):
    """the table of the module docstring"""
    table = {131: (8507, 68213), 221: (8417, 68123), 301: (8337, 68043), 375: (8263, 67969)}
    for d, (r64, r16) in table.items():
        for mode, r in ((FP64, r64), (FP16, r16)):
            assert hook(148, 148 * r, d, mode) == (r, True)
            assert hook(148, 148 * r + 1, d, mode) == (r + 1, False)
    # the benchmark's banks (d' = 301 and smaller) keep the vector in shared memory in both modes
    for N in (200_000, 1_000_000):
        for mode in (FP16, FP64):
            assert hook(148, N, 301, mode)[1]


def test_plan_rejects_bad_arguments(hook, built):
    from cmdiad_b200 import _lib as L
    lib = L.load()
    rpc, in_smem = ctypes.c_int64(), ctypes.c_int()
    assert lib.cmdb_debug_coreset_plan(0, 100, 301, FP16, ctypes.byref(rpc), ctypes.byref(in_smem)) == L.CMDB_ERR_INVALID
    assert lib.cmdb_debug_coreset_plan(148, 0, 301, FP16, ctypes.byref(rpc), ctypes.byref(in_smem)) == L.CMDB_ERR_INVALID
    assert lib.cmdb_debug_coreset_plan(148, 100, 301, 7, ctypes.byref(rpc), ctypes.byref(in_smem)) == L.CMDB_ERR_INVALID
