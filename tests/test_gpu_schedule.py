"""GPU tests of the distance GEMM's schedule with runs of N tiles (banks above 75k rows), against the host restatement in
tests/test_schedule.py: the candidate lists the GEMM writes, the exact rescan of uncertified (query, producer) pairs at
run > 1 on every input path, and the neighbour table of large banks against a brute force."""
import numpy as np
import pytest
import torch

from tests import test_schedule as S

pytestmark = pytest.mark.gpu

P_IMG, FM = 784, (28, 28)
DUP_NOISE = 2e-4    # as in test_gpu_score.py::test_rescan_tier_under_load: far inside the pre-filter's error band


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import Bank
    from cmdiad_b200 import _lib as L
    assert torch.cuda.is_available()
    return dict(Bank=Bank, L=L)


def _grouped_bank(R, D, seed, n_per_kind):
    """Gaussian bank (on the device) with three kinds of near-duplicate groups of 6 rows, all inside one column group:
      "run":  rows r + 256 i (i < 6): one row in each of 6 consecutive N tiles, so a run of >= 3 tiles holds >= 3 of them;
      "run2": rows r + 256 i + {0, 1} (i < 3): two rows in each of 3 consecutive tiles (>= 3 in one run of 2);
      "tile": rows r .. r + 5 of one tile.
    Each kind uses its own column offsets, so groups never share a row.  Returns (bank, {kind: [groups, 6] rows})."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    lib = torch.randn(R, D, generator=gen, device="cuda")
    rng = np.random.Generator(np.random.PCG64(seed))
    nt_full = R // S.BN
    groups = {}
    for kind, span, lo, width in (("run", 6, 0, 42), ("run2", 3, 42, 41), ("tile", 1, 84, 38)):
        t0 = rng.choice(nt_full // span, n_per_kind, replace=False) * span
        off = rng.integers(0, 2, n_per_kind) * S.COLS + lo + rng.integers(0, width, n_per_kind)
        first = t0 * S.BN + off
        if kind == "run":
            step = S.BN * np.arange(6)
        elif kind == "run2":
            step = (S.BN * np.arange(3)[:, None] + np.arange(2)).ravel()
        else:
            step = np.arange(6)
        groups[kind] = first[:, None] + step[None]
    rows = torch.from_numpy(np.concatenate(list(groups.values()))).cuda()
    base = lib[rows[:, 0]]
    lib[rows] = base[:, None] + DUP_NOISE * torch.randn(rows.shape + (D,), generator=gen, device="cuda")
    assert torch.unique(rows).numel() == rows.numel()
    return lib, groups


def _queries(lib, groups, B, P, seed, frac=6):
    """B x P Gaussian queries; every frac-th one sits 0.05 (per dimension) from a group's first row instead.  Returns the
    queries (device) and how many sit next to a group of each kind."""
    D = lib.shape[1]
    gen = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(B * P, D, generator=gen, device="cuda")
    near = torch.arange(0, B * P, frac, device="cuda")
    kinds = list(groups)
    which = np.arange(near.numel()) % len(kinds)
    rng = np.random.Generator(np.random.PCG64(seed))
    src = np.array([groups[kinds[w]][rng.integers(0, len(groups[kinds[w]])), 0] for w in which])
    q[near] = lib[torch.from_numpy(src).cuda()] + 0.05 * torch.randn(near.numel(), D, generator=gen, device="cuda")
    return q.view(B, P, D).contiguous(), {k: int((which == i).sum()) for i, k in enumerate(kinds)}


def _flat(res, name):
    return np.concatenate([getattr(r, name) for r in res])


def _cert_bound(lib, q):
    """E of the certificate (score_tail.cu, as in test_gpu_score.py::_measure_error_model) per query row, float64"""
    D = lib.shape[1]
    l64, q64 = lib.double(), q.double()
    eb = 13 - int(torch.frexp(lib.abs().max()).exponent)
    bh = (lib * 2.0 ** eb).half().double() * 2.0 ** -eb
    eq = 13 - torch.frexp(q.abs().amax(1)).exponent.double()
    qh = (q * torch.exp2(eq)[:, None].float()).half().double() * torch.exp2(-eq)[:, None]
    bmax, ebmax = l64.norm(dim=1).max(), (l64 - bh).norm(dim=1).max()
    qn, qe = q64.norm(dim=1), (q64 - qh).norm(dim=1)
    acc = (D // 16 + 1) * 17 * 2.0 ** -23
    return 2 * (qe * (bmax + ebmax) + qn * ebmax + acc * (qn + qe) * (bmax + ebmax)) + (D + 16) * 2.0 ** -24 * (qn + bmax) ** 2


def _check_lists(b, lib, q_flat, chunks, what):
    """The GEMM's candidate lists of the last call against the restated schedule: every kept row lies in the rows its
    producer saw for that M tile (under that chunk launch's stride and run), a producer with rows kept at least one,
    v1 <= v2, and on a sample of queries the kept row is the smallest of its producer's rows within 2E"""
    import ctypes
    R = lib.shape[0]
    P = q_flat.shape[0]
    n_prod = S.EG * S.G_B200
    cand = np.zeros((n_prod, P, 4), np.float32)
    assert b._lib.cmdb_debug_read_candidates(b._h, cand.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n_prod), ctypes.c_int(P)) == 0
    v1, v2 = cand[:, :, 0], cand[:, :, 2]
    i1, i2 = cand[:, :, 1].copy().view(np.int32), cand[:, :, 3].copy().view(np.int32)
    assert ((i2 < 0) | ((i1 >= 0) & (v1 <= v2))).all(), what
    assert (i1 < R).all() and (i2 < R).all()
    E = _cert_bound(lib, q_flat).cpu().numpy()
    rows = np.arange(R)
    lib64 = lib.double()
    for first, mt in chunks:
        la = S.Launch(R, mt)
        q0, q1 = first * S.BM, min(P, (first + mt) * S.BM)
        qs = np.arange(q0, q1)
        m = qs // S.BM - first
        for i in (i1, i2):
            blk = i[:, q0:q1]
            ok = blk >= 0
            prod = la.owner[np.where(ok, blk, 0) // S.BN // la.run, m[None]] * S.EG + (np.where(ok, blk, 0) % S.BN) // S.COLS
            bad = ok & (prod != np.arange(n_prod)[:, None])
            assert not bad.any(), (what, first, mt, la.run, np.argwhere(bad)[:5])
        # producers whose row set for the tile is not empty kept a row; the others kept none
        for mm in range(mt):
            sel = slice(q0 + mm * S.BM, min(q1, q0 + (mm + 1) * S.BM))
            pid = la.row_owner(mm, rows) * S.EG + (rows % S.BN) // S.COLS
            has = np.bincount(pid, minlength=n_prod) > 0
            assert ((i1[:, sel] >= 0) == has[:, None]).all(), (what, first, mm)
        # kept row = smallest of its producer's rows, up to the pre-filter's error (2E between any two rows' values)
        sample = np.unique(np.linspace(q0, q1 - 1, 6).astype(np.int64))
        for qi in sample:
            d = ((lib64 - q_flat[qi].double()) ** 2).sum(1)
            mm = qi // S.BM - first
            pid = torch.from_numpy(la.row_owner(mm, rows) * S.EG + (rows % S.BN) // S.COLS).cuda()
            smin = torch.full((n_prod,), float("inf"), dtype=torch.float64, device="cuda").scatter_reduce(0, pid, d, "amin")
            kept = torch.from_numpy(i1[:, qi].astype(np.int64)).cuda()
            has = kept >= 0
            excess = (d[kept.clamp(min=0)] - smin)[has]
            assert (excess <= 2 * E[qi]).all(), (what, qi, float(excess.max()), 2 * E[qi])


_RESULT_FIELDS = ("min_idx", "min_val", "s", "s_star", "s_idx", "nn_idx", "m_star_knn", "w", "s_map")


def _same(a, b, tag, fields=_RESULT_FIELDS):
    for i in range(len(a)):
        for name in fields:
            assert (getattr(a[i], name) == getattr(b[i], name)).all(), (tag, i, name)


# (bank rows, D, images): 16 images host 2/3 (4 chunks), device and pending 5; 3 images host 1/4; 6 images host 7/8
CASES = [(200_000, 64, 16), (200_000, 64, 3), (400_000, 64, 6)]


@pytest.mark.parametrize("R,D,B", CASES)
def test_rescans_and_candidate_lists_at_long_runs(env, R, D, B):
    """Certified scoring with uncertified pairs whose hidden rows lie in other tiles of the same run: on the device,
    pinned-host (chunked, full != last run) and pending (one chunk) paths the answers equal the exact scan bit for bit
    and the re-weighting equals the CUDA-core implementation's; the candidate lists follow the restated schedule."""
    L = env["L"]
    lib, groups = _grouped_bank(R, D, seed=R // 1000 + D, n_per_kind=120)
    q, near = _queries(lib, groups, B, P_IMG, seed=R // 1000 + B)
    q_flat = q.view(-1, D)
    pinned = q.cpu().pin_memory()
    b = env["Bank"](D, R)
    b.append(lib)
    b.finalize()
    b.set_score_impl(L.SCORE_SIMT)
    ref = b.score_batch(pinned, FM, 224)
    b.set_score_impl(L.SCORE_TCGEN05)
    ex_val, ex_idx = np.empty(B * P_IMG, np.float32), np.empty(B * P_IMG, np.int64)
    qh = q_flat.cpu().numpy()
    assert b._lib.cmdb_debug_exact_min(b._h, qh.ctypes.data, B * P_IMG, ex_val.ctypes.data, ex_idx.ctypes.data) == 0
    layout = {"device": S.stage_chunks(B * P_IMG, True), "host": S.stage_chunks(B * P_IMG, False),
              "pending": S.stage_chunks(B * P_IMG, False, pending=True)}
    nt = (R + S.BN - 1) // S.BN

    def check(res, what, table):
        st = b.score_stats()
        ch = layout[what]
        runs = [S.gemm_run(nt, mt, S.G_B200) for _, mt in ch]
        print(f"{R} x {D}, {B} img {what}{' (table)' if table else ''}: {len(ch)} chunk(s) of {ch[0][1]}/{ch[-1][1]} M tiles, "
              f"run {runs[0]}/{runs[-1]}, near groups {near}, {st}")
        assert st["mode"] == 0 and not st["gemm_fallback"] and st["queries"] == B * P_IMG, st
        assert st["rescan_pairs"] >= near["tile"], st          # a query next to a one-tile group queues that producer
        bad = np.nonzero((_flat(res, "min_idx") != ex_idx) | (_flat(res, "min_val") != ex_val))[0]
        assert bad.size == 0, (what, bad.size, bad[:8])
        _same(ref, res, f"{what} vs exact-scan implementation", ("s", "s_idx", "nn_idx", "s_map"))

    check(b.score_batch(q, FM, 224), "device", False)
    check(b.score_batch(pinned, FM, 224), "host", False)
    t1 = b.score_batch_async(pinned, FM, 224)
    t2 = b.score_batch_async(pinned, FM, 224)     # submitted while t1 is outstanding: one chunk
    r1, r2 = t1.wait(), t2.wait()
    check(r2, "pending", False)
    _same(ref, r1, "async, nothing pending", ("min_idx", "min_val", "s", "s_idx", "nn_idx", "s_map"))
    # the batched re-weighting without a table rewrites M tile 0 of every list: read the min phase's lists with the table
    b.build_knn()
    for what, src in (("host", pinned), ("device", q)):
        check(b.score_batch(src, FM, 224), what, True)
        _check_lists(b, lib, q_flat, layout[what], what)
    b.close()


def _brute_top3(lib):
    """three nearest rows of every row: float32 candidates (top 8, TF32 off) re-evaluated in float64, ordered by
    (distance, row).  Returns rows [R, 4] and float64 d^2 [R, 4] (the 4th for near-ties)"""
    R = lib.shape[0]
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        n2 = (lib * lib).sum(1)
        rows, d64 = [], []
        for r0 in range(0, R, 2048):
            a = lib[r0:r0 + 2048]
            d2 = n2[r0:r0 + 2048, None] + n2[None] - 2.0 * (a @ lib.T)
            idx = torch.topk(d2, 8, dim=1, largest=False).indices
            ex = ((a.double()[:, None, :] - lib[idx].double()) ** 2).sum(-1)
            rows.append(idx.cpu().numpy()), d64.append(ex.cpu().numpy())
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    rows, d64 = np.concatenate(rows), np.concatenate(d64)
    order = np.lexsort((rows, d64), axis=1)[:, :4]
    return np.take_along_axis(rows, order, 1), np.take_along_axis(d64, order, 1)


def _table(b, R):
    keys = b.read_knn(0, R).numpy().view(np.uint64)
    return (keys & np.uint64(0xffffffff)).astype(np.int64), (keys >> np.uint64(32)).astype(np.uint32).view(np.float32), keys


# 200k x 768: table GEMM run 5 on all 25 chunks (ragged last chunk of 3392 rows); 150k x 128: run 3 / 2, re-weighting run 2
@pytest.mark.parametrize("R,D", [(200_000, 768), (150_000, 128)])
def test_knn_table_on_large_banks(env, R, D):
    """Every row of the neighbour table against a brute force, with near-duplicate groups spread over runs (the certificate's
    bad-producer walk) and exact duplicate rows (first neighbour = lowest duplicate); build_knn_rows over ranges that start
    off the 128- and 8192-row grids gives the same keys; at 150k the batched tensor-core re-weighting without a table
    equals the single-image CUDA-core sweep and the table lookup."""
    lib, groups = _grouped_bank(R, D, seed=7 + D, n_per_kind=60)
    rng = np.random.Generator(np.random.PCG64(D))
    used = np.zeros(R, bool)
    used[np.concatenate([g.ravel() for g in groups.values()])] = True
    free = np.nonzero(~used)[0]
    pick = rng.choice(free, 600, replace=False)
    src, dst = np.minimum(pick[:300], pick[300:]), np.maximum(pick[:300], pick[300:])
    lib[torch.from_numpy(dst).cuda()] = lib[torch.from_numpy(src).cuda()]
    b = env["Bank"](D, R)
    b.append(lib)
    b.finalize()
    if D == 128:
        # each image: patches next to random bank rows, one farther patch next to a group -> m_star is a group member
        P, fm = 100, (10, 10)
        gen = torch.Generator(device="cuda").manual_seed(11)
        near_rows = torch.from_numpy(rng.integers(0, R, (6, P))).cuda()
        patches = lib[near_rows] + 1e-3 * torch.randn(6, P, D, generator=gen, device="cuda")
        gsel = np.concatenate([groups[k][:2, 0] for k in groups])
        patches[:, 37] = lib[torch.from_numpy(gsel).cuda()] + 0.05 * torch.randn(6, D, generator=gen, device="cuda")
        patches = patches.cpu()
        batch_tensor = b.score_batch(patches, fm, 64)
        print(f"{R} x {D}: batched re-weighting GEMM run {S.gemm_run((R + S.BN - 1) // S.BN, 1, S.G_B200)}")
        assert all(int(r.nn_idx[0]) in set(np.concatenate([g.ravel() for g in groups.values()]).tolist()) for r in batch_tensor)
        singles = [b.score(patches[i], fm, 64) for i in range(6)]
        _same(batch_tensor, singles, "tensor-core re-weighting vs CUDA-core sweep")
    b.build_knn()
    rows_t, d2_t, keys = _table(b, R)
    ref_rows, ref_d64 = _brute_top3(lib)
    agree = (np.sort(rows_t, 1) == np.sort(ref_rows[:, :3], 1)).all(1)
    tie = ref_d64[:, 2] * (1 + 1e-5) >= ref_d64[:, 3]
    chunks = S.table_chunks(0, R)
    print(f"{R} x {D} table: {len(chunks)} chunks, last {chunks[-1][1]} rows, run "
          f"{S.gemm_run((R + S.BN - 1) // S.BN, 64, S.G_B200)}/{S.gemm_run((R + S.BN - 1) // S.BN, (chunks[-1][1] + 127) // 128, S.G_B200)}; "
          f"{int((~agree).sum())} rows differ from the brute force only by a 3rd/4th near-tie")
    assert (agree | tie).all(), np.nonzero(~(agree | tie))[0][:10]
    # d^2 of the table's own rows, float64
    lt = lib.double()
    ex = np.concatenate([((lt[r0:r0 + 4096, None, :] - lt[torch.from_numpy(rows_t[r0:r0 + 4096]).cuda()]) ** 2).sum(-1).cpu().numpy()
                         for r0 in range(0, R, 4096)])
    np.testing.assert_allclose(d2_t, ex, rtol=1e-5, atol=1e-6)
    first = np.arange(R)
    first[dst] = src
    assert (rows_t[:, 0] == first).all() and (d2_t[:, 0] == 0).all()     # a row's first neighbour: its lowest duplicate
    assert all(dst[i] in rows_t[src[i]] for i in range(len(src)))
    for k, g in groups.items():   # a group member's two other neighbours are members of its own group
        assert (rows_t[g][..., 1:, None] == g[:, None, None, :]).any(-1).all(), k
    if D == 128:
        _same(batch_tensor, b.score_batch(patches, fm, 64), "tensor-core re-weighting vs table lookup")
    # per-rank ranges of build_knn_sharded, boundaries off the 128- and 8192-row grids
    b.finalize()
    cuts = [0, 61_111, 130_333, R]
    for a, e in zip(cuts[:-1], cuts[1:]):
        b.build_knn_rows(a, e - a)
    assert (_table(b, R)[2] == keys).all()
    b.close()
