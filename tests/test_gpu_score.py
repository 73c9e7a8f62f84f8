"""GPU parity tests (through the C ABI): fused distance GEMM + min/argmin, s*/m*/top-3 re-weighting, upsample + blur,
and the method-class mirror end to end against the reference's golden outputs."""
import numpy as np
import pytest
import torch

from tests import cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(built):
    from cmdiad_b200 import Bank, upsample_blur
    from cmdiad_b200 import _lib as L
    from oracle import restate as O
    assert torch.cuda.is_available()
    return dict(Bank=Bank, L=L, O=O, upsample_blur=upsample_blur)


def _bank(env, lib, impl=None):
    b = env["Bank"](lib.shape[1], lib.shape[0])
    b.append(lib)
    b.finalize()
    if impl is not None:
        b.set_score_impl(impl)
    return b


# Post-blur tolerance against the reference's final map, in 8-bit quantisation steps of the map (max / 255).  Our
# min_val is the exact direct-form float32 distance, the reference's is the mm-form of torch.cdist (|a|^2 + |b|^2 - 2ab,
# relative error ~1e-6 from cancellation): pixels whose pre-blur value sits within that noise of an 8-bit boundary land
# one level apart, and the integer blur spreads such a pixel over its neighbourhood with per-pass rounding.  Measured on
# the golden cases and at the 200k headline size (bench.py parity block): at most 2.4 steps, on at most 0.002 % of the
# pixels of an image (most images: bit-identical maps up to the last ulp of max / 255).
MAP_MAX_LSB = 2.5
MAP_FRAC_OVER_HALF_LSB = 0.0005


def _check_map(env, r, ref_map):
    """The blur quantises to 8 bits, so ulp-level differences of the pre-blur map move whole contour lines by one
    level.  Exactness is asserted where it is attainable (integer blur given the same 8-bit image: blur(my pre-blur
    map) must equal my output bit for bit); against the reference's final map the bound is in quantisation steps."""
    mine, _ = env["O"].knn_blur_restated(r.s_map_pre)
    assert (mine == r.s_map).all()
    lsb = ref_map.max() / 255.0
    diff = np.abs(r.s_map - ref_map)
    print(f"post-blur map vs reference: max {diff.max() / lsb:.3f} LSB, pixels > 0.5 LSB: {(diff > 0.5 * lsb).mean():.5%}, "
          f">= 1.5 LSB: {(diff >= 1.5 * lsb).mean():.5%}")
    assert diff.max() <= MAP_MAX_LSB * lsb and (diff > 0.5 * lsb).mean() <= MAP_FRAC_OVER_HALF_LSB


def _check_against_oracle(env, r, ref, P):
    ok, nbad = cases.tie_aware_idx_ok(r.min_idx, ref["min_idx"], ref["dist"].numpy())
    assert ok and nbad <= max(1, P // 500), f"{nbad} argmin mismatches"
    np.testing.assert_allclose(r.min_val, ref["min_val"], rtol=1e-4)  # north_star tolerance
    assert int(r.s_idx[0]) == ref["s_idx"]
    np.testing.assert_allclose(r.s_star[0], ref["s_star"], rtol=1e-4)
    assert set(r.nn_idx[1:].tolist()) == set(ref["nn_idx"][1:].tolist())
    np.testing.assert_allclose(np.sort(r.m_star_knn), np.sort(ref["m_star_knn"]), rtol=1e-4)
    np.testing.assert_allclose(r.s[0], ref["s"], rtol=1e-4)
    np.testing.assert_allclose(r.s_map_pre, ref["s_map_pre"], rtol=1e-4)
    _check_map(env, r, ref["s_map"])


def _diagnose(b, patch, bank_rows, r, ref, what):
    """printed when a parity assertion fails: which queries, against the exact device scan, a float64 brute force and a
    second scoring call of the same patch"""
    P = patch.shape[0]
    ex_val, ex_idx = np.empty(P, np.float32), np.empty(P, np.int64)
    q = np.ascontiguousarray(patch)
    b._lib.cmdb_debug_exact_min(b._h, q.ctypes.data, P, ex_val.ctypes.data, ex_idx.ctypes.data)
    d64 = np.sqrt(((patch.astype(np.float64)[:, None, :] - bank_rows.astype(np.float64)[None]) ** 2).sum(-1))
    tv, ti = d64.min(1), d64.argmin(1)
    again = b.score(patch, (int(np.sqrt(P)),) * 2, 224, full=True)
    w = np.nonzero(np.abs(r.min_val - tv) > 2e-5 * tv)[0]
    print(f"DIAG {what}: stats {b.score_stats()}; {len(w)} queries off the float64 brute force: {w.tolist()}")
    print(f"DIAG bank rows on the device equal the host rows: {np.array_equal(b.read().numpy(), bank_rows)}")
    for i in w[:40]:
        print(f"DIAG   q {i}: ours {r.min_val[i]!r} row {r.min_idx[i]} | second call {again.min_val[i]!r} row {again.min_idx[i]} | "
              f"exact scan {ex_val[i]!r} row {ex_idx[i]} | torch {ref['min_val'][i]!r} row {ref['min_idx'][i]} | f64 {tv[i]!r} row {ti[i]}")


@pytest.mark.parametrize("impl", ["tcgen05", "simt"])
def test_score_golden_rgb_case(env, golden, impl):
    """the reference's own outputs (frozen in tests/golden/rgb_case.npz) for 2 test images against a 784-row coreset"""
    O, L = env["O"], env["L"]
    g = golden["rgb_case"]
    lib = cases.rgb_normalised_lib(golden)
    bank_rows = lib[g["coreset_idx_TF32"]]
    b = _bank(env, bank_rows, L.SCORE_TCGEN05 if impl == "tcgen05" else L.SCORE_SIMT)
    for t in range(cases.RGB_CASE["n_test"]):
        patch = ((torch.from_numpy(cases.rgb_test_patch(t)) - torch.tensor(g["rgb_mean"])) / torch.tensor(g["rgb_std"])).numpy()
        r = b.score(patch, (28, 28), 224, full=True)
        ref = O.score_restated(patch, bank_rows, (28, 28), 224)
        try:
            _check_against_oracle(env, r, ref, 784)
        except AssertionError:
            _diagnose(b, patch, bank_rows, r, ref, f"golden rgb image {t} ({impl})")
            raise
        assert (r.min_idx == g[f"t{t}_min_idx"]).mean() >= 0.998
        np.testing.assert_allclose(r.min_val, g[f"t{t}_min_val"], rtol=1e-4)
        np.testing.assert_allclose(r.s[0], g[f"t{t}_s"], rtol=1e-4)
        _check_map(env, r, g[f"t{t}_s_map"][0])
    b.close()


@pytest.mark.parametrize("R,P,fm,D", [(1000, 784, 28, 768), (257, 3136, 56, 768), (5000, 3136, 56, 1152),
                                      (2048, 784, 28, 1920), (3, 784, 28, 768), (70000, 784, 28, 768),
                                      (513, 100, 10, 64)])
def test_score_shapes_vs_oracle(env, R, P, fm, D):
    """ragged bank sizes (not multiples of the 256-row tile), P > 1024 (several GEMM launches), all BASELINE dims"""
    from cmdiad_b200 import synth
    O = env["O"]
    cent = synth.centroids(D, 256)
    lib = synth.patches(R, D, seed=R + P, cent=cent)
    patch = synth.patches(P, D, seed=R + P + 1, anomalous_frac=0.01, cent=cent)
    b = _bank(env, lib)
    r = b.score(patch, (fm, fm), 224, full=True)
    ref = O.score_restated(patch, lib, (fm, fm), 224)
    _check_against_oracle(env, r, ref, P)
    b.close()


def test_score_tcgen05_equals_simt(env):
    """the certified tensor-core path and the exact CUDA-core scan must give identical outputs bit for bit"""
    from cmdiad_b200 import synth
    L = env["L"]
    lib = synth.patches(30000, 768, seed=5, dist="G")
    patch = synth.patches(784, 768, seed=6, dist="G")
    b = _bank(env, lib)
    r1 = b.score(patch, (28, 28), 224, full=True)
    b.set_score_impl(L.SCORE_SIMT)
    r2 = b.score(patch, (28, 28), 224, full=True)
    assert (r1.min_idx == r2.min_idx).all() and (r1.min_val == r2.min_val).all()
    assert r1.s[0] == r2.s[0] and (r1.s_map == r2.s_map).all()
    b.close()


@pytest.mark.parametrize("B,P,fm,D", [(5, 784, 28, 768), (3, 3136, 56, 768), (40, 100, 10, 128), (18, 784, 28, 1920)])
def test_score_batch_equals_single_calls(env, B, P, fm, D):
    """cmdb_score_batch (one GEMM sweep + one re-weighting sweep for B images, internal sub-batches) must give exactly
    the per-image results of B separate cmdb_score calls"""
    from cmdiad_b200 import synth
    cent = synth.centroids(D, 128)
    lib = synth.patches(3000, D, seed=21, cent=cent)
    patches = np.stack([synth.patches(P, D, seed=300 + i, anomalous_frac=0.01, cent=cent) for i in range(B)])
    b = _bank(env, lib)
    batch = b.score_batch(patches, (fm, fm), 224, full=True)
    assert len(batch) == B
    for i in (0, 1, B // 2, B - 1):
        one = b.score(patches[i], (fm, fm), 224, full=True)
        for name in ("s", "s_star", "s_idx", "min_val", "min_idx", "nn_idx", "m_star_knn", "w", "s_map", "s_map_pre", "s_map_u8"):
            assert (getattr(batch[i], name) == getattr(one, name)).all(), (i, name)
    # device-resident input gives the same result
    dev = b.score_batch(torch.from_numpy(patches).cuda(), (fm, fm), 224)
    assert all((dev[i].s_map == batch[i].s_map).all() and dev[i].s[0] == batch[i].s[0] for i in range(B))
    b.close()


@pytest.mark.parametrize("R,D,dist", [(3000, 768, "G"), (20000, 768, "C"), (700, 128, "G")])
def test_bank_knn_table(env, R, D, dist):
    """cmdb_bank_build_knn (SURVEY 8f-1): the table of every bank row's three nearest rows must equal a brute force, and
    scoring with the table (re-weighting = lookup) must reproduce scoring without it bit for bit."""
    import ctypes
    from cmdiad_b200 import synth
    cent = synth.centroids(D, 128) if dist == "C" else None
    lib = synth.patches(R, D, seed=81, dist=dist, cent=cent)
    P, fm = (784, 28) if D == 768 else (100, 10)
    patches = np.stack([synth.patches(P, D, seed=600 + i, dist=dist, anomalous_frac=0.01, cent=cent) for i in range(6)])
    b = _bank(env, lib)
    before_batch = b.score_batch(patches, (fm, fm), 224, full=True)
    before_single = b.score(patches[0], (fm, fm), 224, full=True)
    b.build_knn()
    n_chk = min(R, 1500)
    keys = np.zeros((n_chk, 3), np.uint64)
    assert b._lib.cmdb_debug_read_knn(b._h, keys.ctypes.data_as(ctypes.c_void_p), ctypes.c_longlong(0), ctypes.c_longlong(n_chk)) == 0
    rows = (keys & np.uint64(0xffffffff)).astype(np.int64)
    d2 = (keys >> np.uint64(32)).astype(np.uint32).view(np.float32)
    t = torch.from_numpy(lib).double()
    ref_d2 = torch.cdist(t[:n_chk], t, compute_mode="donot_use_mm_for_euclid_dist") ** 2
    ref_v, ref_i = torch.topk(ref_d2, 3, dim=1, largest=False)
    assert (rows[:, 0] == np.arange(n_chk)).all() and (d2[:, 0] == 0).all()       # a row is its own nearest neighbour
    np.testing.assert_allclose(d2, ref_v.numpy(), rtol=1e-5, atol=1e-6)
    agree = (np.sort(rows, 1) == np.sort(ref_i.numpy(), 1)).all(1)
    gap_ok = (ref_d2.gather(1, ref_i)[:, 2] * (1 + 1e-5) >= torch.sort(ref_d2, 1).values[:, 3]).numpy()  # 3rd/4th near-tie
    assert (agree | gap_ok).all(), int((~(agree | gap_ok)).sum())
    _assert_same_results(before_batch, b.score_batch(patches, (fm, fm), 224, full=True), "table vs tensor-core re-weighting")
    after_single = b.score(patches[0], (fm, fm), 224, full=True)
    for name in _RESULT_FIELDS:
        assert (getattr(before_single, name) == getattr(after_single, name)).all(), name
    b.finalize()          # a new finalize drops the table
    _assert_same_results(before_batch, b.score_batch(patches, (fm, fm), 224, full=True), "after re-finalize")
    b.close()


def test_async_submit_wait_pipeline(env):
    """cmdb_score_batch_submit / _wait: three batches outstanding (three result blocks, two compute lanes); results equal
    the synchronous call, in submission order and out of order, host and device inputs, pipeline depth 2 and 3; a fourth
    submit is refused."""
    from cmdiad_b200 import synth
    cent = synth.centroids(768, 128)
    lib = synth.patches(20000, 768, seed=71, cent=cent)
    b = _bank(env, lib)
    batches = [np.stack([synth.patches(784, 768, seed=500 + 10 * k + i, anomalous_frac=0.01, cent=cent) for i in range(6)])
               for k in range(7)]
    ref = [b.score_batch(x, (28, 28), 224, full=True) for x in batches]
    for dev in (False, True):
        xs = [torch.from_numpy(x).cuda() if dev else torch.from_numpy(x).pin_memory() for x in batches]
        for depth in (2, 3):
            got, pending = [], []
            for x in xs:
                pending.append(b.score_batch_async(x, (28, 28), 224, full=True))
                if len(pending) == depth:
                    got.append(pending.pop(0).wait())
            while pending:
                got.append(pending.pop(0).wait())
            for k in range(len(batches)):
                _assert_same_results(ref[k], got[k], f"async batch {k} dev={dev} depth={depth}")
    t0 = b.score_batch_async(batches[0], (28, 28), 224)
    t1 = b.score_batch_async(batches[1], (28, 28), 224)
    t2 = b.score_batch_async(batches[2], (28, 28), 224)
    with pytest.raises(RuntimeError):
        b.score_batch_async(batches[3], (28, 28), 224)
    with pytest.raises(RuntimeError):
        b.score_batch(batches[3], (28, 28), 224)
    r1, r2, r0 = t1.wait(), t2.wait(), t0.wait()   # out of order
    for name in ("min_idx", "min_val", "s", "nn_idx", "s_map"):
        assert all((getattr(r0[i], name) == getattr(ref[0][i], name)).all() for i in range(6))
        assert all((getattr(r1[i], name) == getattr(ref[1][i], name)).all() for i in range(6))
        assert all((getattr(r2[i], name) == getattr(ref[2][i], name)).all() for i in range(6))
    assert all((a.s_map == c.s_map).all() for a, c in zip(b.score_batch(batches[3], (28, 28), 224), ref[3]))
    b.close()


_RESULT_FIELDS = ("min_idx", "min_val", "s", "s_star", "s_idx", "nn_idx", "m_star_knn", "w", "s_map")


def _assert_same_results(a, b, tag):
    for i in range(len(a)):
        for name in _RESULT_FIELDS:
            assert (getattr(a[i], name) == getattr(b[i], name)).all(), (tag, i, name)


@pytest.mark.parametrize("dist,R,D,P,fm", [("C", 60000, 768, 784, 28), ("G", 30000, 768, 784, 28),
                                            ("C", 20000, 1920, 784, 28), ("C", 9000, 128, 100, 10),
                                            ("C", 40000, 768, 3136, 56)])
def test_gemm_modes_give_identical_results(env, dist, R, D, P, fm):
    """The default certified pre-filter (hi.hi GEMM + error-bound certificate + 3-term fallback), the FP32-equivalent
    3-term GEMM, the uncertified pre-filter and the exact CUDA-core scan must agree bit for bit."""
    from cmdiad_b200 import synth
    L = env["L"]
    cent = synth.centroids(D, 256) if dist == "C" else None
    lib = synth.patches(R, D, seed=33, dist=dist, cent=cent)
    n_img = 5   # >= 4 images: the re-weighting runs on the tensor cores in mode 0 and on CUDA cores in the other modes
    patches = np.stack([synth.patches(P, D, seed=400 + i, dist=dist, anomalous_frac=0.01, cent=cent) for i in range(n_img)])
    b = _bank(env, lib)
    cert = b.score_batch(patches, (fm, fm), 224, full=True)
    st = b.score_stats()
    assert st["mode"] == 0 and st["queries"] == n_img * P
    print("certified pre-filter:", st)
    assert st["fallback_queries"] <= 0.25 * st["queries"] and not st["gemm_fallback"], st   # certificate + rescan carry the load
    b.set_prefilter_terms(3)
    full = b.score_batch(patches, (fm, fm), 224, full=True)
    assert b.score_stats()["mode"] == 3
    _assert_same_results(cert, full, "certified vs 3-term")
    b.set_prefilter_terms(1)
    _assert_same_results(cert, b.score_batch(patches, (fm, fm), 224, full=True), "certified vs uncertified 1-term")
    b.set_score_impl(L.SCORE_SIMT)
    _assert_same_results(cert, b.score_batch(patches, (fm, fm), 224, full=True), "certified vs exact scan")
    b.close()


@pytest.mark.parametrize("R", [3, 5, 255, 256, 257, 700])
def test_tiny_banks_all_paths_agree(env, R):
    """Edge shapes: banks smaller than one GEMM tile / than the number of producers, D = 64, 7x7 feature maps, batches
    (tensor-core re-weighting) and single images (CUDA-core sweep): certified mode == exact scan == oracle restatement."""
    from cmdiad_b200 import synth
    L, O = env["L"], env["O"]
    D, P, fm = 64, 49, 7
    lib = synth.patches(R, D, seed=900 + R, dist="G")
    patches = np.stack([synth.patches(P, D, seed=950 + i, dist="G") for i in range(3)])
    b = _bank(env, lib)
    cert = b.score_batch(patches, (fm, fm), 64, full=True)
    assert b.score_stats()["mode"] == 0
    singles = [b.score(patches[i], (fm, fm), 64, full=True) for i in range(3)]
    _assert_same_results(cert, singles, "batch vs single")
    b.set_score_impl(L.SCORE_SIMT)
    _assert_same_results(cert, b.score_batch(patches, (fm, fm), 64, full=True), "certified vs exact scan")
    for i in range(3):
        ref = O.score_restated(patches[i], lib, (fm, fm), 64)
        ok, nbad = cases.tie_aware_idx_ok(cert[i].min_idx, ref["min_idx"], ref["dist"].numpy())
        assert ok and nbad <= 1
        np.testing.assert_allclose(cert[i].min_val, ref["min_val"], rtol=1e-4)
        assert set(cert[i].nn_idx.tolist()) == set(ref["nn_idx"].tolist())
        np.testing.assert_allclose(cert[i].s[0], ref["s"], rtol=1e-4)
    b.close()


def _exact_scan(b, patch):
    P = patch.shape[0]
    ex_val, ex_idx = np.empty(P, np.float32), np.empty(P, np.int64)
    q = np.ascontiguousarray(patch, np.float32)
    assert b._lib.cmdb_debug_exact_min(b._h, q.ctypes.data, P, ex_val.ctypes.data, ex_idx.ctypes.data) == 0
    return ex_val, ex_idx


@pytest.mark.parametrize("B,fm", [(3, 28), (32, 128)])
def test_exact_scan_mode_on_a_row_offset_handle(env, B, fm):
    """The CUDA-core mode on a handle holding global rows [k, k + R): min_idx are global rows, equal to the exact scan of
    the same rows at offset 0 plus k; every row is stored twice and the lower copy wins.  32 images of 128 x 128 patches
    are 524 288 query rows, more than 65 535 groups of 8."""
    L = env["L"]
    D, R, k = 64, 1000, 123_457
    g = np.random.Generator(np.random.PCG64(B))
    half = g.standard_normal((R // 2, D), dtype=np.float32)
    patches = half[g.integers(0, R // 2, (B, fm * fm))] + 0.3 * g.standard_normal((B, fm * fm, D), dtype=np.float32)
    b = env["Bank"](D, R, row_offset=k)
    b.append(np.concatenate([half, half]))
    b.finalize()
    b.set_score_impl(L.SCORE_SIMT)
    res = b.score_batch(patches, (fm, fm), 64)
    b.set_row_offset(0)
    ex_val, ex_idx = _exact_scan(b, patches.reshape(-1, D))
    assert (ex_idx < R // 2).all()
    assert (np.concatenate([r.min_idx for r in res]) == ex_idx + k).all()
    assert (np.concatenate([r.min_val for r in res]) == ex_val).all()
    assert all(r.s_star[0] == r.min_val.max() and r.s_idx[0] == int(np.argmax(r.min_val)) for r in res)
    b.close()


def test_certificate_fallback_on_near_duplicates(env):
    """Groups of near-duplicate bank rows defeat an 11-bit pre-filter: the certificate must notice (fallback > 0).  While the
    unresolved (query, producer) pairs fit the work list they are rescanned exactly and the answers equal the exact scan of
    the whole bank; a bank with hundreds of indistinguishable rows per query overflows it, goes through the 3-term GEMM
    tier and then switches itself to the direct mode."""
    from cmdiad_b200 import synth
    g = np.random.Generator(np.random.PCG64(5))
    unique = synth.patches(8000, 768, seed=49, dist="G")
    base = synth.patches(200, 768, seed=50, dist="G")
    dup = np.concatenate([base + 2e-4 * g.standard_normal(base.shape, dtype=np.float32) for _ in range(40)], 0)
    lib = np.concatenate([unique, dup], 0)
    lib = lib[g.permutation(lib.shape[0])]
    near_dup = np.stack([base[g.integers(0, 200, 784)] + 0.05 * synth.patches(784, 768, seed=60 + i, dist="G") for i in range(2)])
    near_unique = unique[:784] + 0.05 * synth.patches(784, 768, seed=70, dist="G")
    b = _bank(env, lib)
    # mixed batch: image 0 keeps its certificate, image 1 needs the exact rescan tier
    mixed = np.stack([near_unique, near_dup[0], near_unique[::-1].copy()])
    r_mixed = b.score_batch(mixed, (28, 28), 224, full=True)
    st = b.score_stats()
    assert st["mode"] == 0 and 700 <= st["fallback_queries"] <= 784 + 80 and not st["gemm_fallback"], st
    assert st["direct_calls_left"] == 0
    for i in range(3):
        ex_val, ex_idx = _exact_scan(b, mixed[i])
        assert (r_mixed[i].min_idx == ex_idx).all() and (r_mixed[i].min_val == ex_val).all(), i
    b.close()
    # 400 indistinguishable rows per query: far more pairs than the work list holds -> 3-term GEMM tier, then direct mode
    dup = np.concatenate([base + 2e-4 * g.standard_normal(base.shape, dtype=np.float32) for _ in range(400)], 0)
    lib = np.concatenate([unique, dup], 0)
    lib = lib[g.permutation(lib.shape[0])]
    b = _bank(env, lib)
    cert = b.score_batch(near_dup, (28, 28), 224, full=True)
    st = b.score_stats()
    assert st["mode"] == 0 and st["fallback_queries"] > 0.5 * st["queries"] and st["gemm_fallback"], st
    again = b.score_batch(near_dup, (28, 28), 224, full=True)
    st2 = b.score_stats()
    assert st2["mode"] == 3 and st2["direct_calls_left"] == 31, st2
    b.set_prefilter_terms(3)
    full = b.score_batch(near_dup, (28, 28), 224, full=True)
    _assert_same_results(cert, full, "certified(fallback) vs 3-term")
    _assert_same_results(again, full, "adaptive direct vs 3-term")
    ex_val, _ = _exact_scan(b, near_dup[0])
    # 400 rows within 1e-4 of each other: below the resolution of ANY |a|^2 + |b|^2 - 2ab evaluation in float32 (the
    # reference's mm-form included), so this tier returns one of them, not necessarily the exact minimum
    np.testing.assert_allclose(cert[0].min_val, ex_val, rtol=1e-3)
    b.close()


def test_rescan_tier_under_load(env):
    """Groups of 12 near-duplicates: a fifth of the queries has two band rows in one producer, few enough for the exact
    rescan tier (no GEMM fallback).  Results must equal the exact CUDA-core scan."""
    from cmdiad_b200 import synth
    L = env["L"]
    g = np.random.Generator(np.random.PCG64(9))
    base = synth.patches(1500, 768, seed=52, dist="G")
    lib = np.concatenate([base + 2e-4 * g.standard_normal(base.shape, dtype=np.float32) for _ in range(12)], 0)
    lib = lib[g.permutation(lib.shape[0])]
    patches = np.stack([base[g.integers(0, 1500, 784)] + 0.05 * synth.patches(784, 768, seed=65 + i, dist="G") for i in range(3)])
    b = _bank(env, lib)
    cert = b.score_batch(patches, (28, 28), 224, full=True)
    st = b.score_stats()
    print("rescan tier:", st)
    assert st["mode"] == 0 and st["rescan_pairs"] >= 100 and not st["gemm_fallback"], st
    b.set_score_impl(L.SCORE_SIMT)
    exact = b.score_batch(patches, (28, 28), 224, full=True)
    for i in range(3):   # min_val / min_idx are certified identical; the re-weighting keys too
        for name in ("min_idx", "min_val", "s", "s_idx", "nn_idx", "s_map"):
            assert (getattr(cert[i], name) == getattr(exact[i], name)).all(), (i, name)
    b.close()


def _measure_error_model(env, lib, patch, fm):
    """(accumulation error / model, total error / certificate bound) of the pre-filter GEMM's epilogue values, measured
    against a float64 evaluation of the same fp16 operands; also returns the bank for further checks"""
    import ctypes
    R, D = lib.shape
    P = patch.shape[0]
    b = _bank(env, lib)
    b.set_prefilter_terms(1)
    b.score(patch, (fm, fm), 224)
    n_cta = 296   # producers = (CTA, accumulator column half)
    cand = np.zeros((n_cta, P, 4), np.float32)
    rc = b._lib.cmdb_debug_read_candidates(b._h, cand.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n_cta), ctypes.c_int(P))
    assert rc == 0
    val = cand[:, :, 0]
    idx = cand[:, :, 1].copy().view(np.int32)
    ok = idx >= 0
    assert ok.any()
    # the fp16 operands exactly as the library builds them (power-of-two scales, round to nearest even)
    with np.errstate(over="ignore", under="ignore"):
        eb = 13 - int(np.frexp(np.abs(lib).max())[1])
        bh = (lib * np.float32(2.0 ** eb)).astype(np.float16).astype(np.float64) * 2.0 ** -eb
        eq = 13 - np.frexp(np.abs(patch).max(1))[1].astype(np.int64)
        qh = (patch * (2.0 ** eq)[:, None].astype(np.float32)).astype(np.float16).astype(np.float64) * (2.0 ** -eq)[:, None]
    bn = (lib.astype(np.float64) ** 2).sum(1).astype(np.float32).astype(np.float64)
    qhn, bhn = np.linalg.norm(qh, axis=1), np.linalg.norm(bh, axis=1)
    worst_acc, worst_total = 0.0, 0.0
    acc_model = (D // 16 + 1) * 17 * 2.0 ** -23
    qn = np.linalg.norm(patch.astype(np.float64), axis=1)
    qe = np.linalg.norm(patch.astype(np.float64) - qh, axis=1)
    bmax, ebmax = np.linalg.norm(lib.astype(np.float64), axis=1).max(), np.linalg.norm(lib.astype(np.float64) - bh, axis=1).max()
    for c in range(0, n_cta, 7):
        qs = np.nonzero(ok[c])[0]
        if qs.size == 0:
            continue
        rows = idx[c, qs]
        dot = np.einsum("ij,ij->i", qh[qs], bh[rows])
        v64 = bn[rows] - 2.0 * dot
        err = np.abs(val[c, qs].astype(np.float64) - v64)
        # accumulation error alone (the final fma rounds once more: 2^-24 |v|)
        worst_acc = max(worst_acc, float(((err - 2.0 ** -24 * np.abs(v64)) / (2 * acc_model * qhn[qs] * bhn[rows])).max()))
        exact = ((patch[qs].astype(np.float64) - lib[rows].astype(np.float64)) ** 2).sum(1)
        E = 2 * (qe[qs] * (bmax + ebmax) + qn[qs] * ebmax + acc_model * (qn[qs] + qe[qs]) * (bmax + ebmax)) \
            + (D + 16) * 2.0 ** -24 * (qn[qs] + bmax) ** 2
        worst_total = max(worst_total, float((np.abs(val[c, qs] + qn[qs] ** 2 - exact) / E).max()))
    return worst_acc, worst_total, b


def test_prefilter_error_model(env):
    """The certificate rests on (a) Cauchy-Schwarz bounds of the fp16 operand rounding -- mathematics -- and (b) a model
    of the tensor-core accumulation error, (D/16 + 1) * 17 * 2^-23 * ||q_hi|| ||b_hi||.  (b) is measured here: the GEMM
    epilogue's values are compared with a float64 evaluation of the same fp16 operands."""
    from cmdiad_b200 import synth
    D, R, P = 768, 20000, 784
    lib = synth.patches(R, D, seed=91)
    patch = synth.patches(P, D, seed=92, anomalous_frac=0.02)
    worst_acc, worst_total, b = _measure_error_model(env, lib, patch, 28)
    print(f"accumulation error / model = {worst_acc:.4f}, total error / certificate bound = {worst_total:.4f}")
    assert worst_acc < 0.25, worst_acc      # the model keeps >= 4x margin over what the hardware does
    assert worst_total < 0.5, worst_total
    b.close()


def _adversarial(kind, R, P, D, seed, range_bits=14, dup=8):
    """inputs built to stress the certificate (VERDICT r1 weak 5): the accumulation model is empirical, so it is probed
    where alignment / truncation inside the tensor core hurts most"""
    g = np.random.Generator(np.random.PCG64(seed))
    if kind == "wide_range":      # 2^-14 .. 1 inside every row: small addends are aligned against large partial sums
        lib = g.standard_normal((R, D), dtype=np.float32) * np.exp2(-range_bits * g.random((R, D), dtype=np.float32))
        patch = g.standard_normal((P, D), dtype=np.float32) * np.exp2(-range_bits * g.random((P, D), dtype=np.float32))
    elif kind == "subnormal_residue":  # one spike per row: everything else lands in fp16's subnormal range after scaling
        lib = g.standard_normal((R, D), dtype=np.float32) * np.float32(3e-8)
        patch = g.standard_normal((P, D), dtype=np.float32) * np.float32(3e-8)
        lib[np.arange(R), g.integers(0, D, R)] = g.choice([-1.0, 1.0], R).astype(np.float32)
        patch[np.arange(P), g.integers(0, D, P)] = g.choice([-1.0, 1.0], P).astype(np.float32)
    elif kind == "cancelling":    # products alternate in sign and cancel: a.b ~ 0 with |a||b| large
        half = D // 2
        x = g.standard_normal((P, half), dtype=np.float32) + 3
        y = g.standard_normal((R, half), dtype=np.float32) + 3
        patch = np.concatenate([x, -x], 1)[:, g.permutation(D)]
        lib = np.concatenate([y, y * (1 + 1e-3 * g.standard_normal((R, half), dtype=np.float32))], 1)[:, g.permutation(D)]
        patch = np.ascontiguousarray(patch, dtype=np.float32)
        lib = np.ascontiguousarray(lib, dtype=np.float32)
    elif kind == "near_duplicates":   # many rows within float32 noise of each other: the band never empties
        base = g.standard_normal((R // dup, D), dtype=np.float32)
        lib = np.repeat(base, dup, 0) * (1 + 1e-6 * g.standard_normal((R // dup * dup, 1), dtype=np.float32))
        patch = base[g.integers(0, R // dup, P)] + 1e-3 * g.standard_normal((P, D), dtype=np.float32)
    else:
        raise ValueError(kind)
    return np.ascontiguousarray(lib, np.float32), np.ascontiguousarray(patch, np.float32)


@pytest.mark.parametrize("D", [768, 1920])
@pytest.mark.parametrize("kind", ["wide_range", "subnormal_residue", "cancelling", "near_duplicates"])
def test_certificate_under_adversarial_inputs(env, kind, D):
    """mode 0 (certified pre-filter, tensor cores) must equal the exact CUDA-core scan bit for bit on inputs chosen to
    break an optimistic accumulation model, and the measured error must stay below half of the certificate's bound"""
    L = env["L"]
    R, P, fm = 6000, 256, 16
    lib, patch = _adversarial(kind, R, P, D, seed=sum(map(ord, kind)) + D)
    worst_acc, worst_total, b = _measure_error_model(env, lib, patch, fm)
    print(f"{kind} D={D}: accumulation error / model = {worst_acc:.4f}, total error / certificate bound = {worst_total:.4f}")
    assert worst_acc < 0.5 and worst_total < 0.5, (worst_acc, worst_total)
    b.set_prefilter_terms(0)
    cert = b.score(patch, (fm, fm), 224)
    stats = b.score_stats()
    # the exact scan the certificate promises equality with: every (query, row) distance by the re-check arithmetic
    # (warp_sqdist), lowest row on ties
    ex_val, ex_idx = _exact_scan(b, patch)
    bad = np.nonzero((cert.min_idx != ex_idx) | (cert.min_val != ex_val))[0]
    assert bad.size == 0, (kind, D, stats, bad[:5], cert.min_idx[bad[:5]], ex_idx[bad[:5]], cert.min_val[bad[:5]], ex_val[bad[:5]])
    # mode 3 (FP32-equivalent split, exact re-check of the 4 best candidates) carries no certificate: with more than 4 rows
    # inside float32 noise of the minimum it may return another of the tied rows -- values still agree to rounding
    b.set_prefilter_terms(3)
    full3 = b.score(patch, (fm, fm), 224)
    n3 = int(((full3.min_idx != ex_idx) | (full3.min_val != ex_val)).sum())
    print(f"{kind} D={D}: mode 0 == exact scan on all {P} queries ({stats['fallback_queries']} uncertified, {stats['rescan_pairs']} "
          f"rescanned pairs, gemm fallback {stats['gemm_fallback']}); mode 3 differs on {n3}")
    if kind in ("wide_range", "cancelling"):   # no engineered near-ties: mode 3 must agree as well
        assert n3 == 0
    b.close()


def test_certificate_hypothesis_sweep(env):
    """VERDICT r1 item 9: a property sweep over the adversarial families -- bank size (ragged against the 256-row tile),
    dimension, query count, dynamic range inside the rows, duplication factor (up to 40-fold: far more in-band rows than the
    certificate kernel's 24-row query lists, so the surplus goes through the rescan queue) and seed are drawn by hypothesis
    (derandomised: the same examples in every run).  Property: the default mode equals the exact scan of the whole bank,
    value and row, on every query."""
    from hypothesis import given, settings, HealthCheck, strategies as st

    @settings(max_examples=40, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(kind=st.sampled_from(["wide_range", "subnormal_residue", "cancelling", "near_duplicates"]),
           D=st.sampled_from([256, 768, 1152, 1920]), n=st.integers(8, 220), side=st.sampled_from([8, 10, 16]),
           range_bits=st.integers(2, 20), dup=st.sampled_from([2, 8, 40]), seed=st.integers(0, 10_000))
    def prop(kind, D, n, side, range_bits, dup, seed):
        R, P = n * dup, side * side
        lib, patch = _adversarial(kind, R, P, D, seed, range_bits=range_bits, dup=dup)
        b = _bank(env, lib)
        cert = b.score(patch, (side, side), 64)
        stats = b.score_stats()
        ex_val, ex_idx = _exact_scan(b, patch)
        bad = np.nonzero((cert.min_idx != ex_idx) | (cert.min_val != ex_val))[0]
        b.close()
        assert bad.size == 0, (kind, D, R, P, range_bits, dup, seed, stats, bad[:5], cert.min_idx[bad[:5]], ex_idx[bad[:5]])

    prop()


def test_score_duplicate_rows_lowest_index(env):
    """exact ties in the bank: argmin must be the lowest row (torch.min semantics, features.py:227)"""
    from cmdiad_b200 import synth
    base = synth.patches(700, 768, seed=1, dist="G")
    lib = np.concatenate([base, base], 0)
    patch = base[:784 // 2].repeat(2, 0) + 0.01 * synth.patches(784, 768, seed=2, dist="G")
    b = _bank(env, lib)
    r = b.score(patch, (28, 28), 224)
    assert (r.min_idx < 700).all()
    b.close()


def test_score_large_values_are_rescaled(env):
    """the fp16 split is scaled per bank / per image, so unnormalised magnitudes still work"""
    from cmdiad_b200 import synth
    O = env["O"]
    lib = synth.patches(2000, 768, seed=3) * 3.0e4
    patch = synth.patches(784, 768, seed=4, anomalous_frac=0.01) * 3.0e4
    b = _bank(env, lib)
    r = b.score(patch, (28, 28), 224, full=True)
    ref = O.score_restated(patch, lib, (28, 28), 224)
    assert (r.min_idx == ref["min_idx"]).mean() > 0.995
    np.testing.assert_allclose(r.min_val, ref["min_val"], rtol=1e-4)
    b.close()


def test_upsample_blur_bit_exact(env):
    """bilinear (features.py:294) + KNNGaussianBlur (utils/utils.py:71-83): identical bits given identical input"""
    O = env["O"]
    g = np.random.Generator(np.random.PCG64(12))
    for h in (28, 56):
        m = (np.abs(g.standard_normal((h, h))) * 7 + 3).astype(np.float32)
        out, pre, u8 = env["upsample_blur"](m, 224)
        assert (pre == O.bilinear_restated(m, 224)).all()
        ref, ref_u8 = O.knn_blur_restated(pre)
        assert (u8 == ref_u8).all() and (out == ref).all()
        t = torch.nn.functional.interpolate(torch.from_numpy(m).view(1, 1, h, h), size=(224, 224), mode="bilinear")
        assert (pre == t[0, 0].numpy()).all()
    # non-square maps, output sizes that leave row bands empty or ragged, the maximum in the first / last band: the
    # global max is folded from per-band maxima and has to equal the max of the whole upsampled map bit for bit
    for (fh, fw, hw) in ((7, 13, 8), (28, 28, 100), (14, 56, 250), (3, 3, 256), (56, 56, 17)):
        for peak in ("first", "last", "none"):
            m = (np.abs(g.standard_normal((fh, fw))) * 2 + 1).astype(np.float32)
            if peak == "first":
                m[0, fw // 2] = 40.0
            elif peak == "last":
                m[fh - 1, 0] = 40.0
            out, pre, u8 = env["upsample_blur"](m, hw)
            t = torch.nn.functional.interpolate(torch.from_numpy(m).view(1, 1, fh, fw), size=(hw, hw), mode="bilinear")
            # (bit-exactness of the bilinear weights is pinned for the reference's 28 / 56 -> 224 only)
            np.testing.assert_allclose(pre, t[0, 0].numpy(), rtol=2e-5, atol=1e-5, err_msg=str((fh, fw, hw, peak)))
            ref, ref_u8 = O.knn_blur_restated(pre)
            assert (u8 == ref_u8).all() and (out == ref).all(), (fh, fw, hw, peak)


def test_score_errors(env):
    L = env["L"]
    b = env["Bank"](768, 100)
    b.append(np.ones((100, 768), np.float32))
    with pytest.raises(L.CmdbError) as e:
        b.score(np.ones((784, 768), np.float32), (28, 28))
    assert e.value.status == L.CMDB_ERR_STATE  # not finalized
    b.finalize()
    with pytest.raises(L.CmdbError):
        b.score(np.ones((784, 768), np.float32), (28, 27))  # dims do not match P
    b.close()


def test_double_bank_pipeline_matches_reference_golden(env, golden):
    """DoubleRGBPointFeatures end to end through the mirror classes: cross-wired statistics, two coresets, late-fusion
    head, compute_s_s_map -- against tests/golden/dual_case.npz produced by the unmodified reference"""
    from cmdiad_b200 import DoubleRGBPointFeatures, default_args
    g = golden["dual_case"]
    # torch.mean / torch.std on the host depend on the machine's thread count in the last ulp, so the reference's own
    # scalars (frozen in the golden file) are injected; the device statistics are checked against them separately
    fixed = {"xyz": (g["xyz_mean"], None), "rgb": (None, g["rgb_std"])}
    m = DoubleRGBPointFeatures(default_args(coreset_dtype="TF32", random_state=0), parity_stats=fixed,
                               bank_capacity_rows=3 * 3136)
    xyz_train, rgb_train = cases.dual_train()
    for x, r in zip(xyz_train, rgb_train):
        m.add_sample_to_mem_bank({"xyz": x, "rgb": r}, class_name="synthetic")
    dev_mean = m._banks["xyz"].stats()[0]
    dev_std = m._banks["rgb"].stats()[1]
    assert abs(dev_mean - float(g["xyz_mean"])) <= 1e-5 * abs(float(g["xyz_mean"])) + 1e-8
    assert abs(dev_std - float(g["rgb_std"])) <= 1e-6 * float(g["rgb_std"])
    m.run_coreset()
    for k in ("xyz_mean", "xyz_std", "rgb_mean", "rgb_std"):
        assert np.float32(getattr(m, k)) == g[k], k
    assert m.patch_xyz_lib.shape[0] == int(g["n_xyz"]) and m.patch_rgb_lib.shape[0] == int(g["n_rgb"])
    assert (m.coreset_idx.numpy() == g["coreset_idx_rgb"]).all()
    assert (m.patch_xyz_lib[::53].numpy() == g["xyz_lib_sample"]).all()
    for x, r in zip(xyz_train, rgb_train):
        m.add_sample_to_late_fusion_mem_bank({"xyz": x, "rgb": r})
    np.testing.assert_allclose(torch.cat(m.s_lib, 0).numpy(), g["s_lib"], rtol=1e-4)
    m.run_late_fusion()
    xt, rt = cases.dual_test()
    m.predict({"xyz": xt, "rgb": rt}, torch.zeros(1, 224, 224), 0, ["synthetic/0.png"])
    np.testing.assert_allclose(m.image_preds[0], g["image_pred"], rtol=1e-3)
    np.testing.assert_allclose(m.predictions[0], g["prediction"], rtol=1e-3, atol=1e-3 * np.abs(g["prediction"]).max())
    m.close()


def test_full_size_bank_properties(env):
    """BASELINE size (200k x 768, P = 784): parity through a GPU brute force on the same inputs (the float32 [P,R]
    matrix the reference would build) plus size-independent properties"""
    from cmdiad_b200 import synth
    R, D, P = 200_000, 768, 784
    cent = synth.centroids(D)
    lib = np.concatenate([synth.patches(50_000, D, seed=900 + i, cent=cent) for i in range(4)], 0)
    patch = synth.patches(P, D, seed=950, anomalous_frac=0.01, cent=cent)
    b = _bank(env, lib)
    r = b.score(patch, (28, 28), 224, full=True)
    dist = torch.cdist(torch.from_numpy(patch).cuda(), torch.from_numpy(lib).cuda(), compute_mode="donot_use_mm_for_euclid_dist")
    mv, mi = torch.min(dist, dim=1)
    mv, mi = mv.cpu().numpy(), mi.cpu().numpy()
    bad = np.nonzero(r.min_idx != mi)[0]
    dist_c = dist.cpu().numpy()
    for p in bad:
        assert abs(dist_c[p, r.min_idx[p]] - dist_c[p, mi[p]]) <= 2e-6 * dist_c[p, mi[p]]
    assert len(bad) <= 2
    np.testing.assert_allclose(r.min_val, mv, rtol=1e-5)
    # properties: a bank row scores 0 against itself; s_star is the max of min_val; appending the patch to the bank
    # makes every min distance 0
    assert r.s_star[0] == r.min_val.max() and r.s_idx[0] == int(np.argmax(r.min_val))
    self_r = b.score(lib[1000:1784], (28, 28), 224)
    assert (self_r.min_idx == np.arange(1000, 1784)).all() and (self_r.min_val == 0).all()
    b.close()
