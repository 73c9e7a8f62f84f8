"""CPU suite, part 1: the oracle (oracle/restate.py + coreset_oracle.c) against the golden vectors frozen from the
unmodified reference, and -- when the reference tree is present -- against the reference itself."""
import numpy as np
import pytest
import torch

from oracle import ref_loader as R
from oracle import restate as O
from tests import cases


def test_projection_matches_golden(built, golden):
    g = golden["rgb_case"]
    lib = cases.rgb_normalised_lib(golden)
    csr = O.sparse_components(lib.shape[0], lib.shape[1], 0.9, 0)
    assert csr[3] == int(g["proj_dim"])
    z = O.project_restated(lib[g["proj_rows"]], *csr)
    assert (z == g["proj_sample"]).all()  # bit-exact float64


def test_coreset_fp64_matches_golden(built, golden):
    g = golden["rgb_case"]
    lib = cases.rgb_normalised_lib(golden)
    z = O.project_restated(lib, *O.sparse_components(lib.shape[0], lib.shape[1], 0.9, 0))
    n = int(0.1 * lib.shape[0])
    idx = O.coreset_restated(z, n, "TF32")
    assert idx[0] == 0 and len(set(idx.tolist())) == n
    assert (idx == g["coreset_idx_TF32"]).all()


def test_coreset_fp16_teacher_forced_against_cpu_reference(built, golden):
    """The golden FP16 indices come from the reference run on the build container's CPU, whose half-norm summation
    order differs from the CUDA order the oracle restates (and the reference uses on a GPU).  Free-running they agree
    as sets; teacher-forced, every disagreement must be a near-tie."""
    g = golden["rgb_case"]
    lib = cases.rgb_normalised_lib(golden)
    z = O.project_restated(lib, *O.sparse_components(lib.shape[0], lib.shape[1], 0.9, 0))
    ref = g["coreset_idx_FP16"]
    n = len(ref)
    free = O.coreset_restated(z, n, "FP16")
    assert free[0] == 0
    assert len(set(free.tolist()) & set(ref.tolist())) / n > 0.97
    forced = O.coreset_restated(z, n, "FP16", force_idx=ref)
    assert (forced != ref).mean() < 0.02


def test_coreset_literal_torch_equals_oracle_fp64(built):
    g = np.random.Generator(np.random.PCG64(5))
    z = g.standard_normal((1500, 150))
    lit = O.coreset_torch_literal(torch.from_numpy(z), 100, "TF32").numpy()
    assert (lit == O.coreset_restated(z, 100, "TF32")).all()


@pytest.mark.parametrize("d", [32, 64, 100, 127, 128, 129, 130, 131, 198, 221, 301])
def test_canonical_order_is_a_valid_sum(built, d):
    """the canonical order only re-associates: against float64 exact it is within float32 accumulation error"""
    g = np.random.Generator(np.random.PCG64(d))
    z = g.standard_normal((64, d)).astype(np.float16)
    last = g.standard_normal(d).astype(np.float16)
    got = O.rownorms_restated(z, last).astype(np.float64)
    diff = (z.astype(np.float32) - last.astype(np.float32)).astype(np.float16).astype(np.float64)
    exact = np.sqrt((diff ** 2).sum(1))
    np.testing.assert_allclose(got, exact, rtol=2e-3)  # half rounding of the result dominates
    z64 = g.standard_normal((64, d))
    l64 = g.standard_normal(d)
    np.testing.assert_allclose(O.rownorms_restated(z64, l64), np.sqrt(((z64 - l64) ** 2).sum(1)), rtol=1e-13)


def test_scoring_matches_golden(built, golden):
    g = golden["rgb_case"]
    lib = cases.rgb_normalised_lib(golden)
    bank = lib[g["coreset_idx_TF32"]]
    for t in range(cases.RGB_CASE["n_test"]):
        patch = ((torch.from_numpy(cases.rgb_test_patch(t)) - torch.tensor(g["rgb_mean"])) / torch.tensor(g["rgb_std"])).numpy()
        r = O.score_restated(patch, bank, (28, 28), 224)
        assert (r["min_idx"] == g[f"t{t}_min_idx"]).all()
        assert (r["min_val"] == g[f"t{t}_min_val"]).all()
        assert np.float32(r["s"]) == g[f"t{t}_s"]
        assert (r["s_map"] == g[f"t{t}_s_map"][0]).all()  # bilinear + blur restatement, bit-exact


def test_bilinear_and_blur_against_torch_and_pillow(built):
    from PIL import Image, ImageFilter
    g = np.random.Generator(np.random.PCG64(3))
    for h in (28, 56):
        m = torch.from_numpy((np.abs(g.standard_normal((h, h))) * 10 + 5).astype(np.float32))
        ref = torch.nn.functional.interpolate(m.view(1, 1, h, h), size=(224, 224), mode="bilinear")[0, 0].numpy()
        assert (O.bilinear_restated(m.numpy(), 224) == ref).all()
    for _ in range(3):
        img = g.integers(0, 256, (224, 224), dtype=np.uint8)
        ref = np.asarray(Image.fromarray(img, mode="L").filter(ImageFilter.GaussianBlur(4)))
        assert (O.pil_gaussian_blur_restated(img) == ref).all()
    assert abs(float(O.pil_box_radius(4)) - 3.4375) < 1e-6


def test_projection_against_sklearn(built):
    from sklearn import random_projection
    g = np.random.Generator(np.random.PCG64(9))
    x = g.standard_normal((600, 768), dtype=np.float32)
    z_ref = random_projection.SparseRandomProjection(eps=0.9, random_state=0).fit_transform(torch.from_numpy(x))
    z = O.project_restated(x, *O.sparse_components(600, 768, 0.9, 0))
    assert z_ref.dtype == np.float64 and (np.asarray(z_ref) == z).all()
    with pytest.raises(ValueError):
        O.sparse_components(10 ** 7, 64, 0.9, 0)  # d' > D: sklearn raises, the reference skips the projection


def test_oracle_against_live_reference(built, golden):
    """restatement vs the unmodified reference classes on a fresh seed (not just the inputs of rgb_case): the
    reference's outputs are frozen in tests/golden/fresh_seed_case.npz (oracle/make_golden.py); where the reference
    tree is present it is also run live"""
    from cmdiad_b200 import synth
    frozen = golden["fresh_seed_case"]
    train = synth.image_bank(3, 784, 768, seed=77)
    cat = torch.cat([torch.from_numpy(x) for x in train], 0)
    mean, std = O.bank_stats_restated(cat)
    lib = O.normalize_restated(cat, mean, std).numpy()
    z = O.project_restated(lib, *O.sparse_components(lib.shape[0], 768, 0.9, 0))
    idx = O.coreset_restated(z, int(0.1 * lib.shape[0]), "TF32")
    assert (idx == frozen["coreset_idx"]).all()
    patch = ((torch.from_numpy(synth.patches(784, 768, 5, anomalous_frac=0.01)) - mean) / std)
    r = O.score_restated(patch.numpy(), lib[idx], (28, 28), 224)
    assert np.float32(r["s"]) == frozen["s"] and (r["s_map"] == frozen["s_map"]).all()
    if not R.reference_available():
        return
    m = R.make_method("RGBFeatures", coreset_dtype="TF32", random_state=0)
    for x in train:
        m.patch_rgb_lib.append(torch.from_numpy(x))
    with R.cuda_to_cpu_if_needed():
        m.run_coreset()
    assert (idx == m.coreset_idx.numpy()).all()
    dist = m.calculate_dist(patch, m.patch_rgb_lib)
    s, s_map = m.compute_single_s_s_map(patch, dist, (28, 28), modal="rgb")
    assert np.float32(r["s"]) == np.float32(s) and (r["s_map"] == s_map[0].numpy()).all()


def test_cdist_guard_recovers_from_a_faulty_sgemm(monkeypatch):
    """oracle.restate.cdist_guarded: the GPU boxes' host BLAS returned float32 mm-form distances at ~1e-4 relative accuracy in
    the first sgemm of ~5 % of fresh processes (a float64 brute force and the device agreed with each other to 1e-7).  The
    guard re-evaluates the row minima in float64 and repeats the call; a healthy cdist is returned untouched after one call."""
    import torch
    from cmdiad_b200 import synth
    from oracle import restate as O
    cent = synth.centroids(768, 64)
    a = torch.from_numpy(synth.patches(200, 768, seed=1, cent=cent))
    b = torch.from_numpy(synth.patches(3000, 768, seed=2, cent=cent))
    good = torch.cdist(a, b)
    real, calls = torch.cdist, []

    def flaky(x, y, *args, **kw):
        calls.append(1)
        d = real(x, y, *args, **kw)
        if len(calls) == 1:   # the first call of the "process": every distance off by up to 2e-4 relative
            g = torch.Generator().manual_seed(0)
            d = d * (1 + 2e-4 * (2 * torch.rand(d.shape, generator=g) - 1))
        return d

    monkeypatch.setattr(torch, "cdist", flaky)
    out = O.cdist_guarded(a, b)
    assert len(calls) == 2 and torch.equal(out, good)
    calls.clear()
    calls.append(1)   # healthy from the start: exactly one more call, result untouched
    out = O.cdist_guarded(a, b)
    assert len(calls) == 2 and torch.equal(out, good)
    # degenerate inputs do not loop or fail: a query equal to a bank row (distance 0), and a single bank row
    monkeypatch.setattr(torch, "cdist", real)
    assert float(O.cdist_guarded(b[:1], b).min()) < 0.05
    assert O.cdist_guarded(a, b[:1]).shape == (200, 1)
