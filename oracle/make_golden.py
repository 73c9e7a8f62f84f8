"""TEST INFRASTRUCTURE ONLY -- freezes golden vectors from the UNMODIFIED reference (run in the build container).

    python -m oracle.make_golden                       # writes tests/golden/*.npz
    python -m oracle.make_golden --from-restatement    # only au_pro_case / fresh_seed_case, without the reference

The reference ships no tests, fixtures or golden vectors (SURVEY.md section 4), so parity is pinned on outputs of the
reference's own code (feature_extractors/features.py, multiple_features.py, utils/utils.py) imported through
oracle/ref_loader.py and fed seeded synthetic patches (cmdiad_b200/synth.py).  Inputs are regenerated from seeds in the
tests; only outputs are stored.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cmdiad_b200 import synth  # noqa: E402
from oracle import ref_loader as R  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

RGB_CASE = dict(n_train=10, P=784, D=768, seed=11, n_test=2, fmap=28)
DUAL_CASE = dict(n_train=3, P_xyz=3136, P_rgb=784, D=768, seed=23, fmap_xyz=56, fmap_rgb=28)


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x))


def golden_rgb():
    c = RGB_CASE
    out = {}
    train = synth.image_bank(c["n_train"], c["P"], c["D"], c["seed"])
    for mode in ("FP16", "TF32"):
        torch.manual_seed(0)
        m = R.make_method("RGBFeatures", coreset_dtype=mode, random_state=0)
        for x in train:
            m.patch_rgb_lib.append(_t(x))               # multiple_features.py:35
        with R.cuda_to_cpu_if_needed():
            m.run_coreset()                              # multiple_features.py:37-48
        out[f"coreset_idx_{mode}"] = m.coreset_idx.numpy()
        out["rgb_mean"] = m.rgb_mean.numpy()
        out["rgb_std"] = m.rgb_std.numpy()
    # projection output (float64) sampled on a fixed row stride
    from sklearn import random_projection
    lib = (torch.cat([_t(x) for x in train], 0) - m.rgb_mean) / m.rgb_std
    z = random_projection.SparseRandomProjection(eps=0.9, random_state=0).fit_transform(lib)
    out["proj_rows"] = np.arange(0, lib.shape[0], 97)
    out["proj_sample"] = np.asarray(z)[out["proj_rows"]]
    out["proj_dim"] = np.int64(z.shape[1])
    # scoring: the bank is the TF32-mode (float64) coreset -- the mode whose indices every platform reproduces
    for t in range(c["n_test"]):
        patch = _t(synth.patches(c["P"], c["D"], c["seed"] * 1000 + 500 + t, anomalous_frac=0.01,
                                 cent=synth.centroids(c["D"])))
        patch = (patch - m.rgb_mean) / m.rgb_std        # multiple_features.py:90
        dist = m.calculate_dist(patch, m.patch_rgb_lib)  # :91
        min_val, min_idx = torch.min(dist, dim=1)
        s, s_map = m.compute_single_s_s_map(patch, dist, (c["fmap"], c["fmap"]), modal="rgb")  # :94
        out[f"t{t}_min_val"] = min_val.numpy()
        out[f"t{t}_min_idx"] = min_idx.numpy()
        out[f"t{t}_s"] = np.float32(s)
        out[f"t{t}_s_map"] = s_map.numpy()
    np.savez_compressed(os.path.join(OUT, "rgb_case.npz"), **out)
    print("rgb_case:", {k: getattr(v, "shape", v) for k, v in out.items()})


def golden_dual():
    """DoubleRGBPointFeatures end to end (multiple_features.py:800-1015): cross-wired statistics, two banks, late
    fusion head, compute_s_s_map outputs."""
    c = DUAL_CASE
    out = {}
    torch.manual_seed(0)
    m = R.make_method("DoubleRGBPointFeatures", coreset_dtype="TF32", random_state=0)
    xyz_train = synth.image_bank(c["n_train"], c["P_xyz"], c["D"], c["seed"])
    rgb_train = synth.image_bank(c["n_train"], c["P_rgb"], c["D"], c["seed"] + 1)
    for x, r in zip(xyz_train, rgb_train):
        m.patch_xyz_lib.append(_t(x))                   # multiple_features.py:870-871
        m.patch_rgb_lib.append(_t(r))
    with R.cuda_to_cpu_if_needed():
        m.run_coreset()                                  # :873-895
    for k in ("xyz_mean", "xyz_std", "rgb_mean", "rgb_std"):
        out[k] = getattr(m, k).numpy()
    out["coreset_idx_rgb"] = m.coreset_idx.numpy()       # the attribute is overwritten by the rgb call (:890)
    out["n_xyz"] = np.int64(m.patch_xyz_lib.shape[0])
    out["n_rgb"] = np.int64(m.patch_rgb_lib.shape[0])
    out["xyz_lib_sample"] = m.patch_xyz_lib[::53].numpy()
    # late-fusion pass over the train images (:897-927 minus the backbone call)
    for x, r in zip(xyz_train, rgb_train):
        xp = (_t(x) - m.xyz_mean) / m.xyz_std
        rp = (_t(r) - m.rgb_mean) / m.rgb_std
        s_x, map_x = m.compute_single_s_s_map(xp, m.calculate_dist(xp, m.patch_xyz_lib), (56, 56), modal="xyz")
        s_r, map_r = m.compute_single_s_s_map(rp, m.calculate_dist(rp, m.patch_rgb_lib), (28, 28), modal="rgb")
        s = torch.tensor([[m.args.xyz_s_lambda * s_x, m.args.rgb_s_lambda * s_r]])
        s_map = torch.cat([m.args.xyz_smap_lambda * map_x, m.args.rgb_smap_lambda * map_r],
                          dim=0).squeeze().reshape(2, -1).permute(1, 0)
        m.s_lib.append(s)
        m.s_map_lib.append(s_map)
    out["s_lib"] = torch.cat(m.s_lib, 0).numpy()
    m.run_late_fusion()                                  # features.py:352-358
    cent = synth.centroids(c["D"])
    xt = _t(synth.patches(c["P_xyz"], c["D"], c["seed"] * 1000 + 700, anomalous_frac=0.01, cent=cent))
    rt = _t(synth.patches(c["P_rgb"], c["D"], c["seed"] * 1000 + 701, anomalous_frac=0.01, cent=cent))
    mask = torch.zeros(1, 224, 224)
    m.compute_s_s_map(xt, rt, mask, 0, None, None, None, None, None, ["synthetic/0.png"])  # :967-1015
    out["image_pred"] = np.asarray(m.image_preds[0])
    out["prediction"] = np.asarray(m.predictions[0])
    np.savez_compressed(os.path.join(OUT, "dual_case.npz"), **out)
    print("dual_case:", {k: getattr(v, "shape", v) for k, v in out.items()})


# --------------------------------------------------------------------------------------------------------------------
# outputs of the live-reference comparisons of tests/test_metrics.py and tests/test_oracle.py, frozen so that those
# comparisons also run where the reference is absent.  Both tests assert bit-identity between the reference and
# cmdiad_b200.metrics / oracle.restate on exactly these inputs, so --from-restatement computes the same values without
# the reference.  The committed files were made that way, from code that passed both live tests (commit 03de1db; the
# metrics and oracle code is unchanged since).
# --------------------------------------------------------------------------------------------------------------------
AU_PRO_CASES = ((0, False), (1, True), (2, False), (3, True))   # (seed, quantised) of test_metrics._maps
AU_PRO_SETTINGS = ((0.3, 100), (0.01, 100), (0.3, 37))         # (integration_limit, num_thresholds)
FRESH_SEED_CASE = dict(n_train=3, P=784, D=768, seed=77, patch_seed=5, fmap=28)


def au_pro_key(seed, limit, nth):
    return f"seed{seed}_limit{limit}_n{nth}"


def golden_au_pro(use_reference=True):
    """calculate_au_pro (utils/au_pro_util.py) on the seeded maps of tests/test_metrics.py: value and curve"""
    from tests.test_metrics import _maps
    if use_reference:
        from tests.test_metrics import _reference_au_pro
        calc, source = _reference_au_pro().calculate_au_pro, "reference utils/au_pro_util.py"
    else:
        from cmdiad_b200 import metrics
        calc, source = metrics.au_pro, "cmdiad_b200.metrics.au_pro (bit-identical to the reference on these inputs)"
    out = {"source": np.str_(source)}
    for seed, quantised in AU_PRO_CASES:
        gts, preds = _maps(seed, quantised=quantised)
        for limit, nth in AU_PRO_SETTINGS:
            au, (fprs, pros) = calc(gts, preds, integration_limit=limit, num_thresholds=nth)
            k = au_pro_key(seed, limit, nth)
            out[f"{k}_au_pro"] = np.float64(au)
            out[f"{k}_fprs"] = np.asarray(fprs, dtype=np.float64)
            out[f"{k}_pros"] = np.asarray(pros, dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "au_pro_case.npz"), **out)
    print("au_pro_case:", len(out) - 1, "arrays from", source)


def golden_fresh_seed(use_reference=True):
    """RGBFeatures run_coreset (TF32 mode) + calculate_dist + compute_single_s_s_map on a seed none of the other golden
    cases uses; the statistics come from oracle.restate as in tests/test_oracle.py"""
    from oracle import restate as O
    c = FRESH_SEED_CASE
    train = synth.image_bank(c["n_train"], c["P"], c["D"], seed=c["seed"])
    cat = torch.cat([_t(x) for x in train], 0)
    mean, std = O.bank_stats_restated(cat)
    patch = (_t(synth.patches(c["P"], c["D"], c["patch_seed"], anomalous_frac=0.01)) - mean) / std
    fmap = (c["fmap"], c["fmap"])
    if use_reference:
        m = R.make_method("RGBFeatures", coreset_dtype="TF32", random_state=0)
        for x in train:
            m.patch_rgb_lib.append(_t(x))
        with R.cuda_to_cpu_if_needed():
            m.run_coreset()
        idx = m.coreset_idx.numpy()
        s, s_map = m.compute_single_s_s_map(patch, m.calculate_dist(patch, m.patch_rgb_lib), fmap, modal="rgb")
        s, s_map, source = np.float32(s), s_map[0].numpy(), "reference RGBFeatures"
    else:
        lib = O.normalize_restated(cat, mean, std).numpy()
        z = O.project_restated(lib, *O.sparse_components(lib.shape[0], c["D"], 0.9, 0))
        idx = O.coreset_restated(z, int(0.1 * lib.shape[0]), "TF32")
        r = O.score_restated(patch.numpy(), lib[idx], fmap, 224)
        s, s_map, source = np.float32(r["s"]), r["s_map"], "oracle.restate (bit-identical to the reference on these inputs)"
    np.savez_compressed(os.path.join(OUT, "fresh_seed_case.npz"), coreset_idx=np.asarray(idx, dtype=np.int64), s=s,
                        s_map=np.asarray(s_map, dtype=np.float32), source=np.str_(source))
    print("fresh_seed_case: from", source)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "--from-restatement" in sys.argv[1:]:
        golden_au_pro(use_reference=False)
        golden_fresh_seed(use_reference=False)
    else:
        golden_rgb()
        golden_dual()
        golden_au_pro()
        golden_fresh_seed()
