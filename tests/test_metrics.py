"""CPU suite: cmdiad_b200/metrics.py (SURVEY 8f-3) against the unmodified reference utils/au_pro_util.py (live, when
the reference tree is present) and against values frozen from it."""
import importlib.util
import os

import numpy as np
import pytest

from cmdiad_b200 import metrics
from oracle import ref_loader as R


def _maps(seed, n_img=6, hw=64, quantised=False):
    """anomaly maps with a few blob-shaped defects (some touching diagonally: 8-connectivity matters) + noise"""
    g = np.random.Generator(np.random.PCG64(seed))
    preds, gts = [], []
    for i in range(n_img):
        gt = np.zeros((hw, hw), dtype=np.float32)
        pred = g.random((hw, hw)).astype(np.float32) * 0.5
        for _ in range(int(g.integers(0, 4)) if i else 2):
            cy, cx, r = g.integers(6, hw - 6), g.integers(6, hw - 6), g.integers(2, 6)
            yy, xx = np.ogrid[:hw, :hw]
            blob = (yy - cy) ** 2 + (xx - cx) ** 2 <= r * r
            gt[blob] = 1
            pred[blob] += g.random() * 0.8
        if i == 1:  # two pixels that only touch diagonally
            gt[2, 2] = gt[3, 3] = 1
        if quantised:   # the blurred score maps have <= 256 levels: many ties between scores and thresholds
            pred = np.floor(pred * 20) / 20
        preds.append(pred)
        gts.append(gt)
    return gts, preds


def _reference_au_pro():
    spec = importlib.util.spec_from_file_location("ref_au_pro_util", os.path.join(R.REFERENCE_ROOT, "utils", "au_pro_util.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.filterwarnings("ignore::DeprecationWarning")
@pytest.mark.parametrize("seed,quantised", [(0, False), (1, True), (2, False), (3, True)])
def test_au_pro_bit_exact_against_live_reference(golden, seed, quantised):
    """value and curve against the reference's calculate_au_pro: its outputs on these inputs are frozen in
    tests/golden/au_pro_case.npz (oracle/make_golden.py); where the reference tree is present it is also run live"""
    frozen = golden["au_pro_case"]
    ref = _reference_au_pro() if R.reference_available() else None
    gts, preds = _maps(seed, quantised=quantised)
    for limit, nth in ((0.3, 100), (0.01, 100), (0.3, 37)):
        got, (gf, gp) = metrics.au_pro(gts, preds, integration_limit=limit, num_thresholds=nth)
        k = f"seed{seed}_limit{limit}_n{nth}"
        assert (frozen[f"{k}_fprs"] == gf).all() and (frozen[f"{k}_pros"] == gp).all(), k
        assert got == float(frozen[f"{k}_au_pro"]), (k, got)
        if ref is not None:
            want, (wf, wp) = ref.calculate_au_pro(gts, preds, integration_limit=limit, num_thresholds=nth)
            assert (np.asarray(wf) == gf).all() and (np.asarray(wp) == gp).all()
            assert got == want, (seed, limit, nth, got, want)


def test_au_pro_frozen_values():
    """values produced by the reference's calculate_au_pro on these inputs (frozen so the check travels without it)"""
    expect = {(0, False, 0.3): 0.7840381111818155, (0, False, 0.01): 0.7114581276946017,
              (1, True, 0.3): 0.5781859588205034, (1, True, 0.01): 0.5021305225386857}
    for (seed, q, limit), want in expect.items():
        gts, preds = _maps(seed, quantised=q)
        got, _ = metrics.au_pro(gts, preds, integration_limit=limit)
        assert got == want, (seed, q, limit, got.hex() if hasattr(got, "hex") else got)


def test_trapezoid_and_edge_cases():
    x = np.array([0.0, 0.1, 0.2, 0.5, 1.0])
    y = np.array([0.0, 0.5, 0.6, 0.9, 1.0])
    assert metrics.trapezoid(x, y) == np.sum(0.5 * (y[1:] + y[:-1]) * (x[1:] - x[:-1]))
    # x_max between two samples: the last segment is interpolated
    full_to_02 = 0.5 * 0.5 * 0.1 + 0.5 * 1.1 * 0.1
    y03 = 0.6 + (0.9 - 0.6) * (0.3 - 0.2) / (0.5 - 0.2)
    np.testing.assert_allclose(metrics.trapezoid(x, y, x_max=0.3), full_to_02 + 0.5 * (0.6 + y03) * 0.1, rtol=1e-15)
    assert metrics.trapezoid(x, y, x_max=0.2) == metrics.trapezoid(x[:3], y[:3])
    # no anomalous region at all: the reference divides by the component count (au_pro_util.py:192) -> same error here
    gts, preds = [np.zeros((8, 8), np.float32)], [np.arange(64, dtype=np.float32).reshape(8, 8)]
    with pytest.raises(ZeroDivisionError):
        metrics.au_pro(gts, preds)
    if R.reference_available():
        with pytest.raises(ZeroDivisionError):
            _reference_au_pro().calculate_au_pro(gts, preds)
    img, pix = metrics.image_and_pixel_rocauc([0, 1, 1, 0], [0.1, 0.9, 0.8, 0.3], [[0, 1], [1, 0]], [[0.2, 0.7], [0.9, 0.1]])
    assert img == 1.0 and pix == 1.0


def test_pro_curve_from_integer_counts_equals_direct_evaluation():
    """the host half of the device-side evaluation (metrics.device_pixel_metrics): given the exact integer counts the GPU
    returns (emulated with numpy here), the curve and both integrals must equal the direct evaluation bit for bit"""
    for seed, q in ((0, False), (1, True)):
        gts, preds = _maps(seed, quantised=q)
        preds = [p.astype(np.float64) for p in preds]
        labels, n_comp = metrics.label_components(gts)
        flat = np.stack([p.reshape(-1) for p in preds])
        ok = np.sort(flat[labels == 0])
        pos = np.linspace(0, len(ok) - 1, num=100, dtype=int)
        thr = ok[pos]
        le = np.stack([(flat[labels == c + 1][:, None] <= thr[None, :]).sum(0) for c in range(n_comp)])
        sizes = np.array([(labels == c + 1).sum() for c in range(n_comp)])
        fprs, pros = metrics.pro_curve_from_counts(pos, len(ok), le, sizes)
        wf, wp = metrics.pro_curve(preds, gts)
        assert (fprs == wf).all() and (pros == wp).all()
        for lim in (0.3, 0.01):
            assert metrics.trapezoid(fprs, pros, x_max=lim) / lim == metrics.au_pro(gts, preds, lim)[0]
        # exact Mann-Whitney form of the pixel AUROC (what cmdb_eval_pixel_metrics returns as the integer 2U)
        y, s = (labels > 0).reshape(-1), flat.reshape(-1)
        neg = np.sort(s[~y])
        two_u = int((np.searchsorted(neg, s[y], side="left") + np.searchsorted(neg, s[y], side="right")).sum())
        from sklearn.metrics import roc_auc_score
        assert abs(two_u / (2.0 * y.sum() * (~y).sum()) - roc_auc_score(y, s)) < 1e-12
