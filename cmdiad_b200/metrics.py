"""Evaluation metrics of the reference's calculate_metrics (features.py:302-324; SURVEY 8f-3), vectorised.

The reference accumulates 50 176 Python scalars per test image (`pixel_preds.extend`, multiple_features.py:998) and
walks every ground-truth component once per threshold in Python (utils/au_pro_util.py:157-201).  Here predictions stay
numpy arrays and the PRO curve is evaluated with one `searchsorted` per component for all thresholds at once.  The
arithmetic (which counts are taken, the order of the float64 additions, the trapezoid with its interpolated last
segment) follows the reference, so the values are bit-identical -- tests/test_metrics.py checks that against the
unmodified reference module.
"""
import numpy as np
from scipy.ndimage import label
from sklearn.metrics import roc_auc_score


def pro_curve(predictions, gts, num_thresholds=100):
    """PRO curve (utils/au_pro_util.py:104-201): false-positive rates and mean per-region overlaps at `num_thresholds`
    thresholds taken at equidistant ranks of the sorted anomaly-free scores.  predictions / gts: sequences of 2-D arrays."""
    assert len(predictions) == len(gts)
    structure = np.ones((3, 3), dtype=int)        # 8-connectivity (au_pro_util.py:129)
    ok_scores, components = [], []
    for gt, pred in zip(gts, predictions):
        gt, pred = np.asarray(gt), np.asarray(pred)
        labeled, n = label(gt, structure)
        ok_scores.append(pred[labeled == 0])
        for k in range(n):
            components.append(np.sort(pred[labeled == (k + 1)]))
    # the reference collects the anomaly-free scores in a float64 buffer (np.zeros default dtype) before sorting
    ok = np.sort(np.concatenate(ok_scores).astype(np.float64)) if ok_scores else np.zeros(0)
    pos = np.linspace(0, len(ok) - 1, num=num_thresholds, dtype=int)
    thr = ok[pos]
    fprs = 1.0 - (pos + 1) / len(ok)
    # overlap of a component at threshold t = 1 - #{scores <= t} / size  (GroundTruthComponent.compute_overlap)
    overlaps = np.empty((len(components), len(thr)), dtype=np.float64)
    for i, c in enumerate(components):
        overlaps[i] = 1.0 - np.searchsorted(c, thr, side="right") / len(c)
    # `pro += overlap` over the components in order, then `/= len`: a sequential float64 sum
    if not components:  # the reference divides by len(ground_truth_components) (au_pro_util.py:192): same error here
        raise ZeroDivisionError("float division by zero: no ground-truth component in any mask")
    pros = np.cumsum(overlaps, axis=0)[-1] / len(components)
    fprs = np.concatenate([[1.0], fprs])[::-1]
    pros = np.concatenate([[1.0], pros])[::-1]
    return fprs, pros


def trapezoid(x, y, x_max=None):
    """au_pro_util.py:52-101: trapezoid rule with an interpolated last segment at x_max (non-finite points dropped)"""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    keep = np.isfinite(x) & np.isfinite(y)
    x, y = x[keep], y[keep]
    correction = 0.0
    if x_max is not None:
        if x_max not in x:
            ins = int(np.searchsorted(x, x_max, side="right"))   # bisect.bisect
            assert 0 < ins < len(x)
            y_interp = y[ins - 1] + ((y[ins] - y[ins - 1]) * (x_max - x[ins - 1]) / (x[ins] - x[ins - 1]))
            correction = 0.5 * (y_interp + y[ins - 1]) * (x_max - x[ins - 1])
        m = x <= x_max
        x, y = x[m], y[m]
    return np.sum(0.5 * (y[1:] + y[:-1]) * (x[1:] - x[:-1])) + correction


def au_pro(gts, predictions, integration_limit=0.3, num_thresholds=100):
    """calculate_au_pro (au_pro_util.py:204-224): area under the PRO curve up to `integration_limit`, normalised"""
    fprs, pros = pro_curve(predictions, gts, num_thresholds)
    return trapezoid(fprs, pros, x_max=integration_limit) / integration_limit, (fprs, pros)


def image_and_pixel_rocauc(image_labels, image_preds, pixel_labels, pixel_preds):
    """features.py:314-319"""
    return (roc_auc_score(np.asarray(image_labels), np.asarray(image_preds)),
            roc_auc_score(np.asarray(pixel_labels).reshape(-1), np.asarray(pixel_preds).reshape(-1)))


# ---- device-side evaluation (SURVEY 8f-3): cmdb_eval_pixel_metrics does the sorting / counting on the GPU ----------------
def label_components(gts):
    """scipy.ndimage.label with the 8-connectivity structure of au_pro_util.py:129 for every mask, numbered through the
    whole set in image order.  Returns (int32 labels [n, H*W], n_components)."""
    structure = np.ones((3, 3), dtype=int)
    out, base = [], 0
    for gt in gts:
        labeled, n = label(np.asarray(gt), structure)
        lab = labeled.astype(np.int32)
        lab[lab > 0] += base
        out.append(lab.reshape(-1))
        base += n
    return np.stack(out), base


def pro_curve_from_counts(pos, n_ok, le_counts, sizes):
    """the PRO curve of utils/au_pro_util.py:157-201 from exact integer counts (same float64 operations, same order)"""
    if len(sizes) == 0:
        raise ZeroDivisionError("float division by zero: no ground-truth component in any mask")
    fprs = 1.0 - (pos + 1) / n_ok
    overlaps = 1.0 - le_counts / sizes[:, None]                       # 1.0 - index / len(scores) per component
    pros = np.cumsum(overlaps, axis=0)[-1] / len(sizes)               # pro += overlap in component order, then /= len
    return np.concatenate([[1.0], fprs])[::-1], np.concatenate([[1.0], pros])[::-1]


def device_pixel_metrics(fusion, gts, num_thresholds=100, limits=(0.3, 0.01)):
    """pixel AUROC + AU-PRO (features.py:322-324) of the maps kept in `fusion`'s device-side result store (one per mask in
    `gts`, in predict order).  Returns dict(pixel_rocauc, au_pro={limit: value}, curve=(fprs, pros))."""
    import ctypes

    from . import _lib as L
    lib = L.load()
    labels, n_comp = label_components(gts)
    hw = fusion._eval_hw
    if labels.shape != (fusion.eval_count(), hw * hw):   # the library reads one label per stored pixel
        raise ValueError(f"one {hw}x{hw} ground-truth mask per stored map: {fusion.eval_count()} maps, masks {labels.shape}")
    labels = np.ascontiguousarray(labels)
    n_ok = int((labels == 0).sum())
    pos = np.linspace(0, n_ok - 1, num=num_thresholds, dtype=int).astype(np.int64)
    thr = np.empty(num_thresholds, np.float64)
    le = np.empty((max(1, n_comp), num_thresholds), np.int64)
    sizes = np.empty(max(1, n_comp), np.int64)
    two_u, n_pos, n_neg = ctypes.c_uint64(), ctypes.c_int64(), ctypes.c_int64()
    L.check(lib.cmdb_eval_pixel_metrics(fusion.banks[0]._h, labels.ctypes.data, n_comp, pos.ctypes.data, num_thresholds,
                                        thr.ctypes.data, le.ctypes.data, sizes.ctypes.data, ctypes.byref(two_u),
                                        ctypes.byref(n_pos), ctypes.byref(n_neg)))
    fprs, pros = pro_curve_from_counts(pos, n_ok, le[:n_comp], sizes[:n_comp])
    auc = two_u.value / (2.0 * n_pos.value * n_neg.value) if n_pos.value and n_neg.value else float("nan")
    return dict(pixel_rocauc=auc, au_pro={lim: trapezoid(fprs, pros, x_max=lim) / lim for lim in limits}, curve=(fprs, pros),
                thresholds=thr, n_pos=n_pos.value, n_neg=n_neg.value)
