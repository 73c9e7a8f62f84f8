"""GPU tests of the kernels around the distance path against exact host references computed from the same values:
the device-side pixel metrics (cmdb_eval_pixel_metrics, csrc/eval.cu), the late-fusion head with one to three
modalities (fuse_head_kernel, csrc/api.cu) and the bank statistics (cmdb_bank_stats, csrc/bank.cu).

The metrics are driven through the test-only loader cmdb_debug_eval_load, which appends chosen float64 maps to the
result store, so ties, sign mixes and 10 M-pixel stores cost one host-to-device copy.  Every exact check compares
integers or float64 bit patterns."""
import ctypes
import math
import zlib
from fractions import Fraction

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib(built):
    from cmdiad_b200 import _lib as L
    assert torch.cuda.is_available()
    return L.load()


@pytest.fixture(scope="module")
def fus(lib):
    """a late-fusion head over one tiny bank: only its result store is used"""
    from cmdiad_b200 import Bank
    from cmdiad_b200.fusion import LateFusion
    b = Bank(64, 64)
    yield LateFusion([b], [1.0], [1.0], [1.0], [0.0], [1.0], [0.0])
    b.close()


# ---- pixel metrics: loader, raw call, exact reference ---------------------------------------------------------------
def _load(fus, maps):
    from cmdiad_b200 import _lib as L
    maps = np.ascontiguousarray(maps, np.float64)
    # the head computes (v - off) + off in round-to-nearest and never stores -0.0; the sort keys order -0.0 below +0.0
    assert not np.any((maps == 0) & np.signbit(maps))
    L.check(L.load().cmdb_debug_eval_load(fus.banks[0]._h, maps.ctypes.data, maps.shape[0]))


def _store(fus, maps, capacity=None):
    fus.eval_reserve(capacity or maps.shape[0], maps.shape[-1])
    _load(fus, maps)


def _raw(fus, labels, n_comp, pos, n_thr=None):
    """cmdb_eval_pixel_metrics with explicit labels / ranks: thresholds, per-component <= counts, sizes, 2U, n_pos, n_neg"""
    from cmdiad_b200 import _lib as L
    labels = np.ascontiguousarray(labels, np.int32)
    pos = np.ascontiguousarray(pos, np.int64)
    n_thr = len(pos) if n_thr is None else n_thr
    thr = np.empty(max(1, n_thr), np.float64)
    le = np.empty((max(1, n_comp), max(1, n_thr)), np.int64)
    sizes = np.empty(max(1, n_comp), np.int64)
    two_u, n_pos, n_neg = ctypes.c_uint64(), ctypes.c_int64(), ctypes.c_int64()
    L.check(L.load().cmdb_eval_pixel_metrics(fus.banks[0]._h, labels.ctypes.data, int(n_comp), pos.ctypes.data, int(n_thr),
                                             thr.ctypes.data, le.ctypes.data, sizes.ctypes.data, ctypes.byref(two_u),
                                             ctypes.byref(n_pos), ctypes.byref(n_neg)))
    return dict(thr=thr[:n_thr], le=le[:n_comp], sizes=sizes[:n_comp], two_u=two_u.value, n_pos=n_pos.value, n_neg=n_neg.value)


def _reference(scores, labels, n_comp, pos):
    """the same quantities from the float64 values on the host, with numpy sorts and searches"""
    scores, labels = np.asarray(scores, np.float64).reshape(-1), np.asarray(labels).reshape(-1)
    ok = np.sort(scores[labels == 0])
    thr = ok[pos]
    an, lab = scores[labels > 0], labels[labels > 0]
    order = np.argsort(lab, kind="stable")
    lab, comp_scores = lab[order], an[order]
    sizes = np.bincount(lab, minlength=n_comp + 1)[1:].astype(np.int64)
    bounds = np.concatenate([[0], np.cumsum(sizes)])
    le = np.zeros((n_comp, len(pos)), np.int64)
    for c in range(n_comp):
        le[c] = np.searchsorted(np.sort(comp_scores[bounds[c]:bounds[c + 1]]), thr, side="right")
    # Mann-Whitney with ties counted one half: 2U = sum over anomalous pixels of #{ok < x} + #{ok <= x}
    two_u = int(np.searchsorted(ok, an, side="left").sum()) + int(np.searchsorted(ok, an, side="right").sum())
    return dict(thr=thr, le=le, sizes=sizes, two_u=two_u, n_pos=int(an.size), n_neg=int(ok.size))


def _assert_exact(got, ref):
    assert (got["thr"].view(np.uint64) == ref["thr"].view(np.uint64)).all()
    assert got["le"].shape == ref["le"].shape and (got["le"] == ref["le"]).all()
    assert (got["sizes"] == ref["sizes"]).all()
    assert (got["two_u"], got["n_pos"], got["n_neg"]) == (ref["two_u"], ref["n_pos"], ref["n_neg"])


def _check(fus, maps, gts, n_thr, curve=True):
    """exact counts of the device against the host reference; then the AU-PRO of device_pixel_metrics bit-identical to
    metrics.au_pro and its pixel AUROC against sklearn.  Returns the raw device result."""
    from sklearn.metrics import roc_auc_score

    from cmdiad_b200 import metrics
    labels, n_comp = metrics.label_components(gts)
    n_neg = int((labels == 0).sum())
    pos = np.linspace(0, n_neg - 1, num=n_thr, dtype=int).astype(np.int64)
    got = _raw(fus, labels, n_comp, pos)
    _assert_exact(got, _reference(maps, labels, n_comp, pos))
    if curve:
        dev = metrics.device_pixel_metrics(fus, gts, num_thresholds=n_thr)
        for lim in (0.3, 0.01):
            host, _ = metrics.au_pro(gts, list(maps), integration_limit=lim, num_thresholds=n_thr)
            assert dev["au_pro"][lim] == host, (lim, dev["au_pro"][lim], host)
        # 2U is exact; sklearn's trapezoid over its ROC curve differs from U / (n_pos n_neg) by rounding only
        auc = roc_auc_score((labels.reshape(-1) > 0).astype(np.int8), np.asarray(maps).reshape(-1))
        assert abs(dev["pixel_rocauc"] - auc) <= 1e-12, (dev["pixel_rocauc"], auc)
    return got


def _blobs(g, n, hw, max_blobs=3):
    yy, xx = np.ogrid[:hw, :hw]
    out = []
    for _ in range(n):
        m = np.zeros((hw, hw), np.uint8)
        for _ in range(int(g.integers(0, max_blobs + 1))):
            cy, cx = g.integers(0, hw, 2)
            r = int(g.integers(1, max(2, hw // 8)))
            m[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 1
        out.append(m)
    if not any(m.any() for m in out):
        out[0][hw // 2, hw // 2] = 1
    return out


def _quantised(g, n, hw):
    """256 levels x a per-image scale, like the blurred maps: dense ties, thresholds equal to component scores"""
    return g.integers(0, 256, (n, hw, hw)).astype(np.float64) * g.uniform(0.5, 4.0, n)[:, None, None]


def _magnitudes(g, n, hw):
    """both signs, magnitudes from the smallest subnormal to 1e300, with repeated values"""
    v = 10.0 ** g.uniform(-322, 300, n * hw * hw) * np.where(g.random(n * hw * hw) < 0.5, -1.0, 1.0)
    tiny = np.nextafter(0.0, 1.0)
    v[:8] = [tiny, -tiny, 3 * tiny, -3 * tiny, 1e300, -1e300, 0.0, 2.2250738585072014e-308]
    dup = g.choice(v.size, v.size // 8, replace=False)
    v[dup] = v[g.choice(v.size, dup.size)]
    return v.reshape(n, hw, hw)


@pytest.mark.parametrize("case", ["hw8", "hw8_few_negatives", "hw37", "constant", "negative", "mixed_sign", "magnitudes",
                                  "one_threshold", "4096_thresholds"])
def test_pixel_metrics_exact_small(fus, case):
    g = np.random.Generator(np.random.PCG64(zlib.crc32(case.encode())))
    n_thr = 100
    if case == "hw8":                   # 64 pixels per image: less than one warp slice of the sort
        maps, gts = g.standard_normal((3, 8, 8)), _blobs(g, 3, 8, 1)
    elif case == "hw8_few_negatives":   # fewer anomaly-free pixels than thresholds: linspace repeats ranks
        maps, gts = _quantised(g, 2, 8), [np.ones((8, 8), np.uint8), np.zeros((8, 8), np.uint8)]
        gts[1][:5] = 1
        assert (np.concatenate(gts) == 0).sum() < n_thr
    elif case == "hw37":                # ragged pixel count
        maps, gts = _quantised(g, 5, 37), _blobs(g, 5, 37)
    elif case == "constant":            # every pixel ties
        maps, gts = np.full((4, 32, 32), 0.75), _blobs(g, 4, 32)
    elif case == "negative":
        maps, gts = -(_quantised(g, 4, 32) + 0.25), _blobs(g, 4, 32)
    elif case == "mixed_sign":
        maps, gts = _quantised(g, 4, 32) - 300.0, _blobs(g, 4, 32)
    elif case == "magnitudes":
        maps, gts = _magnitudes(g, 4, 32), _blobs(g, 4, 32)
    elif case == "one_threshold":
        maps, gts, n_thr = _quantised(g, 3, 16), _blobs(g, 3, 16), 1
    else:
        maps, gts, n_thr = _quantised(g, 6, 64), _blobs(g, 6, 64), 4096
    _store(fus, maps)
    # one threshold leaves the whole PRO curve above the integration limits: the reference's trapezoid rejects it
    got = _check(fus, maps, gts, n_thr, curve=n_thr > 1)
    if case == "constant":
        assert got["two_u"] == got["n_pos"] * got["n_neg"]
        assert (got["le"] == got["sizes"][:, None]).all() and (got["thr"] == 0.75).all()
    if case == "hw8_few_negatives":
        assert len(np.unique(np.linspace(0, got["n_neg"] - 1, num=n_thr, dtype=int))) < n_thr


@pytest.mark.parametrize("n_images,n_thr", [(100, 100), (200, 4096)])
def test_pixel_metrics_exact_large(fus, n_images, n_thr):
    """224 x 100 images (5.0 M pixels: more than 1024 scan tiles, several tile counts per scan thread) and 224 x 200 images
    (10.0 M pixels: past the block cap of the sort grid, where each warp's slice grows)"""
    g = np.random.Generator(np.random.PCG64(n_images))
    maps, gts = _quantised(g, n_images, 224), _blobs(g, n_images, 224)
    _store(fus, maps)
    _check(fus, maps, gts, n_thr)


def test_pixel_metrics_components(fus):
    """a one-pixel component, the diagonal 8-connected pair, a component covering a whole image, and masks touching the
    border of consecutive images (they stay separate components)"""
    hw = 32
    g = np.random.Generator(np.random.PCG64(3))
    gts = [np.zeros((hw, hw), np.uint8) for _ in range(5)]
    gts[0][5, 5] = 1
    gts[0][10, 10] = gts[0][11, 11] = 1
    gts[1][:] = 1
    gts[2][-1, :] = 1
    gts[3][0, :] = 1
    maps = _quantised(g, 5, hw)
    _store(fus, maps)
    got = _check(fus, maps, gts, 100)
    assert got["sizes"].tolist() == [1, 2, hw * hw, hw, hw]


def test_pixel_metrics_without_components(fus):
    from cmdiad_b200 import metrics
    g = np.random.Generator(np.random.PCG64(4))
    maps, gts = _quantised(g, 3, 16), [np.zeros((16, 16), np.uint8)] * 3
    _store(fus, maps)
    got = _check(fus, maps, gts, 100, curve=False)
    assert got["n_pos"] == 0 and got["two_u"] == 0 and got["le"].shape == (0, 100)
    with pytest.raises(ZeroDivisionError):
        metrics.au_pro(gts, list(maps))
    with pytest.raises(ZeroDivisionError):
        metrics.device_pixel_metrics(fus, gts)


def test_result_store_fill_reset_and_repeat(fus):
    from cmdiad_b200 import metrics
    g = np.random.Generator(np.random.PCG64(5))
    maps, gts = _quantised(g, 10, 32), _blobs(g, 10, 32)
    # reserved for 10, filled with 7: only those 7 are counted
    fus.eval_reserve(10, 32)
    _load(fus, maps[:4])
    _load(fus, maps[4:7])
    assert fus.eval_count() == 7
    partial = _check(fus, maps[:7], gts[:7], 100)
    assert partial["n_pos"] + partial["n_neg"] == 7 * 32 * 32
    with pytest.raises(ValueError):   # masks of a different size than the stored maps
        metrics.device_pixel_metrics(fus, [np.zeros((64, 64), np.uint8)] * 7)
    # two calls on the same store: identical results
    again = _check(fus, maps[:7], gts[:7], 100)
    for k in partial:
        assert np.array_equal(np.asarray(partial[k]), np.asarray(again[k]))
    # reset and refill with other maps == a fresh store
    fus.eval_reset()
    assert fus.eval_count() == 0
    other = _quantised(g, 7, 32) - 100.0
    _load(fus, other)
    refilled = _check(fus, other, gts[:7], 100)
    _store(fus, other)
    fresh = _check(fus, other, gts[:7], 100)
    for k in fresh:
        assert np.array_equal(np.asarray(refilled[k]), np.asarray(fresh[k]))


def test_pixel_metrics_argument_checks(fus):
    """every malformed call raises CmdbError before any kernel runs; a valid call afterwards still gives the exact result"""
    from cmdiad_b200 import metrics
    from cmdiad_b200._lib import CmdbError
    g = np.random.Generator(np.random.PCG64(6))
    maps, gts = _quantised(g, 2, 16), _blobs(g, 2, 16)
    fus.eval_reserve(2, 16)
    labels, n_comp = metrics.label_components(gts)
    pos = np.linspace(0, int((labels == 0).sum()) - 1, num=10, dtype=int)
    with pytest.raises(CmdbError):   # empty store
        _raw(fus, labels, n_comp, pos)
    with pytest.raises(CmdbError):   # more images than reserved
        _load(fus, np.zeros((3, 16, 16)))
    _load(fus, maps)
    n_neg = int((labels == 0).sum())
    bad_high, bad_neg = labels.copy(), labels.copy()
    bad_high[1, 7] = n_comp + 1
    bad_neg[0, 3] = -1
    for args in [(bad_high, n_comp, pos), (bad_neg, n_comp, pos), (labels, n_comp, pos[::-1].copy()),
                 (labels, n_comp, np.array([0, n_neg])), (labels, n_comp, pos, 0), (labels, n_comp, np.zeros(4097, np.int64))]:
        with pytest.raises(CmdbError):
            _raw(fus, *args)
    torch.cuda.synchronize()
    _assert_exact(_raw(fus, labels, n_comp, pos), _reference(maps, labels, n_comp, pos))


def test_pixel_metrics_through_the_head(lib):
    """the store filled by the real fused head: a negative segmentation coefficient (negative maps: the sign branch of the
    sort key) and a zero one (an all-zero block of the store), read back and checked against the exact reference"""
    from cmdiad_b200 import Bank, synth
    from cmdiad_b200.fusion import LateFusion
    bank = Bank(64, 600)
    bank.append(synth.patches(600, 64, 11, k=32))
    bank.finalize()
    neg = LateFusion([bank], [1.0], [0.1], [1.0], [0.5], [-1.7], [0.3])
    zero = LateFusion([bank], [1.0], [0.1], [1.0], [0.5], [0.0], [0.3])
    patches = torch.from_numpy(np.stack([synth.patches(64, 64, 20 + i, anomalous_frac=0.05, k=32) for i in range(6)]))
    neg.eval_reserve(6, 224)
    r_neg = neg.score_batch([patches[:3]], [(8, 8)], 224, keep_on_device=True)
    r_zero = zero.score_batch([patches[3:]], [(8, 8)], 224, keep_on_device=True)
    maps, s = neg.eval_read()
    assert neg.eval_count() == 6 and (maps == np.concatenate([r_neg.s_map, r_zero.s_map])).all()
    assert not np.any((maps == 0) & np.signbit(maps)) and (maps[:3] < 0).any() and (maps[:3] <= 0).all() and (maps[3:] == 0).all()
    g = np.random.Generator(np.random.PCG64(7))
    _check(neg, maps, _blobs(g, 6, 224), 100)
    bank.close()


# ---- late-fusion head, one to three modalities ------------------------------------------------------------------------
HEADS = {   # s_lambda, smap_lambda, detect_coef, detect_offset, seg_coef, seg_offset
    "one": ([3.7], [0.1], [-2.5], 0.7, [1.9e3], -0.4),
    "two": ([0.1, 3.7], [3.7, 0.1], [0.8, -1.1], 2.0, [-0.6, 2.2e2], 3.0),
    "three": ([0.1, 3.7, 1.0], [0.1, 3.7, 0.1], [1.3, -0.7, 4.1e3], 0.3, [-1.3, 0.7, 2.5e3], 0.25),
    "three_zero": ([3.7, 0.1, 0.1], [3.7, 0.1, 3.7], [0.0, 2.0, -3.0], -1.5, [0.9, 0.0, -1e4], 7.0),
}


@pytest.fixture(scope="module")
def three_banks(lib):
    """three finalised banks with different P (fh x fw), D and row counts, and 3 test images per modality"""
    from cmdiad_b200 import Bank, synth
    spec = [(7, 64, 400), (8, 128, 500), (10, 192, 600)]
    banks, patches, dims = [], [], []
    for m, (side, dim, rows) in enumerate(spec):
        b = Bank(dim, rows)
        b.append(synth.patches(rows, dim, 30 + m, k=32))
        b.finalize()
        banks.append(b)
        patches.append(torch.from_numpy(np.stack([synth.patches(side * side, dim, 40 + 3 * m + i, anomalous_frac=0.05, k=32)
                                                  for i in range(3)])))
        dims.append((side, side))
    yield banks, patches, dims
    for b in banks:
        b.close()


def _fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))   # exact a*b + c, one rounding (int / int is correctly rounded)


def _head_inputs(banks, patches, dims, lam_s, lam_m, out_hw):
    """per modality the float32 products of the reference, lam * torch.from_numpy(map) / lam * s, as float64"""
    xs, xm = [], []
    for m in range(len(lam_s)):
        r = banks[m].score_batch(patches[m], dims[m], out_hw)
        xs.append(np.array([(lam_s[m] * torch.from_numpy(r[i].s)).numpy()[0] for i in range(len(r))]).astype(np.float64))
        xm.append(np.stack([(lam_m[m] * torch.from_numpy(r[i].s_map)).numpy() for i in range(len(r))]).astype(np.float64))
    return xs, xm


@pytest.mark.parametrize("name", list(HEADS))
def test_fused_head_against_exact_restatement_and_sklearn(three_banks, name):
    """s and s_map of the device head == the documented expression evaluated exactly (out_hw 32), and within 2 ulp of
    SGDOneClassSVM.score_samples (out_hw 224).  Map: x0*c0, fma(x0,c0, x1*c1), fma(x2,c2, fma(x0,c0, x1*c1)); image score:
    a sequential fma over the columns; both followed by (v - off) + off."""
    from sklearn.linear_model import SGDOneClassSVM

    from cmdiad_b200.fusion import LateFusion
    lam_s, lam_m, det, det_off, seg, seg_off = HEADS[name]
    M = len(lam_s)
    banks, patches, dims = (x[:M] for x in three_banks)
    fus = LateFusion(banks, lam_s, lam_m, det, det_off, seg, seg_off)

    res = fus.score_batch(patches, dims, out_hw=32)
    xs, xm = _head_inputs(banks, patches, dims, lam_s, lam_m, 32)
    assert (res.s_modal == np.stack(xs, 1).astype(np.float32)).all()
    want_s = np.empty(len(res))
    for i in range(len(res)):
        v = xs[0][i] * det[0]
        for m in range(1, M):
            v = _fma(xs[m][i], det[m], v)
        want_s[i] = (v - det_off) + det_off
        want = np.empty(32 * 32)
        for p, x in enumerate(np.stack([xm[m][i].reshape(-1) for m in range(M)], 1)):
            if M == 1:
                v = x[0] * seg[0]
            elif M == 2:
                v = _fma(x[0], seg[0], x[1] * seg[1])
            else:
                v = _fma(x[2], seg[2], _fma(x[0], seg[0], x[1] * seg[1]))
            want[p] = (v - seg_off) + seg_off
        bad = np.flatnonzero(want.view(np.uint64) != res.s_map[i].reshape(-1).view(np.uint64))
        assert bad.size == 0, (i, bad[:5], want[bad[:5]], res.s_map[i].reshape(-1)[bad[:5]])
    assert (want_s.view(np.uint64) == res.s.view(np.uint64)).all(), (want_s, res.s)

    # sklearn on the reference's layout: X = cat(maps).reshape(M, -1).permute(1, 0) (a column-major [npix, M] view)
    res = fus.score_batch(patches, dims, out_hw=224)
    xs, xm = _head_inputs(banks, patches, dims, lam_s, lam_m, 224)
    g = np.random.Generator(np.random.PCG64(0))
    heads = []
    for coef, off in ((det, det_off), (seg, seg_off)):
        h = SGDOneClassSVM().fit(g.standard_normal((8, M)))
        h.coef_, h.offset_ = np.array(coef, np.float64), np.array([off], np.float64)
        heads.append(h)
    same = []
    for i in range(len(res)):
        X = torch.from_numpy(np.stack([x[i] for x in xm]).astype(np.float32)).reshape(M, -1).permute(1, 0)
        want_map = heads[1].score_samples(X)
        want_s = heads[0].score_samples(torch.tensor([[float(x[i]) for x in xs]], dtype=torch.float32))[0]
        got_map = res.s_map[i].reshape(-1)
        ulp = np.abs(got_map - want_map) / np.spacing(np.maximum(np.abs(got_map), np.abs(want_map)))
        # nothing pins the BLAS's order of the column products: a different order moves a result by about an ulp
        assert ulp.max() <= 2 and abs(res.s[i] - want_s) <= 2 * np.spacing(abs(want_s)), (i, ulp.max(), res.s[i], want_s)
        same.append(float((got_map == want_map).mean()))
    print(f"fused head '{name}' ({M} modalities): maps bit-identical to sklearn on {min(same):.4%} of pixels (worst image)")


# ---- bank statistics ----------------------------------------------------------------------------------------------
_Z = {}


def _normal(rows, dim):
    if (rows, dim) not in _Z:
        _Z[(rows, dim)] = np.random.Generator(np.random.PCG64(rows)).standard_normal((rows, dim), dtype=np.float32)
    return _Z[(rows, dim)]


@pytest.mark.parametrize("rows,dim", [(5000, 192), (200_000, 768)])
@pytest.mark.parametrize("offset", [0.0, 1e2, 1e3, 1e4])
def test_bank_stats_against_exact_sums(lib, rows, dim, offset):
    """mean / unbiased std of a bank with mean/std = offset against exact rational sums.  The values are float32 on the grid
    2^-k of the largest binade (x = Q * 2^-k, |Q| < 2^24), so sum(x) and the two-pass sum((x - mean)^2) are exact
    integers over powers of two -- the exact counterpart of math.fsum, affordable at 1.5e8 elements."""
    from cmdiad_b200 import Bank
    z = _normal(rows, dim)
    k = 24 - math.frexp(abs(offset) + float(np.abs(z).max()) + 1.0)[1]
    c = int(offset * 2 ** k)
    assert c == offset * 2 ** k
    n = rows * dim
    b = Bank(dim, rows)
    sum_d = sum_d2 = sum_absq = 0
    for r0 in range(0, rows, 20_000):
        d = np.rint(z[r0:r0 + 20_000].astype(np.float64) * 2.0 ** k).astype(np.int64)
        q = c + d
        assert np.abs(q).max() < 2 ** 24
        x = (q * 2.0 ** -k).astype(np.float32)
        assert (x.astype(np.float64) * 2.0 ** k == q).all()
        b.append(x)
        sum_d += int(d.sum())
        sum_d2 += sum((d * d).sum(axis=1).tolist())   # a row sum stays below 2^63; the total is a Python integer
        sum_absq += int(np.abs(q).sum())
    mean, std, s, sq = b.stats()
    mean_ref = float(Fraction(n * c + sum_d, n * 2 ** k))
    var_ref = Fraction(n * sum_d2 - sum_d * sum_d, n * (n - 1) * 4 ** k)   # sum((x - mean)^2) / (n - 1), exactly
    std_ref = math.sqrt(float(var_ref))
    sq_ref = float(Fraction(sum_d2 + 2 * c * sum_d + n * c * c, 4 ** k))
    mean_abs = float(Fraction(sum_absq, n * 2 ** k))
    # float64 accumulation of up to 1.5e8 terms: rounding error far below 1e-13 when the variance is summed from the
    # deviations; the one-pass (sumsq - sum * mean) cancels by (mean / std)^2 and misses it from mean/std = 1e2 on
    assert abs(std - std_ref) <= 1e-13 * std_ref, (offset, std, std_ref, abs(std - std_ref) / std_ref)
    # at offset 0 the mean is a cancelling sum: bound its error by the data's magnitude, not by itself
    assert abs(mean - mean_ref) <= 1e-13 * mean_abs, (offset, mean, mean_ref)
    assert abs(sq - sq_ref) <= 1e-13 * sq_ref, (offset, sq, sq_ref)
    # a fixed reduction order: repeated calls are bit-identical
    for _ in range(3):
        m2, s2, sum2, sq2 = b.stats()
        assert np.array([sum2, sq2, m2, s2]).view(np.uint64).tolist() == np.array([s, sq, mean, std]).view(np.uint64).tolist()
    print(f"offset {offset:g} {rows}x{dim}: std relative error {abs(std - std_ref) / std_ref:.2e}")
    b.close()
