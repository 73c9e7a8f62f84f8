"""CPU suite: integration/cmdiad_b200.patch applies to the reference and the patched reference is a working drop-in.

Needs the reference tree (oracle/ref_loader.py).  The patched tree is a scratch copy under tmp_path; nothing is copied
into the repository."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import ref_loader as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATCH = os.path.join(ROOT, "integration", "cmdiad_b200.patch")

pytestmark = pytest.mark.skipif(not R.reference_available(), reason=R.SKIP_REASON)


def _scratch_copy(tmp_path):
    dst = tmp_path / "ref"
    shutil.copytree(R.REFERENCE_ROOT, dst, ignore=shutil.ignore_patterns(".git", "*.png", "*.jpg", "*.pdf"))
    subprocess.run(["git", "init", "-q", "."], cwd=dst, check=True)
    return str(dst)


def test_patch_applies_and_touches_only_the_seams(tmp_path):
    ref = _scratch_copy(tmp_path)
    subprocess.run(["git", "apply", "--check", PATCH], cwd=ref, check=True)
    subprocess.run(["git", "apply", PATCH], cwd=ref, check=True)
    text = open(PATCH, newline="").read()
    added = [ln for ln in text.splitlines() if ln.startswith("+") and not ln.startswith("+++")]
    removed = [ln for ln in text.splitlines() if ln.startswith("-") and not ln.startswith("---")]
    assert len(removed) == 0 and len(added) == 12, (len(added), len(removed))   # additions only: no reference line changes
    assert [ln for ln in text.splitlines() if ln.startswith("+++")] == ["+++ b/feature_extractors/features.py"]
    # the method bodies the runner calls are byte-identical in multiple_features.py (not touched at all)
    a = open(os.path.join(R.REFERENCE_ROOT, "feature_extractors", "multiple_features.py"), "rb").read()
    b = open(os.path.join(ref, "feature_extractors", "multiple_features.py"), "rb").read()
    assert a == b


def _drive(ref_root, out, cls):
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_dropin_driver.py"), ref_root, out, cls], env=env,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    return dict(np.load(out))


@pytest.mark.timeout(1500)
@pytest.mark.parametrize("cls", ["RGBFeatures", "DoubleRGBPointFeatures"])
def test_patched_reference_equals_stock_reference(tmp_path, cls):
    """the reference's own __init__ / add_sample_to_mem_bank / run_coreset / add_sample_to_late_fusion_mem_bank /
    run_late_fusion / predict / calculate_metrics bodies run over the three seams (device-backed lists + BankLib via
    __torch_function__, get_coreset_idx_randomp, calculate_dist + compute_single_s_s_map).  With the CPU checker behind
    the seams the patched run must equal the stock run bit for bit."""
    ref = _scratch_copy(tmp_path)
    subprocess.run(["git", "apply", PATCH], cwd=ref, check=True)
    stock = _drive(R.REFERENCE_ROOT, str(tmp_path / "stock.npz"), cls)
    patched = _drive(ref, str(tmp_path / "patched.npz"), cls)
    assert not bool(stock["patched"]) and bool(patched["patched"])
    for k in ("coreset_idx", "image_preds", "predictions", "pixel_rocauc", "au_pro", "rgb_mean", "rgb_std", "lib_rgb_shape",
              "lib_rgb_head"):
        assert (stock[k] == patched[k]).all(), k
    calls = str(patched["calls_rgb"]).split(",")
    # the seams were really exercised: rows appended to the bank, statistics / normalise / coreset / gather on it, scoring
    # through the fused call (finalize + neighbour table once, before the first score)
    assert calls[:4] == ["append"] * 4 and "stats" in calls and "normalize" in calls and "coreset_select" in calls
    assert calls.index("gather") < calls.index("finalize") < calls.index("build_knn") < calls.index("score")
    assert calls.count("finalize") == 1 and calls.count("score") == 6   # 4 train images + 2 test images
