"""TEST INFRASTRUCTURE ONLY -- loads the UNMODIFIED reference (evenrose/CMDIAD) in-process.

The repository does not contain the reference: place a checkout of it at oracle/_ref/ (git-ignored) or point
CMDIAD_REFERENCE_ROOT at one.  Nothing under -m gpu tests, smoke() or bench.py may call this.  It is used by
oracle/make_golden.py to freeze golden vectors under tests/golden/ and by the CPU test-suite to validate
oracle/restate.py against the real reference code; those tests skip where the reference is absent.

Recipe (SURVEY.md Appendix C): register empty stand-in modules for the seven imports this image lacks
(cupy, cupyx.scipy.spatial.distance, matplotlib.pyplot, timm, knn_cuda, pointnet2_ops, tifffile), import
feature_extractors.{features,multiple_features} unmodified, build method objects with __new__ (skipping the backbone
constructor, features.py:22-32) and set the attributes features.py:34-121 would have set.
"""
import contextlib
import os
import sys
import types
from argparse import Namespace

import torch

REFERENCE_ROOT = os.environ.get("CMDIAD_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))
SKIP_REASON = "needs the unmodified reference tree (oracle/_ref/ or CMDIAD_REFERENCE_ROOT), which the repository does not ship"


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "feature_extractors", "features.py"))


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent:
        setattr(_stub(parent), child, m)
    return m


_loaded = None


def load_reference():
    """Returns (features_module, multiple_features_module) of the unmodified reference."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    for name in ("cupy", "cupyx", "cupyx.scipy", "cupyx.scipy.spatial", "cupyx.scipy.spatial.distance",
                 "matplotlib", "matplotlib.pyplot", "tifffile", "pointnet2_ops", "pointnet2_ops.pointnet2_utils"):
        try:
            __import__(name)
        except Exception:
            _stub(name)
    try:
        import timm  # noqa: F401
    except Exception:
        _stub("timm")
        _stub("timm.models")
        _stub("timm.models.layers", DropPath=object)
    try:
        import knn_cuda  # noqa: F401
    except Exception:
        _stub("knn_cuda", KNN=object)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import feature_extractors.features as F
    import feature_extractors.multiple_features as MF
    _loaded = (F, MF)
    return _loaded


def default_args(**over):
    """Hot-path knobs with the defaults of main.py:85-189."""
    a = dict(dist_method_s="l2", dist_method_coreset="l2", coreset_dtype="FP16", f_coreset=0.1, coreset_eps=0.9,
             random_state=0, rgb_s_lambda=0.1, rgb_smap_lambda=0.1, xyz_s_lambda=1.0, xyz_smap_lambda=1.0,
             fusion_s_lambda=1.0, fusion_smap_lambda=1.0, main_modality="", gt_size=224, save_seg_results=False,
             save_raw_results=False, use_depth=False, save_feature_for_fusion=False, save_frgb_xyz=False,
             save_rgb_fxyz=False, ocsvm_nu=0.5, ocsvm_maxiter=1000)
    a.update(over)
    return Namespace(**a)


def make_method(cls_name="RGBFeatures", **arg_over):
    """Instantiate a reference method class without its backbones (features.py:22-121 minus 25-32, 91-112)."""
    F, MF = load_reference()
    from sklearn import linear_model
    from utils.utils import KNNGaussianBlur
    cls = getattr(MF, cls_name)
    args = default_args(**arg_over)
    obj = cls.__new__(cls)
    torch.nn.Module.__init__(obj)
    obj.args = args
    obj.device = "cpu"
    obj.class_name = None
    obj.gt_size = args.gt_size
    obj.f_coreset = args.f_coreset
    obj.coreset_eps = args.coreset_eps
    obj.coreset_dtype = args.coreset_dtype
    obj.random_state = args.random_state
    obj.blur = KNNGaussianBlur(4)
    obj.n_reweight = 3
    for lib in ("patch_xyz_lib", "patch_rgb_lib", "patch_fusion_lib", "patch_lib", "patch_share_lib",
                "patch_non_share_lib", "s_lib", "s_map_lib", "image_preds", "image_labels", "pixel_preds",
                "pixel_labels", "gts", "predictions", "img_name"):
        setattr(obj, lib, [])
    for s in ("xyz", "rgb", "fusion"):
        setattr(obj, f"{s}_mean", 0)
        setattr(obj, f"{s}_std", 0)
    obj.detect_fuser = linear_model.SGDOneClassSVM(random_state=42, nu=args.ocsvm_nu, max_iter=args.ocsvm_maxiter)
    obj.seg_fuser = linear_model.SGDOneClassSVM(random_state=42, nu=args.ocsvm_nu, max_iter=args.ocsvm_maxiter)
    return obj


@contextlib.contextmanager
def cuda_to_cpu_if_needed():
    """get_coreset_idx_randomp hard-codes .to("cuda") (features.py:397-399); redirect when no GPU is present."""
    if torch.cuda.is_available():
        yield
        return
    orig = torch.Tensor.to

    def to(self, *a, **k):
        a = tuple("cpu" if (isinstance(x, str) and x.startswith("cuda")) else x for x in a)
        if isinstance(k.get("device"), str) and k["device"].startswith("cuda"):
            k["device"] = "cpu"
        return orig(self, *a, **k)

    torch.Tensor.to = to
    try:
        yield
    finally:
        torch.Tensor.to = orig
