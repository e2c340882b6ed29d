"""Makes the reference's import paths resolve to this package.

`dropin_pkgs/` holds two tiny shadow packages with the reference's module names:
    metrics/CD/chamfer3D/dist_chamfer_3D.py, metrics/CD/fscore.py, metrics/__init__.py
    pointnet2_ops/pointnet2_utils.py
Put DROPIN_PATH ahead of the reference tree on sys.path (install_dropin() does it) and
models/SVDFormer.py, models_PointSea/PointSea.py and utils/loss_utils.py import unchanged.

`dropin_fallback/` holds torch_scatter (PointSea's renderer, models_PointSea/mv_utils_zs.py:1,130), which only covers
the one reduction PointSea uses.  A user's own torch_scatter must keep precedence, so DROPIN_FALLBACK_PATH goes at the
END of sys.path: the shim is found only when no torch_scatter is installed.
"""
import os.path as osp
import sys

DROPIN_PATH = osp.join(osp.dirname(osp.abspath(__file__)), "dropin_pkgs")
DROPIN_FALLBACK_PATH = osp.join(osp.dirname(osp.abspath(__file__)), "dropin_fallback")


def install_dropin():
    if DROPIN_PATH not in sys.path:
        sys.path.insert(0, DROPIN_PATH)
    if DROPIN_FALLBACK_PATH not in sys.path:
        sys.path.append(DROPIN_FALLBACK_PATH)
    # drop any already-imported reference modules of the same names
    for name in list(sys.modules):
        if name == "metrics" or name.startswith("metrics.") or name == "pointnet2_ops" or name.startswith("pointnet2_ops."):
            mod = sys.modules[name]
            f = getattr(mod, "__file__", None) or ""
            if not f.startswith(DROPIN_PATH):
                del sys.modules[name]
    return DROPIN_PATH
