"""B200-native point-geometry hot path of SVDFormer / PointSea.

Public surface = the reference's op boundary (SURVEY.md 8b):
    chamfer_3DDist, chamfer_3DFunction                       (metrics/CD/chamfer3D/dist_chamfer_3D.py)
    furthest_point_sample, gather_operation, grouping_operation, ball_query,
    three_nn, three_interpolate, QueryAndGroup, GroupAll      (pointnet2_ops/pointnet2_utils.py)
    query_knn, fps_subsample, query_knn_point, index_points, group_local, sample_and_group_knn,
    EdgeConv (+ edge_features)                                (models/model_utils.py)
    calc_cd, calc_dcd, fscore                                 (utils/loss_utils.py, metrics/CD/fscore.py)
    losses.chamfer, chamfer_sqrt, chamfer_single_side, chamfer_single_side_sqrt  (utils/loss_utils.py:10-31)
    seprate_point_cloud (+ patch_helpers)                     (utils/helpers.py:62-123, ShapeNet-55/34 cropping)
`install_dropin()` makes `import metrics.CD.chamfer3D.dist_chamfer_3D` and
`import pointnet2_ops.pointnet2_utils` resolve to this package so the reference's models and
losses run unchanged, and `import torch_scatter` too where no torch_scatter is installed
(svdformer_pointsea_b200.scatter: PointSea's scatter-max).
"""
from ._lib import PointSeaError, LIB_PATH, load as load_library  # noqa: F401
from .chamfer import chamfer_3DDist, chamfer_3DFunction, chamfer_forward, chamfer_backward, chamfer_sums, chamfer_host, chamfer_host_async, HostStep, chamfer_host_step, ChamferStep  # noqa: F401
from .pointnet2_utils import (  # noqa: F401
    furthest_point_sample, gather_operation, grouping_operation, ball_query, three_nn, three_interpolate,
    FurthestPointSampling, GatherOperation, GroupingOperation, BallQuery, ThreeNN, ThreeInterpolate,
    QueryAndGroup, GroupAll, query_knn, fps_subsample,
)
from .model_ops import (  # noqa: F401
    query_knn_point, index_points, group_local, edge_features, EdgeConv, sample_and_group_knn, knn_self, patch_model_utils,
)
from .metrics import calc_cd, calc_dcd, fscore, chamfer_metrics_raw, chamfer_metrics_grad_raw, patch_loss_utils  # noqa: F401
# `chamfer` itself stays at losses.chamfer: as a package attribute it would hide the `chamfer` submodule
# (`import svdformer_pointsea_b200.chamfer as C` binds the attribute)
from .losses import ChamferLossFunction, chamfer_loss, chamfer_sqrt, chamfer_single_side, chamfer_single_side_sqrt  # noqa: F401
from .crop import seprate_point_cloud, crop_split_raw, fps_ragged_raw, patch_helpers  # noqa: F401
from .dropin import install_dropin, DROPIN_PATH, DROPIN_FALLBACK_PATH  # noqa: F401

__version__ = "0.1.0"
