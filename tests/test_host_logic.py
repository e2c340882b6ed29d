"""Host-side logic that needs no GPU: the reference-facing module surface, the drop-in shadow
packages, argument validation, and the fail-loudly behaviour of the product path."""
import os.path as osp
import sys

import pytest
import torch

from conftest import REFERENCE, ROOT
import svdformer_pointsea_b200 as ps
from svdformer_pointsea_b200 import _lib as L


def test_public_surface_matches_the_reference_names():
    for name in ("chamfer_3DDist", "chamfer_3DFunction", "furthest_point_sample", "gather_operation",
                 "grouping_operation", "ball_query", "three_nn", "three_interpolate", "QueryAndGroup", "GroupAll",
                 "query_knn", "fps_subsample"):
        assert hasattr(ps, name), name


def test_dropin_modules_resolve_to_this_package():
    ps.install_dropin()
    import metrics.CD.chamfer3D.dist_chamfer_3D as d
    from metrics.CD.fscore import fscore
    from pointnet2_ops.pointnet2_utils import (furthest_point_sample, gather_operation, ball_query, three_nn,  # noqa: F401
                                               three_interpolate, grouping_operation)
    assert d.chamfer_3DDist is ps.chamfer_3DDist and d.chamfer_3DFunction is ps.chamfer_3DFunction
    assert furthest_point_sample is ps.furthest_point_sample
    d1 = torch.tensor([[0.0, 0.00005, 1.0]])
    d2 = torch.tensor([[0.0, 0.0, 0.0, 1.0]])
    f, p1, p2 = fscore(d1, d2)
    assert abs(p1.item() - 2 / 3) < 1e-6 and abs(p2.item() - 0.75) < 1e-6
    assert abs(f.item() - 2 * (2 / 3) * 0.75 / (2 / 3 + 0.75)) < 1e-6
    f0, _, _ = fscore(torch.ones(1, 3), torch.ones(1, 3))
    assert f0.item() == 0.0  # 0/0 -> 0 as in the reference


def test_cpu_tensors_are_rejected_not_silently_computed():
    x = torch.rand(2, 16, 3)
    for fn in (lambda: ps.furthest_point_sample(x, 4), lambda: ps.chamfer_3DDist()(x, x),
               lambda: ps.query_knn(4, x, x), lambda: ps.ball_query(0.1, 4, x, x),
               lambda: ps.gather_operation(x.transpose(1, 2).contiguous(), torch.zeros(2, 4, dtype=torch.int32)),
               lambda: ps.grouping_operation(x.transpose(1, 2).contiguous(), torch.zeros(2, 4, 2, dtype=torch.int32))):
        with pytest.raises(RuntimeError, match="CUDA tensor"):
            fn()


def test_require_checks_dtype_rank_contiguity():
    with pytest.raises(L.PointSeaError, match="CUDA"):
        L.require(torch.zeros(2, 3), "t", torch.float32, 2)
    with pytest.raises(L.PointSeaError, match="torch.Tensor"):
        L.require([1, 2], "t", torch.float32, 1)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(L, "_lib", None)
    monkeypatch.setattr(L, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(L.PointSeaError, match="no CPU or PyTorch fallback"):
        L.load()


def test_reference_loss_utils_imports_unchanged_when_reference_present():
    """utils/loss_utils.py:3-6 imports models.model_utils (which needs our six pointnet2 names) and
    metrics.CD.* — with the drop-in ahead on sys.path the import works without building anything.
    Runs where a checkout of the reference (not part of this repository) is present."""
    ref = REFERENCE
    if not osp.isdir(ref):
        pytest.skip(f"needs a checkout of the reference at {ref} (or set POINTSEA_REFERENCE)")
    ps.install_dropin()
    added = ref not in sys.path
    if added:
        sys.path.append(ref)
    try:
        for m in [k for k in sys.modules if k == "utils" or k.startswith("utils.") or k == "models" or k.startswith("models.")]:
            del sys.modules[m]
        try:
            import utils.loss_utils as lu
        except ImportError as e:  # an unrelated third-party dependency of the models (timm, einops, ...)
            pytest.skip(f"reference import needs an absent dependency: {e}")
        assert lu.chamfer_dist.__class__ is ps.chamfer_3DDist
        import models.model_utils as mu
        assert mu.furthest_point_sample is ps.furthest_point_sample
        assert mu.grouping_operation is ps.grouping_operation
    finally:
        if added:
            sys.path.remove(ref)
        for m in [k for k in sys.modules if k == "utils" or k.startswith("utils.") or k == "models" or k.startswith("models.")]:
            del sys.modules[m]


def test_bench_reference_arm_contract():
    """--impl reference prints one JSON line with the same metric/unit and a cpu_baseline."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, osp.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "chamfer_fwd_bwd_gpair_per_s" and line["unit"] == "Gpair/s"
    assert line["cpu_baseline"]["cores"] >= 1 and line["e2e"]["h2d_bytes_per_step"] == 0


def test_next_row_surface_and_cpu_rejection():
    """SURVEY 8(f) names exist with the reference's signatures and refuse CPU tensors (no fallback)."""
    import inspect
    for name in ("query_knn_point", "index_points", "group_local", "sample_and_group_knn", "EdgeConv", "edge_features",
                 "calc_cd", "calc_dcd", "fscore", "patch_model_utils", "patch_loss_utils", "chamfer_host_step"):
        assert hasattr(ps, name), name
    assert list(inspect.signature(ps.query_knn_point).parameters) == ["k", "xyz", "new_xyz"]
    assert list(inspect.signature(ps.sample_and_group_knn).parameters) == ["xyz", "points", "npoint", "k", "use_xyz", "idx"]
    assert list(inspect.signature(ps.group_local).parameters) == ["xyz", "k", "return_idx"]
    assert list(inspect.signature(ps.calc_cd).parameters) == ["output", "gt", "calc_f1", "return_raw", "normalize", "separate"]
    assert list(inspect.signature(ps.calc_dcd).parameters) == ["x", "gt", "alpha", "n_lambda", "return_raw", "non_reg"]
    x = torch.rand(2, 32, 3)
    f = torch.rand(2, 8, 32)
    for fn in (lambda: ps.query_knn_point(4, x, x), lambda: ps.query_knn_point(4, torch.rand(2, 32, 8), torch.rand(2, 32, 8)),
               lambda: ps.edge_features(f, 4), lambda: ps.index_points(x, torch.zeros(2, 5, dtype=torch.long)),
               lambda: ps.sample_and_group_knn(x.transpose(1, 2).contiguous(), None, 8, 4),
               lambda: ps.calc_cd(x, x), lambda: ps.calc_dcd(x, x), lambda: ps.fscore(torch.rand(2, 5), torch.rand(2, 6))):
        with pytest.raises(ps.PointSeaError):
            fn()
    # EdgeConv keeps the reference's parameter names (state_dict compatibility: models/model_utils.py:856-866)
    keys = set(ps.EdgeConv(3, 64, 16).state_dict().keys())
    assert {"conv.0.weight", "conv.1.running_mean", "conv.3.weight", "conv.6.bias"} <= keys


def test_pipelined_sums_and_numa_helper_never_raise_without_a_gpu():
    from svdformer_pointsea_b200.dist import bind_to_gpu_numa_node
    assert bind_to_gpu_numa_node(0) is None or isinstance(bind_to_gpu_numa_node(0), set)


def test_host_buffer_entry_points_validate_before_touching_a_device():
    """chamfer_host / chamfer_host_async: shape and dtype errors are raised on the host (they do not need a GPU),
    and without a CUDA device both refuse to run (no CPU path)."""
    import inspect
    assert list(inspect.signature(ps.chamfer_host_async).parameters) == ["xyz1", "xyz2", "graddist1", "graddist2", "out", "chunk",
                                                                          "device", "sums_out", "comm"]
    a, b = torch.zeros(2, 8, 3), torch.zeros(2, 9, 3)
    for fn in (ps.chamfer_host, ps.chamfer_host_async):
        with pytest.raises(ps.PointSeaError, match="expects"):
            fn(a, torch.zeros(3, 9, 3))
        with pytest.raises(ps.PointSeaError, match="both graddist1 and graddist2"):
            fn(a, b, graddist1=torch.zeros(2, 8))
        with pytest.raises(ps.PointSeaError, match="contiguous"):
            fn(a.double(), b)
        if not torch.cuda.is_available():
            with pytest.raises(ps.PointSeaError, match="needs a CUDA device"):
                fn(a, b)
    step = ps.HostStep(0, 0, (a,), None, None)  # an empty submission: joining it is a no-op that needs no library call
    assert step.ticket == 0


def test_fps_flags_and_graphed_loss_fail_on_the_host_before_any_device_work():
    """ps_fps_sample_ex rejects flag bits it does not know (argument check, no device needed); GraphedLoss has no CPU
    path and says so."""
    import ctypes
    from svdformer_pointsea_b200 import _lib as L
    from svdformer_pointsea_b200.dist import GraphedLoss
    lib = L.load()
    rc = lib.ps_fps_sample_ex(None, None, None, 1, 8, 2, 0x40, 0, None)
    assert rc != 0 and b"unknown flags" in lib.ps_last_error()
    assert lib.ps_fps_sample_ex(None, None, None, 0, 8, 2, 1, 0, None) == 0  # empty batch: nothing to do, PS_FPS_CORUN accepted
    if not torch.cuda.is_available():
        with pytest.raises(ps.PointSeaError, match="CUDA device"):
            GraphedLoss([(1, 8, 3), (1, 16, 3), (1, 32, 3)], (1, 32, 3))
