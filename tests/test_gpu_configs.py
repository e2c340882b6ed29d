"""BASELINE.json configs 4 and 5 as GPU tests (VERDICT r1 item 6).

C4  the reference's UNMODIFIED models (models/SVDFormer.py, models_PointSea/PointSea.py) and losses
    (utils/loss_utils.get_loss / get_loss_PM) run on top of this repo's ops through the drop-in import paths, and
    the loss is compared bit-for-bit with the same model on the reference's own CUDA ops (oracle/_ref).  The two
    arms bind the same module names, so each runs in its own process (tools/bench_configs.py c4 --arm ...).
    The reference is not part of this repository: these tests run where a checkout of it is present
    (POINTSEA_REFERENCE, else BASELINE.json's reference_path; build() then builds its CUDA ops into oracle/_ref), and
    skip otherwise.
C5  one cloud of 131072 points: Chamfer (symmetric kernel, 64 A tiles) and FPS -> 16384 (cluster of 16 CTAs)
    against the reference kernels as the CPU oracle restates them (bit-exact to the reference's own outputs in
    tests/golden/), bit-exact.
"""
import hashlib
import json
import os
import os.path as osp
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import REFERENCE, ROOT, load_golden, make_cloud
from oracle import oracle as O

pytestmark = pytest.mark.gpu
REF_TREE = REFERENCE


def _c4(arm, knn, model="svdformer", loss="get_loss", batch=2):
    if not osp.isdir(REF_TREE):
        pytest.skip(f"needs a checkout of the reference at {REF_TREE} (or set POINTSEA_REFERENCE)")
    if not osp.exists(osp.join(ROOT, "oracle", "_ref", "ref_pointnet2_ext.so")):
        pytest.skip("oracle/_ref not built (python __graft_entry__.py build builds it beside a reference checkout)")
    p = subprocess.run([sys.executable, osp.join(ROOT, "tools", "bench_configs.py"), "c4", "--arm", arm, "--knn", knn, "--iters", "1",
                        "--batch", str(batch), "--model", model, "--loss", loss], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, POINTSEA_REFERENCE_TREE=REF_TREE))
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert p.returncode == 0 and lines, (p.stderr or p.stdout)[-3000:]
    d = json.loads(lines[-1])
    assert "loss_hex" in d, d
    return d


def test_c4_svdformer_loss_is_bit_identical_to_the_reference_ops():
    """models/SVDFormer.py + utils/loss_utils.get_loss, B=2, random-init weights (seed 1): our ops through the drop-in
    paths, with and without patch_model_utils (every call site fused), against the reference's CUDA ops."""
    ref = _c4("ref", "torch")
    ours = _c4("ours", "torch")
    fused = _c4("ours", "all")
    assert ours["loss_hex"] == ref["loss_hex"] and ours["losses_hex"] == ref["losses_hex"], (ours["loss"], ref["loss"])
    assert fused["loss_hex"] == ref["loss_hex"] and fused["losses_hex"] == ref["losses_hex"], (fused["loss"], ref["loss"])


def test_c4_get_loss_pm_path_matches_the_reference_ops():
    """utils/loss_utils.get_loss_PM (core/train_55.py:154, core/train_geospec.py:108): the single-sided term included."""
    ref = _c4("ref", "torch", loss="get_loss_PM")
    ours = _c4("ours", "all", loss="get_loss_PM")
    assert ours["loss_hex"] == ref["loss_hex"], (ours["loss"], ref["loss"])


def test_c4_pointsea_imports_and_runs_over_the_dropin():
    """models_PointSea/PointSea.py:3-5 imports gather_operation, model_utils (six pointnet2 names) and chamfer_3DDist
    from the reference's module paths; with torch_scatter stood in by torch.scatter_reduce_ the model runs on our
    ops and its loss equals the reference-ops arm."""
    ref = _c4("ref", "torch", model="pointsea")
    ours = _c4("ours", "torch", model="pointsea")
    assert ours["loss_hex"] == ref["loss_hex"], (ours["loss"], ref["loss"])


def test_c5_chamfer_131072_vs_live_reference():
    """A point's distance and index depend on that point and the other cloud alone, so the oracle's forward runs on a
    fixed sample of 1024 points of each cloud; the backward is checked everywhere."""
    import svdformer_pointsea_b200 as ps
    g = torch.Generator().manual_seed(1234 + 5)
    a, b = make_cloud(g, 1, 131072), make_cloud(g, 1, 131072)
    d1, d2, i1, i2 = ps.chamfer_forward(a.cuda(), b.cuda())
    rows = np.sort(np.random.default_rng(5).choice(131072, 1024, replace=False))
    od1, _, oi1, _ = O.chamfer_fwd(a[:, rows].numpy(), b.numpy())
    od2, _, oi2, _ = O.chamfer_fwd(b[:, rows].numpy(), a.numpy())
    assert np.array_equal(i1[:, rows].cpu().numpy(), oi1) and np.array_equal(i2[:, rows].cpu().numpy(), oi2)
    assert np.array_equal(d1[:, rows].cpu().numpy(), od1) and np.array_equal(d2[:, rows].cpu().numpy(), od2)
    gd1, gd2 = torch.randn(1, 131072, generator=g), torch.randn(1, 131072, generator=g)
    g1, g2 = ps.chamfer_backward(a.cuda(), b.cuda(), gd1.cuda(), gd2.cuda(), i1, i2)
    og1, og2 = O.chamfer_bwd(a.numpy(), b.numpy(), gd1.numpy(), gd2.numpy(), i1.cpu().numpy(), i2.cpu().numpy())
    for x, y in ((g1.cpu().numpy(), og1), (g2.cpu().numpy(), og2)):  # atomics in another order: 1e-5 relative (north star)
        assert np.allclose(x, y, rtol=1e-5, atol=1e-6 * float(np.abs(y).max()))


def test_c5_fps_131072_to_16384_vs_live_reference():
    """The oracle's indices for this input are stored (tests/golden/c5.npz, tests/golden/make_golden_c5.py): FPS over
    131072 points takes the oracle minutes on one core."""
    import svdformer_pointsea_b200 as ps
    z = load_golden("c5")
    g = torch.Generator().manual_seed(1234 + 5)
    xyz = make_cloud(g, 2, 131072, dup=3000, near_origin=40)  # duplicates and origin-skipped points included
    assert hashlib.sha256(xyz.numpy().tobytes()).hexdigest() == str(z["fps.xyz_sha256"]), "the seeded input changed"
    got = ps.furthest_point_sample(xyz.cuda(), 16384)
    assert np.array_equal(got.cpu().numpy(), z["fps.idx"])
