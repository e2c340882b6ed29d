"""Golden vectors for the SURVEY 8(f) "next" rows, generated on a B200 from the reference's own
CUDA ops (oracle/_ref) combined by the reference's torch expressions (restated in oracle/oracle.py
with file:line citations; tests/test_reference_python.py checks those restatements against the
reference's Python wherever a checkout of it is present).

    python tests/golden/make_golden_next.py OUT_DIR

  next.npz            committed fixture: sample_and_group_knn, EdgeConv edge features (C=3 and
                      feature space), calc_cd / fscore / calc_dcd
  featknn_study.npz   scratch (not committed): raw matmul / sum rows for the arithmetic study of
                      the feature-space kNN (cuBLAS K=64/256 accumulation, torch row sums)
"""
import os
import os.path as osp
import sys

import numpy as np
import torch

ROOT = osp.dirname(osp.dirname(osp.dirname(osp.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, osp.dirname(osp.abspath(__file__)))
from make_golden import cloud, load_ext  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    ch = load_ext("ref_chamfer_3D")
    pn = load_ext("ref_pointnet2_ext")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    cases = {}

    # ---- sample_and_group_knn (models/model_utils.py:322-358) -----------------------------------
    g = torch.Generator().manual_seed(1234 + 11)
    for name, (B, N, npoint, k, f, dup) in {"sg": (2, 512, 128, 16, 5, 0), "sgdup": (2, 600, 64, 8, 0, 150)}.items():
        xyz_f = cloud(g, B, N, dup=dup)                       # (B,N,3)
        xyz = xyz_f.permute(0, 2, 1).contiguous().to(dev)     # (B,3,N)
        pts = torch.randn(B, f, N, generator=g).to(dev) if f else None
        xyz_flipped = xyz.permute(0, 2, 1).contiguous()
        fidx = pn.furthest_point_sampling(xyz_flipped, npoint)
        new_xyz = pn.gather_points(xyz, fidx)
        idx = O.torch_knn(k, xyz_flipped, new_xyz.permute(0, 2, 1).contiguous())
        grouped_xyz = pn.group_points(xyz, idx)
        grouped_xyz -= new_xyz.unsqueeze(3).repeat(1, 1, 1, k)
        new_points = torch.cat([grouped_xyz, pn.group_points(pts, idx)], 1) if f else grouped_xyz
        cases.update({f"{name}.xyz": xyz.cpu().numpy(), f"{name}.npoint": np.int32(npoint), f"{name}.k": np.int32(k),
                      f"{name}.new_xyz": new_xyz.cpu().numpy(), f"{name}.idx": idx.cpu().numpy(),
                      f"{name}.grouped_xyz": grouped_xyz.cpu().numpy(), f"{name}.new_points": new_points.cpu().numpy()})
        if f:
            cases[f"{name}.points"] = pts.cpu().numpy()

    # ---- EdgeConv front (models/model_utils.py:807-826, 869-877) --------------------------------
    study = {}
    g = torch.Generator().manual_seed(1234 + 12)
    for name, (B, C, N, k, dup) in {"edge3": (2, 3, 1024, 16, 0), "edge3dup": (2, 3, 700, 16, 200),
                                    "edge64": (2, 64, 512, 8, 0), "edge256": (1, 256, 512, 4, 0),
                                    "edge64post": (2, 64, 384, 8, 0)}.items():
        if C == 3:
            x = cloud(g, B, N, dup=dup).permute(0, 2, 1).contiguous()
        else:
            x = torch.randn(B, C, N, generator=g)
            if name.endswith("post"):  # post-activation-like features: non-negative, many exact zeros
                x = torch.relu(x)
        X = x.to(dev)
        feat, idx = O.torch_edge_features(X, k)
        torch.cuda.synchronize()
        cases.update({f"{name}.k": np.int32(k), f"{name}.idx": idx.int().cpu().numpy()})
        if name != "edge256":  # 0.5 MB of noise: tests/conftest.py redraws it from this seed sequence
            cases[f"{name}.x"] = x.numpy()
        if N * k * C <= 200000:
            cases[f"{name}.feat"] = feat.cpu().numpy()
        xt = X.transpose(2, 1).contiguous()
        study[f"{name}.x"] = x.numpy()
        study[f"{name}.idx"] = idx.int().cpu().numpy()
        study[f"{name}.dot"] = torch.matmul(xt, xt.permute(0, 2, 1))[:, :64].cpu().numpy()
        study[f"{name}.m2dot"] = (-2 * torch.matmul(xt, xt.permute(0, 2, 1)))[:, :64].cpu().numpy()
        study[f"{name}.sumsq"] = torch.sum(xt ** 2, -1).cpu().numpy()
        study[f"{name}.dist"] = O.torch_square_distance(xt, xt)[:, :64].cpu().numpy()
        vals, _ = O.torch_square_distance(xt, xt).topk(k, largest=False)
        study[f"{name}.topk_vals"] = vals.cpu().numpy()

    # ---- calc_cd / fscore / calc_dcd (utils/loss_utils.py:98-155, metrics/CD/fscore.py) ---------
    g = torch.Generator().manual_seed(1234 + 13)
    for name, (B, n_x, n_gt, dup, scale) in {"dcd": (3, 512, 700, 0, 1.0), "dcddup": (2, 640, 512, 200, 1.0),
                                             "dcdnear": (2, 400, 400, 0, 0.02)}.items():
        gt = cloud(g, B, n_gt, dup=dup)
        x = cloud(g, B, n_x, dup=min(dup, n_x - 1) if dup else 0)
        if name == "dcdnear":  # prediction = gt + small noise, so exp(-alpha d) and the F-score are non-trivial
            x = gt + scale * 0.1 * torch.randn(B, n_gt, 3, generator=g)
        X, GT = x.to(dev), gt.to(dev)
        n_x_, n_gt_ = X.shape[1], GT.shape[1]
        # calc_dcd -> calc_cd(x, gt): cham_loss(gt=x_arg, output=gt_arg): first argument of calc_cd is `output`
        # calc_cd(output, gt) calls cham_loss(gt, output) (utils/loss_utils.py:101); calc_dcd passes (x, gt) as
        # (output, gt), so dist1/idx1 are per gt point and dist2/idx2 per x point (:136-139)
        d1 = torch.zeros(B, n_gt_, device=dev); d2 = torch.zeros(B, n_x_, device=dev)
        i1 = torch.zeros(B, n_gt_, device=dev, dtype=torch.int32); i2 = torch.zeros(B, n_x_, device=dev, dtype=torch.int32)
        ch.forward(GT, X, d1, d2, i1, i2)
        cd_p, cd_t = O.torch_cd_terms(d1, d2)
        f1, p1, p2 = O.torch_fscore(d1, d2)
        f1b, _, _ = O.torch_fscore(d1, d2, threshold=0.01)
        dcd = O.torch_dcd_from_raw(d1, d2, i1, i2, n_x_, n_gt_)
        dcd_nr = O.torch_dcd_from_raw(d1, d2, i1, i2, n_x_, n_gt_, alpha=40, n_lambda=0.5, non_reg=True)
        torch.cuda.synchronize()
        cases.update({f"{name}.x": x.numpy(), f"{name}.gt": gt.numpy(), f"{name}.dist1": d1.cpu().numpy(),
                      f"{name}.dist2": d2.cpu().numpy(), f"{name}.idx1": i1.cpu().numpy(), f"{name}.idx2": i2.cpu().numpy(),
                      f"{name}.cd_p": cd_p.cpu().numpy(), f"{name}.cd_t": cd_t.cpu().numpy(), f"{name}.f1": f1.cpu().numpy(),
                      f"{name}.p1": p1.cpu().numpy(), f"{name}.p2": p2.cpu().numpy(), f"{name}.f1_t01": f1b.cpu().numpy(),
                      f"{name}.dcd": dcd.cpu().numpy(), f"{name}.dcd_nonreg": dcd_nr.cpu().numpy()})
    np.savez_compressed(osp.join(out_dir, "next.npz"), **cases)
    np.savez_compressed(osp.join(out_dir, "featknn_study.npz"), **study)
    print("next-row golden vectors written to", out_dir, "| torch", torch.__version__, "| gpu", torch.cuda.get_device_name(0))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else osp.join(ROOT, "gpurun_out", "golden"))
