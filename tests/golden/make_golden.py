"""Generate tests/golden/*.npz from the REFERENCE's own CUDA ops (oracle/_ref) on a B200.

Needs oracle/_ref/*.so (oracle/build_ref.py builds them from a checkout of the reference) and a B200:
    python tests/golden/make_golden.py OUT_DIR
then copy OUT_DIR/*.npz into tests/golden/ and commit them.

Every case stores its seeded inputs next to the reference outputs, so the fixtures are
self-contained.  kNN has no reference kernel: its golden output is the reference's torch
expression (models/model_utils.py:258-286, restated in oracle.torch_knn) evaluated by torch on
the same GPU (cuBLAS + torch sort), plus the raw distance rows for the arithmetic study.
"""
import importlib.util
import os
import os.path as osp
import sys

import numpy as np
import torch

ROOT = osp.dirname(osp.dirname(osp.dirname(osp.abspath(__file__))))
sys.path.insert(0, ROOT)
REF_DIR = osp.join(ROOT, "oracle", "_ref")


def load_ext(name):
    path = osp.join(REF_DIR, name + ".so")
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cloud(g, B, N, dup=0, near_origin=0):
    """rand-0.5 cloud; `dup` > 0 pads by duplicating points the way UpSamplePoints does
    (utils/data_transforms.py:153-172); `near_origin` plants points inside the FPS skip ball."""
    x = torch.rand(B, N, 3, generator=g) - 0.5
    if dup:
        uniq = N - dup
        for b in range(B):
            src = torch.randint(0, uniq, (dup,), generator=g)
            x[b, uniq:] = x[b, src]
    if near_origin:
        for b in range(B):
            pos = torch.randperm(N, generator=g)[:near_origin]
            x[b, pos] = (torch.rand(near_origin, 3, generator=g) - 0.5) * 0.03
    return x.contiguous()


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    ch = load_ext("ref_chamfer_3D")
    pn = load_ext("ref_pointnet2_ext")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    # ---- Chamfer forward + backward (chamfer3D.cu) ------------------------------------------
    cases = {}
    g = torch.Generator().manual_seed(1234 + 1)
    for name, (B, N, M, dup) in {"small": (3, 300, 700, 0), "tiles": (2, 1024, 1537, 0),
                                 "dups": (2, 512, 640, 200), "tiny": (1, 1, 5, 0)}.items():
        a, b = cloud(g, B, N, dup=min(dup, N - 1) if dup else 0), cloud(g, B, M, dup=dup)
        if dup:  # make the two clouds share exact points too (zero distances, cross-cloud ties)
            b[:, :100] = a[:, :100]
        gd1, gd2 = torch.randn(B, N, generator=g), torch.randn(B, M, generator=g)
        A, Bc = a.to(dev), b.to(dev)
        d1 = torch.zeros(B, N, device=dev); d2 = torch.zeros(B, M, device=dev)
        i1 = torch.zeros(B, N, device=dev, dtype=torch.int32); i2 = torch.zeros(B, M, device=dev, dtype=torch.int32)
        ch.forward(A, Bc, d1, d2, i1, i2)
        g1 = torch.zeros(B, N, 3, device=dev); g2 = torch.zeros(B, M, 3, device=dev)
        ch.backward(A, Bc, g1, g2, gd1.to(dev), gd2.to(dev), i1, i2)
        torch.cuda.synchronize()
        for k, v in dict(xyz1=a, xyz2=b, gd1=gd1, gd2=gd2, dist1=d1, dist2=d2, idx1=i1, idx2=i2, g1=g1, g2=g2).items():
            cases[f"{name}.{k}"] = v.cpu().numpy()
    np.savez_compressed(osp.join(out_dir, "chamfer.npz"), **cases)

    # ---- FPS (sampling_gpu.cu) --------------------------------------------------------------
    cases = {}
    g = torch.Generator().manual_seed(1234 + 2)
    for name, (B, N, npoint, dup, no) in {"n1000": (3, 1000, 128, 0, 0), "dups2048": (2, 2048, 512, 548, 0),
                                          "bs256": (2, 300, 64, 0, 2), "origin": (2, 5000, 200, 0, 40),
                                          "n16384": (1, 16384, 256, 0, 3), "npow2": (2, 512, 512, 100, 1),
                                          "tiny": (2, 7, 7, 0, 0)}.items():
        x = cloud(g, B, N, dup=dup, near_origin=no)
        idx = pn.furthest_point_sampling(x.to(dev), npoint)
        torch.cuda.synchronize()
        cases[f"{name}.xyz"] = x.numpy()
        cases[f"{name}.idx"] = idx.cpu().numpy()
    np.savez_compressed(osp.join(out_dir, "fps.npz"), **cases)

    # ---- gather / group / ball query / 3-NN / interpolate -----------------------------------
    cases = {}
    g = torch.Generator().manual_seed(1234 + 3)
    B, C, N, M = 2, 5, 333, 77
    feat = torch.randn(B, C, N, generator=g)
    idx = torch.randint(0, N, (B, M), generator=g, dtype=torch.int32)
    go = torch.randn(B, C, M, generator=g)
    cases.update({"gather.feat": feat.numpy(), "gather.idx": idx.numpy(), "gather.go": go.numpy(),
                  "gather.out": pn.gather_points(feat.to(dev), idx.to(dev)).cpu().numpy(),
                  "gather.grad": pn.gather_points_grad(go.to(dev), idx.to(dev), N).cpu().numpy()})
    B, C, N, S, K = 2, 6, 256, 64, 16
    feat = torch.randn(B, C, N, generator=g)
    idx = torch.randint(0, N, (B, S, K), generator=g, dtype=torch.int32)
    go = torch.randn(B, C, S, K, generator=g)
    cases.update({"group.feat": feat.numpy(), "group.idx": idx.numpy(), "group.go": go.numpy(),
                  "group.out": pn.group_points(feat.to(dev), idx.to(dev)).cpu().numpy(),
                  "group.grad": pn.group_points_grad(go.to(dev), idx.to(dev), N).cpu().numpy()})
    B, N, S = 2, 700, 96
    xyz, new_xyz = cloud(g, B, N), cloud(g, B, S)
    for r, ns in ((0.2, 16), (0.05, 8), (0.6, 32)):
        out = pn.ball_query(new_xyz.to(dev), xyz.to(dev), r, ns)
        cases[f"ball.r{r}.ns{ns}.idx"] = out.cpu().numpy()
    cases.update({"ball.xyz": xyz.numpy(), "ball.new_xyz": new_xyz.numpy()})
    B, n, m, C = 2, 150, 64, 7
    unknown, known = cloud(g, B, n), cloud(g, B, m, dup=10)
    d2, ix = pn.three_nn(unknown.to(dev), known.to(dev))
    w = torch.rand(B, n, 3, generator=g)
    w = w / w.sum(-1, keepdim=True)
    pts = torch.randn(B, C, m, generator=g)
    go = torch.randn(B, C, n, generator=g)
    cases.update({"three.unknown": unknown.numpy(), "three.known": known.numpy(), "three.dist2": d2.cpu().numpy(),
                  "three.idx": ix.cpu().numpy(), "three.weight": w.numpy(), "three.points": pts.numpy(),
                  "three.go": go.numpy(),
                  "three.out": pn.three_interpolate(pts.to(dev), ix, w.to(dev)).cpu().numpy(),
                  "three.grad": pn.three_interpolate_grad(go.to(dev), ix, w.to(dev), m).cpu().numpy()})
    torch.cuda.synchronize()
    np.savez_compressed(osp.join(out_dir, "pointnet2.npz"), **cases)

    # ---- kNN: the reference's torch expression on this GPU ------------------------------------
    from oracle import oracle as O
    cases = {}
    g = torch.Generator().manual_seed(1234 + 4)
    torch.backends.cuda.matmul.allow_tf32 = False  # torch default; stated for the record
    for name, (B, N, S, k, dup, inc) in {"k16": (2, 2048, 512, 16, 0, True), "dups": (2, 1024, 256, 16, 300, True),
                                         "noself": (2, 512, 512, 8, 0, False), "small": (1, 100, 40, 20, 0, True),
                                         "k40": (1, 600, 64, 40, 0, True)}.items():
        xyz = cloud(g, B, N, dup=dup)
        new_xyz = xyz[:, :S].contiguous() if name in ("noself", "dups") else cloud(g, B, S)
        X, Q = xyz.to(dev), new_xyz.to(dev)
        idx = O.torch_knn(k, X, Q, include_self=inc)
        dist = -2 * torch.matmul(Q, X.permute(0, 2, 1))
        dist += torch.sum(Q ** 2, -1).view(B, S, 1)
        dist += torch.sum(X ** 2, -1).view(B, 1, N)
        torch.cuda.synchronize()
        cases[f"{name}.xyz"] = xyz.numpy()
        cases[f"{name}.new_xyz"] = new_xyz.numpy()
        cases[f"{name}.idx"] = idx.cpu().numpy()
        cases[f"{name}.k"] = np.int32(k)
        cases[f"{name}.include_self"] = np.int32(inc)
        if name in ("small", "dups"):
            rows = slice(None)
            if name == "dups":  # a seeded sample of 8 query rows keeps the file small
                cases[f"{name}.rows"] = np.sort(np.random.default_rng(0).choice(S, 8, replace=False)).astype(np.int32)
                rows = torch.as_tensor(cases[f"{name}.rows"], dtype=torch.long, device=dev)
            cases[f"{name}.dist"] = dist[:, rows].cpu().numpy()
            cases[f"{name}.dot"] = torch.matmul(Q, X.permute(0, 2, 1))[:, rows].cpu().numpy()
            cases[f"{name}.qq"] = torch.sum(Q ** 2, -1).cpu().numpy()
    np.savez_compressed(osp.join(out_dir, "knn.npz"), **cases)
    print("golden vectors written to", out_dir, "| torch", torch.__version__, "| gpu", torch.cuda.get_device_name(0))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else osp.join(ROOT, "gpurun_out", "golden"))
