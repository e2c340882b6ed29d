"""BASELINE.json configs 4 and 5 on a B200 (not part of bench.py's contract; results go to profiles/).

C4  full SVDFormer PCN forward + Chamfer loss, random-init weights (seed 1), B=32 split over the
    ranks, the reference's UNMODIFIED models/SVDFormer.py + utils/loss_utils.py on top of
      arm "ours": this repo's ops through the drop-in import paths
      arm "ref" : the reference's own CUDA ops (oracle/_ref/*.so) through the reference's own
                  Python wrappers
    The reference tree is not part of this repository: stage it (git-ignored) with
        cp -r /root/reference baseline/_ref/reference
    before `gpurun`.  Each arm runs in its own process (they bind the same module names).
    PointSea's renderer imports torch_scatter (models_PointSea/mv_utils_zs.py:1,130).  --torch-scatter stub (default)
    stands it in by Tensor.scatter_reduce_ in both arms; --torch-scatter dropin makes the "ours" arm import it through
    install_dropin()'s fallback path (svdformer_pointsea_b200.scatter, the sm_100a scatter-max) instead.
    --loss-impl fused makes the "ours" arm call patch_loss_utils(utils.loss_utils, training=True), so get_loss /
    get_loss_PM run their Chamfer terms on the fused ops; the result reports how many calls reached them.
C5  stress: Chamfer fwd+bwd and FPS 131072 -> 16384 on B=8 clouds of 131072 points (split over the
    ranks), parity against the reference kernels on rank 0, NCCL all-reduce of the loss sums.

usage:  python tools/bench_configs.py c4 [--arm ours|ref|both] [--iters 5] [--model pointsea --torch-scatter stub|dropin]
                                           [--loss-impl composed|fused]
        python tools/bench_configs.py c5
        torchrun --nproc-per-node G tools/bench_configs.py c5      (sharded)
"""
import argparse
import importlib.util
import json
import os
import os.path as osp
import subprocess
import sys
import types

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, ROOT)
REF_TREE = os.environ.get("POINTSEA_REFERENCE_TREE", osp.join(ROOT, "baseline", "_ref", "reference"))
REF_SO = osp.join(ROOT, "oracle", "_ref")

import torch  # noqa: E402


def load_ext(name):
    spec = importlib.util.spec_from_file_location(name, osp.join(REF_SO, name + ".so"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def dist_setup():
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, torch.device("cuda", local)


def ev_time(fn, iters, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


# ------------------------------------------------------------------------------------------- C4
def install_torch_scatter_stub():
    """torch_scatter is a third-party package absent from this image; models_PointSea/mv_utils_zs.py:1,130 uses one
    call, scatter(src, index, dim, out=..., reduce="max").  A torch stand-in (test harness only)."""
    if "torch_scatter" in sys.modules:
        return
    m = types.ModuleType("torch_scatter")

    def scatter(src, index, dim=-1, out=None, dim_size=None, reduce="sum"):
        red = {"max": "amax", "min": "amin", "sum": "sum", "add": "sum", "mean": "mean", "mul": "prod"}[reduce]
        if out is None:
            shape = list(src.shape)
            shape[dim] = int(dim_size if dim_size is not None else index.max().item() + 1)
            out = torch.zeros(shape, device=src.device, dtype=src.dtype)
            return out.scatter_reduce_(dim, index, src, reduce=red, include_self=False)
        return out.scatter_reduce_(dim, index, src, reduce=red, include_self=True)

    m.scatter = scatter
    sys.modules["torch_scatter"] = m


def c4_arm(arm, iters, knn, batch=32, model_name="svdformer", loss_name="get_loss", torch_scatter="stub",
           loss_impl="composed"):
    rank, world, dev = dist_setup()
    if not osp.isdir(REF_TREE):
        print(json.dumps({"config": "C4", "arm": arm, "unavailable": f"{REF_TREE} not staged"}))
        return
    # shims for third-party API drift only (the reference files stay untouched)
    m = types.ModuleType("torchvision.models.utils")
    m.load_state_dict_from_url = torch.hub.load_state_dict_from_url
    sys.modules["torchvision.models.utils"] = m
    if arm == "ours":
        import svdformer_pointsea_b200 as ps
        ps.install_dropin()
        sys.path.append(REF_TREE)
    else:
        import torch.utils.cpp_extension as ce
        ref_ch, ref_pn = load_ext("ref_chamfer_3D"), load_ext("ref_pointnet2_ext")
        real_load = ce.load

        def fake_load(name, *a, **k):  # the reference JIT-builds at import; hand it the prebuilt objects
            if name == "chamfer_3D":
                return ref_ch
            if name == "emd":
                return types.ModuleType("emd")
            return real_load(name, *a, **k)
        ce.load = fake_load
        sys.path.insert(0, osp.join(REF_TREE, "pointnet2_ops_lib"))
        sys.path.insert(0, REF_TREE)
        sys.modules["pointnet2_ops._ext"] = ref_pn
        import pointnet2_ops  # noqa: F401  (binds the reference wrappers to the reference kernels)
        pointnet2_ops._ext = ref_pn
    from types import SimpleNamespace as NS
    if arm != "ours" or torch_scatter == "stub":
        install_torch_scatter_stub()
    # no network on the box: PointSea asks torchvision for ImageNet weights (PointSea.py:40); random init instead
    import torchvision.models as tvm
    _resnet18 = tvm.resnet18
    tvm.resnet18 = lambda *a, weights=None, **k: _resnet18(*a, weights=None, **k)
    if model_name == "pointsea":
        import models_PointSea.model_utils as mu
    else:
        import models.model_utils as mu
    if knn == "ours" and arm == "ours":
        import svdformer_pointsea_b200 as ps
        mu.query_knn = ps.query_knn  # the optional one-line swap of INTEGRATION.md
    if knn == "all" and arm == "ours":
        import svdformer_pointsea_b200 as ps
        ps.patch_model_utils(mu)     # every call-site function (kNN, sample_and_group_knn, EdgeConv front, ...)
    if model_name == "pointsea":
        from models_PointSea.PointSea import Model
    else:
        from models.SVDFormer import Model  # after the patch: it does `from models.model_utils import *`
    import utils.loss_utils as lu
    fused_calls = [0]
    if loss_impl == "fused" and arm == "ours":
        import svdformer_pointsea_b200 as ps
        from svdformer_pointsea_b200 import losses
        ps.patch_loss_utils(lu, training=True)

        def counted(fn):
            def call(*a, **k):
                fused_calls[0] += 1
                return fn(*a, **k)
            return call
        # count the calls that reach the rebound names, so a loss that does not look them up shows 0
        for name in losses.TRAINING_LOSSES:
            setattr(lu, name, counted(getattr(lu, name)))
    if loss_name == "get_loss_PM":
        def get_loss(preds, gt, sqrt=True):
            return lu.get_loss_PM(preds, partial, gt, sqrt=sqrt)
    else:
        get_loss = lu.get_loss
    cfg = NS(NETWORK=NS(step1=4, step2=8, merge_points=512, local_points=512, view_distance=0.7),
             DATASET=NS(TEST_DATASET="ShapeNet"))
    torch.manual_seed(1)
    model = Model(cfg).to(dev)
    model.train()
    B = batch // world
    g = torch.Generator().manual_seed(1234 + 4)
    partial_all = (torch.rand(batch, 2048, 3, generator=g) - 0.5)
    gt_all = (torch.rand(batch, 16384, 3, generator=g) - 0.5)
    partial = partial_all[rank * B:(rank + 1) * B].contiguous().to(dev)
    gt = gt_all[rank * B:(rank + 1) * B].contiguous().to(dev)
    if model_name == "pointsea":
        import models_PointSea.mv_utils_zs as mv
        render = mv.PCViews_Real(TRANS=-cfg.NETWORK.view_distance)
    else:
        render = mu.PCViews(TRANS=-cfg.NETWORK.view_distance, RESOLUTION=224)
    out = {}

    if world > 1 and arm == "ours" and loss_name == "get_loss_PM":
        from svdformer_pointsea_b200.dist import get_loss_PM_sharded

        def get_loss(preds, gt, sqrt=True):  # noqa: F811
            return get_loss_PM_sharded(preds, partial, gt, sqrt=sqrt)
    elif world > 1 and arm == "ours":
        # batch-sharded loss: the reference's get_loss over the GLOBAL batch = local Chamfer terms + ONE all-reduce
        # of their partial sums (svdformer_pointsea_b200.dist.get_loss_sharded), identical on every rank
        from svdformer_pointsea_b200.dist import get_loss_sharded as get_loss  # noqa: F811

    def make_depth():
        img = render.get_img(partial)
        return img if model_name == "pointsea" else torch.unsqueeze(img, 1)

    def step():
        with torch.no_grad():
            depth = make_depth()
            preds = model(partial, depth)
            loss, losses = get_loss(preds, gt, sqrt=True)
        out["loss"], out["losses"] = loss, losses

    ts = ev_time(step, iters)
    # time only the loss (FPS x2 + Chamfer x3), the part the reference runs un-parallelised
    with torch.no_grad():
        depth = make_depth()
        preds = model(partial, depth)
    tl = ev_time(lambda: get_loss(preds, gt, sqrt=True), iters)
    res = {"config": "C4 SVDFormer PCN fwd + Chamfer loss", "arm": arm, "knn": knn if arm == "ours" else "torch",
           "world": world, "B_per_gpu": B, "ms_step_min": round(min(ts), 3), "ms_step_median": round(sorted(ts)[len(ts) // 2], 3),
           "ms_loss_min": round(min(tl), 3), "loss": float(out["loss"]), "losses": [float(x) for x in out["losses"]],
           "loss_hex": float(out["loss"]).hex(), "losses_hex": [float(x).hex() for x in out["losses"]],
           "model": model_name, "loss_fn": loss_name, "batch": batch}
    if loss_impl == "fused" and arm == "ours":
        res["loss_impl"] = "fused"
        res["fused_loss_calls"] = fused_calls[0]
    if "torch_scatter" in sys.modules:  # where PointSea's scatter came from: the stub (no file) or a package
        res["torch_scatter"] = getattr(sys.modules["torch_scatter"], "__file__", None) or "stub"
    if rank == 0:
        print(json.dumps(res))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def c4(args):
    arms = ["ours", "ref"] if args.arm == "both" else [args.arm]
    if args.arm != "both":
        return c4_arm(args.arm, args.iters, args.knn, args.batch, args.model, args.loss, args.torch_scatter,
                      args.loss_impl)
    lines = []
    for arm, knn in (("ours", "torch"), ("ours", "ours"), ("ours", "all"), ("ref", "torch")):
        p = subprocess.run([sys.executable, __file__, "c4", "--arm", arm, "--iters", str(args.iters), "--knn", knn, "--batch", str(args.batch),
                            "--model", args.model, "--loss", args.loss, "--torch-scatter", args.torch_scatter,
                            "--loss-impl", args.loss_impl],
                           capture_output=True, text=True)
        last = [ln for ln in p.stdout.strip().splitlines() if ln.startswith("{")]
        if not last:
            print(json.dumps({"config": "C4", "arm": arm, "error": (p.stderr or p.stdout)[-600:]}))
            continue
        print(last[-1])
        lines.append(json.loads(last[-1]))
    ours = [x for x in lines if x.get("arm") == "ours" and x.get("knn") == "torch" and "loss" in x]
    ref = [x for x in lines if x.get("arm") == "ref" and "loss" in x]
    if ours and ref:
        rel = abs(ours[0]["loss"] - ref[0]["loss"]) / abs(ref[0]["loss"])
        print(json.dumps({"config": "C4", "loss_rel_diff_ours_vs_ref": rel, "speedup_step": ref[0]["ms_step_min"] / ours[0]["ms_step_min"],
                          "speedup_loss": ref[0]["ms_loss_min"] / ours[0]["ms_loss_min"]}))


# ------------------------------------------------------------------------------------------- C5
def c5(args):
    import svdformer_pointsea_b200 as ps
    from svdformer_pointsea_b200.dist import LossSums, chamfer_loss_terms, combine_chamfer
    rank, world, dev = dist_setup()
    Btot, N, npoint = 8, 131072, 16384
    B = Btot // world
    g = torch.Generator().manual_seed(1234 + 5)
    a_all = (torch.rand(Btot, N, 3, generator=g) - 0.5)
    b_all = (torch.rand(Btot, N, 3, generator=g) - 0.5)
    a = a_all[rank * B:(rank + 1) * B].contiguous().to(dev)
    b = b_all[rank * B:(rank + 1) * B].contiguous().to(dev)
    gd = torch.ones(B, N, device=dev) / N
    hold = {}

    def chamfer_step():
        d1, d2, i1, i2 = ps.chamfer_forward(a, b)
        sums = LossSums(dev)
        chamfer_loss_terms(sums, "cd", d1, d2, sqrt=True)
        hold["loss"] = combine_chamfer(sums.reduce(), "cd", True)
        hold["g"] = ps.chamfer_backward(a, b, gd, gd, i1, i2)
        hold["out"] = (d1, d2, i1, i2)

    tc = ev_time(chamfer_step, args.iters, warm=1)
    tf = ev_time(lambda: hold.__setitem__("fps", ps.furthest_point_sample(a, npoint)), args.iters, warm=1)
    res = {"config": "C5 stress B=8 N=131072", "world": world, "B_per_gpu": B,
           "chamfer_fwd_bwd_ms": round(min(tc), 3), "chamfer_gpair_per_s_whole_job": round(2.0 * Btot * N * N / (min(tc) * 1e-3) / 1e9, 1),
           "fps_ms": round(min(tf), 3), "fps_sampled_pts_per_s_whole_job": round(Btot * npoint / (min(tf) * 1e-3), 1),
           "fps_us_per_iteration": round(min(tf) * 1e3 / (npoint - 1), 4), "loss": float(hold["loss"])}
    if rank == 0 and osp.exists(osp.join(REF_SO, "ref_chamfer_3D.so")) and not args.no_check:
        ref_ch, ref_pn = load_ext("ref_chamfer_3D"), load_ext("ref_pointnet2_ext")
        d1, d2, i1, i2 = hold["out"]
        r = [torch.zeros_like(d1), torch.zeros_like(d2), torch.zeros_like(i1), torch.zeros_like(i2)]
        tr = ev_time(lambda: ref_ch.forward(a, b, *r), 1, warm=0)
        res["parity_chamfer_idx_exact"] = bool(torch.equal(i1, r[2]) and torch.equal(i2, r[3]))
        res["parity_chamfer_dist_exact"] = bool(torch.equal(d1, r[0]) and torch.equal(d2, r[1]))
        res["ref_cuda_chamfer_fwd_ms"] = round(tr[0], 2)
        t0 = ev_time(lambda: hold.__setitem__("rfps", ref_pn.furthest_point_sampling(a, npoint)), 1, warm=0)
        res["parity_fps_exact"] = bool(torch.equal(hold["fps"], hold["rfps"]))
        res["ref_cuda_fps_ms"] = round(t0[0], 2)
    if rank == 0:
        print(json.dumps(res))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("config", choices=["c4", "c5"])
    ap.add_argument("--arm", default="both", choices=["ours", "ref", "both"])
    ap.add_argument("--knn", default="torch", choices=["torch", "ours", "all"])
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--batch", type=int, default=32, help="c4: total clouds")
    ap.add_argument("--model", default="svdformer", choices=["svdformer", "pointsea"])
    ap.add_argument("--loss", default="get_loss", choices=["get_loss", "get_loss_PM"])
    ap.add_argument("--torch-scatter", default="stub", choices=["stub", "dropin"],
                    help="c4 pointsea: arm ours imports torch_scatter from the drop-in instead of the stand-in")
    ap.add_argument("--loss-impl", default="composed", choices=["composed", "fused"],
                    help="c4: arm ours runs utils/loss_utils' Chamfer losses on the fused ops (patch_loss_utils training=True)")
    a = ap.parse_args()
    {"c4": c4, "c5": c5}[a.config](a)
