"""Fused Chamfer training losses against the composition they replace: python tools/chamfer_loss_time.py [--out PATH]

composed: chamfer_3DFunction + the torch expression of utils/loss_utils.py:10-31, backward through torch's autograd
fused:    svdformer_pointsea_b200.losses (ps_chamfer_loss_fwd / ps_chamfer_loss_bwd)
Times are forward + backward, eager, median of 21 with the L2 cache overwritten before each, CUDA events, the two arms
taking turns; *_fwd_ms is the forward alone under no_grad.  The ground truth does not require grad.  Shapes: the three terms get_loss runs at B = 32 (prediction vs thinned ground truth,
as tools/c4loss_time.py) and get_loss_PM's partial-matching term (partial 2048, which does not require grad, vs the
16384-point prediction), every kind at each; then a whole get_loss (sqrt=True: the FPS chain plus three terms, as
tests/test_dist_gloo.py:214-232 restates it) at B = 32 and B = 4.  Kernels per call come from a separate
torch.profiler run.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os.path as osp
import subprocess
import sys

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import svdformer_pointsea_b200 as ps  # noqa: E402
from svdformer_pointsea_b200 import losses  # noqa: E402
from svdformer_pointsea_b200.pointnet2_utils import fps_subsample  # noqa: E402

dev = torch.device("cuda:0")
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
KINDS = ["cd", "cd_sqrt", "single", "single_sqrt"]
FUSED = {"cd": losses.chamfer, "cd_sqrt": losses.chamfer_sqrt, "single": losses.chamfer_single_side,
         "single_sqrt": losses.chamfer_single_side_sqrt}


def composed(kind):
    def f(p1, p2):
        d1, d2, _, _ = ps.chamfer_3DFunction.apply(p1.contiguous(), p2.contiguous())
        if kind == "cd":
            return torch.mean(d1) + torch.mean(d2)
        if kind == "cd_sqrt":
            return (torch.mean(torch.sqrt(d1)) + torch.mean(torch.sqrt(d2))) / 2
        if kind == "single":
            return torch.mean(d1)
        return torch.mean(torch.sqrt(d1))
    return f


def timed(fns, n=21, warm=3):
    """Median ms of each function; the functions take turns, so drift on the shared host hits them alike."""
    for _ in range(warm):
        for fn in fns:
            fn()
    torch.cuda.synchronize()
    ts = [[] for _ in fns]
    for _ in range(n):
        for fn, t in zip(fns, ts):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize(); t.append(e0.elapsed_time(e1))
    return [round(sorted(t)[n // 2], 4) for t in ts]


def kernels(fn):
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return sum(1 for nm in names if not nm.startswith(("Memcpy", "Memset")))


def step(loss_fn, leaves):
    def run():
        loss_fn().backward()
        for t in leaves:
            t.grad = None
    return run


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=osp.join(osp.dirname(osp.dirname(osp.abspath(__file__))), "profiles", "chamfer_loss.jsonl"))
    args = ap.parse_args()
    rows = [{"gpu": gpu_info(), "torch": torch.__version__,
             "timing": "fwd+bwd eager, median of 21, arms alternated, L2 overwritten, CUDA events"}]
    g = torch.Generator().manual_seed(1238)
    B = 32
    # (term, N, M, which cloud requires grad): get_loss's cdc / cd1 / cd2 and get_loss_PM's pm
    terms = [("cdc", 512, 512, 0), ("cd1", 2048, 2048, 0), ("cd2", 16384, 16384, 0), ("pm", 2048, 16384, 1)]
    for term, N, M, grad_side in terms:
        clouds = [(torch.rand(B, n, 3, generator=g) - 0.5).to(dev) for n in (N, M)]
        clouds[grad_side].requires_grad_(True)
        leaf = [clouds[grad_side]]
        for kind in KINDS:
            row = {"term": term, "B": B, "N": N, "M": M, "grad": "xyz%d" % (grad_side + 1), "kind": kind}
            runs = [step(lambda fn=fn: fn(*clouds), leaf) for fn in (composed(kind), FUSED[kind])]
            row["composed_ms"], row["fused_ms"] = timed(runs)
            row["composed_kernels"], row["fused_kernels"] = kernels(runs[0]), kernels(runs[1])
            row["speedup"] = round(row["composed_ms"] / row["fused_ms"], 3)

            def fwd_only(fn):
                def run():
                    with torch.no_grad():
                        fn(*clouds)
                return run
            row["composed_fwd_ms"], row["fused_fwd_ms"] = timed([fwd_only(composed(kind)), fwd_only(FUSED[kind])])
            rows.append(row)
            print(json.dumps(row), flush=True)
    for B in (32, 4):
        gt = (torch.rand(B, 16384, 3, generator=g) - 0.5).to(dev)
        preds = [(torch.rand(B, n, 3, generator=g) - 0.5).to(dev).requires_grad_(True) for n in (512, 2048, 16384)]

        def get_loss(cd):
            Pc, P1, P2 = preds
            gt_1 = fps_subsample(gt, P1.shape[1])
            gt_c = fps_subsample(gt_1, Pc.shape[1])
            return cd(Pc, gt_c) + cd(P1, gt_1) + cd(P2, gt)

        row = {"term": "get_loss sqrt=True", "B": B}
        runs = [step(lambda cd=cd: get_loss(cd), preds) for cd in (composed("cd_sqrt"), losses.chamfer_sqrt)]
        row["composed_ms"], row["fused_ms"] = timed(runs)
        row["composed_kernels"], row["fused_kernels"] = kernels(runs[0]), kernels(runs[1])
        row["speedup"] = round(row["composed_ms"] / row["fused_ms"], 3)
        rows.append(row)
        print(json.dumps(row), flush=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
