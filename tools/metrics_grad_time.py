"""Forward + backward of the differentiable calc_dcd / calc_cd against the reference's torch expressions over the
Chamfer drop-in (what a user has without ps_chamfer_metrics_bwd), and ps_chamfer_metrics_bwd alone.

    python tools/metrics_grad_time.py [--iters 100] [--out profiles/metrics_grad.jsonl]

B = 32; 16384 vs 16384 (PCN: gt vs P2) and 2048 vs 16384.  CUDA events around each call, a 256 MB buffer
overwritten between calls (outside the events) so that no input is served from L2, 10 warm-up calls, the arms of
one configuration alternated call by call, median (and 10th / 90th percentiles) of --iters calls.  Both arms' losses
and gradients are checked against each other (1e-5 relative) before anything is timed.  The first line names the
device, its power limit and its maximum SM clock.
"""
import argparse
import json
import os.path as osp
import sys

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import svdformer_pointsea_b200 as ps  # noqa: E402
from oracle import oracle as O  # noqa: E402

DEV = torch.device("cuda:0")


def device_line():
    info = {"device": torch.cuda.get_device_name(DEV), "torch": torch.__version__}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(DEV.index or 0)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:  # the numbers are still written, marked as lacking the power limit
        info["power_limit_w"] = None
        info["nvml_error"] = str(e)
    return info


def ref_dcd_loss(x, gt):
    """utils/loss_utils.py:117-155 over chamfer_3DFunction: cham_loss(gt, x), then the reference's expressions."""
    d1, d2, i1, i2 = ps.chamfer_3DFunction.apply(gt, x)
    return O.torch_dcd_from_raw(d1, d2, i1, i2, x.shape[1], gt.shape[1]).mean()


def ref_cd_loss(x, gt):
    d1, d2, _, _ = ps.chamfer_3DFunction.apply(gt, x)
    return O.torch_cd_terms(d1, d2)[0].mean()


def step(loss_fn, x, gt):
    x.grad = None
    loss = loss_fn(x, gt)
    loss.backward()
    return loss.detach(), x.grad


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def time_arms(arms, iters, flush, warm=10):
    for _ in range(warm):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in arms}
    for _ in range(iters):
        for k, fn in arms.items():
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts[k].append(e0.elapsed_time(e1))
    return {k: {"ms_median": round(float(np.median(v)), 4), "ms_p10": round(float(np.percentile(v, 10)), 4),
                "ms_p90": round(float(np.percentile(v, 90)), 4), "iters": iters} for k, v in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    args = ap.parse_args()
    if args.iters < 50:
        ap.error("--iters must be at least 50")
    lines = [device_line()]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    B = 32
    for n_x, n_gt in ((16384, 16384), (2048, 16384)):
        g = torch.Generator().manual_seed(n_x + n_gt)
        gt = (torch.rand(B, n_gt, 3, generator=g) - 0.5).to(DEV)
        x = (gt[:, torch.randperm(n_gt, generator=g)[:n_x]] + 0.004 * torch.randn(B, n_x, 3, generator=g).to(DEV))
        x = x.contiguous().requires_grad_(True)
        cfg = {"B": B, "n_x": n_x, "n_gt": n_gt}
        dcd_ours = lambda a, b: ps.calc_dcd(a, b)[0].mean()  # noqa: E731
        cd_ours = lambda a, b: ps.calc_cd(a, b)[0].mean()  # noqa: E731
        for what, ours, ref in (("calc_dcd(x, gt)[0].mean() fwd+bwd", dcd_ours, ref_dcd_loss),
                                ("calc_cd(x, gt)[0].mean() fwd+bwd", cd_ours, ref_cd_loss)):
            lo, go = (t.clone() for t in step(ours, x, gt))
            lr, gr = (t.clone() for t in step(ref, x, gt))
            check = {"loss_rel": rel(lo, lr), "grad_rel": rel(go, gr)}
            assert check["loss_rel"] < 1e-5 and check["grad_rel"] < 1e-5, (what, check)
            t = time_arms({"ours": lambda: step(ours, x, gt), "reference": lambda: step(ref, x, gt)}, args.iters, flush)
            lines.append({**cfg, "what": what, "ours": t["ours"], "reference_torch_over_chamfer_dropin": t["reference"],
                          "speedup": round(t["reference"]["ms_median"] / t["ours"]["ms_median"], 2), "check": check})
        # the new kernel alone, every term present (histograms rebuilt) and without the dcd term (no histograms)
        with torch.no_grad():
            d1, d2, i1, i2 = ps.chamfer_forward(gt, x.detach())
            gcoef = torch.rand(B, 5, generator=g).to(DEV)
            graw1, graw2 = torch.randn(B, n_gt, generator=g).to(DEV), torch.randn(B, n_x, generator=g).to(DEV)
        fr1, fr2 = n_gt / n_x, n_x / n_gt
        kern = {"terms=31": lambda: ps.chamfer_metrics_grad_raw(d1, d2, i1, i2, gcoef, 31, frac1=fr1, frac2=fr2),
                "terms=15": lambda: ps.chamfer_metrics_grad_raw(d1, d2, i1, i2, gcoef, 15, frac1=fr1, frac2=fr2),
                "terms=31+raw": lambda: ps.chamfer_metrics_grad_raw(d1, d2, i1, i2, gcoef, 31, graw1, graw2, frac1=fr1,
                                                                    frac2=fr2)}
        t = time_arms(kern, args.iters, flush)
        pts = B * (n_x + n_gt)
        bytes_ = {"terms=31": pts * 16, "terms=15": pts * 8, "terms=31+raw": pts * 20}  # idx x2, dist, graddist (+ graw)
        for k, v in t.items():
            lines.append({**cfg, "what": f"ps_chamfer_metrics_bwd alone, {k}", **v, "bytes": bytes_[k],
                          "GB_per_s": round(bytes_[k] / (v["ms_median"] * 1e-3) / 1e9, 1)})
    for line in lines:
        print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
