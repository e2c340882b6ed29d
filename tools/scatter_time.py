"""PointSea's depth-map scatter-max (models_PointSea/mv_utils_zs.py:130) on ps_scatter_max against torch's own
`out.scatter_reduce_(dim, index, src, "amax", include_self=True)` on the same GPU.

    python tools/scatter_time.py [--iters 200] [--out profiles/scatter_max.jsonl]

Shapes: src (32*3, P) depths into out (96, 224*224) pre-filled with zeros, P = 2048 and 16384, with the pixel index
uniform over the image, clustered into a 40x40 patch (a projected partial cloud) and all on one pixel (the worst
case of contention).  Arms: ours (values only, what a call under no_grad runs), ours with the argmax pass (what a call
with a src that requires grad runs) and torch.  Before timing, each arm's output is checked bit for bit against
torch's.  CUDA events around each call, a 256 MB buffer overwritten between calls (outside the events) so that no
input is served from L2, 10 warm-up calls, the arms alternated call by call, median (and 10th / 90th percentiles) of
--iters calls.  The first line names the device, its power limit and its maximum SM clock.
"""
import argparse
import json
import os.path as osp
import sys

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from svdformer_pointsea_b200.scatter import _scatter_max, scatter  # noqa: E402

DEV = torch.device("cuda:0")
B, H = 96, 224


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


def make_inputs(points, pattern, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed + points)
    src = torch.rand(B, points, generator=g, device=DEV) * 2.0
    if pattern == "uniform":
        index = torch.randint(0, H * H, (B, points), generator=g, device=DEV)
    elif pattern == "patch40":
        y = torch.randint(92, 132, (B, points), generator=g, device=DEV)
        x = torch.randint(92, 132, (B, points), generator=g, device=DEV)
        index = y * H + x
    else:
        index = torch.full((B, points), H * H // 2 + H // 2, dtype=torch.int64, device=DEV)
    return src, index


def arms(src, index):
    """name -> call; every call updates its own zero-filled output in place (max is idempotent, so repeated calls
    leave the same values)."""
    outs = {k: torch.zeros(B, H * H, device=DEV) for k in ("ours", "ours_argmax", "torch")}
    return outs, {
        "ours": lambda: scatter(src, index, 1, out=outs["ours"], reduce="max"),
        "ours_argmax": lambda: _scatter_max(src, index, 1, outs["ours_argmax"], None, True),
        "torch": lambda: outs["torch"].scatter_reduce_(1, index, src, "amax", include_self=True),
    }


def time_arms(fns, iters, flush, warm=10):
    for _ in range(warm):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(iters):
        for k, fn in fns.items():
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
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    args = ap.parse_args()
    if args.iters < 100:
        ap.error("--iters must be at least 100")
    lines = [device_line()]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    for points in (2048, 16384):
        for pattern in ("uniform", "patch40", "one_pixel"):
            src, index = make_inputs(points, pattern)
            outs, fns = arms(src, index)
            for fn in fns.values():
                fn()
            for k in ("ours", "ours_argmax"):
                assert torch.equal(outs[k].view(torch.int32), outs["torch"].view(torch.int32)), (points, pattern, k)
            t = time_arms(fns, args.iters, flush)
            lines.append({"src": [B, points], "out": [B, H * H], "index": pattern, **t,
                          "speedup_values": round(t["torch"]["ms_median"] / t["ours"]["ms_median"], 2),
                          "speedup_with_argmax": round(t["torch"]["ms_median"] / t["ours_argmax"]["ms_median"], 2),
                          "check": "bit-identical"})
    for line in lines:
        print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
