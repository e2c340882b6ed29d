"""ShapeNet-55/34 online cropping (utils/helpers.py:62-123, seprate_point_cloud) per step: the reference's per-cloud
loop against the batched drop-in (svdformer_pointsea_b200.crop) on the same GPU.

    python tools/crop_time.py [--iters 30] [--out profiles/crop.jsonl]

Arms, all called with the same seeds:
  loop_ours      the reference's loop (restated in tests/test_gpu_crop.py) over this repository's per-cloud FPS and
                 gather: what `install_dropin()` gives a user today;
  loop_ref_cuda  the same loop over the reference's own CUDA FPS and gather (oracle/_ref), where that is built;
  dropin         seprate_point_cloud of this repository.
Configurations: B = 32 clouds of N = 8192 points, the training form (crop [2048, 6144], two FPS of 2048 per cloud) and
the test form (int crops 2048 / 4096 / 6144 around one of the test loop's fixed viewpoints).  Before timing, every
arm's outputs are checked bit for bit against the first arm's.  Each call is timed with the host clock from before the
call to a device synchronise after it (the loop blocks on the host, so host time is what a step pays), a 256 MB buffer
is overwritten between calls (outside the timed window), 3 warm-up calls, arms alternated call by call, median and
10th / 90th percentiles of --iters calls.  The first line names the device, its power limit and its maximum SM clock.
"""
import argparse
import importlib.util
import json
import os.path as osp
import random
import sys
import time

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, osp.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from scatter_time import device_line  # noqa: E402
from svdformer_pointsea_b200 import _lib as L  # noqa: E402
from svdformer_pointsea_b200 import crop as C  # noqa: E402
import test_gpu_crop as T  # noqa: E402

DEV = torch.device("cuda:0")
B, N = 32, 8192


def load_ref_fps():
    path = osp.join(ROOT, "oracle", "_ref", "ref_pointnet2_ext.so")
    if not osp.exists(path):
        return None
    spec = importlib.util.spec_from_file_location("ref_pointnet2_ext", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    def fps(data, number):
        idx = mod.furthest_point_sampling(data, number)
        return mod.gather_points(data.transpose(1, 2).contiguous(), idx).transpose(1, 2).contiguous()
    return fps


def seeded(fn, seed):
    def call():
        random.seed(seed)
        torch.manual_seed(seed)
        return fn()
    return call


def time_arms(fns, iters, flush, warm=3):
    for _ in range(warm):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(iters):
        for k, fn in fns.items():
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts[k].append((time.perf_counter() - t0) * 1e3)
    return {k: {"ms_median": round(float(np.median(v)), 3), "ms_p10": round(float(np.percentile(v, 10)), 3),
                "ms_p90": round(float(np.percentile(v, 90)), 3), "iters": iters} for k, v in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    args = ap.parse_args()
    if args.iters < 10:
        ap.error("--iters must be at least 10")
    ref_fps = load_ref_fps()
    lines = [dict(device_line(), loop_ref_cuda="timed" if ref_fps else "oracle/_ref not built: arm left out")]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    g = torch.Generator().manual_seed(0)
    xyz = (torch.rand(B, N, 3, generator=g) - 0.5).to(DEV)

    def loop(fps_fn, crop, kw):
        saved = T.fps
        T.fps = fps_fn
        try:
            return T.reference_seprate_point_cloud(xyz, N, crop, **kw)
        finally:
            T.fps = saved

    for crop, kw in (([2048, 6144], {}), (2048, {"fixed_points": T.VIEWPOINTS[0]}),
                     (4096, {"fixed_points": T.VIEWPOINTS[0]}), (6144, {"fixed_points": T.VIEWPOINTS[0]})):
        fns = {"loop_ours": seeded(lambda: loop(T.fps, crop, kw), 1)}
        if ref_fps:
            fns["loop_ref_cuda"] = seeded(lambda: loop(ref_fps, crop, kw), 1)
        fns["dropin"] = seeded(lambda: C.seprate_point_cloud(xyz, N, crop, **kw), 1)
        outs = {k: fn() for k, fn in fns.items()}
        for k, o in outs.items():
            for a, b in zip(o, outs["loop_ours"]):
                assert T.same_bits(a, b), (crop, k)
        launches = {}
        for k in ("loop_ours", "dropin"):
            L.launch_count(reset=True)
            fns[k]()
            launches[k] = L.launch_count()
        t = time_arms(fns, args.iters, flush)
        line = {"B": B, "N": N, "crop": crop, "fixed_points": "viewpoint [1,1,0]" if kw else None, **t,
                "library_launches": launches, "check": "bit-identical outputs"}
        line["speedup_vs_loop_ours"] = round(t["loop_ours"]["ms_median"] / t["dropin"]["ms_median"], 1)
        if ref_fps:
            line["speedup_vs_loop_ref_cuda"] = round(t["loop_ref_cuda"]["ms_median"] / t["dropin"]["ms_median"], 1)
        lines.append(line)
        print(json.dumps(line), flush=True)
    print(json.dumps(lines[0]), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
