"""Online cropping of ShapeNet-55/34 (utils/helpers.py:62-123, `seprate_point_cloud`) on the sm_100a kernels.

The reference cuts the partial input out of the complete cloud at every training and test step, one cloud at a time:
a host draw and a blocking copy of the centre, a norm, a full argsort and two gathers per cloud, and in the training
form two single-cloud FPS chains per cloud.  Here the whole batch takes two launches and two small uploads:

    crop_split_raw       ps_crop_split: per-cloud torch-exact distance, stable sort, split into crop / kept rows
    fps_ragged_raw       ps_fps_sample_ragged: FPS + gather of every part of a ragged batch in one launch
    seprate_point_cloud  the reference's function: same name, arguments, results and random draws
    patch_helpers        rebinds it inside an imported reference `utils.helpers`

The random draws stay on the host, in the reference's order (per cloud: `random.randint` for a list crop, then
`torch.randn` + `F.normalize` or `random.sample` for the centre), so a seeded run crops the same clouds and leaves
Python's and torch's generators in the same state.
"""
import ctypes
import random

import torch
import torch.nn.functional as F

from . import _lib as L
from .model_ops import _with_reference_fallback

CROP_MIN_N, CROP_MAX_N = 33, 16384  # what one CTA sorts (include/pointsea_b200.h)
FPS_POINTS = 2048                   # the reference's fps(..., 2048) of both parts of a list crop


def _unsupported(msg):
    err = L.PointSeaError(msg)
    err.code = L.PS_ERR_UNSUPPORTED
    return err


def crop_split_raw(xyz, centers, counts, pad_zeros=False, padded=False):
    """xyz (B,N,3) CUDA float32, centers (B,3) host float32, counts: B ints in [0, N] -> (keep, crop).

    padded=False (every count equal to c): packed keep (B,N-c,3) (or (B,N,3) with pad_zeros) and crop (B,c,3).
    padded=True: keep and crop are the two halves of one (2,B,N,3) buffer; row b holds N-counts[b] (N with
    pad_zeros) and counts[b] valid points, in the order the packed form has them."""
    L.require(xyz, "xyz", torch.float32, 3)
    if xyz.size(2) != 3:
        raise L.PointSeaError(f"xyz must be (B,N,3), got {tuple(xyz.shape)}")
    dev = L.same_device(xyz)
    B, N, _ = xyz.shape
    counts = [int(c) for c in counts]
    centers = torch.as_tensor(centers, dtype=torch.float32).reshape(-1).contiguous()
    if len(counts) != B or centers.numel() != 3 * B:
        raise L.PointSeaError(f"crop_split: {B} clouds need {B} counts and {B} centres")
    if padded:
        buf = torch.empty(2, B, N, 3, device=xyz.device, dtype=torch.float32)
        keep, crop = buf[0], buf[1]
        ks = cs = N
    else:
        if len(set(counts)) > 1:
            raise L.PointSeaError("crop_split: packed outputs need equal counts (use padded=True)")
        c = counts[0] if counts else 0
        ks, cs = (N if pad_zeros else N - c), c
        keep = torch.empty(B, ks, 3, device=xyz.device, dtype=torch.float32)
        crop = torch.empty(B, cs, 3, device=xyz.device, dtype=torch.float32)
    cnt = (ctypes.c_int * max(B, 1))(*counts)
    L.check(L.load().ps_crop_split(L.ptr(xyz), centers.data_ptr() if B else None, cnt, keep.data_ptr() or None,
                                   crop.data_ptr() or None, B, N, ks, cs, 1 if pad_zeros else 0, dev,
                                   L.stream_ptr(dev)), "ps_crop_split")
    return keep, crop


def fps_ragged_raw(xyz, sizes, npoint):
    """xyz (B,S,3) CUDA float32, sizes: B ints in [1, S] -> (idx (B,npoint) int32, new_xyz (B,npoint,3)): FPS of the
    first sizes[b] points of every row, each as the reference samples that cloud alone."""
    L.require(xyz, "xyz", torch.float32, 3)
    if xyz.size(2) != 3:
        raise L.PointSeaError(f"xyz must be (B,S,3), got {tuple(xyz.shape)}")
    dev = L.same_device(xyz)
    B, S, _ = xyz.shape
    sizes = [int(n) for n in sizes]
    if len(sizes) != B:
        raise L.PointSeaError(f"fps_ragged: {B} rows need {B} sizes")
    npoint = int(npoint)
    idx = torch.empty(B, npoint, device=xyz.device, dtype=torch.int32)
    new_xyz = torch.empty(B, npoint, 3, device=xyz.device, dtype=torch.float32)
    n = (ctypes.c_int * max(B, 1))(*sizes)
    L.check(L.load().ps_fps_sample_ragged(L.ptr(xyz), n, L.ptr(idx), L.ptr(new_xyz), B, S, npoint, dev,
                                          L.stream_ptr(dev)), "ps_fps_sample_ragged")
    return idx, new_xyz


def draw_crops(B, crop, fixed_points=None):
    """The reference's host draws for B clouds, in its order: (num_crop list, centre list of (1,1,3) CPU tensors)."""
    counts, centers = [], []
    for _ in range(B):
        if isinstance(crop, list):
            num_crop = random.randint(crop[0], crop[1])
        else:
            num_crop = crop
        if fixed_points is None:
            center = F.normalize(torch.randn(1, 1, 3), p=2, dim=-1)
        else:
            if isinstance(fixed_points, list):
                fixed_point = random.sample(fixed_points, 1)[0]
            else:
                fixed_point = fixed_points
            center = fixed_point.reshape(1, 1, 3)
        counts.append(num_crop)
        centers.append(center)
    return counts, centers


def seprate_point_cloud(xyz, num_points, crop, fixed_points=None, padding_zeros=False):
    """utils/helpers.py:62-123.  xyz (B,n,3) CUDA -> (input, crop):
      int crop c:   input (B,n-c,3) (or (B,n,3), cropped points zeroed, with padding_zeros), crop (B,c,3), both in
                    ascending distance from each cloud's centre;
      list [lo,hi]: per cloud c = random.randint(lo, hi), then input = fps(kept part, 2048), crop = fps(cropped part,
                    2048): (B,2048,3) each;
      crop == num_points: (xyz, None).
    Shapes the kernels do not cover raise PointSeaError with code PS_ERR_UNSUPPORTED, with both random generators
    restored to their state at the call, so the reference can take the call over unchanged (patch_helpers)."""
    _, n, c = xyz.shape
    assert n == num_points
    assert c == 3
    if crop == num_points:
        return xyz, None
    if not xyz.is_cuda:
        raise L.PointSeaError("xyz must be a CUDA tensor (CPU not supported)")
    if xyz.dtype != torch.float32:
        raise _unsupported(f"seprate_point_cloud: xyz is {xyz.dtype}, the kernels take float32")
    if xyz.requires_grad and torch.is_grad_enabled():
        raise _unsupported("seprate_point_cloud: no gradient flows through the kernels; xyz requires grad")
    if xyz.size(0) == 0:
        raise _unsupported("seprate_point_cloud: an empty batch (the reference's torch.cat of no clouds raises)")
    if not CROP_MIN_N <= n <= CROP_MAX_N:
        raise _unsupported(f"seprate_point_cloud: {n} points per cloud, the kernels sort {CROP_MIN_N}..{CROP_MAX_N}")
    B = xyz.size(0)
    py_state, torch_state = random.getstate(), torch.get_rng_state()
    try:
        counts, centers = draw_crops(B, crop, fixed_points)
        if any(t.dtype != torch.float32 for t in centers):
            raise _unsupported("seprate_point_cloud: a fixed point that is not float32 changes the distance's dtype")
        if any(not 0 <= k <= n for k in counts):
            raise _unsupported(f"seprate_point_cloud: crop counts {sorted(set(counts))} outside [0, {n}]")
        ctr = torch.cat([t.reshape(1, 3).detach().cpu() for t in centers])
        xyz = xyz.detach().contiguous()
        if not isinstance(crop, list):
            return crop_split_raw(xyz, ctr, counts, pad_zeros=padding_zeros)
        sizes = [n if padding_zeros else n - k for k in counts] + counts
        if min(sizes, default=1) < 1:
            raise _unsupported("seprate_point_cloud: an empty part has no farthest point sample")
        keep, _ = crop_split_raw(xyz, ctr, counts, pad_zeros=padding_zeros, padded=True)
        # both halves of the (2,B,n,3) buffer as 2B rows: every kept part, then every cropped part, in one launch
        _, sampled = fps_ragged_raw(keep.as_strided((2 * B, n, 3), (3 * n, 3, 1)), sizes, FPS_POINTS)
        return sampled[:B], sampled[B:]
    except L.PointSeaError as e:
        if e.code == L.PS_ERR_UNSUPPORTED:
            random.setstate(py_state)
            torch.set_rng_state(torch_state)
        raise


def patch_helpers(module):
    """Rebind `seprate_point_cloud` inside an imported reference `utils.helpers`.  The training and test loops look
    it up there at call time (`helpers.seprate_point_cloud(...)`); inputs the kernels do not cover go to the module's
    own function.  A call site that did `from utils.helpers import seprate_point_cloud` before this ran keeps the
    original (INTEGRATION.md)."""
    if getattr(module, "_pointsea_crop_patched", False):
        return module
    module.seprate_point_cloud = _with_reference_fallback(seprate_point_cloud, getattr(module, "seprate_point_cloud", None))
    module._pointsea_crop_patched = True
    return module
