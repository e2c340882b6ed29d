"""ShapeNet-55/34 online cropping on the B200, bit for bit:
  * ps_crop_split against torch's own norm + argsort + indexing of each cloud, run on the same GPU;
  * ps_fps_sample_ragged against the CPU oracle's FPS of every part on its own;
  * seprate_point_cloud against the reference's loop restated here over this repository's per-cloud FPS (outputs and
    the states of both random generators), and against the checkout's own utils/helpers.py where one is present."""
import importlib.util
import os.path as osp
import random
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import REFERENCE, make_cloud
from oracle import oracle as O
from svdformer_pointsea_b200 import _lib as L
from svdformer_pointsea_b200 import crop as C
from svdformer_pointsea_b200 import pointnet2_utils as pu

pytestmark = pytest.mark.gpu
DEV = "cuda"

# the fixed viewpoints of the ShapeNet-55 test loop (core/test_55.py), passed one at a time as fixed_points
VIEWPOINTS = [torch.Tensor([1, 1, 0]), torch.Tensor([1, 0, 0]), torch.Tensor([1, 0, 1]), torch.Tensor([-1, 0, 0]),
              torch.Tensor([-1, 1, 0]), torch.Tensor([0, 0, 1]), torch.Tensor([0, 1, 1]), torch.Tensor([-1, 0, 1])]


def bits(t):
    return t.contiguous().view(torch.int32)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(bits(a), bits(b))


def torch_split(points, center, num_crop, padding_zeros=False):
    """One cloud of the reference's loop body (utils/helpers.py:62-123): points (1,n,3), center (1,1,3), both CUDA."""
    distance_matrix = torch.norm(center.unsqueeze(2) - points.unsqueeze(1), p=2, dim=-1)
    idx = torch.argsort(distance_matrix, dim=-1, descending=False)[0, 0]
    if padding_zeros:
        input_data = points.clone()
        input_data[0, idx[:num_crop]] = input_data[0, idx[:num_crop]] * 0
    else:
        input_data = points.clone()[0, idx[num_crop:]].unsqueeze(0)
    crop_data = points.clone()[0, idx[:num_crop]].unsqueeze(0)
    return input_data, crop_data


def fps(data, number):
    """The reference's fps: FurthestPointSampling + gather, here over this repository's bit-exact per-cloud ops."""
    idx = pu.furthest_point_sample(data, number)
    return pu.gather_operation(data.transpose(1, 2).contiguous(), idx).transpose(1, 2).contiguous()


def reference_seprate_point_cloud(xyz, num_points, crop, fixed_points=None, padding_zeros=False):
    """utils/helpers.py:62-123 restated (PoinTr's misc.seprate_point_cloud)."""
    _, n, c = xyz.shape
    assert n == num_points
    assert c == 3
    if crop == num_points:
        return xyz, None
    INPUT = []
    CROP = []
    for points in xyz:
        if isinstance(crop, list):
            num_crop = random.randint(crop[0], crop[1])
        else:
            num_crop = crop
        points = points.unsqueeze(0)
        if fixed_points is None:
            center = F.normalize(torch.randn(1, 1, 3), p=2, dim=-1).cuda()
        else:
            if isinstance(fixed_points, list):
                fixed_point = random.sample(fixed_points, 1)[0]
            else:
                fixed_point = fixed_points
            center = fixed_point.reshape(1, 1, 3).cuda()
        input_data, crop_data = torch_split(points, center, num_crop, padding_zeros)
        if isinstance(crop, list):
            INPUT.append(fps(input_data, 2048))
            CROP.append(fps(crop_data, 2048))
        else:
            INPUT.append(input_data)
            CROP.append(crop_data)
    input_data = torch.cat(INPUT, dim=0)
    crop_data = torch.cat(CROP, dim=0)
    return input_data.contiguous(), crop_data.contiguous()


def cloud(kind, B, N, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "uniform":
        x = torch.rand(B, N, 3, generator=g) - 0.5
    elif kind == "dup":  # a coarse grid: most distances are exact ties
        x = torch.randint(0, 6, (B, N, 3), generator=g).float() / 4 - 0.6
    elif kind == "dup_upsampled":  # duplicated points, as the upsampling stages produce
        x = make_cloud(g, B, N, dup=N // 3)
    else:
        raise ValueError(kind)
    return x.contiguous()


def centres_for(kind, xyz, seed):
    B = xyz.size(0)
    g = torch.Generator().manual_seed(seed + 1)
    if kind == "random":
        return [F.normalize(torch.randn(1, 1, 3, generator=g), p=2, dim=-1) for _ in range(B)]
    if kind == "on_point":  # the centre is one of the cloud's points: a distance of exactly 0
        return [xyz[b, (7 * b) % xyz.size(1)].reshape(1, 1, 3).clone() for b in range(B)]
    if kind == "viewpoints":
        return [VIEWPOINTS[b % 8].reshape(1, 1, 3) for b in range(B)]
    raise ValueError(kind)


def check_split(xyz_cpu, centres, counts, pad_zeros):
    xyz = xyz_cpu.to(DEV)
    B, N, _ = xyz.shape
    ctr = torch.cat([c.reshape(1, 3) for c in centres])
    padded = len(set(counts)) > 1
    keep, crop = C.crop_split_raw(xyz, ctr, counts, pad_zeros=pad_zeros, padded=padded)
    for b in range(B):
        want_in, want_crop = torch_split(xyz[b:b + 1], centres[b].to(DEV), counts[b], pad_zeros)
        k = N if pad_zeros else N - counts[b]
        assert same_bits(keep[b, :k], want_in[0]), f"kept part of cloud {b} (N={N}, count {counts[b]})"
        assert same_bits(crop[b, :counts[b]], want_crop[0]), f"cropped part of cloud {b} (N={N}, count {counts[b]})"
    return keep, crop


# 33 and 128/129, 4096/4097: each side of torch's sort algorithm switches above 32 elements (a sort of <= 32 is not
# stable and is not covered); 2048, 8192 (ShapeNet-55), 16384 (PCN) and a size that is no power of two
SIZES = [33, 128, 129, 2048, 4096, 4097, 8192, 10000, 16384]


@pytest.mark.parametrize("N", SIZES)
@pytest.mark.parametrize("kind", ["uniform", "dup"])
def test_crop_split_matches_torch(N, kind):
    xyz = cloud(kind, 4, N, seed=N)
    g = torch.Generator().manual_seed(N + 5)
    counts = [int(v) for v in torch.randint(0, N + 1, (4,), generator=g)]
    check_split(xyz, centres_for("random", xyz, N), counts, pad_zeros=False)
    check_split(xyz, centres_for("random", xyz, N), [N // 4] * 4, pad_zeros=False)


@pytest.mark.parametrize("centre", ["on_point", "viewpoints"])
@pytest.mark.parametrize("kind", ["uniform", "dup", "dup_upsampled"])
def test_crop_split_ties_and_fixed_centres(centre, kind):
    xyz = cloud(kind, 8, 8192, seed=3)
    check_split(xyz, centres_for(centre, xyz, 3), [2048, 4096, 6144, 1, 8191, 3000, 5000, 7000], pad_zeros=False)
    check_split(xyz, centres_for(centre, xyz, 3), [6144] * 8, pad_zeros=False)


@pytest.mark.parametrize("pad_zeros", [False, True])
def test_crop_split_counts_zero_and_all(pad_zeros):
    xyz = cloud("uniform", 3, 2048, seed=9)
    check_split(xyz, centres_for("random", xyz, 9), [0, 2048, 100], pad_zeros=pad_zeros)
    check_split(xyz, centres_for("random", xyz, 9), [0, 0, 0], pad_zeros=pad_zeros)
    check_split(xyz, centres_for("random", xyz, 9), [2048] * 3, pad_zeros=pad_zeros)


@pytest.mark.parametrize("N", [2048, 8192])
def test_crop_split_padding_zeros_special_values(N):
    """points * 0 on the cropped points: NaN and inf give NaN, negative values -0.0; NaN distances sort last."""
    xyz = cloud("uniform", 4, N, seed=21)
    g = torch.Generator().manual_seed(22)
    pos = torch.randint(0, N, (4, 40), generator=g)
    for b in range(4):
        xyz[b, pos[b, :10], 0] = float("nan")
        xyz[b, pos[b, 10:20], 1] = float("inf")
        xyz[b, pos[b, 20:30], 2] = -float("inf")
        xyz[b, pos[b, 30:]] = -xyz[b, pos[b, 30:]].abs()
    centres = centres_for("random", xyz, 21)
    for pad in (True, False):
        check_split(xyz, centres, [N // 2, N - 3, 5, N // 3], pad_zeros=pad)
    keep, _ = check_split(xyz, centres, [N // 2] * 4, pad_zeros=True)
    assert torch.isnan(keep).any() and (bits(keep) == torch.tensor(-2 ** 31, dtype=torch.int32, device=DEV)).any()


def fps_parts(rows, sizes, npoint):
    """Every part through ps_fps_sample_ragged in one call, compared with the oracle's FPS of that part alone."""
    xyz = rows.to(DEV)
    idx, new_xyz = C.fps_ragged_raw(xyz, sizes, npoint)
    for b, n in enumerate(sizes):
        part = rows[b:b + 1, :n].contiguous()
        want = O.fps(part.numpy(), npoint)[0]
        assert np.array_equal(idx[b].cpu().numpy(), want), f"part {b} of {n} points"
        assert same_bits(new_xyz[b].cpu(), part[0, torch.from_numpy(want).long()]), f"coordinates of part {b}"


def test_fps_ragged_across_block_sizes():
    """Lengths on each side of opt_n_threads' steps below 512 and of the kernel sizes above it, n < npoint among them."""
    sizes = [1, 2, 3, 31, 32, 33, 100, 255, 256, 257, 511, 512, 513, 1000, 1024, 1025, 2048, 2049, 4095, 4096, 4097,
             6144, 8192]
    g = torch.Generator().manual_seed(31)
    rows = make_cloud(g, len(sizes), 8192)
    fps_parts(rows, sizes, 2048)
    fps_parts(rows[:8], sizes[:8], 64)


def test_fps_ragged_duplicates_and_skipped_points():
    """Exact ties between duplicated points and points within the origin radius the reference never selects."""
    g = torch.Generator().manual_seed(32)
    dup = make_cloud(g, 4, 6144, dup=2000)
    near = make_cloud(g, 4, 6144, near_origin=500)
    rows = torch.cat([dup, near])
    rows[7, :40] = 0.0  # the start point itself inside the origin radius
    fps_parts(rows, [6144, 5000, 2048, 3001, 6144, 4097, 2500, 300], 2048)
    allnear = (torch.rand(2, 600, 3, generator=g) - 0.5) * 0.03  # no point is ever eligible
    fps_parts(allnear, [600, 450], 64)


def test_fps_ragged_smaller_batches_than_sizes():
    """A small cloud in a batch sized by a large one, and a batch of one part."""
    g = torch.Generator().manual_seed(33)
    rows = make_cloud(g, 3, 8192)
    fps_parts(rows, [8192, 40, 4000], 512)
    fps_parts(rows[:1], [700], 700)


def run_both(fn_a, fn_b, xyz, *args, seed=0, **kw):
    out = []
    for fn in (fn_a, fn_b):
        random.seed(seed)
        torch.manual_seed(seed + 1)
        r = fn(xyz, *args, **kw)
        out.append((r, random.getstate(), torch.get_rng_state()))
    (ra, pa, ta), (rb, pb, tb) = out
    assert pa == pb and torch.equal(ta, tb), "random generator states differ after the call"
    return ra, rb


def assert_same_result(ra, rb):
    assert len(ra) == len(rb) == 2
    for a, b in zip(ra, rb):
        if a is None or b is None:
            assert a is None and b is None
        else:
            assert same_bits(a, b), (tuple(a.shape), tuple(b.shape))


@pytest.mark.parametrize("crop", [[2048, 6144], 2048, 4096, 6144])
@pytest.mark.parametrize("padding_zeros", [False, True])
def test_dropin_matches_the_reference_loop(crop, padding_zeros):
    xyz = cloud("uniform", 6, 8192, seed=41).to(DEV)
    ra, rb = run_both(reference_seprate_point_cloud, C.seprate_point_cloud, xyz, 8192, crop, seed=42,
                      padding_zeros=padding_zeros)
    assert_same_result(ra, rb)
    if isinstance(crop, list):
        assert rb[0].shape == rb[1].shape == (6, 2048, 3)


@pytest.mark.parametrize("fixed", ["single", "list"])
@pytest.mark.parametrize("crop", [[2048, 6144], 4096])
def test_dropin_matches_the_reference_loop_fixed_points(fixed, crop):
    xyz = cloud("dup_upsampled", 4, 8192, seed=43).to(DEV)
    fixed_points = VIEWPOINTS[5] if fixed == "single" else VIEWPOINTS
    ra, rb = run_both(reference_seprate_point_cloud, C.seprate_point_cloud, xyz, 8192, crop, seed=44,
                      fixed_points=fixed_points)
    assert_same_result(ra, rb)


def test_dropin_test_loop_viewpoints():
    """The ShapeNet-55 test loop: each of the eight viewpoints in turn, int crops of 1/4, 1/2 and 3/4."""
    xyz = cloud("uniform", 2, 8192, seed=45).to(DEV)
    for num_crop in (2048, 4096, 6144):
        for item in VIEWPOINTS:
            ra, rb = run_both(reference_seprate_point_cloud, C.seprate_point_cloud, xyz, 8192, num_crop, seed=46,
                              fixed_points=item)
            assert_same_result(ra, rb)


def test_dropin_other_shapes():
    """PCN-sized clouds, a cloud size that is no power of two, and crop == num_points."""
    xyz = cloud("uniform", 3, 16384, seed=47).to(DEV)
    assert_same_result(*run_both(reference_seprate_point_cloud, C.seprate_point_cloud, xyz, 16384, 4096, seed=48))
    xyz = cloud("dup", 3, 5000, seed=49).to(DEV)
    assert_same_result(*run_both(reference_seprate_point_cloud, C.seprate_point_cloud, xyz, 5000, [2048, 2952], seed=50))
    out = C.seprate_point_cloud(xyz, 5000, 5000)
    assert out[0] is xyz and out[1] is None


def test_launch_count_does_not_depend_on_the_batch():
    counts = {}
    for B in (1, 32):
        xyz = cloud("uniform", B, 8192, seed=51).to(DEV)
        for crop in ([2048, 6144], 4096):
            C.seprate_point_cloud(xyz, 8192, crop)  # warm: first calls set kernel attributes
            L.launch_count(reset=True)
            C.seprate_point_cloud(xyz, 8192, crop)
            counts[(B, str(crop))] = L.launch_count()
    assert counts[(1, "[2048, 6144]")] == counts[(32, "[2048, 6144]")] == 2
    assert counts[(1, "4096")] == counts[(32, "4096")] == 1


def stand_in_helpers():
    helpers = types.ModuleType("utils.helpers")
    helpers.seprate_point_cloud = reference_seprate_point_cloud
    return C.patch_helpers(helpers)


def test_patched_name_falls_back_with_the_random_state_restored():
    """Shapes the kernels do not cover go to the module's own function, which must see the generators untouched."""
    helpers = stand_in_helpers()
    xyz = cloud("uniform", 3, 8192, seed=52).to(DEV)
    # a count beyond the cloud (the reference's slicing takes it), found after the centres were drawn
    assert_same_result(*run_both(reference_seprate_point_cloud, helpers.seprate_point_cloud, xyz, 8192, 8300, seed=53))
    # an input that requires grad under grad mode: the reference keeps the graph
    xg = xyz.clone().requires_grad_(True)
    ra, rb = run_both(reference_seprate_point_cloud, helpers.seprate_point_cloud, xg, 8192, 4096, seed=54)
    assert_same_result([t.detach() for t in ra], [t.detach() for t in rb])
    assert rb[0].requires_grad
    with pytest.raises(L.PointSeaError) as e:
        C.seprate_point_cloud(xg, 8192, 4096)
    assert e.value.code == L.PS_ERR_UNSUPPORTED
    with torch.no_grad():
        assert_same_result(*run_both(reference_seprate_point_cloud, helpers.seprate_point_cloud, xg, 8192, 4096,
                                     seed=55))
    # a float64 fixed point promotes the reference's distances to float64
    assert_same_result(*run_both(reference_seprate_point_cloud, helpers.seprate_point_cloud, xyz, 8192, 4096, seed=56,
                                 fixed_points=VIEWPOINTS[0].double()))
    # and a cloud too large for one CTA
    big = cloud("uniform", 1, 20000, seed=57).to(DEV)
    assert_same_result(*run_both(reference_seprate_point_cloud, helpers.seprate_point_cloud, big, 20000, 5000, seed=58))


def reference_helpers():
    path = osp.join(REFERENCE, "utils", "helpers.py")
    if not osp.exists(path):
        pytest.skip(f"needs a checkout of the reference at {REFERENCE} (or set POINTSEA_REFERENCE)")
    import svdformer_pointsea_b200 as ps
    ps.install_dropin()  # its pointnet2_ops import resolves to this repository's bit-exact ops
    spec = importlib.util.spec_from_file_location("reference_utils_helpers", path)
    mod = importlib.util.module_from_spec(spec)
    try:
        spec.loader.exec_module(mod)
    except ImportError as e:
        pytest.skip(f"the reference's utils/helpers.py needs a package missing here: {e}")
    return mod


@pytest.mark.parametrize("crop,fixed", [([2048, 6144], None), (4096, None), (2048, "list"), ([2048, 6144], "single"),
                                        (6144, "pad")])
def test_dropin_matches_the_checkout(crop, fixed):
    ref = reference_helpers()
    xyz = cloud("uniform", 4, 8192, seed=61).to(DEV)
    kw = {"list": dict(fixed_points=VIEWPOINTS), "single": dict(fixed_points=VIEWPOINTS[3]),
          "pad": dict(padding_zeros=True)}.get(fixed, {})
    assert_same_result(*run_both(ref.seprate_point_cloud, C.seprate_point_cloud, xyz, 8192, crop, seed=62, **kw))
