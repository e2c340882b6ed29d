"""Host-side checks of the ShapeNet-55/34 cropping drop-in: ps_crop_split and ps_fps_sample_ragged validate their
arguments before any CUDA call, the host draws follow the reference's order exactly (same crop counts and centres, same
final states of Python's and torch's generators), and patch_helpers rebinds the name inside a helpers-like module."""
import ctypes
import random
import types

import pytest
import torch
import torch.nn.functional as F

from svdformer_pointsea_b200 import _lib as L
from svdformer_pointsea_b200 import crop as C

FAKE = ctypes.c_void_p(0x1000)  # never dereferenced: validation fails first or there is nothing to do
CENTRES = (ctypes.c_float * 6)(0, 0, 1, 1, 0, 0)


def ints(*v):
    return (ctypes.c_int * len(v))(*v)


def split(xyz=FAKE, centers=CENTRES, counts=None, keep=FAKE, crop=FAKE, B=2, N=100, ks=100, cs=100, pad=0):
    lib = L.load()
    rc = lib.ps_crop_split(xyz, centers, ints(10, 20) if counts is None else counts, keep, crop, B, N, ks, cs, pad, 0,
                           None)
    return rc, lib.ps_last_error()


def ragged(xyz=FAKE, n=None, idx=FAKE, new_xyz=FAKE, B=2, stride=100, npoint=16):
    lib = L.load()
    rc = lib.ps_fps_sample_ragged(xyz, ints(50, 100) if n is None else n, idx, new_xyz, B, stride, npoint, 0, None)
    return rc, lib.ps_last_error()


@pytest.mark.parametrize("kw", [dict(B=-1), dict(N=-1), dict(ks=-1), dict(cs=-1)])
def test_crop_split_rejects_negative_sizes(kw):
    rc, msg = split(**kw)
    assert rc == -1 and b"bad sizes" in msg


@pytest.mark.parametrize("missing", ["xyz", "centers", "counts", "keep", "crop"])
def test_crop_split_rejects_null_pointers(missing):
    lib = L.load()
    args = dict(xyz=FAKE, centers=CENTRES, counts=ints(10, 20), keep=FAKE, crop=FAKE)
    args[missing] = None
    rc = lib.ps_crop_split(args["xyz"], args["centers"], args["counts"], args["keep"], args["crop"], 2, 100, 100, 100,
                           0, 0, None)
    assert rc == -1 and b"null pointer" in lib.ps_last_error()


@pytest.mark.parametrize("counts", [(-1, 20), (10, 101)])
def test_crop_split_rejects_counts_outside_the_cloud(counts):
    rc, msg = split(counts=ints(*counts))
    assert rc == -1 and b"outside [0, 100]" in msg


@pytest.mark.parametrize("kw", [dict(ks=89), dict(cs=19), dict(ks=99, pad=1)])
def test_crop_split_rejects_rows_too_short(kw):
    rc, msg = split(**kw)
    assert rc == -1 and b"does not fit" in msg


@pytest.mark.parametrize("N", [0, 32, 16385])
def test_crop_split_unsupported_sizes(N):
    rc, msg = split(N=N, ks=N, cs=N, counts=ints(0, 0))
    assert rc == L.PS_ERR_UNSUPPORTED and b"outside 33..16384" in msg


@pytest.mark.parametrize("counts,pad,missing", [((0, 0), 0, "keep"), ((100, 100), 0, "crop"), ((100, 100), 1, "keep")])
def test_crop_split_needs_every_output_that_has_rows(counts, pad, missing):
    """An output whose rows are all empty may be NULL; one that receives points may not."""
    rc, msg = split(counts=ints(*counts), pad=pad, **{missing: None})
    assert rc == -1 and b"null pointer" in msg


def test_crop_split_empty_batch_is_a_no_op():
    assert split(xyz=None, centers=None, counts=None, keep=None, crop=None, B=0)[0] == 0


@pytest.mark.parametrize("kw", [dict(B=-1), dict(stride=-1), dict(npoint=-1)])
def test_fps_ragged_rejects_negative_sizes(kw):
    rc, msg = ragged(**kw)
    assert rc == -1 and b"bad sizes" in msg


@pytest.mark.parametrize("missing", ["xyz", "n", "idx"])
def test_fps_ragged_rejects_null_pointers(missing):
    lib = L.load()
    args = dict(xyz=FAKE, n=ints(50, 100), idx=FAKE)
    args[missing] = None
    rc = lib.ps_fps_sample_ragged(args["xyz"], args["n"], args["idx"], FAKE, 2, 100, 16, 0, None)
    assert rc == -1 and b"null pointer" in lib.ps_last_error()


@pytest.mark.parametrize("n", [(0, 100), (50, 101), (-3, 10)])
def test_fps_ragged_rejects_sizes_outside_the_row(n):
    rc, msg = ragged(n=ints(*n))
    assert rc == -1 and b"outside [1, stride=100]" in msg


def test_fps_ragged_unsupported_size():
    rc, msg = ragged(n=ints(50, 8193), stride=9000)  # opt_n_threads pads 8193 points to 8704 ranks
    assert rc == L.PS_ERR_UNSUPPORTED and b"8192" in msg


@pytest.mark.parametrize("kw", [dict(B=0), dict(npoint=0)])
def test_fps_ragged_empty_work_is_a_no_op(kw):
    assert ragged(xyz=None, n=None, idx=None, new_xyz=None, **kw)[0] == 0


# ---- host draws -------------------------------------------------------------------------------------------------
VIEWPOINTS = [torch.Tensor([1, 1, 0]), torch.Tensor([1, 0, 0]), torch.Tensor([1, 0, 1]), torch.Tensor([-1, 0, 0]),
              torch.Tensor([-1, 1, 0])]  # the kind of list the test loop passes as fixed_points


def reference_draws(B, crop, fixed_points=None):
    """The draws of utils/helpers.py seprate_point_cloud's loop, restated (the centre stays on the host)."""
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


@pytest.mark.parametrize("crop", [[2048, 6144], 4096])
@pytest.mark.parametrize("fixed", ["none", "single", "list"])
def test_draws_follow_the_reference_order(crop, fixed):
    fixed_points = {"none": None, "single": VIEWPOINTS[2], "list": VIEWPOINTS}[fixed]
    runs = []
    for fn in (reference_draws, C.draw_crops):
        random.seed(11)
        torch.manual_seed(12)
        torch.randn(5)  # a generator already in use
        counts, centers = fn(7, crop, fixed_points)
        runs.append((counts, torch.cat(centers), random.getstate(), torch.get_rng_state()))
    (c0, x0, p0, t0), (c1, x1, p1, t1) = runs
    assert c0 == c1 and torch.equal(x0, x1) and p0 == p1 and torch.equal(t0, t1)
    if isinstance(crop, list):
        assert len(set(c0)) > 1 and all(crop[0] <= k <= crop[1] for k in c0)


@pytest.fixture
def no_device(monkeypatch):
    """Any attempt to reach the native library or a device fails the test."""
    def boom(*a, **k):
        raise AssertionError("touched the device")
    monkeypatch.setattr(L, "load", boom)
    monkeypatch.setattr(L, "same_device", boom)


def test_cpu_tensor_raises_without_drawing(no_device):
    xyz = torch.rand(2, 64, 3)
    random.seed(3)
    torch.manual_seed(4)
    p, t = random.getstate(), torch.get_rng_state()
    with pytest.raises(L.PointSeaError, match="CUDA") as e:
        C.seprate_point_cloud(xyz, 64, [16, 32])
    assert e.value.code is None  # not a shape the reference takes over: the patched name raises too
    assert random.getstate() == p and torch.equal(torch.get_rng_state(), t)


def test_reference_passthrough_and_assertions(no_device):
    xyz = torch.rand(2, 64, 3)
    out, none = C.seprate_point_cloud(xyz, 64, 64)
    assert out is xyz and none is None
    with pytest.raises(AssertionError):
        C.seprate_point_cloud(xyz, 65, 16)
    with pytest.raises(AssertionError):
        C.seprate_point_cloud(torch.rand(2, 64, 4), 64, 16)


def test_patch_helpers_rebinds_with_the_reference_behind(no_device):
    calls = []

    def original(xyz, num_points, crop, fixed_points=None, padding_zeros=False):
        calls.append(crop)
        return "reference"

    helpers = types.ModuleType("utils.helpers")
    helpers.seprate_point_cloud = original
    assert C.patch_helpers(helpers) is helpers
    fn = helpers.seprate_point_cloud
    assert fn.reference is original and fn.pointsea_kernel is C.seprate_point_cloud
    assert C.patch_helpers(helpers).seprate_point_cloud is fn  # idempotent
    with pytest.raises(L.PointSeaError):  # a CPU tensor is an error for the drop-in, not a shape to hand back
        fn(torch.rand(1, 64, 3), 64, 16)
    assert calls == []
