"""Host-side checks of the fused Chamfer training losses: both entry points validate their arguments before any device
work, CPU or non-fp32 clouds and unknown kinds are refused (no CPU fallback), and patch_loss_utils rebinds the four
training losses only when asked."""
import ctypes
import types

import pytest
import torch

import svdformer_pointsea_b200 as ps
from svdformer_pointsea_b200 import _lib as L
from svdformer_pointsea_b200 import losses

FAKE = ctypes.c_void_p(0x1000)  # never dereferenced: validation fails first


def fwd(xyz1=FAKE, xyz2=FAKE, d1=FAKE, d2=FAKE, i1=FAKE, i2=FAKE, sums=FAKE, loss=FAKE, kind=0, B=2, N=8, M=9):
    lib = L.load()
    rc = lib.ps_chamfer_loss_fwd(xyz1, xyz2, d1, d2, i1, i2, sums, loss, kind, B, N, M, 0, None)
    return rc, lib.ps_last_error()


def bwd(xyz1=FAKE, xyz2=FAKE, d1=FAKE, d2=FAKE, i1=FAKE, i2=FAKE, gl=FAKE, g1=FAKE, g2=FAKE, kind=0, B=2, N=8, M=9):
    lib = L.load()
    rc = lib.ps_chamfer_loss_bwd(xyz1, xyz2, d1, d2, i1, i2, gl, g1, g2, kind, B, N, M, 0, None)
    return rc, lib.ps_last_error()


@pytest.mark.parametrize("call", [fwd, bwd])
@pytest.mark.parametrize("B,N,M", [(-1, 8, 9), (2, 0, 9), (2, 8, 0), (2, -4, 9)])
def test_rejects_bad_sizes(call, B, N, M):
    rc, msg = call(B=B, N=N, M=M)
    assert rc == -1 and b"bad sizes" in msg


@pytest.mark.parametrize("call", [fwd, bwd])
@pytest.mark.parametrize("kind", [-1, 4, 100])
def test_rejects_unknown_kind(call, kind):
    for B in (2, 0):  # even when there is no work
        rc, msg = call(kind=kind, B=B)
        assert rc == -1 and b"unknown kind" in msg


@pytest.mark.parametrize("missing", ["xyz1", "xyz2", "d1", "d2", "i1", "i2", "sums", "loss"])
def test_fwd_rejects_null_pointers(missing):
    rc, msg = fwd(**{missing: None})
    assert rc == -1 and b"null pointer" in msg


@pytest.mark.parametrize("missing", ["xyz1", "xyz2", "d1", "d2", "i1", "i2", "gl"])
@pytest.mark.parametrize("kind", [0, 3])
def test_bwd_rejects_null_pointers(missing, kind):
    rc, msg = bwd(kind=kind, **{missing: None})
    assert rc == -1 and b"null pointer" in msg


def test_bwd_rejects_both_gradients_null():
    for B in (2, 0):
        rc, msg = bwd(g1=None, g2=None, B=B)
        assert rc == -1 and b"both null" in msg


def test_bwd_empty_batch_is_a_no_op():
    assert bwd(None, None, None, None, None, None, None, FAKE, None, B=0)[0] == 0
    assert bwd(None, None, None, None, None, None, None, None, FAKE, kind=3, B=0)[0] == 0


@pytest.mark.parametrize("fn", [losses.chamfer, ps.chamfer_sqrt, ps.chamfer_single_side, ps.chamfer_single_side_sqrt])
@pytest.mark.parametrize("grad", [False, True])
def test_cpu_clouds_raise(fn, grad):
    g = torch.Generator().manual_seed(0)
    a = (torch.rand(2, 16, 3, generator=g) - 0.5).requires_grad_(grad)
    b = torch.rand(2, 20, 3, generator=g) - 0.5
    with pytest.raises(ps.PointSeaError):
        fn(a, b)


def test_non_fp32_and_unknown_kind_raise():
    a = torch.zeros(2, 16, 3, dtype=torch.float64)
    with pytest.raises(ps.PointSeaError):
        losses.chamfer(a, a)
    with pytest.raises(ps.PointSeaError, match="unknown Chamfer loss kind"):
        ps.chamfer_loss(torch.zeros(2, 16, 3), torch.zeros(2, 16, 3), "emd")


def test_patch_loss_utils_rebinds_the_training_losses_only_when_asked():
    sentinels = {name: object() for name in losses.TRAINING_LOSSES}
    m = types.ModuleType("fake_loss_utils")
    for name, s in sentinels.items():
        setattr(m, name, s)
    m.get_loss = get_loss = object()
    ps.patch_loss_utils(m)
    assert all(getattr(m, name) is s for name, s in sentinels.items())
    assert m.calc_cd is ps.calc_cd
    ps.patch_loss_utils(m, training=True)
    assert {name: getattr(m, name) for name in sentinels} == {
        "chamfer": losses.chamfer, "chamfer_sqrt": losses.chamfer_sqrt,
        "chamfer_single_side": losses.chamfer_single_side, "chamfer_single_side_sqrt": losses.chamfer_single_side_sqrt}
    assert m.get_loss is get_loss and m.calc_dcd is ps.calc_dcd and m.fscore is ps.fscore


def test_package_keeps_the_chamfer_submodule():
    import svdformer_pointsea_b200.chamfer as C
    assert isinstance(C, types.ModuleType) and C.chamfer_3DFunction is ps.chamfer_3DFunction
