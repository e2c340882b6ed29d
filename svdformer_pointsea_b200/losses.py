"""The Chamfer training losses of utils/loss_utils.py:10-31 as fused autograd ops.

    chamfer                   mean(d1) + mean(d2)
    chamfer_sqrt              (mean(sqrt d1) + mean(sqrt d2)) / 2
    chamfer_single_side       mean(d1)
    chamfer_single_side_sqrt  mean(sqrt d1)

Same names and arguments as the reference.  The forward is the Chamfer forward with its fused loss sums plus one
single-thread launch that writes the 0-dim fp32 loss (ps_chamfer_loss_fwd; the sums are combined in double and
rounded once, so the value may differ from torch's fp32 means in the last bits).  The backward is one call of
ps_chamfer_loss_bwd, which derives every point's distance gradient from the forward's `dist` as torch's autograd of
the expressions above does, and computes gradients only for the clouds that require them.  Measured on a B200
(DESIGN.md §4.10, profiles/chamfer_loss.jsonl): 6-9 kernels per term forward + backward against 11-22 for the
Chamfer Function plus the torch expression.

`patch_loss_utils(module, training=True)` (metrics.py) rebinds the four names inside the reference's
`utils.loss_utils`, whose get_loss / get_loss_PM look them up as module globals when they run.
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib as L
from .chamfer import _check_out

# the PS_LOSS_* values of include/pointsea_b200.h
LOSS_KINDS = {"cd": 0, "cd_sqrt": 1, "single": 2, "single_sqrt": 3}


def _kind(kind):
    if kind not in LOSS_KINDS:
        raise L.PointSeaError(f"unknown Chamfer loss kind {kind!r}; expected one of {sorted(LOSS_KINDS)}")
    return LOSS_KINDS[kind]


def _clouds(xyz1, xyz2):
    L.require(xyz1, "xyz1", torch.float32, 3)
    L.require(xyz2, "xyz2", torch.float32, 3)
    if xyz1.size(2) != 3 or xyz2.size(2) != 3 or xyz1.size(0) != xyz2.size(0):
        raise L.PointSeaError(f"chamfer expects (B,N,3) and (B,M,3), got {tuple(xyz1.shape)} {tuple(xyz2.shape)}")
    return L.same_device(xyz1, xyz2)


def chamfer_loss_forward(xyz1, xyz2, kind):
    """(loss 0-dim, dist1, dist2, idx1, idx2); no autograd.  `kind`: a key of LOSS_KINDS."""
    k = _kind(kind)
    dev = _clouds(xyz1, xyz2)
    B, N, _ = xyz1.shape
    M = xyz2.size(1)
    f = dict(device=xyz1.device, dtype=torch.float32)
    dist1, dist2 = torch.empty(B, N, **f), torch.empty(B, M, **f)
    idx1 = torch.empty(B, N, device=xyz1.device, dtype=torch.int32)
    idx2 = torch.empty(B, M, device=xyz1.device, dtype=torch.int32)
    sums = torch.empty(6, device=xyz1.device, dtype=torch.float64)
    loss = torch.empty((), **f)
    L.check(L.load().ps_chamfer_loss_fwd(L.ptr(xyz1), L.ptr(xyz2), L.ptr(dist1), L.ptr(dist2), L.ptr(idx1), L.ptr(idx2),
                                         L.ptr(sums), loss.data_ptr(), k, B, N, M, dev, L.stream_ptr(dev)),
            "ps_chamfer_loss_fwd")
    return loss, dist1, dist2, idx1, idx2


def chamfer_loss_backward(xyz1, xyz2, dist1, dist2, idx1, idx2, grad_loss, kind, need1=True, need2=True):
    """(gradxyz1 or None, gradxyz2 or None) of the loss `kind` for the upstream gradient `grad_loss` (0-dim)."""
    if not (need1 or need2):
        raise L.PointSeaError("chamfer_loss_backward: no gradient requested")
    k = _kind(kind)
    dev = _clouds(xyz1, xyz2)
    B, N, _ = xyz1.shape
    M = xyz2.size(1)
    for t, name, dtype, shape in ((dist1, "dist1", torch.float32, (B, N)), (dist2, "dist2", torch.float32, (B, M)),
                                  (idx1, "idx1", torch.int32, (B, N)), (idx2, "idx2", torch.int32, (B, M))):
        _check_out(t, name, dtype, shape, xyz1)
    grad_loss = grad_loss.to(device=xyz1.device, dtype=torch.float32).contiguous()
    if grad_loss.numel() != 1:
        raise L.PointSeaError(f"grad_loss must hold one value, got {tuple(grad_loss.shape)}")
    g1 = torch.empty_like(xyz1) if need1 else None
    g2 = torch.empty_like(xyz2) if need2 else None
    if B == 0:  # empty gradients; an empty tensor has no data pointer to pass
        return g1, g2
    L.check(L.load().ps_chamfer_loss_bwd(L.ptr(xyz1), L.ptr(xyz2), L.ptr(dist1), L.ptr(dist2), L.ptr(idx1), L.ptr(idx2),
                                         grad_loss.data_ptr(), L.ptr(g1) if need1 else None,
                                         L.ptr(g2) if need2 else None, k, B, N, M, dev, L.stream_ptr(dev)),
            "ps_chamfer_loss_bwd")
    return g1, g2


class ChamferLossFunction(Function):
    """apply(xyz1, xyz2, kind) -> the 0-dim loss `kind` (a key of LOSS_KINDS), differentiable w.r.t. both clouds.
    Double backward is not supported."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, kind):
        loss, dist1, dist2, idx1, idx2 = chamfer_loss_forward(xyz1, xyz2, kind)
        ctx.kind = kind
        ctx.save_for_backward(xyz1, xyz2, dist1, dist2, idx1, idx2)
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_loss):
        # a cloud that does not require grad gets no buffer: its writes and scatters are skipped
        g1, g2 = chamfer_loss_backward(*ctx.saved_tensors, grad_loss, ctx.kind, ctx.needs_input_grad[0],
                                       ctx.needs_input_grad[1])
        return g1, g2, None


def chamfer_loss(xyz1, xyz2, kind):
    """The Chamfer loss `kind` ("cd", "cd_sqrt", "single", "single_sqrt") of xyz1 (B,N,3) against xyz2 (B,M,3), a 0-dim
    fp32 tensor.  Without grad mode, or when neither cloud requires grad, only the forward runs and nothing is saved."""
    xyz1, xyz2 = xyz1.contiguous(), xyz2.contiguous()  # chamfer_3DDist.forward does the same (dist_chamfer_3D.py:71-72)
    if torch.is_grad_enabled() and (xyz1.requires_grad or xyz2.requires_grad):
        return ChamferLossFunction.apply(xyz1, xyz2, kind)
    return chamfer_loss_forward(xyz1, xyz2, kind)[0]


def chamfer(p1, p2):
    """utils/loss_utils.py `chamfer`: mean(d1) + mean(d2)."""
    return chamfer_loss(p1, p2, "cd")


def chamfer_sqrt(p1, p2):
    """utils/loss_utils.py `chamfer_sqrt`: (mean(sqrt d1) + mean(sqrt d2)) / 2."""
    return chamfer_loss(p1, p2, "cd_sqrt")


def chamfer_single_side(pcd1, pcd2):
    """utils/loss_utils.py `chamfer_single_side`: mean(d1), the pcd1 -> pcd2 side only."""
    return chamfer_loss(pcd1, pcd2, "single")


def chamfer_single_side_sqrt(pcd1, pcd2):
    """utils/loss_utils.py `chamfer_single_side_sqrt`: mean(sqrt d1), the pcd1 -> pcd2 side only."""
    return chamfer_loss(pcd1, pcd2, "single_sqrt")


TRAINING_LOSSES = ("chamfer", "chamfer_sqrt", "chamfer_single_side", "chamfer_single_side_sqrt")
