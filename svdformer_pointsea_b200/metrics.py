"""Evaluation metrics of utils/loss_utils.py and metrics/CD/fscore.py on the sm_100a kernels.

    calc_cd   utils/loss_utils.py:98-115    fscore   metrics/CD/fscore.py:3-16    calc_dcd   utils/loss_utils.py:117-155

Same names, arguments and return lists as the reference.  One Chamfer forward + ONE epilogue kernel
(ps_chamfer_metrics) per call; per-cloud results, so the batch-sharded multi-GPU path needs no collective.

calc_cd and calc_dcd are differentiable w.r.t. both clouds, as the reference's torch expressions are, so the
density-aware Chamfer distance (or cd_p / cd_t) can be part of a training loss.  When grad mode is on and a cloud
requires grad, the forward runs the same two launches (same values) plus five (B,)-sized copies (torch kernels) that
give the per-cloud outputs tensors of their own; the backward is one launch of ps_chamfer_metrics_bwd (gradients of
the distances) + ps_chamfer_bwd (gradients of the points), and only the outputs the loss used contribute.  idx, precisions and the F-score carry no gradient (the reference's are integer tensors or
comparisons).  Otherwise no graph is built.
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib as L
from .chamfer import chamfer_backward, chamfer_forward

FSCORE_THRESHOLD = 0.0001  # metrics/CD/fscore.py:3


def chamfer_metrics_raw(dist1, dist2, idx1=None, idx2=None, threshold=FSCORE_THRESHOLD, alpha=1000.0, n_lambda=1.0,
                        frac1=1.0, frac2=1.0):
    """(B,8) float32: mean sqrt d1, mean sqrt d2, mean d1, mean d2, precision_1, precision_2, fscore, dcd."""
    L.require(dist1, "dist1", torch.float32, 2)
    L.require(dist2, "dist2", torch.float32, 2)
    ts = [dist1, dist2]
    if (idx1 is None) != (idx2 is None):
        raise L.PointSeaError("idx1 and idx2 must both be given or both be None")
    if idx1 is not None:
        L.require(idx1, "idx1", torch.int32, 2)
        L.require(idx2, "idx2", torch.int32, 2)
        ts += [idx1, idx2]
    dev = L.same_device(*ts)
    B, n1 = dist1.shape
    n2 = dist2.size(1)
    out = torch.empty(B, 8, device=dist1.device, dtype=torch.float32)
    L.check(L.load().ps_chamfer_metrics(L.ptr(dist1), L.ptr(dist2), L.ptr(idx1) if idx1 is not None else None,
                                        L.ptr(idx2) if idx2 is not None else None, L.ptr(out), B, n1, n2,
                                        float(threshold), float(alpha), float(n_lambda), float(frac1), float(frac2),
                                        dev, L.stream_ptr(dev)), "ps_chamfer_metrics")
    return out


def chamfer_metrics_grad_raw(dist1, dist2, idx1, idx2, gcoef5, terms, graw1=None, graw2=None, alpha=1000.0, n_lambda=1.0,
                             frac1=1.0, frac2=1.0):
    """(graddist1 (B,n1), graddist2 (B,n2)) from the per-cloud upstream gradients gcoef5 (B,5) of mean sqrt d1,
    mean sqrt d2, mean d1, mean d2, dcd (`terms`: bitmask of the columns present) and of the raw distances
    (graw1 / graw2 or None).  idx1/idx2 are needed for the dcd term (bit 4) only."""
    L.require(dist1, "dist1", torch.float32, 2)
    L.require(dist2, "dist2", torch.float32, 2)
    ts = [dist1, dist2]
    for t, name, dtype in ((idx1, "idx1", torch.int32), (idx2, "idx2", torch.int32), (gcoef5, "gcoef5", torch.float32),
                           (graw1, "graw1", torch.float32), (graw2, "graw2", torch.float32)):
        if t is not None:
            ts.append(L.require(t, name, dtype, 2))
    dev = L.same_device(*ts)
    B, n1 = dist1.shape
    n2 = dist2.size(1)
    gd1, gd2 = torch.empty_like(dist1), torch.empty_like(dist2)
    L.check(L.load().ps_chamfer_metrics_bwd(L.ptr(dist1), L.ptr(dist2), L.ptr(idx1) if idx1 is not None else None,
                                            L.ptr(idx2) if idx2 is not None else None,
                                            L.ptr(gcoef5) if gcoef5 is not None else None, int(terms),
                                            L.ptr(graw1) if graw1 is not None else None,
                                            L.ptr(graw2) if graw2 is not None else None, L.ptr(gd1), L.ptr(gd2), B, n1, n2,
                                            float(alpha), float(n_lambda), float(frac1), float(frac2), dev,
                                            L.stream_ptr(dev)), "ps_chamfer_metrics_bwd")
    return gd1, gd2


class ChamferMetricsFunction(Function):
    """cham_loss(gt, output) followed by the epilogue, differentiable w.r.t. gt and output.

    apply(gt, output, dcd) with dcd = None (calc_cd) or (alpha, n_lambda, frac_21, frac_12) (calc_dcd) returns
    mean sqrt d1, mean sqrt d2, mean d1, mean d2, dcd (each (B,), separate tensors), the (B,8) block of
    ps_chamfer_metrics, dist1, dist2, idx1, idx2.  The block, idx1/idx2 and (without dcd) the dcd output are not
    differentiable; dist1/dist2 are, as chamfer_3DFunction's."""

    @staticmethod
    def forward(ctx, gt, output, dcd):
        ctx.set_materialize_grads(False)
        dist1, dist2, idx1, idx2 = chamfer_forward(gt, output)
        if dcd is None:
            m = chamfer_metrics_raw(dist1, dist2)
        else:
            alpha, n_lambda, frac1, frac2 = dcd
            m = chamfer_metrics_raw(dist1, dist2, idx1, idx2, alpha=alpha, n_lambda=n_lambda, frac1=frac1, frac2=frac2)
        # five small copies: each differentiable output is a tensor of its own, not a view of the (B,8) block
        terms = [m[:, k].clone(memory_format=torch.contiguous_format) for k in (0, 1, 2, 3, 7)]
        ctx.dcd = dcd
        ctx.save_for_backward(gt, output, dist1, dist2, idx1, idx2)
        ctx.mark_non_differentiable(m, idx1, idx2, *([terms[4]] if dcd is None else []))
        return (*terms, m, dist1, dist2, idx1, idx2)

    @staticmethod
    @once_differentiable
    def backward(ctx, g_sqrt1, g_sqrt2, g_mean1, g_mean2, g_dcd, _g_m, g_dist1, g_dist2, _g_idx1, _g_idx2):
        gt, output, dist1, dist2, idx1, idx2 = ctx.saved_tensors
        grads = (g_sqrt1, g_sqrt2, g_mean1, g_mean2, g_dcd)
        terms = sum(1 << k for k, g in enumerate(grads) if g is not None)
        gcoef5 = None
        if terms:
            gcoef5 = torch.zeros(dist1.size(0), 5, device=dist1.device, dtype=torch.float32)
            for k, g in enumerate(grads):
                if g is not None:
                    gcoef5[:, k] = g
        alpha, n_lambda, frac1, frac2 = ctx.dcd if ctx.dcd is not None else (1000.0, 1.0, 1.0, 1.0)  # unread without bit 4
        raw = [None if g is None else g.to(torch.float32).contiguous() for g in (g_dist1, g_dist2)]
        gd1, gd2 = chamfer_metrics_grad_raw(dist1, dist2, idx1, idx2, gcoef5, terms, raw[0], raw[1], alpha=alpha,
                                            n_lambda=n_lambda, frac1=frac1, frac2=frac2)
        g_gt, g_output = chamfer_backward(gt, output, gd1, gd2, idx1, idx2)
        return (g_gt if ctx.needs_input_grad[0] else None), (g_output if ctx.needs_input_grad[1] else None), None


def _needs_graph(*clouds):
    return torch.is_grad_enabled() and any(c.requires_grad for c in clouds)


def fscore(dist1, dist2, threshold=FSCORE_THRESHOLD):
    """metrics/CD/fscore.py:3-16 -> (fscore, precision_1, precision_2), each (B,)."""
    m = chamfer_metrics_raw(dist1.detach().contiguous(), dist2.detach().contiguous(), threshold=threshold)
    return m[:, 6], m[:, 4], m[:, 5]


def calc_cd(output, gt, calc_f1=False, return_raw=False, normalize=False, separate=False):
    """utils/loss_utils.py:98-115 (differentiable w.r.t. output and gt, as the reference's)."""
    if _needs_graph(output, gt):
        s1, s2, q1, q2, _, m, dist1, dist2, idx1, idx2 = ChamferMetricsFunction.apply(gt.contiguous(), output.contiguous(), None)
    else:
        dist1, dist2, idx1, idx2 = chamfer_forward(gt.detach().contiguous(), output.detach().contiguous())
        m = chamfer_metrics_raw(dist1, dist2)
        s1, s2, q1, q2 = m[:, 0], m[:, 1], m[:, 2], m[:, 3]
    cd_p = (s1 + s2) / 2
    cd_t = q1 + q2
    if separate:
        res = [torch.cat([s1.unsqueeze(0), s2.unsqueeze(0)]), torch.cat([q1.unsqueeze(0), q2.unsqueeze(0)])]
    else:
        res = [cd_p, cd_t]
    if calc_f1:
        res.append(m[:, 6])
    if return_raw:
        res.extend([dist1, dist2, idx1, idx2])
    return res


def calc_dcd(x, gt, alpha=1000, n_lambda=1, return_raw=False, non_reg=False):
    """utils/loss_utils.py:117-155: density-aware Chamfer distance -> [loss (B,), cd_p, cd_t (, raw...)],
    differentiable w.r.t. x and gt (the hit counts are detached, as in the reference)."""
    x = x.float()
    gt = gt.float()
    n_x, n_gt = x.shape[1], gt.shape[1]
    assert x.shape[0] == gt.shape[0]
    if non_reg:
        frac_12 = max(1, n_x / n_gt)
        frac_21 = max(1, n_gt / n_x)
    else:
        frac_12 = n_x / n_gt
        frac_21 = n_gt / n_x
    # calc_cd(x, gt) -> cham_loss(gt, x): dist1/idx1 per gt point, dist2/idx2 per x point (:131-139)
    if _needs_graph(x, gt):
        s1, s2, q1, q2, loss, _, dist1, dist2, idx1, idx2 = ChamferMetricsFunction.apply(
            gt.contiguous(), x.contiguous(), (alpha, n_lambda, frac_21, frac_12))
        res = [loss, (s1 + s2) / 2, q1 + q2]
    else:
        dist1, dist2, idx1, idx2 = chamfer_forward(gt.detach().contiguous(), x.detach().contiguous())
        m = chamfer_metrics_raw(dist1, dist2, idx1, idx2, alpha=alpha, n_lambda=n_lambda, frac1=frac_21, frac2=frac_12)
        res = [m[:, 7], (m[:, 0] + m[:, 1]) / 2, m[:, 2] + m[:, 3]]
    if return_raw:
        res.extend([dist1, dist2, idx1, idx2])
    return res


def patch_loss_utils(module, training=False):
    """Rebind calc_cd / calc_dcd / fscore inside an imported reference `utils.loss_utils` (evaluation loops call
    them through that module: core/test_pcn.py:64, core/eval_55.py:74).

    training=True also rebinds chamfer / chamfer_sqrt / chamfer_single_side / chamfer_single_side_sqrt to the fused
    ops of `losses`.  The reference's get_loss / get_loss_PM (:33-85) look these names up as module globals when they
    run, so they then run on the fused ops unchanged."""
    module.calc_cd = calc_cd
    module.calc_dcd = calc_dcd
    module.fscore = fscore
    if training:
        from . import losses
        for name in losses.TRAINING_LOSSES:
            setattr(module, name, getattr(losses, name))
    return module
