"""torch_scatter.scatter with reduce="max" on the sm_100a kernel of csrc/scatter.cu (ps_scatter_max).

PointSea's renderer draws its depth maps with one call (models_PointSea/mv_utils_zs.py:1,130):
    scatter(src, index, dim, out=..., reduce="max")
This module follows torch_scatter 2.x for that call: the index is broadcast to src as torch_scatter.utils.broadcast
does, `out` is updated in place and returned, a fresh output is 0 where nothing arrives, and the result is
differentiable with respect to src (the gradient goes to the argmax positions).  Ties send the whole gradient to the
lowest position, deterministically; torch_scatter's arg pass lets the last writer win, and torch.scatter_reduce's
backward splits the gradient between tied positions.  Other reductions are not provided: an installed torch_scatter
takes precedence over the drop-in of svdformer_pointsea_b200.dropin (DROPIN_FALLBACK_PATH) and covers them.
"""
import torch

from . import _lib as L


def _broadcast(index, src, dim):
    """torch_scatter.utils.broadcast(index, src, dim)."""
    if index.dim() == 1:
        for _ in range(dim):
            index = index.unsqueeze(0)
    for _ in range(index.dim(), src.dim()):
        index = index.unsqueeze(-1)
    return index.expand(src.size())


def _scatter_max(src, index, dim, out, shape, want_arg):
    """src, index contiguous (index broadcast to src); out None (fresh output of `shape`) or contiguous float32.
    Returns (out, argmax or None)."""
    fresh = out is None
    if fresh:
        out = torch.empty(shape, dtype=torch.float32, device=src.device)
    outer = 1
    for s in src.shape[:dim]:
        outer *= s
    inner = 1
    for s in src.shape[dim + 1:]:
        inner *= s
    arg = torch.empty(out.shape, dtype=torch.int64, device=out.device) if want_arg else None
    dev = L.same_device(src, index, out)
    L.check(L.load().ps_scatter_max(L.ptr(src), L.ptr(index), L.ptr(out), L.ptr(arg) if arg is not None else None,
                                    outer, src.shape[dim], inner, out.shape[dim], 1 if fresh else 0, dev,
                                    L.stream_ptr(dev)), "ps_scatter_max")
    return out, arg


class ScatterMax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, index, dim, out, shape):
        if out is not None:
            ctx.mark_dirty(out)
        out, arg = _scatter_max(src, index, dim, out, shape, True)
        ctx.mark_non_differentiable(arg)
        ctx.save_for_backward(arg)
        ctx.dim, ctx.src_shape = dim, src.shape
        return out, arg

    @staticmethod
    def backward(ctx, grad_out, _grad_arg):
        (arg,) = ctx.saved_tensors
        shape = list(ctx.src_shape)
        shape[ctx.dim] += 1  # positions without a source (arg == E) land in the extra slot, which is cut off
        grad = grad_out.new_zeros(shape).scatter_(ctx.dim, arg, grad_out)
        return grad.narrow(ctx.dim, 0, shape[ctx.dim] - 1), None, None, None, None


def scatter(src, index, dim=-1, out=None, dim_size=None, reduce="sum"):
    """torch_scatter.scatter for reduce="max": src float32, index int64 (broadcast to src along `dim`), on one CUDA
    device; the work goes on that device's current stream.  With `out` (contiguous float32, src's shape except along
    `dim`) the max includes out's values and out is updated in place and returned; otherwise the output has
    `dim_size` (default index.max() + 1) positions along `dim` and 0 where nothing arrives.  Index values outside
    [0, size along dim) are skipped."""
    if reduce != "max":
        raise NotImplementedError(
            f"svdformer_pointsea_b200.scatter covers reduce='max', the call PointSea's renderer makes; got "
            f"reduce={reduce!r}. An installed torch_scatter takes precedence over this drop-in and provides the other "
            "reductions.")
    for t, name in ((src, "src"), (index, "index")):
        if not isinstance(t, torch.Tensor):
            raise L.PointSeaError(f"{name} must be a torch.Tensor")
    if src.dtype != torch.float32:
        raise L.PointSeaError(f"src must be a float32 tensor, got {src.dtype}")
    if index.dtype != torch.int64:
        raise L.PointSeaError(f"index must be an int64 tensor, got {index.dtype}")
    if not src.is_cuda or not index.is_cuda:
        raise L.PointSeaError("src and index must be CUDA tensors (CPU not supported)")
    if src.dim() == 0:
        raise L.PointSeaError("src must have at least one dimension")
    if not -src.dim() <= dim < src.dim():
        raise IndexError(f"dim {dim} out of range for a {src.dim()}-dimensional src")
    dim = dim + src.dim() if dim < 0 else dim
    index = _broadcast(index, src, dim).contiguous()
    src = src.contiguous()
    if out is None:
        shape = list(src.shape)
        if dim_size is not None:
            shape[dim] = int(dim_size)
        else:
            shape[dim] = int(index.max()) + 1 if index.numel() > 0 else 0
    else:
        if not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or out.device != src.device:
            raise L.PointSeaError(f"out must be a float32 tensor on {src.device}")
        if not out.is_contiguous():
            raise L.PointSeaError("out must be a contiguous tensor")
        if out.dim() != src.dim() or any(a != b for d, (a, b) in enumerate(zip(out.shape, src.shape)) if d != dim):
            raise L.PointSeaError(f"out has shape {tuple(out.shape)}; expected {tuple(src.shape)} except along dim {dim}")
        if out.requires_grad:
            raise L.PointSeaError("out must not require grad: it carries no gradient")
        shape = None
    if torch.is_grad_enabled() and src.requires_grad:
        return ScatterMax.apply(src, index, dim, out, shape)[0]
    res = _scatter_max(src, index, dim, out, shape, False)[0]
    if out is not None:  # written through a raw pointer: let autograd see the in-place update, as mark_dirty does
        torch.autograd.graph.increment_version(out)
    return res
