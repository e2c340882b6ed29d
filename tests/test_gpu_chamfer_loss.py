"""The fused Chamfer training losses (ps_chamfer_loss_fwd / ps_chamfer_loss_bwd) against the reference's own expressions
(utils/loss_utils.py:10-31) evaluated with torch autograd over (a) chamfer_3DFunction live on the same GPU and (b) a CPU
Function over the oracle's Chamfer forward / backward.

Bars: the loss within 1e-6 relative (the fused loss sums in double, torch's means in fp32); gradients within 1e-5 of
the reference's, relative to its largest finite magnitude, with NaN and inf in identical positions; where no atomics
are involved (single-side kinds, only xyz1 requiring grad) the gradient is bit-identical to the composition.
"""
import json
import os
import os.path as osp
import subprocess
import sys

import numpy as np
import pytest
import torch
from torch.autograd import Function

from conftest import REFERENCE, ROOT, make_cloud
from oracle import oracle as O

pytestmark = pytest.mark.gpu

import svdformer_pointsea_b200 as ps  # noqa: E402
from svdformer_pointsea_b200 import _lib as L  # noqa: E402
from svdformer_pointsea_b200 import losses  # noqa: E402

DEV = "cuda:0"
KINDS = ["cd", "cd_sqrt", "single", "single_sqrt"]
FUSED = {"cd": losses.chamfer, "cd_sqrt": losses.chamfer_sqrt, "single": losses.chamfer_single_side,
         "single_sqrt": losses.chamfer_single_side_sqrt}


# ---------------------------------------------------------------- the reference's expressions (utils/loss_utils.py:10-31)
def ref_loss(kind, chamfer, p1, p2):
    d1, d2, _, _ = chamfer(p1, p2)
    if kind == "cd":
        return torch.mean(d1) + torch.mean(d2)
    if kind == "cd_sqrt":
        d1 = torch.mean(torch.sqrt(d1))
        d2 = torch.mean(torch.sqrt(d2))
        return (d1 + d2) / 2
    if kind == "single":
        return torch.mean(d1)
    return torch.mean(torch.sqrt(d1))


def live(p1, p2):
    return ps.chamfer_3DFunction.apply(p1.contiguous(), p2.contiguous())


class OracleChamfer(Function):
    """chamfer_3DFunction on the CPU oracle (pinned bit for bit to the reference's kernels by the goldens)."""

    @staticmethod
    def forward(ctx, xyz1, xyz2):
        d1, d2, i1, i2 = O.chamfer_fwd(xyz1.detach().numpy(), xyz2.detach().numpy())
        ctx.save_for_backward(xyz1, xyz2, torch.from_numpy(i1), torch.from_numpy(i2))
        return tuple(torch.from_numpy(a) for a in (d1, d2, i1, i2))

    @staticmethod
    def backward(ctx, gd1, gd2, _gi1, _gi2):
        xyz1, xyz2, i1, i2 = ctx.saved_tensors
        g1, g2 = O.chamfer_bwd(xyz1.detach().numpy(), xyz2.detach().numpy(), gd1.contiguous().numpy(),
                               gd2.contiguous().numpy(), i1.numpy(), i2.numpy())
        return torch.from_numpy(g1), torch.from_numpy(g2)


# ---------------------------------------------------------------- helpers
def assert_close_loss(got, want, what):
    got, want = float(got), float(want)
    assert abs(got - want) <= 1e-6 * abs(want), f"{what}: loss {got!r} vs {want!r}"


def assert_grad_close(got, want, what):
    if want is None:
        assert got is None, what
        return
    assert got is not None, what
    got, want = got.detach().cpu().double().numpy(), want.detach().cpu().double().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN positions differ"
    assert np.array_equal(np.isposinf(got), np.isposinf(want)) and np.array_equal(np.isneginf(got), np.isneginf(want)), \
        f"{what}: inf positions differ"
    fin = np.isfinite(want)
    if fin.any():
        r = np.abs(got[fin] - want[fin]).max() / max(np.abs(want[fin]).max(), 1e-30)
        assert r < 1e-5, f"{what}: rel {r:.3g}"


def run(fn, a0, b0, grad, device=DEV):
    """fn(a, b).backward() with the clouds requiring grad per `grad` ("both", "xyz1", "xyz2"): (loss, a.grad, b.grad)."""
    a = a0.detach().to(device).requires_grad_(grad in ("both", "xyz1"))  # a fresh leaf, also where .to() is a no-op
    b = b0.detach().to(device).requires_grad_(grad in ("both", "xyz2"))
    loss = fn(a, b)
    loss.backward()
    return loss.detach(), a.grad, b.grad


def pair(seed, B, N, M):
    g = torch.Generator().manual_seed(seed)
    return make_cloud(g, B, N, dup=N // 16), make_cloud(g, B, M)


SHAPES = [(3, 37, 53), (2, 301, 1037), (4, 2048, 2048), (2, 2048, 16384), (1, 16384, 16384)]
GRADS = ["both", "xyz1", "xyz2"]


# ---------------------------------------------------------------- (a) live composition on the same GPU
@pytest.mark.parametrize("grad", GRADS)
@pytest.mark.parametrize("B,N,M", SHAPES)
@pytest.mark.parametrize("kind", KINDS)
def test_matches_the_composition(kind, B, N, M, grad):
    a, b = pair(B * 7 + N + M, B, N, M)
    want = run(lambda p, q: ref_loss(kind, live, p, q), a, b, grad)
    got = run(FUSED[kind], a, b, grad)
    assert got[0].dim() == 0 and got[0].dtype == torch.float32
    assert_close_loss(got[0], want[0], f"{kind} {B}x{N}x{M}")
    assert_grad_close(got[1], want[1], f"{kind} {B}x{N}x{M} {grad} d/dxyz1")
    assert_grad_close(got[2], want[2], f"{kind} {B}x{N}x{M} {grad} d/dxyz2")
    if kind.startswith("single") and grad == "xyz1":
        assert torch.equal(got[1], want[1]), "no atomics: the gradient is the composition's, bit for bit"


# ---------------------------------------------------------------- (b) CPU oracle
@pytest.mark.parametrize("grad", GRADS)
@pytest.mark.parametrize("kind", KINDS)
def test_matches_the_oracle(kind, grad):
    a, b = pair(21, 2, 300, 260)
    want = run(lambda p, q: ref_loss(kind, OracleChamfer.apply, p, q), a, b, grad, device="cpu")
    got = run(FUSED[kind], a, b, grad)
    assert_close_loss(got[0], want[0], kind)
    assert_grad_close(got[1], want[1], f"{kind} {grad} d/dxyz1")
    assert_grad_close(got[2], want[2], f"{kind} {grad} d/dxyz2")


@pytest.mark.parametrize("B,N,M", [(2, 300, 700), (2, 2048, 16384)])
@pytest.mark.parametrize("kind", KINDS)
def test_shared_points_give_nan_and_inf_where_the_composition_does(kind, B, N, M):
    """xyz1 an exact subset of xyz2: d1 = 0 everywhere, d2 = 0 at the shared points."""
    g = torch.Generator().manual_seed(N + M)
    b = make_cloud(g, B, M)
    a = b[:, torch.randperm(M, generator=g)[:N]].contiguous()
    want = run(lambda p, q: ref_loss(kind, live, p, q), a, b, "both")
    got = run(FUSED[kind], a, b, "both")
    assert_close_loss(got[0], want[0], kind)
    assert_grad_close(got[1], want[1], f"{kind} d/dxyz1")
    assert_grad_close(got[2], want[2], f"{kind} d/dxyz2")
    if kind.endswith("sqrt"):
        assert not torch.isfinite(got[1]).all(), "the d = 0 case is exercised"
    else:
        assert torch.isfinite(got[1]).all() and torch.isfinite(got[2]).all()


def test_weighted_sums_of_several_kinds():
    """Upstream gradients other than 1, several loss nodes on the same clouds, both argument orders."""
    a, b = pair(5, 3, 2048, 4096)
    c = pair(6, 3, 512, 16)[0]
    w = (torch.rand(6, generator=torch.Generator().manual_seed(3)) * 3 - 1).tolist()

    def total(fns):
        def f(p, q):
            return (w[0] * fns["cd"](p, q) + w[1] * fns["cd_sqrt"](q, p) + w[2] * fns["single"](p, q)
                    + w[3] * fns["single_sqrt"](q, p) + w[4] * fns["cd_sqrt"](p[:, :512], c.to(p.device))
                    + w[5] * fns["single"](p, q) * fns["cd"](p, q))
        return f

    ref = {k: (lambda k: lambda p, q: ref_loss(k, live, p, q))(k) for k in KINDS}
    for grad in GRADS:
        want = run(total(ref), a, b, grad)
        got = run(total(FUSED), a, b, grad)
        assert_close_loss(got[0], want[0], f"mix {grad}")
        assert_grad_close(got[1], want[1], f"mix {grad} d/dxyz1")
        assert_grad_close(got[2], want[2], f"mix {grad} d/dxyz2")


@pytest.mark.parametrize("B,N,M", [(3, 37, 53), (32, 512, 512), (4, 2048, 16384)])
@pytest.mark.parametrize("kind", KINDS)
def test_loss_is_reproducible_and_independent_of_grad_mode(kind, B, N, M):
    a, b = pair(9, B, N, M)
    a, b = a.to(DEV), b.to(DEV)
    first = FUSED[kind](a, b)
    assert torch.equal(FUSED[kind](a, b), first)
    with torch.no_grad():
        assert torch.equal(FUSED[kind](a.requires_grad_(True), b), first)
    assert torch.equal(FUSED[kind](a, b).detach(), first)  # a requires grad: the autograd Function
    a.requires_grad_(False)


def test_launch_counts():
    """Forward: the Chamfer forward's launches plus one.  Backward: plain stores and, when a scattered term lands in a
    requested buffer, one atomic pass."""
    for B, N, M in [(3, 37, 53), (4, 2048, 16384)]:
        a, b = pair(2, B, N, M)
        a, b = a.to(DEV), b.to(DEV)
        sums = torch.empty(6, device=DEV, dtype=torch.float64)
        L.launch_count(reset=True)
        ps.chamfer_forward(a, b, sums=sums)
        n_fwd = L.launch_count()
        for kind in KINDS:
            L.launch_count(reset=True)
            loss, d1, d2, i1, i2 = losses.chamfer_loss_forward(a, b, kind)
            assert L.launch_count() == n_fwd + 1, kind
            one = torch.ones((), device=DEV)
            for need1, need2 in ((True, True), (True, False), (False, True)):
                L.launch_count(reset=True)
                losses.chamfer_loss_backward(a, b, d1, d2, i1, i2, one, kind, need1, need2)
                scatters = need2 or (need1 and not kind.startswith("single"))
                assert L.launch_count() == (2 if scatters else 1), (kind, need1, need2)


def bwd_into(a, b, d1, d2, i1, i2, kind, g1, g2):
    """ps_chamfer_loss_bwd into caller-owned buffers (None: NULL), with an upstream gradient of 1."""
    one = torch.ones((), device=DEV)
    B, N, M = a.size(0), a.size(1), b.size(1)
    L.check(L.load().ps_chamfer_loss_bwd(L.ptr(a), L.ptr(b), L.ptr(d1), L.ptr(d2), L.ptr(i1), L.ptr(i2), L.ptr(one),
                                         None if g1 is None else L.ptr(g1), None if g2 is None else L.ptr(g2),
                                         losses.LOSS_KINDS[kind], B, N, M, 0, L.stream_ptr(0)), "ps_chamfer_loss_bwd")


@pytest.mark.parametrize("kind", KINDS)
def test_buffers_are_fully_overwritten(kind):
    """Gradient buffers filled with NaN before the call: nothing of their old contents survives, and a cloud that no
    term reaches gets exact zeros (xyz2 of a single-side loss whose xyz1 does not require grad still gets d1's scatter)."""
    a, b = pair(4, 2, 700, 1300)
    a, b = a.to(DEV), b.to(DEV)
    _, d1, d2, i1, i2 = losses.chamfer_loss_forward(a, b, kind)
    g1, g2 = torch.full_like(a, float("nan")), torch.full_like(b, float("nan"))
    bwd_into(a, b, d1, d2, i1, i2, kind, g1, g2)
    assert torch.isfinite(g1).all() and torch.isfinite(g2).all()
    want1, want2 = losses.chamfer_loss_backward(a, b, d1, d2, i1, i2, torch.ones((), device=DEV), kind)
    assert_grad_close(g1, want1, f"{kind} d/dxyz1")
    assert_grad_close(g2, want2, f"{kind} d/dxyz2")
    g2_only = torch.full_like(b, float("nan"))
    bwd_into(a, b, d1, d2, i1, i2, kind, None, g2_only)
    assert_grad_close(g2_only, want2, f"{kind} d/dxyz2 alone")
    if kind.startswith("single"):
        hit = torch.zeros(2, 1300, dtype=torch.bool, device=DEV)
        hit.scatter_(1, i1.long(), True)
        assert (~hit).any() and torch.equal(g2_only[~hit], torch.zeros_like(g2_only[~hit]))
    g1_only = torch.full_like(a, float("nan"))
    bwd_into(a, b, d1, d2, i1, i2, kind, g1_only, None)
    assert_grad_close(g1_only, want1, f"{kind} d/dxyz1 alone")


@pytest.mark.parametrize("kind", KINDS)
def test_empty_batch(kind):
    """B = 0: a NaN loss (torch.mean of an empty tensor) and empty gradients, as the composition gives."""
    want = run(lambda p, q: ref_loss(kind, live, p, q), torch.zeros(0, 64, 3), torch.zeros(0, 80, 3), "both")
    got = run(FUSED[kind], torch.zeros(0, 64, 3), torch.zeros(0, 80, 3), "both")
    assert torch.isnan(want[0]) and torch.isnan(got[0])
    assert got[1].shape == (0, 64, 3) and got[2].shape == (0, 80, 3)


@pytest.mark.parametrize("kind", KINDS)
def test_cuda_graph_capture_matches_eager(kind):
    a0, b0 = pair(31, 4, 2048, 16384)
    a1, b1 = pair(32, 4, 2048, 16384)
    sa, sb = a0.to(DEV).requires_grad_(True), b0.to(DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            torch.autograd.grad(FUSED[kind](sa, sb), [sa])
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = FUSED[kind](sa, sb)
        (ga,) = torch.autograd.grad(loss, [sa])
    with torch.no_grad():
        sa.copy_(a1.to(DEV))
        sb.copy_(b1.to(DEV))
    graph.replay()
    torch.cuda.synchronize()
    want_loss, want_ga, _ = run(FUSED[kind], a1, b1, "xyz1")
    assert torch.equal(loss, want_loss)
    assert_grad_close(ga, want_ga, f"graph {kind}")
    if kind.startswith("single"):
        assert torch.equal(ga, want_ga)


def test_double_backward_is_refused():
    a, b = pair(1, 2, 300, 400)
    a = a.to(DEV).requires_grad_(True)
    (g,) = torch.autograd.grad(losses.chamfer(a, b.to(DEV)), [a], create_graph=True)
    with pytest.raises(RuntimeError):
        g.sum().backward()


STAND_IN_LOSS_UTILS = '''
import torch
from svdformer_pointsea_b200 import chamfer_3DFunction, fps_subsample

def _cd(p1, p2):
    return chamfer_3DFunction.apply(p1.contiguous(), p2.contiguous())

def chamfer(p1, p2):
    d1, d2, _, _ = _cd(p1, p2)
    return torch.mean(d1) + torch.mean(d2)

def chamfer_sqrt(p1, p2):
    d1, d2, _, _ = _cd(p1, p2)
    d1 = torch.mean(torch.sqrt(d1))
    d2 = torch.mean(torch.sqrt(d2))
    return (d1 + d2) / 2

def chamfer_single_side(pcd1, pcd2):
    d1, d2, _, _ = _cd(pcd1, pcd2)
    return torch.mean(d1)

def chamfer_single_side_sqrt(pcd1, pcd2):
    d1, d2, _, _ = _cd(pcd1, pcd2)
    return torch.mean(torch.sqrt(d1))

def get_loss(pcds_pred, gt, sqrt=True):
    CD = chamfer_sqrt if sqrt else chamfer
    Pc, P1, P2 = pcds_pred
    gt_2 = fps_subsample(gt, P1.shape[1])
    gt_c = fps_subsample(gt_2, Pc.shape[1])
    cdc, cd1, cd2 = CD(Pc, gt_c), CD(P1, gt_2), CD(P2, gt)
    return cdc + cd1 + cd2, [cdc, cd1, cd2]

def get_loss_PM(pcds_pred, partial, gt, sqrt=True):
    PM = chamfer_single_side_sqrt if sqrt else chamfer_single_side
    loss_all, losses = get_loss(pcds_pred, gt, sqrt)
    return loss_all + PM(partial, pcds_pred[-1]), losses
'''


@pytest.mark.parametrize("sqrt", [True, False])
def test_patched_stand_in_loss_utils_runs_get_loss_on_the_fused_ops(sqrt):
    """A module shaped like utils/loss_utils.py (its get_loss / get_loss_PM pick the Chamfer losses up as module
    globals at call time): after patch_loss_utils(training=True) the same functions give the same loss and gradients,
    and no chamfer_3DFunction runs any more."""
    import types
    g = torch.Generator().manual_seed(77)
    gt = make_cloud(g, 4, 16384).to(DEV)
    partial = make_cloud(g, 4, 2048).to(DEV)
    preds0 = [make_cloud(g, 4, n).to(DEV) for n in (512, 2048, 16384)]
    res = []
    for training in (False, True):
        m = types.ModuleType("stand_in_loss_utils")
        exec(STAND_IN_LOSS_UTILS, m.__dict__)
        if training:
            ps.patch_loss_utils(m, training=True)
            m._cd = None  # the composition is unreachable now
        preds = [p.clone().requires_grad_(True) for p in preds0]
        loss, parts = m.get_loss_PM(preds, partial, gt, sqrt=sqrt)
        loss.backward()
        res.append((loss.detach(), [p.grad for p in preds]))
    assert_close_loss(res[1][0], res[0][0], "get_loss_PM")
    for k in range(3):
        assert_grad_close(res[1][1][k], res[0][1][k], f"get_loss_PM d/dP{k}")


# ---------------------------------------------------------------- C4: the reference's get_loss / get_loss_PM
def _c4(arm, loss, impl):
    if not osp.isdir(REFERENCE):
        pytest.skip(f"needs a checkout of the reference at {REFERENCE} (or set POINTSEA_REFERENCE)")
    if not osp.exists(osp.join(ROOT, "oracle", "_ref", "ref_pointnet2_ext.so")):
        pytest.skip("oracle/_ref not built (python __graft_entry__.py build builds it beside a reference checkout)")
    p = subprocess.run([sys.executable, osp.join(ROOT, "tools", "bench_configs.py"), "c4", "--arm", arm, "--iters", "1",
                        "--batch", "2", "--loss", loss, "--loss-impl", impl], capture_output=True, text=True,
                       timeout=900, env=dict(os.environ, POINTSEA_REFERENCE_TREE=REFERENCE))
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert p.returncode == 0 and lines, (p.stderr or p.stdout)[-3000:]
    d = json.loads(lines[-1])
    assert "loss" in d, d
    return d


@pytest.mark.parametrize("loss", ["get_loss", "get_loss_PM"])
def test_c4_reference_loss_on_the_fused_ops(loss):
    ref = _c4("ref", loss, "composed")
    ours = _c4("ours", loss, "fused")
    assert ours["fused_loss_calls"] > 0, "the reference's loss did not pick up the rebound names"
    assert abs(ours["loss"] - ref["loss"]) <= 1e-6 * abs(ref["loss"]), (ours["loss"], ref["loss"])
    for x, y in zip(ours["losses"], ref["losses"]):
        assert abs(x - y) <= 1e-6 * abs(y), (ours["losses"], ref["losses"])
