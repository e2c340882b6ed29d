"""Gradients of calc_cd / calc_dcd (ps_chamfer_metrics_bwd + ps_chamfer_bwd) against torch autograd over the
reference's own expressions (oracle.torch_cd_terms, oracle.torch_dcd_from_raw, utils/loss_utils.py:98-155), on top of
(a) chamfer_3DFunction live on the same GPU and (b) a CPU Function over the oracle's Chamfer forward / backward.

Bars: gradients w.r.t. both clouds within 1e-5 of the reference's, relative to its largest finite magnitude; NaN and
inf entries in identical positions (a sqrt term at d = 0 is NaN in the reference and must be here too).
"""
import types

import numpy as np
import pytest
import torch
from torch.autograd import Function

from conftest import make_cloud
from oracle import oracle as O

pytestmark = pytest.mark.gpu

import svdformer_pointsea_b200 as ps  # noqa: E402

DEV = "cuda:0"


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def assert_grad_close(got, want, what):
    if want is None:
        assert got is None, what
        return
    got, want = got.detach().cpu().double().numpy(), want.detach().cpu().double().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN positions differ"
    assert np.array_equal(np.isposinf(got), np.isposinf(want)) and np.array_equal(np.isneginf(got), np.isneginf(want)), \
        f"{what}: inf positions differ"
    fin = np.isfinite(want)
    if fin.any():
        r = rel(got[fin], want[fin])
        assert r < 1e-5, f"{what}: rel {r:.3g}"


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
        g1, g2 = O.chamfer_bwd(xyz1.detach().numpy(), xyz2.detach().numpy(), gd1.numpy(), gd2.numpy(), i1.numpy(), i2.numpy())
        return torch.from_numpy(g1), torch.from_numpy(g2)


# ---------------------------------------------------------------- the reference's calc_cd / calc_dcd, restated
def ref_calc_cd(output, gt, chamfer, calc_f1=False, return_raw=False, separate=False):
    dist1, dist2, idx1, idx2 = chamfer(gt, output)
    cd_p, cd_t = O.torch_cd_terms(dist1, dist2)
    if separate:
        res = [torch.cat([torch.sqrt(dist1).mean(1).unsqueeze(0), torch.sqrt(dist2).mean(1).unsqueeze(0)]),
               torch.cat([dist1.mean(1).unsqueeze(0), dist2.mean(1).unsqueeze(0)])]
    else:
        res = [cd_p, cd_t]
    if calc_f1:
        res.append(O.torch_fscore(dist1, dist2)[0])
    if return_raw:
        res.extend([dist1, dist2, idx1, idx2])
    return res


def ref_calc_dcd(x, gt, chamfer, alpha=1000, n_lambda=1, return_raw=False, non_reg=False):
    x, gt = x.float(), gt.float()
    cd_p, cd_t, dist1, dist2, idx1, idx2 = ref_calc_cd(x, gt, chamfer, return_raw=True)
    loss = O.torch_dcd_from_raw(dist1, dist2, idx1, idx2, x.shape[1], gt.shape[1], alpha, n_lambda, non_reg)
    res = [loss, cd_p, cd_t]
    if return_raw:
        res.extend([dist1, dist2, idx1, idx2])
    return res


def outputs(impl, x, gt, p):
    """Every differentiable output of calc_dcd(x, gt, **p, return_raw=True), calc_cd(x, gt) and
    calc_cd(x, gt, separate=True)."""
    if impl == "ours":
        loss, cd_p, cd_t, d1, d2, _, _ = ps.calc_dcd(x, gt, return_raw=True, **p)
        cc_p, cc_t = ps.calc_cd(x, gt)
        sq, mn = ps.calc_cd(x, gt, separate=True)
    else:
        loss, cd_p, cd_t, d1, d2, _, _ = ref_calc_dcd(x, gt, impl, return_raw=True, **p)
        cc_p, cc_t = ref_calc_cd(x, gt, impl)
        sq, mn = ref_calc_cd(x, gt, impl, separate=True)
    return {"dcd": loss, "cd_p": cd_p, "cd_t": cd_t, "d1": d1, "d2": d2, "cc_p": cc_p, "cc_t": cc_t, "sq": sq, "mn": mn}


LOSSES = {
    "dcd": lambda o, w: o["dcd"].mean(),
    "cd_p": lambda o, w: o["cd_p"].mean(),
    "cd_t": lambda o, w: o["cd_t"].mean(),
    "calc_cd_p": lambda o, w: o["cc_p"].mean(),
    "calc_cd_t": lambda o, w: o["cc_t"].mean(),
    "sep_sqrt1": lambda o, w: o["sq"][0].mean(),
    "sep_sqrt2": lambda o, w: o["sq"][1].mean(),
    "sep_mean1": lambda o, w: o["mn"][0].mean(),
    "sep_mean2": lambda o, w: o["mn"][1].mean(),
    "mix": lambda o, w: (w["c"][0] * o["dcd"] + w["c"][1] * o["cd_p"] + w["c"][2] * o["cd_t"] + w["c"][3] * o["sq"][0]
                         + w["c"][4] * o["sq"][1] + w["c"][5] * o["mn"][0] + w["c"][6] * o["mn"][1]
                         + w["c"][7] * o["cc_p"] + w["c"][8] * o["cc_t"]).sum(),
    "raw_dcd": lambda o, w: (w["r1"] * o["d1"]).sum() + (w["r2"] * o["d2"]).sum() + o["dcd"].mean(),
    "raw_only": lambda o, w: (w["r1"] * o["d1"]).mean() + (w["r2"] * o["d2"]).mean(),
}
FINITE_LOSSES = ["dcd", "cd_t", "calc_cd_t", "sep_mean1", "sep_mean2"]  # no sqrt term: finite even where d = 0


def weights(seed, B, n_x, n_gt, device):
    g = torch.Generator().manual_seed(seed)
    w = {"c": torch.rand(9, B, generator=g) * 2 - 0.5, "r1": torch.rand(B, n_gt, generator=g) - 0.5,
         "r2": torch.rand(B, n_x, generator=g) - 0.5}
    return {k: v.to(device) for k, v in w.items()}


def all_grads(impl, x0, gt0, p, names, w):
    x = x0.clone().requires_grad_(True)
    gt = gt0.clone().requires_grad_(True)
    o = outputs(impl, x, gt, p)
    return {n: torch.autograd.grad(LOSSES[n](o, w), [x, gt], retain_graph=True) for n in names}


def compare(got, want, tag):
    for name in want:
        assert_grad_close(got[name][0], want[name][0], f"{tag} {name} d/dx")
        assert_grad_close(got[name][1], want[name][1], f"{tag} {name} d/dgt")


def clouds(seed, B, n_x, n_gt, kind):
    """gt (B,n_gt,3) and x (B,n_x,3): x near gt with exact duplicates ("dup", so hit counts > 1 and Chamfer ties), or
    an exact subset of gt ("subset", so distances are exactly 0)."""
    g = torch.Generator().manual_seed(seed)
    gt = make_cloud(g, B, n_gt)
    if kind == "subset":
        return gt[:, torch.randperm(n_gt, generator=g)[:n_x]].contiguous(), gt
    x = gt[:, torch.randperm(n_gt, generator=g)[:n_x]] if n_x <= n_gt else make_cloud(g, B, n_x)
    x = x + 0.004 * torch.randn(x.shape, generator=g)
    dup = n_x // 8
    x[:, n_x - dup:] = x[:, :dup]
    return x.contiguous(), gt


PARAMS = {"default": {}, "nonreg": dict(alpha=40, n_lambda=0.5, non_reg=True), "lambda2": dict(n_lambda=2),
          "lambda1.7": dict(n_lambda=1.7)}
SHAPES = [(4, 2048, 2048), (2, 16384, 16384), (2, 8192, 16384), (1, 30000, 25000)]


# ---------------------------------------------------------------- (a) live reference on the same GPU
@pytest.mark.parametrize("B,n_x,n_gt", SHAPES)
@pytest.mark.parametrize("pname", list(PARAMS))
def test_grads_vs_live_reference(B, n_x, n_gt, pname):
    """All losses; the last shape runs the global-memory histograms (n_x + n_gt > 40960)."""
    x, gt = clouds(n_x + n_gt, B, n_x, n_gt, "dup")
    x, gt = x.to(DEV), gt.to(DEV)
    w = weights(B + n_x, B, n_x, n_gt, DEV)
    want = all_grads(ps.chamfer_3DFunction.apply, x, gt, PARAMS[pname], list(LOSSES), w)
    got = all_grads("ours", x, gt, PARAMS[pname], list(LOSSES), w)
    compare(got, want, f"{pname} {B}x{n_x}x{n_gt}")


@pytest.mark.parametrize("B,n_x,n_gt", [(4, 2048, 2048), (2, 8192, 16384), (1, 25000, 30000)])
def test_grads_where_distances_are_zero(B, n_x, n_gt):
    """x an exact subset of gt: a loss with a sqrt term is NaN in the reference's positions, the others finite."""
    x, gt = clouds(n_x * 3 + n_gt, B, n_x, n_gt, "subset")
    x, gt = x.to(DEV), gt.to(DEV)
    w = weights(B + n_gt, B, n_x, n_gt, DEV)
    p = PARAMS["default"]
    want = all_grads(ps.chamfer_3DFunction.apply, x, gt, p, list(LOSSES), w)
    got = all_grads("ours", x, gt, p, list(LOSSES), w)
    compare(got, want, f"subset {B}x{n_x}x{n_gt}")
    assert torch.isnan(got["cd_p"][0]).any() and torch.isnan(got["mix"][1]).any()  # the case is exercised
    for name in FINITE_LOSSES:
        assert all(torch.isfinite(g).all() for g in got[name]), name


# ---------------------------------------------------------------- (b) CPU oracle
@pytest.mark.parametrize("kind", ["dup", "subset"])
@pytest.mark.parametrize("pname", list(PARAMS))
def test_grads_vs_oracle(kind, pname):
    B, n_x, n_gt = 2, 300, 256 if kind == "dup" else 700
    x, gt = clouds(17, B, n_x, n_gt, kind)
    w = weights(5, B, n_x, n_gt, "cpu")
    want = all_grads(OracleChamfer.apply, x, gt, PARAMS[pname], list(LOSSES), w)
    got = all_grads("ours", x.to(DEV), gt.to(DEV), PARAMS[pname], list(LOSSES), {k: v.to(DEV) for k, v in w.items()})
    compare(got, want, f"oracle {kind} {pname}")


# ---------------------------------------------------------------- autograd plumbing
@pytest.mark.parametrize("which", ["x", "gt"])
def test_one_cloud_requiring_grad(which):
    B, n_x, n_gt = 3, 2048, 4096
    x0, gt0 = clouds(3, B, n_x, n_gt, "dup")
    res = {}
    for impl in ("ours", ps.chamfer_3DFunction.apply):
        x, gt = x0.to(DEV).requires_grad_(which == "x"), gt0.to(DEV).requires_grad_(which == "gt")
        o = outputs(impl, x, gt, PARAMS["nonreg"])
        (o["dcd"].mean() + 0.5 * o["cd_p"].sum() + o["cd_t"].mean()).backward()
        res[impl == "ours"] = (x.grad, gt.grad)
    assert (res[True][0] is None) == (which == "gt") and (res[True][1] is None) == (which == "x")
    assert_grad_close(res[True][0], res[False][0], "x")
    assert_grad_close(res[True][1], res[False][1], "gt")


def test_forward_values_identical_with_and_without_grad():
    x0, gt0 = clouds(11, 3, 3000, 2500, "dup")
    x0, gt0 = x0.to(DEV), gt0.to(DEV)
    for p in PARAMS.values():
        calls = [lambda x, gt: ps.calc_dcd(x, gt, return_raw=True, **p),
                 lambda x, gt: ps.calc_cd(x, gt, calc_f1=True, return_raw=True),
                 lambda x, gt: ps.calc_cd(x, gt, calc_f1=True, separate=True)]
        for call in calls:
            with torch.no_grad():
                want = call(x0, gt0)
            got = call(x0.clone().requires_grad_(True), gt0.clone().requires_grad_(True))
            plain = call(x0, gt0)  # grad mode on, nothing requires grad: the no-graph path
            for a, b, c in zip(got, want, plain):
                assert torch.equal(a.detach(), b) and torch.equal(c, b)


@pytest.mark.parametrize("grad", ["x", "gt", "both", "none"])
def test_requires_grad_matches_reference(grad):
    x0, gt0 = clouds(12, 2, 1024, 1500, "dup")
    flags = {}
    for impl in ("ours", ps.chamfer_3DFunction.apply):
        x = x0.to(DEV).requires_grad_(grad in ("x", "both"))
        gt = gt0.to(DEV).requires_grad_(grad in ("gt", "both"))
        if impl == "ours":
            res = [ps.calc_dcd(x, gt, return_raw=True), ps.calc_cd(x, gt, calc_f1=True, return_raw=True),
                   ps.calc_cd(x, gt, calc_f1=True, separate=True)]
        else:
            res = [ref_calc_dcd(x, gt, impl, return_raw=True), ref_calc_cd(x, gt, impl, calc_f1=True, return_raw=True),
                   ref_calc_cd(x, gt, impl, calc_f1=True, separate=True)]
        flags[impl == "ours"] = [[t.requires_grad for t in r] for r in res]
    assert flags[True] == flags[False]
    if grad != "none":
        assert flags[True][0] == [True, True, True, True, True, False, False]


def test_gradients_flow_through_patched_loss_utils():
    """A DCD term added to a training loss through a patched utils.loss_utils contributes its gradient."""
    m = ps.patch_loss_utils(types.ModuleType("fake_loss_utils"))
    x0, gt0 = clouds(13, 4, 2048, 16384, "dup")
    grads = []
    for calc_dcd in (m.calc_dcd, lambda x, gt: ref_calc_dcd(x, gt, ps.chamfer_3DFunction.apply)):
        x = x0.to(DEV).requires_grad_(True)
        gt = gt0.to(DEV)
        loss = (x ** 2).mean() + 0.5 * calc_dcd(x, gt)[0].mean()
        loss.backward()
        grads.append(x.grad)
    assert_grad_close(grads[0], grads[1], "patched calc_dcd")
    assert not torch.equal(grads[0], 2 * x0.to(DEV) / x0.numel())  # the DCD term did contribute
