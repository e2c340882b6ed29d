"""The torch_scatter drop-in (svdformer_pointsea_b200.scatter, ps_scatter_max) against torch on the same GPU.

Values are compared bit for bit (as int32 views, so NaN patterns count too) with
    out.scatter_reduce_(dim, index, src, "amax", include_self=True)                        when `out=` is given
    full(-FLT_MAX).scatter_reduce_(..., include_self=True).masked_fill_(== -FLT_MAX, 0)      for a fresh output
the second being torch_scatter's own rule.  A max does not depend on the order of the updates, so nothing here has a
tolerance.  The last test runs PointSea end to end with torch_scatter resolved to the drop-in.
"""
import json
import os
import os.path as osp
import subprocess
import sys

import pytest
import torch

from conftest import REFERENCE, ROOT
from svdformer_pointsea_b200.scatter import _scatter_max, scatter

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
LOWEST = -torch.finfo(torch.float32).max


def bits(t):
    return t.contiguous().view(torch.int32)


def assert_bits_equal(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    assert torch.equal(bits(a), bits(b)), (a - b).abs().max()


def ref_max(src, full_index, dim, out=None, dim_size=None):
    """torch's scatter_reduce over an index already of src's shape; out None: torch_scatter's fresh rule."""
    if out is not None:
        return out.clone().scatter_reduce_(dim, full_index, src, "amax", include_self=True)
    shape = list(src.shape)
    shape[dim] = dim_size
    r = torch.full(shape, LOWEST, device=src.device).scatter_reduce_(dim, full_index, src, "amax", include_self=True)
    return r.masked_fill_(r == LOWEST, 0.0)


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


# (name, src shape, dim, index builder: (src, D, g) -> (index passed, index of src's shape), D)
def _full(src, D, g):
    i = torch.randint(0, D, src.shape, generator=g, device=DEV)
    return i, i


def _one_d(src, D, g):  # 1-D index along dim 1 of a 3-D src: unsqueezed in front and at the end, then expanded
    i = torch.randint(0, D, (src.shape[1],), generator=g, device=DEV)
    return i, i.view(1, -1, 1).expand_as(src)


def _fewer_dims(src, D, g):  # (a, E) index for an (a, E, c) src: unsqueezed at the end
    i = torch.randint(0, D, src.shape[:2], generator=g, device=DEV)
    return i, i.unsqueeze(-1).expand_as(src)


CASES = [
    ("2d_dim1", (8, 2048), 1, _full, 4096),
    ("2d_dim-1", (8, 2048), -1, _full, 64),
    ("2d_dim0", (3000, 6), 0, _full, 50),
    ("3d_inner5", (4, 300, 5), 1, _full, 37),
    ("3d_dim-1", (4, 3, 300), -1, _full, 17),
    ("1d_index_broadcast", (4, 300, 5), 1, _one_d, 40),
    ("index_fewer_dims", (4, 300, 5), 1, _fewer_dims, 40),
    ("1d_src", (5000,), 0, _full, 100),
]


@pytest.mark.parametrize("name,shape,dim,make_index,D", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("mode", ["out", "fresh_dim_size", "fresh_inferred"])
def test_values_bit_identical_to_torch(name, shape, dim, make_index, D, mode):
    g = gen(sum(map(ord, name)))
    src = torch.randn(shape, generator=g, device=DEV)
    index, full = make_index(src, D, g)
    d = dim % src.dim()
    if mode == "out":
        oshape = list(shape)
        oshape[d] = D
        out = torch.randn(oshape, generator=g, device=DEV)
        want = ref_max(src, full, d, out=out)
        got = scatter(src, index, dim, out=out, reduce="max")
        assert got is out
    else:
        size = D if mode == "fresh_dim_size" else int(full.max()) + 1
        want = ref_max(src, full, d, dim_size=size)
        got = scatter(src, index, dim, dim_size=size if mode == "fresh_dim_size" else None, reduce="max")
    assert_bits_equal(got, want)


@pytest.mark.parametrize("pattern", ["uniform", "patch40", "one_pixel"])
@pytest.mark.parametrize("points", [2048, 16384])
def test_pointsea_render_shape(pattern, points):
    """mv_utils_zs.py:130: src (32*3, points) of depths into out (96, 224*224) pre-filled with zeros."""
    g = gen(points)
    B, H = 96, 224
    src = torch.rand(B, points, generator=g, device=DEV) * 2.0
    if pattern == "uniform":
        index = torch.randint(0, H * H, (B, points), generator=g, device=DEV)
    elif pattern == "patch40":
        y = torch.randint(92, 132, (B, points), generator=g, device=DEV)
        x = torch.randint(92, 132, (B, points), generator=g, device=DEV)
        index = y * H + x
    else:
        index = torch.full((B, points), H * H // 2 + H // 2, dtype=torch.int64, device=DEV)
    out = torch.zeros(B, H * H, device=DEV)
    want = ref_max(src, index, 1, out=out)
    got = scatter(src, index, 1, out=out, reduce="max")
    assert got is out
    assert_bits_equal(got, want)


def test_non_contiguous_src_and_index():
    g = gen(7)
    base = torch.randn(600, 8, generator=g, device=DEV)
    src = base.t()  # (8, 600), not contiguous
    index = torch.randint(0, 33, (600, 8), generator=g, device=DEV).t()
    assert not src.is_contiguous() and not index.is_contiguous()
    assert_bits_equal(scatter(src, index, 1, dim_size=33, reduce="max"),
                      ref_max(src.contiguous(), index.contiguous(), 1, dim_size=33))
    out = torch.randn(8, 33, generator=g, device=DEV)
    assert_bits_equal(scatter(src, index, 1, out=out.clone(), reduce="max"), ref_max(src, index, 1, out=out))


def test_empty_src():
    src = torch.empty(4, 0, device=DEV)
    index = torch.empty(4, 0, dtype=torch.int64, device=DEV)
    assert scatter(src, index, 1, reduce="max").shape == (4, 0)
    r = scatter(src, index, 1, dim_size=7, reduce="max")
    assert r.shape == (4, 7) and torch.equal(bits(r), torch.zeros(4, 7, dtype=torch.int32, device=DEV))
    out = torch.randn(4, 7, device=DEV)
    keep = out.clone()
    assert scatter(src, index, 1, out=out, reduce="max") is out and torch.equal(bits(out), bits(keep))


@pytest.mark.parametrize("fresh", [True, False])
def test_heavy_collisions_and_ties(fresh):
    """Everything to one slot (and to a few slots), values from a small set so that most are tied."""
    g = gen(11)
    for D, n in ((1, 200000), (3, 100000)):
        src = torch.randint(-3, 4, (2, n), generator=g, device=DEV).float() * 0.5
        index = torch.randint(0, D, (2, n), generator=g, device=DEV)
        out = None if fresh else torch.randn(2, D, generator=g, device=DEV)
        want = ref_max(src, index, 1, out=out, dim_size=D)
        got = scatter(src, index, 1, out=None if fresh else out.clone(), dim_size=D, reduce="max")
        assert_bits_equal(got, want)


@pytest.mark.parametrize("fresh", [True, False])
def test_infinities_and_nan_propagation(fresh):
    g = gen(13)
    src = torch.randn(3, 4000, generator=g, device=DEV)
    index = torch.randint(0, 50, (3, 4000), generator=g, device=DEV)
    src[0, :10] = float("inf")
    src[1, 100:400] = float("-inf")
    src[2, 7] = float("nan")
    src[2, 900] = float("nan")
    index[1] = torch.where(index[1] == 49, 48, index[1])
    index[1, 100:400] = 49  # slot 49 of row 1 receives only -inf
    out = None if fresh else torch.randn(3, 50, generator=g, device=DEV)
    want = ref_max(src, index, 1, out=out, dim_size=50)
    got = scatter(src, index, 1, out=None if fresh else out.clone(), dim_size=50, reduce="max")
    assert torch.isnan(got[2, index[2, 7]]) and torch.isnan(got[2, index[2, 900]])
    assert_bits_equal(got, want)  # torch keeps float("nan")'s pattern, which is the canonical one


def test_negative_nan_and_all_negative_infinity_slots():
    """A negative NaN pattern still reads NaN.  A slot that receives only -inf reads 0 in a fresh output, as in
    torch_scatter: max(-FLT_MAX, -inf) is its initial value, which the fresh rule turns into 0."""
    src = torch.tensor([[1.0, -2.0, 3.0, float("-inf"), float("-inf")]], device=DEV)
    src[0, 1] = torch.tensor([-4194304], dtype=torch.int32).view(torch.float32)[0]  # bits 0xffc00000: -NaN
    assert torch.isnan(src[0, 1]) and bits(src)[0, 1] < 0
    index = torch.tensor([[0, 0, 1, 2, 2]], device=DEV)
    r = scatter(src, index, 1, dim_size=4, reduce="max")
    assert torch.isnan(r[0, 0])
    assert r[0, 1].item() == 3.0 and bits(r)[0, 2].item() == 0 and bits(r)[0, 3].item() == 0
    out = torch.full((1, 4), float("-inf"), device=DEV)  # with out=, -inf stays -inf
    assert scatter(src, index, 1, out=out, reduce="max")[0, 2].item() == float("-inf")


def test_nan_already_in_out_is_kept():
    """A NaN in a caller's `out=` survives any src value, whatever its bit pattern (0xffc00000 is the x86 default NaN
    of 0/0 on the CPU)."""
    out = torch.zeros(2, 3, device=DEV)
    out.view(torch.int32)[0, 0] = -4194304  # 0xffc00000: negative NaN
    out.view(torch.int32)[1, 1] = 0x7fc00001  # positive NaN with another payload
    src = torch.tensor([[5.0, -5.0, 1.0], [7.0, -7.0, 2.0]], device=DEV)
    index = torch.tensor([[0, 0, 2], [1, 1, 2]], device=DEV)
    r = scatter(src, index, 1, out=out, reduce="max")
    assert torch.isnan(r[0, 0]) and torch.isnan(r[1, 1])
    assert bits(r)[1, 1].item() == 0x7fc00001  # a positive pattern is left as it is, as torch leaves it
    assert r[0, 2].item() == 1.0 and r[1, 2].item() == 2.0 and r[0, 1].item() == 0.0


def test_in_place_update_bumps_the_version_counter():
    """Without grad, `out` is written through a raw pointer; its version counter still moves, so autograd detects the
    update of a tensor an earlier op saved for backward."""
    a = torch.rand(2, 10, device=DEV, requires_grad=True)
    out = torch.zeros(2, 10, device=DEV)
    y = (a * out).sum()  # saves out for backward
    v = out._version
    with torch.no_grad():
        scatter(torch.rand(2, 30, device=DEV), torch.randint(0, 10, (2, 30), device=DEV), 1, out=out, reduce="max")
    assert out._version > v
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        y.backward()


def test_negative_zero_and_lowest_in_a_fresh_output():
    """-0.0 must read -0.0 (not -FLT_MAX, not 0); all-negative slots read their max; a max of exactly -FLT_MAX reads 0
    (torch_scatter's masked_fill(out == lowest, 0))."""
    src = torch.tensor([[-0.0, -5.0, -3.0, LOWEST, -1e-30, -0.0]], device=DEV)
    index = torch.tensor([[0, 1, 1, 2, 3, 3]], device=DEV)
    r = scatter(src, index, 1, dim_size=5, reduce="max")
    assert bits(r)[0].tolist() == bits(torch.tensor([-0.0, -3.0, 0.0, -0.0, 0.0], device=DEV)).tolist()
    # +0 beats -0 whatever the order
    r = scatter(torch.tensor([[-0.0, 0.0, -0.0]], device=DEV), torch.zeros(1, 3, dtype=torch.int64, device=DEV), 1,
                reduce="max")
    assert bits(r).item() == 0


@pytest.mark.parametrize("fresh", [True, False])
def test_out_of_range_indices_are_skipped(fresh):
    """Negative indices and indices >= the size along dim are skipped: the result equals torch on the in-range subset
    and nothing outside `out` is written (out sits inside a larger buffer with guard bands)."""
    g = gen(17)
    A, E, D = 6, 3000, 40
    src = torch.randn(A, E, generator=g, device=DEV)
    index = torch.randint(-45, 85, (A, E), generator=g, device=DEV)
    valid = (index >= 0) & (index < D)
    assert (~valid).sum() > 1000
    # torch must not see an out-of-range index: those entries go to slot 0 as -inf, which never raises a max
    ref_index = torch.where(valid, index, 0)
    ref_src = torch.where(valid, src, torch.full_like(src, float("-inf")))
    guard = 4096
    buf = torch.full((guard + A * D + guard,), 12345.0, device=DEV)
    out = buf[guard:guard + A * D].view(A, D)
    if fresh:
        want = ref_max(ref_src, ref_index, 1, dim_size=D)
        got = scatter(src, index, 1, dim_size=D, reduce="max")
    else:
        out.normal_(generator=g)
        want = ref_max(ref_src, ref_index, 1, out=out)
        got = scatter(src, index, 1, out=out, reduce="max")
        assert got is out
    assert_bits_equal(got, want)
    assert torch.all(buf[:guard] == 12345.0) and torch.all(buf[guard + A * D:] == 12345.0)
    # the argmax never names an out-of-range entry (those sit in slot 0 of the reference as -inf, never equal to its max)
    res, arg = _scatter_max(src, index, 1, None, [A, D], True)
    assert torch.equal(arg, expected_argmax(ref_src, ref_index, 1, res))


def test_current_stream_is_used():
    g = gen(19)
    src = torch.randn(16, 20000, generator=g, device=DEV)
    index = torch.randint(0, 300, (16, 20000), generator=g, device=DEV)
    want = ref_max(src, index, 1, dim_size=300)
    s = torch.cuda.Stream(DEV)
    s.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(s):
        got = scatter(src, index, 1, dim_size=300, reduce="max")
        done = torch.cuda.Event()
        done.record(s)
    done.synchronize()
    assert_bits_equal(got, want)


def expected_argmax(src, full_index, dim, result):
    """Lowest position along dim of a src element equal to its slot's result (NaN matching NaN), E if none."""
    E = src.shape[dim]
    shape = [1] * src.dim()
    shape[dim] = E
    pos = torch.arange(E, device=src.device).view(shape).expand_as(src)
    r = result.gather(dim, full_index)
    eq = (src == r) | (torch.isnan(src) & torch.isnan(r))
    cand = torch.where(eq, pos, torch.full_like(pos, E))
    return torch.full(result.shape, E, dtype=torch.int64, device=src.device).scatter_reduce_(
        dim, full_index, cand, "amin", include_self=True)


@pytest.mark.parametrize("fresh", [True, False])
@pytest.mark.parametrize("shape,dim", [((8, 3000), 1), ((4, 500, 3), 1), ((700, 5), 0)])
def test_gradient_matches_torch_autograd_without_ties(fresh, shape, dim):
    g = gen(23)
    D = 97
    n = 1
    for s in shape:
        n *= s
    # distinct positive values: no ties among src, none with a zero-filled out
    src0 = (torch.randperm(n, generator=torch.Generator().manual_seed(5)).float().view(shape) + 1.0).to(DEV)
    index = torch.randint(0, D, shape, generator=g, device=DEV)
    oshape = list(shape)
    oshape[dim] = D
    w = torch.randn(oshape, generator=g, device=DEV)
    src = src0.clone().requires_grad_(True)
    out = None if fresh else torch.zeros(oshape, device=DEV)
    r = scatter(src, index, dim, out=out, dim_size=D, reduce="max")
    (r * w).sum().backward()
    src_t = src0.clone().requires_grad_(True)
    r_t = torch.zeros(oshape, device=DEV).scatter_reduce(dim, index, src_t, "amax", include_self=False)
    (r_t * w).sum().backward()
    assert_bits_equal(r.detach(), r_t.detach())
    assert torch.equal(src.grad, src_t.grad)


@pytest.mark.parametrize("fresh", [True, False])
def test_ties_send_the_whole_gradient_to_the_lowest_position(fresh):
    g = gen(29)
    A, E, D = 5, 6000, 30
    src0 = torch.randint(0, 4, (A, E), generator=g, device=DEV).float()
    index = torch.randint(0, D, (A, E), generator=g, device=DEV)
    gw = torch.randn(A, D, generator=g, device=DEV)
    grads, args = [], []
    for _ in range(2):
        src = src0.clone().requires_grad_(True)
        out = None if fresh else torch.full((A, D), 2.0, device=DEV)
        r = scatter(src, index, 1, out=out, dim_size=D, reduce="max")
        (r * gw).sum().backward()
        grads.append(src.grad)
        args.append(_scatter_max(src0, index, 1, None if fresh else torch.full((A, D), 2.0, device=DEV), [A, D], True)[1])
    arg = expected_argmax(src0, index, 1, r.detach())
    assert torch.equal(args[0], arg)
    pos = torch.arange(E, device=DEV).expand(A, E)
    want = torch.where(pos == arg.gather(1, index), gw.gather(1, index), torch.zeros_like(src0))
    assert torch.equal(grads[0], want)
    # deterministic: two identical calls give bit-identical argmax and gradients
    assert torch.equal(args[0], args[1]) and torch.equal(bits(grads[0]), bits(grads[1]))


def test_in_place_with_grad_returns_out():
    src = torch.rand(4, 100, device=DEV, requires_grad=True)
    index = torch.randint(0, 10, (4, 100), device=DEV)
    out = torch.zeros(4, 10, device=DEV)
    r = scatter(src, index, 1, out=out, reduce="max")
    assert r is out and r.requires_grad
    r.sum().backward()
    assert src.grad.sum().item() == float((out > 0).sum().item())
    with pytest.raises(RuntimeError, match="not require grad"):
        scatter(src, index, 1, out=torch.zeros(4, 10, device=DEV, requires_grad=True), reduce="max")


def test_refused_outputs():
    src = torch.rand(4, 100, device=DEV)
    index = torch.randint(0, 10, (4, 100), device=DEV)
    for bad in (torch.zeros(4, 10, device=DEV, dtype=torch.float64), torch.zeros(10, 4, device=DEV).t(),
                torch.zeros(5, 10, device=DEV), torch.zeros(4, 10)):
        with pytest.raises(RuntimeError):
            scatter(src, index, 1, out=bad, reduce="max")


def _c4_pointsea(arm, torch_scatter):
    if not osp.isdir(REFERENCE):
        pytest.skip(f"needs a checkout of the reference at {REFERENCE} (or set POINTSEA_REFERENCE)")
    if not osp.exists(osp.join(ROOT, "oracle", "_ref", "ref_pointnet2_ext.so")):
        pytest.skip("oracle/_ref not built (python __graft_entry__.py build builds it beside a reference checkout)")
    p = subprocess.run([sys.executable, osp.join(ROOT, "tools", "bench_configs.py"), "c4", "--arm", arm, "--knn", "torch",
                        "--iters", "1", "--batch", "2", "--model", "pointsea", "--torch-scatter", torch_scatter],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, POINTSEA_REFERENCE_TREE=REFERENCE))
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert p.returncode == 0 and lines, (p.stderr or p.stdout)[-3000:]
    d = json.loads(lines[-1])
    assert "loss_hex" in d, d
    return d


def test_c4_pointsea_runs_on_the_torch_scatter_dropin():
    """models_PointSea/PointSea.py with `import torch_scatter` resolved through install_dropin()'s fallback path: the
    depth maps come from ps_scatter_max, and the loss equals the reference-ops arm as hex floats."""
    ours = _c4_pointsea("ours", "dropin")
    ref = _c4_pointsea("ref", "stub")
    assert osp.join("dropin_fallback", "torch_scatter") in ours["torch_scatter"], ours["torch_scatter"]
    assert ours["loss_hex"] == ref["loss_hex"], (ours["loss"], ref["loss"])
