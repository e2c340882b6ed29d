"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the committed golden
vectors (outputs of the reference's own CUDA kernels, to which the oracle is pinned bit for bit).

Bars (BASELINE.json north_star): indices bit-exact (FPS, argmin, ball query, 3-NN, kNN);
Chamfer distances bit-exact in practice (same rounding order), asserted to 1e-5 relative;
gradients within 1e-5 relative (the reference accumulates with atomics in arbitrary order).
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, make_cloud
from oracle import oracle as O

pytestmark = pytest.mark.gpu

import svdformer_pointsea_b200 as ps  # noqa: E402
from svdformer_pointsea_b200 import pointnet2_utils as pu  # noqa: E402

DEV = "cuda:0"
RTOL = 1e-5


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def assert_close_rel(a, b, rtol=RTOL, what=""):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    scale = max(np.abs(b).max(), 1e-30)
    err = np.abs(a - b).max() / scale
    assert err <= rtol, f"{what}: max rel err {err:.3e} > {rtol}"


# ---------------------------------------------------------------- Chamfer
@pytest.mark.parametrize("B,N,M,dup", [(2, 100, 200, 0), (3, 300, 700, 0), (2, 1024, 1537, 0), (2, 512, 640, 200),
                                       (1, 1, 5, 0), (2, 5, 1, 0), (1, 2049, 4100, 0), (4, 64, 4096, 0)])
def test_chamfer_fwd_bwd_vs_oracle(B, N, M, dup):
    g = torch.Generator().manual_seed(100 + N + M)
    a, b = make_cloud(g, B, N, dup=min(dup, max(N - 1, 0))), make_cloud(g, B, M, dup=min(dup, max(M - 1, 0)))
    if dup:
        b[:, :100] = a[:, :100]
    gd1, gd2 = torch.randn(B, N, generator=g), torch.randn(B, M, generator=g)
    d1, d2, i1, i2 = ps.chamfer_forward(a.to(DEV), b.to(DEV))
    od1, od2, oi1, oi2 = O.chamfer_fwd(a.numpy(), b.numpy())
    assert np.array_equal(i1.cpu().numpy(), oi1), "idx1 differs from the oracle"
    assert np.array_equal(i2.cpu().numpy(), oi2), "idx2 differs from the oracle"
    assert np.array_equal(d1.cpu().numpy(), od1) and np.array_equal(d2.cpu().numpy(), od2), "distances not bit-exact"
    g1, g2 = ps.chamfer_backward(a.to(DEV), b.to(DEV), gd1.to(DEV), gd2.to(DEV), i1, i2)
    og1, og2 = O.chamfer_bwd(a.numpy(), b.numpy(), gd1.numpy(), gd2.numpy(), oi1, oi2)
    assert_close_rel(g1.cpu().numpy(), og1, what="gradxyz1")
    assert_close_rel(g2.cpu().numpy(), og2, what="gradxyz2")


@pytest.mark.parametrize("sym,q", [("2", "16"), ("2", "8"), ("2", "4"), ("1", "8"), ("1", "4"), ("1", "2"), ("0", "8"),
                                   ("6", "8"), ("3", "8"), ("7", "8")])
@pytest.mark.parametrize("B,N,M,dup", [(2, 2048, 4096, 700), (3, 5000, 1300, 300), (1, 16384, 2048, 548),
                                       (2, 1024, 1024, 1000), (1, 2050, 257, 0), (1, 300, 9000, 100)])
def test_chamfer_symmetric_and_two_pass_kernels_agree_with_oracle(B, N, M, dup, sym, q, monkeypatch):
    """Both forward kernels (single-pass symmetric, two-pass) at every register blocking, with
    heavy duplication inside and across the clouds (exact ties on both sides)."""
    monkeypatch.setenv("PS_CHAMFER_SYM", sym)
    monkeypatch.setenv("PS_CHAMFER_SYM_Q", q)
    g = torch.Generator().manual_seed(900 + N + M)
    a, b = make_cloud(g, B, N, dup=min(dup, N - 1)), make_cloud(g, B, M, dup=min(dup, M - 1))
    n_shared = min(N, M) // 3
    b[:, :n_shared] = a[:, N - n_shared:]  # cross-cloud exact matches at different indices
    d1, d2, i1, i2 = ps.chamfer_forward(a.to(DEV), b.to(DEV))
    od1, od2, oi1, oi2 = O.chamfer_fwd(a.numpy(), b.numpy())
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(i2.cpu().numpy(), oi2)
    assert np.array_equal(d1.cpu().numpy(), od1) and np.array_equal(d2.cpu().numpy(), od2)


@pytest.mark.parametrize("sym", ["1", "6", "3", "7"])
@pytest.mark.parametrize("split", ["2304", "1100", "4608"])
def test_chamfer_units_spanning_several_tiles(sym, split, monkeypatch):
    """Units longer than one shared-memory tile (forced split length): the argmin group remembered by the scan may
    lie in an earlier tile (re-evaluated from global memory), tiles end ragged, duplicates tie across tiles."""
    monkeypatch.setenv("PS_CHAMFER_SYM", sym)
    monkeypatch.setenv("PS_CHAMFER_SPLIT", split)
    g = torch.Generator().manual_seed(77)
    a, b = make_cloud(g, 2, 4096, dup=1500), make_cloud(g, 2, 4608, dup=3000)
    b[:, 4000:4500] = a[:, 100:600]
    d1, d2, i1, i2 = ps.chamfer_forward(a.to(DEV), b.to(DEV))
    od1, od2, oi1, oi2 = O.chamfer_fwd(a.numpy(), b.numpy())
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(i2.cpu().numpy(), oi2)
    assert np.array_equal(d1.cpu().numpy(), od1) and np.array_equal(d2.cpu().numpy(), od2)


@pytest.mark.parametrize("B,N,M,chunk,bwd", [(5, 300, 700, 2, True), (4, 1024, 2048, 0, True), (3, 64, 4096, 1, False),
                                              (7, 2048, 512, 3, True), (1, 10, 20, 8, True)])
def test_chamfer_host_pipeline_matches_device_entry_points_bitwise(B, N, M, chunk, bwd):
    """ps_chamfer_host (host buffers, chunked 3-stream pipeline) == device entry points, bit for bit,
    for every chunking including ragged last chunks; and it matches the oracle."""
    g = torch.Generator().manual_seed(4000 + N + M)
    a, b = make_cloud(g, B, N).pin_memory(), make_cloud(g, B, M).pin_memory()
    gd1, gd2 = torch.randn(B, N, generator=g).pin_memory(), torch.randn(B, M, generator=g).pin_memory()
    out = ps.chamfer_host(a, b, gd1 if bwd else None, gd2 if bwd else None, chunk=chunk)
    d1, d2, i1, i2 = ps.chamfer_forward(a.to(DEV), b.to(DEV))
    for h, d in zip(out[:4], (d1, d2, i1, i2)):
        assert torch.equal(h, d.cpu())
    od1, od2, oi1, oi2 = O.chamfer_fwd(a.numpy(), b.numpy())
    assert np.array_equal(out[2].numpy(), oi1) and np.array_equal(out[3].numpy(), oi2)
    assert np.array_equal(out[0].numpy(), od1) and np.array_equal(out[1].numpy(), od2)
    if bwd:
        og1, og2 = O.chamfer_bwd(a.numpy(), b.numpy(), gd1.numpy(), gd2.numpy(), oi1, oi2)
        assert_close_rel(out[4].numpy(), og1, what="gradxyz1 (host)")
        assert_close_rel(out[5].numpy(), og2, what="gradxyz2 (host)")
    # second call reuses the staging slots; pageable (non-pinned) buffers also work
    out2 = ps.chamfer_host(a.clone(), b.clone(), chunk=chunk)
    assert torch.equal(out2[0], out[0]) and torch.equal(out2[3], out[3])


def test_chamfer_host_async_keeps_several_steps_in_flight_bitwise():
    """ps_chamfer_host_submit / ps_chamfer_host_wait: steps submitted back to back on the library's two lanes (step
    i+1 uploads and computes while step i downloads) return exactly what the stream-ordered call returns, for
    different clouds per step, rotating buffer sets, with and without the backward, and through both ways of
    joining a step (host synchronize, stream wait)."""
    g = torch.Generator().manual_seed(4242)
    B, N, M, NSTEPS, NSETS = 6, 700, 1500, 9, 3
    clouds = [(make_cloud(g, B, N).pin_memory(), make_cloud(g, B, M).pin_memory(),
               torch.randn(B, N, generator=g).pin_memory(), torch.randn(B, M, generator=g).pin_memory()) for _ in range(NSTEPS)]
    want, want_sums = [], []
    for a, b, ga, gb in clouds:
        ws = torch.empty(6, dtype=torch.float64).pin_memory()
        want.append(tuple(x.clone() for x in ps.chamfer_host(a, b, ga, gb, sums_out=ws)))
        want_sums.append(ws.clone())
    outs = [[torch.empty(B, N).pin_memory(), torch.empty(B, M).pin_memory(), torch.empty(B, N, dtype=torch.int32).pin_memory(),
             torch.empty(B, M, dtype=torch.int32).pin_memory(), torch.empty(B, N, 3).pin_memory(), torch.empty(B, M, 3).pin_memory()]
            for _ in range(NSETS)]
    sums = [torch.empty(6, dtype=torch.float64).pin_memory() for _ in range(NSETS)]
    pending, done = None, 0
    for i, (a, b, ga, gb) in enumerate(clouds):
        step = ps.chamfer_host_async(a, b, ga, gb, out=outs[i % NSETS], sums_out=sums[i % NSETS])
        assert step.ticket != 0
        if pending is not None:
            got = pending.synchronize()
            for h, w in zip(got[:4], want[i - 1][:4]):
                assert torch.equal(h, w)
            for h, w in zip(got[4:], want[i - 1][4:]):  # the backward accumulates with atomics: order-dependent rounding
                assert_close_rel(h.numpy(), w.numpy(), what="gradient (async)")
            assert torch.equal(pending.sums, want_sums[i - 1])
            done += 1
        pending = step
    # the last one through a stream wait: a kernel queued behind it sees the finished host buffer
    pending.wait()
    torch.cuda.current_stream().synchronize()
    for h, w in zip(pending.out[:4], want[-1][:4]):
        assert torch.equal(h, w)
    assert_close_rel(pending.out[5].numpy(), want[-1][5].numpy(), what="gradient (async, stream join)")
    assert done == NSTEPS - 1
    # three in flight (four lanes): joined in submission order
    import collections
    q3, k = collections.deque(), 0
    outs4 = outs + [[torch.empty_like(x).pin_memory() for x in outs[0]]]
    for i, (a, b, ga, gb) in enumerate(clouds):
        q3.append((i, ps.chamfer_host_async(a, b, ga, gb, out=outs4[i % 4])))
        if len(q3) == 3:
            j, st = q3.popleft()
            for h, w in zip(st.synchronize()[:4], want[j][:4]):
                assert torch.equal(h, w)
            k += 1
    while q3:
        j, st = q3.popleft()
        for h, w in zip(st.synchronize()[:4], want[j][:4]):
            assert torch.equal(h, w)
        k += 1
    assert k == NSTEPS
    # forward only, library-allocated outputs, two in flight at once
    s1 = ps.chamfer_host_async(clouds[0][0], clouds[0][1])
    s2 = ps.chamfer_host_async(clouds[1][0], clouds[1][1])
    for h, w in zip(s2.synchronize(), want[1][:4]):
        assert torch.equal(h, w)
    for h, w in zip(s1.synchronize(), want[0][:4]):
        assert torch.equal(h, w)
    # the stream-ordered call still works in between (lane 0) and empty batches are no-ops
    again = ps.chamfer_host(clouds[2][0], clouds[2][1])
    assert torch.equal(again[0], want[2][0])
    e = ps.chamfer_host_async(torch.zeros(0, 8, 3), torch.zeros(0, 9, 3))
    assert e.ticket == 0 and e.synchronize()[0].numel() == 0


def test_chamfer_host_async_mixed_shapes_many_steps():
    """A longer run of the asynchronous pair as a race guard: four steps in flight, shapes changing from step to step
    (the lanes' staging slots grow, cached graphs are evicted and retargeted), fresh output buffers half of the
    time; every distance and index is compared with the stream-ordered call."""
    import collections
    g = torch.Generator().manual_seed(77)
    shapes = [(4, 512, 3000), (7, 2048, 1024), (2, 300, 300), (5, 1500, 6000)]
    data, want = [], []
    for B, N, M in shapes:
        a, b = make_cloud(g, B, N, dup=N // 5).pin_memory(), make_cloud(g, B, M).pin_memory()
        data.append((a, b))
        want.append(tuple(x.clone() for x in ps.chamfer_host(a, b)))
    outs = [[[torch.empty(B, N).pin_memory(), torch.empty(B, M).pin_memory(), torch.empty(B, N, dtype=torch.int32).pin_memory(),
              torch.empty(B, M, dtype=torch.int32).pin_memory()] for _ in range(5)] for B, N, M in shapes]
    order = torch.randint(0, len(shapes), (120,), generator=g).tolist()
    pend, checked = collections.deque(), 0
    for i, k in enumerate(order):
        out = outs[k][i % 5] if i % 2 else None
        pend.append((k, ps.chamfer_host_async(data[k][0], data[k][1], out=out)))
        if len(pend) == 4:
            kk, st = pend.popleft()
            for h, w in zip(st.synchronize(), want[kk]):
                assert torch.equal(h, w), f"step {checked} shape {shapes[kk]}"
            checked += 1
    while pend:
        kk, st = pend.popleft()
        for h, w in zip(st.synchronize(), want[kk]):
            assert torch.equal(h, w)
        checked += 1
    assert checked == len(order)


def test_chamfer_host_async_pageable_buffers_small_clouds_and_sums():
    """Corners of the asynchronous pair: pageable (non-pinned) host tensors (the copies then stage synchronously, the
    results must still be right), clouds small enough for the two-pass forward kernel, loss sums with and without the
    backward, and both submission modes (PS_HOST_ASYNC=lanes: the chunked graph per lane)."""
    import os
    g = torch.Generator().manual_seed(31)
    for mode in ("fifo", "lanes"):
        os.environ["PS_HOST_ASYNC"] = mode
        try:
            for B, N, M, bwd in ((3, 200, 150, True), (2, 64, 900, False), (4, 1024, 3000, True)):
                a, b = make_cloud(g, B, N), make_cloud(g, B, M)  # pageable
                ga, gb = torch.randn(B, N, generator=g), torch.randn(B, M, generator=g)
                ws = torch.empty(6, dtype=torch.float64).pin_memory()
                want = ps.chamfer_host(a, b, ga if bwd else None, gb if bwd else None, sums_out=ws)
                s1 = torch.empty(6, dtype=torch.float64)  # pageable as well
                s2 = torch.empty(6, dtype=torch.float64).pin_memory()
                st1 = ps.chamfer_host_async(a, b, ga if bwd else None, gb if bwd else None, sums_out=s1)
                st2 = ps.chamfer_host_async(a.pin_memory(), b.pin_memory(), sums_out=s2)
                o1, o2 = st1.synchronize(), st2.synchronize()
                for h, w in zip(o1[:4], want[:4]):
                    assert torch.equal(h, w)
                for h, w in zip(o2[:4], want[:4]):
                    assert torch.equal(h, w)
                if bwd:
                    assert_close_rel(o1[4].numpy(), want[4].numpy(), what="gradxyz1 (async, pageable)")
                    assert_close_rel(o1[5].numpy(), want[5].numpy(), what="gradxyz2 (async, pageable)")
                assert torch.allclose(s1, ws, rtol=1e-13, atol=0) and torch.allclose(s2, ws, rtol=1e-13, atol=0)
        finally:
            os.environ.pop("PS_HOST_ASYNC", None)


def test_chamfer_host_rejects_device_tensors_and_bad_shapes():
    a = torch.zeros(2, 8, 3, device=DEV)
    with pytest.raises(ps.PointSeaError):
        ps.chamfer_host(a, a)
    with pytest.raises(ps.PointSeaError):
        ps.chamfer_host(torch.zeros(2, 8, 3), torch.zeros(3, 8, 3))
    with pytest.raises(ps.PointSeaError):
        ps.chamfer_host(torch.zeros(2, 8, 3), torch.zeros(2, 8, 3), graddist1=torch.zeros(2, 8))


def test_chamfer_sums_match_torch_reductions():
    g = torch.Generator().manual_seed(12)
    a, b = make_cloud(g, 3, 777).to(DEV), make_cloud(g, 3, 1500).to(DEV)
    d1, d2, _, _ = ps.chamfer_forward(a, b)
    s = ps.chamfer_sums(d1, d2).cpu().numpy()
    want = [torch.sqrt(d1).double().sum().item(), torch.sqrt(d2).double().sum().item(), d1.double().sum().item(), d2.double().sum().item()]
    assert np.allclose(s[:4], want, rtol=1e-9) and s[4] == d1.numel() and s[5] == d2.numel()
    from svdformer_pointsea_b200.dist import chamfer_metric_means
    m = chamfer_metric_means(d1, d2)
    assert abs(m["sqrt_d1"].item() - torch.sqrt(d1).double().mean().item()) < 1e-12


def test_chamfer_golden():
    z = load_golden("chamfer")
    for name in ("small", "tiles", "dups", "tiny"):
        a, b = t(z[f"{name}.xyz1"]), t(z[f"{name}.xyz2"])
        d1, d2, i1, i2 = ps.chamfer_forward(a, b)
        assert np.array_equal(i1.cpu().numpy(), z[f"{name}.idx1"]), name
        assert np.array_equal(i2.cpu().numpy(), z[f"{name}.idx2"]), name
        assert_close_rel(d1.cpu().numpy(), z[f"{name}.dist1"], what=name + ".dist1")
        assert_close_rel(d2.cpu().numpy(), z[f"{name}.dist2"], what=name + ".dist2")
        g1, g2 = ps.chamfer_backward(a, b, t(z[f"{name}.gd1"]), t(z[f"{name}.gd2"]), i1, i2)
        assert_close_rel(g1.cpu().numpy(), z[f"{name}.g1"], what=name + ".g1")
        assert_close_rel(g2.cpu().numpy(), z[f"{name}.g2"], what=name + ".g2")


def test_chamfer_autograd_module_and_dropin():
    ps.install_dropin()
    from metrics.CD.chamfer3D import dist_chamfer_3D
    g = torch.Generator().manual_seed(7)
    a = make_cloud(g, 2, 256).to(DEV).requires_grad_(True)
    b = make_cloud(g, 2, 300).to(DEV).requires_grad_(True)
    d1, d2, i1, i2 = dist_chamfer_3D.chamfer_3DDist()(a, b)
    assert i1.dtype == torch.int32 and i2.dtype == torch.int32 and d1.is_contiguous()
    loss = torch.mean(torch.sqrt(d1)) + torch.mean(d2)
    loss.backward()
    # autograd of the direct form on the CPU as the gradient oracle
    ac, bc = a.detach().cpu().requires_grad_(True), b.detach().cpu().requires_grad_(True)
    td1, td2, _, _ = O.torch_chamfer(ac, bc)
    (torch.mean(torch.sqrt(td1)) + torch.mean(td2)).backward()
    assert_close_rel(a.grad.cpu().numpy(), ac.grad.numpy(), rtol=1e-4, what="autograd grad a")
    assert_close_rel(b.grad.cpu().numpy(), bc.grad.numpy(), rtol=1e-4, what="autograd grad b")


def test_chamfer_vs_reference_cuda_full_size():
    """C1 shape (B=32, 2048 vs 16384) against the reference kernel as the CPU oracle restates it (bit-exact to the
    reference's own outputs in tests/golden/chamfer.npz), all 32 clouds."""
    g = torch.Generator().manual_seed(1234 + 1)
    a, b = make_cloud(g, 32, 2048, dup=548), make_cloud(g, 32, 16384)
    d1, d2, i1, i2 = ps.chamfer_forward(a.to(DEV), b.to(DEV))
    gd1, gd2 = torch.randn(d1.shape, generator=g), torch.randn(d2.shape, generator=g)
    g1, g2 = ps.chamfer_backward(a.to(DEV), b.to(DEV), gd1.to(DEV), gd2.to(DEV), i1, i2)
    od1, od2, oi1, oi2 = O.chamfer_fwd(a.numpy(), b.numpy())
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(i2.cpu().numpy(), oi2), "argmin indices differ from the reference kernel"
    assert np.array_equal(d1.cpu().numpy(), od1) and np.array_equal(d2.cpu().numpy(), od2), "distances differ from the reference kernel"
    og1, og2 = O.chamfer_bwd(a.numpy(), b.numpy(), gd1.numpy(), gd2.numpy(), oi1, oi2)
    assert_close_rel(g1.cpu().numpy(), og1, what="g1 vs ref")
    assert_close_rel(g2.cpu().numpy(), og2, what="g2 vs ref")


def test_chamfer_properties_full_size():
    """Size-independent properties at the stress-ish size: dist equals the distance to the
    reported index, self-Chamfer is zero with identity indices, result is permutation-consistent."""
    g = torch.Generator().manual_seed(5)
    a, b = make_cloud(g, 4, 16384).to(DEV), make_cloud(g, 4, 16384).to(DEV)
    d1, d2, i1, i2 = ps.chamfer_forward(a, b)
    nn = torch.gather(b, 1, i1.long()[..., None].expand(-1, -1, 3))
    diff = nn - a
    recomputed = torch.addcmul(torch.addcmul(diff[..., 1] * diff[..., 1], diff[..., 0], diff[..., 0]), diff[..., 2], diff[..., 2])
    assert_close_rel(d1.cpu().numpy(), recomputed.cpu().numpy(), rtol=1e-6, what="dist1 == |a - b[idx1]|^2")
    s1, s2, j1, j2 = ps.chamfer_forward(a, a.clone())
    assert torch.count_nonzero(s1) == 0 and torch.count_nonzero(s2) == 0
    ar = torch.arange(16384, device=DEV, dtype=torch.int32).expand(4, -1)
    assert torch.equal(j1, ar) and torch.equal(j2, ar)
    # swapping the arguments swaps the outputs
    e1, e2, k1, k2 = ps.chamfer_forward(b, a)
    assert torch.equal(e1, d2) and torch.equal(e2, d1) and torch.equal(k1, i2) and torch.equal(k2, i1)


# ---------------------------------------------------------------- FPS
@pytest.mark.parametrize("B,N,npoint,dup,no", [(3, 1000, 128, 0, 0), (2, 2048, 512, 548, 0), (2, 300, 64, 0, 2),
                                               (2, 5000, 200, 0, 40), (2, 512, 512, 100, 1), (2, 7, 7, 0, 0),
                                               (1, 1, 1, 0, 0), (2, 33, 20, 5, 0), (1, 16384, 300, 0, 3),
                                               (40, 1024, 64, 0, 0)])
def test_fps_vs_oracle(B, N, npoint, dup, no):
    g = torch.Generator().manual_seed(200 + N + npoint)
    x = make_cloud(g, B, N, dup=dup, near_origin=no)
    got = ps.furthest_point_sample(x.to(DEV), npoint)
    assert got.dtype == torch.int32 and tuple(got.shape) == (B, npoint)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), npoint))


@pytest.mark.parametrize("threads", [128, 256])
@pytest.mark.parametrize("cluster", [1, 2, 4, 8, 16])
def test_fps_every_cluster_size(cluster, threads, monkeypatch):
    """Every exchange variant of the kernel (single CTA; st.async push from every warp; two-level)
    at both CTA sizes must give the reference's indices, ties included."""
    monkeypatch.setenv("PS_FPS_CLUSTER", str(cluster))
    monkeypatch.setenv("PS_FPS_THREADS", str(threads))
    g = torch.Generator().manual_seed(300 + cluster)
    x = make_cloud(g, 3, 4096, dup=500, near_origin=5)
    got = ps.furthest_point_sample(x.to(DEV), 256)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), 256))
    x = make_cloud(g, 2, min(20000, 4000 * cluster), dup=1000, near_origin=9)
    got = ps.furthest_point_sample(x.to(DEV), 300)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), 300))
    x = make_cloud(g, 2, 300, dup=40, near_origin=2)  # bs = 256 < 512, mostly padding ranks
    got = ps.furthest_point_sample(x.to(DEV), 100)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), 100))


@pytest.mark.parametrize("B,N,npoint,dup,no", [(3, 16384, 700, 0, 5), (2, 16384, 2048, 4000, 0), (2, 9999, 500, 1000, 30),
                                               (2, 4096, 4096, 0, 0), (3, 1000, 128, 0, 0), (2, 33, 20, 5, 0), (1, 1, 1, 0, 0),
                                               (2, 7, 7, 0, 0), (150, 2048, 96, 0, 1)])
def test_fps_bucket_pruned_kernel_vs_oracle(B, N, npoint, dup, no, monkeypatch):
    """fps_pruned_kernel forced for every shape it accepts (N <= 16384): duplicates (ties by rank), points inside
    the skip ball (left out of the buckets), ragged last buckets, more clouds than SMs, npoint == N."""
    monkeypatch.setenv("PS_FPS_PRUNE", "1")
    g = torch.Generator().manual_seed(5200 + N + npoint)
    x = make_cloud(g, B, N, dup=dup, near_origin=no)
    got = ps.furthest_point_sample(x.to(DEV), npoint)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), npoint))


@pytest.mark.parametrize("B,N,npoint", [(32, 16384, 300), (4, 16384, 2048), (32, 2048, 512), (3, 5000, 77), (150, 8192, 400)])
def test_fps_corun_hint_changes_the_kernel_not_the_samples(B, N, npoint):
    """ps_fps_sample_ex(PS_FPS_CORUN): the variant that leaves the SMs' shared memory to a neighbouring kernel returns
    the same indices and coordinates as the default plan and as the oracle."""
    from svdformer_pointsea_b200.pointnet2_utils import fps_sample_raw
    g = torch.Generator().manual_seed(640 + N)
    x = make_cloud(g, B, N, dup=N // 10, near_origin=3)
    xd = x.to(DEV)
    i0, p0 = fps_sample_raw(xd, npoint)
    i1, p1 = fps_sample_raw(xd, npoint, corun=True)
    assert torch.equal(i0, i1) and torch.equal(p0, p1)
    assert np.array_equal(i1[:2].cpu().numpy(), O.fps(x[:2].numpy(), npoint))
    assert torch.equal(p1, torch.gather(xd, 1, i1.long().unsqueeze(-1).expand(-1, -1, 3)))


def test_fps_bucket_pruned_kernel_shapes_of_real_clouds_and_the_give_up_path(monkeypatch):
    """(1) points on a thin surface and in tight clusters (where the pruning bites hardest, and bucket boxes are
    degenerate in one axis); (2) clouds squeezed into one grid cell by a far outlier, or made of one repeated point:
    forced (PS_FPS_PRUNE=1), the pruned kernel ploughs on; with its give-up path on (=2, what the launcher does when
    it picks the pruned kernel for a batch of many waves) it hands exactly those clouds to the cluster kernel behind
    it; unset / 0: the planner's own choice and the cluster kernels alone."""
    g = torch.Generator().manual_seed(91)
    N, B, M = 8192, 150, 400
    sphere = torch.randn(1, N, 3, generator=g)
    sphere = sphere / sphere.norm(dim=2, keepdim=True) * 0.4
    plane = torch.rand(1, N, 3, generator=g) - 0.5
    plane[..., 2] = 0.25
    clusters = (torch.randint(0, 5, (1, N, 1), generator=g).float() - 2) * 0.2 + torch.randn(1, N, 3, generator=g) * 0.003
    outlier = torch.randn(1, N, 3, generator=g) * 1e-3 + 0.3
    outlier[0, 17] = torch.tensor([900.0, -700.0, 800.0])
    same = torch.full((1, N, 3), 0.37)
    kinds = [sphere, plane, clusters, outlier, same, make_cloud(g, 1, N, dup=3000, near_origin=7)]
    clouds = torch.cat([kinds[i % len(kinds)] if i < 12 else kinds[i % len(kinds)].roll(i, 1) for i in range(B)], 0).contiguous()
    want = O.fps(clouds.numpy(), M)
    for mode in ("1", "2", None, "0"):
        if mode is None:
            monkeypatch.delenv("PS_FPS_PRUNE", raising=False)
        else:
            monkeypatch.setenv("PS_FPS_PRUNE", mode)
        got = ps.furthest_point_sample(clouds.to(DEV), M)
        assert np.array_equal(got.cpu().numpy(), want), f"PS_FPS_PRUNE={mode}"
    monkeypatch.delenv("PS_FPS_PRUNE", raising=False)
    sub = ps.fps_subsample(clouds.to(DEV), M)  # fused coordinates output through the same kernels
    assert torch.equal(sub.cpu(), torch.gather(clouds, 1, torch.from_numpy(want).long()[..., None].expand(-1, -1, 3)))


def test_fps_generic_fallback_beyond_register_capacity():
    g = torch.Generator().manual_seed(77)
    x = make_cloud(g, 1, 140000, near_origin=4)
    got = ps.furthest_point_sample(x.to(DEV), 40)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), 40))


def test_fps_all_points_inside_skip_ball():
    x = (torch.rand(2, 600, 3, generator=torch.Generator().manual_seed(3)) - 0.5) * 0.02
    got = ps.furthest_point_sample(x.to(DEV), 16)
    assert np.array_equal(got.cpu().numpy(), O.fps(x.numpy(), 16))
    assert int(got.abs().sum()) == 0  # the reference's tree returns index 0 every time


def test_fps_golden():
    z = load_golden("fps")
    for name in ("n1000", "dups2048", "bs256", "origin", "n16384", "npow2", "tiny"):
        x = z[f"{name}.xyz"]
        want = z[f"{name}.idx"]
        got = ps.furthest_point_sample(t(x), want.shape[1])
        assert np.array_equal(got.cpu().numpy(), want), name


def test_fps_vs_reference_cuda_full_size():
    """C2 shape (B=32, 16384 -> 2048) against the reference kernel as the CPU oracle restates it (bit-exact to the
    reference's own outputs in tests/golden/fps.npz), all 32 clouds, + fused call site."""
    g = torch.Generator().manual_seed(1234 + 2)
    x = make_cloud(g, 32, 16384, near_origin=3)
    xd = x.to(DEV)
    got = ps.furthest_point_sample(xd, 2048)
    want = O.fps(x.numpy(), 2048)
    assert np.array_equal(got.cpu().numpy(), want)
    sub = ps.fps_subsample(xd, 2048)
    assert torch.equal(sub, torch.gather(xd, 1, torch.from_numpy(want).to(DEV).long()[..., None].expand(-1, -1, 3)))


# ---------------------------------------------------------------- gather / group
@pytest.mark.parametrize("B,C,N,M", [(2, 5, 333, 77), (3, 3, 16384, 2048), (2, 64, 2048, 512), (1, 1, 9, 1), (2, 7, 100, 401)])
def test_gather_fwd_bwd(B, C, N, M):
    g = torch.Generator().manual_seed(400 + N)
    feat = torch.randn(B, C, N, generator=g)
    idx = torch.randint(0, N, (B, M), generator=g, dtype=torch.int32)
    go = torch.randn(B, C, M, generator=g)
    f = feat.to(DEV).requires_grad_(True)
    out = ps.gather_operation(f, idx.to(DEV))
    assert np.array_equal(out.detach().cpu().numpy(), O.gather(feat.numpy(), idx.numpy()))
    out.backward(go.to(DEV))
    assert_close_rel(f.grad.cpu().numpy(), O.gather_grad(go.numpy(), idx.numpy(), N), what="gather grad")


@pytest.mark.parametrize("B,C,N,S,K", [(2, 6, 256, 64, 16), (2, 128, 2048, 256, 16), (2, 3, 2048, 512, 16),
                                       (1, 2, 50, 7, 3), (2, 9, 300, 33, 5), (1, 4, 70000, 64, 8),
                                       (2, 8, 3000, 1024, 16), (1, 5, 7000, 2048, 16), (1, 4, 512, 1100, 32),
                                       (2, 12, 1024, 40000, 1)])
def test_group_fwd_bwd(B, C, N, S, K):
    g = torch.Generator().manual_seed(500 + N + S)
    feat = torch.randn(B, C, N, generator=g)
    idx = torch.randint(0, N, (B, S, K), generator=g, dtype=torch.int32)
    go = torch.randn(B, C, S, K, generator=g)
    f = feat.to(DEV).requires_grad_(True)
    out = ps.grouping_operation(f, idx.to(DEV))
    assert out.is_contiguous() and tuple(out.shape) == (B, C, S, K)
    assert np.array_equal(out.detach().cpu().numpy(), O.group(feat.numpy(), idx.numpy()))
    out.backward(go.to(DEV))
    assert_close_rel(f.grad.cpu().numpy(), O.group_grad(go.numpy(), idx.numpy(), N), what="group grad")


def test_group_output_can_be_modified_in_place():
    """models/model_utils.py:345 does `grouped_xyz -= ...` on the op's output."""
    g = torch.Generator().manual_seed(9)
    feat = torch.randn(2, 3, 128, generator=g).to(DEV).requires_grad_(True)
    idx = torch.randint(0, 128, (2, 16, 4), generator=g, dtype=torch.int32).to(DEV)
    out = ps.grouping_operation(feat, idx)
    out -= 1.0
    out.sum().backward()
    assert feat.grad is not None


def test_gather_group_golden_and_reference():
    z = load_golden("pointnet2")
    out = pu.gather_raw(t(z["gather.feat"]), t(z["gather.idx"]))
    assert np.array_equal(out.cpu().numpy(), z["gather.out"])
    assert_close_rel(pu.gather_grad_raw(t(z["gather.go"]), t(z["gather.idx"]), z["gather.feat"].shape[2]).cpu().numpy(),
                     z["gather.grad"], what="gather grad golden")
    out = pu.group_raw(t(z["group.feat"]), t(z["group.idx"]))
    assert np.array_equal(out.cpu().numpy(), z["group.out"])
    assert_close_rel(pu.group_grad_raw(t(z["group.go"]), t(z["group.idx"]), z["group.feat"].shape[2]).cpu().numpy(),
                     z["group.grad"], what="group grad golden")


def test_group_vs_reference_cuda_full_size():
    """Against the reference kernel as the CPU oracle restates it (pinned by tests/golden/pointnet2.npz)."""
    g = torch.Generator().manual_seed(1234 + 3)
    feat = torch.randn(8, 128, 2048, generator=g)
    idx = torch.randint(0, 2048, (8, 2048, 16), generator=g, dtype=torch.int32)
    assert np.array_equal(pu.group_raw(feat.to(DEV), idx.to(DEV)).cpu().numpy(), O.group(feat.numpy(), idx.numpy()))
    go = torch.randn(8, 128, 2048, 16, generator=g)
    assert_close_rel(pu.group_grad_raw(go.to(DEV), idx.to(DEV), 2048).cpu().numpy(), O.group_grad(go.numpy(), idx.numpy(), 2048),
                     what="group grad vs ref")


# ---------------------------------------------------------------- ball query / 3-NN / interpolate
@pytest.mark.parametrize("r,ns", [(0.2, 16), (0.05, 8), (0.6, 32), (0.0, 4), (2.0, 3)])
def test_ball_query_vs_oracle(r, ns):
    g = torch.Generator().manual_seed(600)
    xyz, new_xyz = make_cloud(g, 2, 2500), make_cloud(g, 2, 130)
    got = ps.ball_query(r, ns, xyz.to(DEV), new_xyz.to(DEV))
    assert np.array_equal(got.cpu().numpy(), O.ball_query(new_xyz.numpy(), xyz.numpy(), r, ns))


def test_ball_three_golden():
    z = load_golden("pointnet2")
    for r, ns in ((0.2, 16), (0.05, 8), (0.6, 32)):
        got = pu.ball_query_raw(t(z["ball.new_xyz"]), t(z["ball.xyz"]), r, ns)
        assert np.array_equal(got.cpu().numpy(), z[f"ball.r{r}.ns{ns}.idx"]), (r, ns)
    d2, ix = pu.three_nn_raw(t(z["three.unknown"]), t(z["three.known"]))
    assert np.array_equal(ix.cpu().numpy(), z["three.idx"])
    assert np.array_equal(d2.cpu().numpy(), z["three.dist2"])
    out = pu.three_interpolate_raw(t(z["three.points"]), ix, t(z["three.weight"]))
    assert np.array_equal(out.cpu().numpy(), z["three.out"])
    gr = pu.three_interpolate_grad_raw(t(z["three.go"]), ix, t(z["three.weight"]), z["three.points"].shape[2])
    assert_close_rel(gr.cpu().numpy(), z["three.grad"], what="three_interpolate grad golden")


@pytest.mark.parametrize("B,n,m", [(2, 150, 64), (1, 3000, 5000), (2, 10, 2), (1, 5, 1)])
def test_three_nn_interpolate_vs_oracle(B, n, m):
    g = torch.Generator().manual_seed(700 + n)
    unknown, known = make_cloud(g, B, n), make_cloud(g, B, m, dup=min(10, m - 1))
    dist, ix = ps.three_nn(unknown.to(DEV), known.to(DEV))
    od, oi = O.three_nn(unknown.numpy(), known.numpy())
    assert np.array_equal(ix.cpu().numpy(), oi)
    assert np.array_equal(dist.cpu().numpy(), np.sqrt(od))
    C = 5
    pts = torch.randn(B, C, m, generator=g)
    w = torch.rand(B, n, 3, generator=g)
    f = pts.to(DEV).requires_grad_(True)
    out = ps.three_interpolate(f, ix, w.to(DEV))
    assert np.array_equal(out.detach().cpu().numpy(), O.three_interpolate(pts.numpy(), oi, w.numpy()))
    go = torch.randn(B, C, n, generator=g)
    out.backward(go.to(DEV))
    assert_close_rel(f.grad.cpu().numpy(), O.three_interpolate_grad(go.numpy(), oi, w.numpy(), m), what="interp grad")


# ---------------------------------------------------------------- kNN
@pytest.mark.parametrize("B,N,S,k,dup,inc", [(2, 2048, 512, 16, 0, True), (2, 1024, 256, 16, 300, True),
                                             (2, 512, 512, 8, 0, False), (1, 100, 40, 20, 0, True),
                                             (1, 600, 64, 40, 0, True), (1, 5000, 33, 16, 0, True),
                                             (1, 300, 10, 100, 0, True), (1, 16, 4, 16, 0, True)])
def test_knn_vs_oracle(B, N, S, k, dup, inc):
    g = torch.Generator().manual_seed(800 + N + k)
    xyz = make_cloud(g, B, N, dup=dup)
    new_xyz = xyz[:, :S].contiguous() if (dup or not inc) else make_cloud(g, B, S)
    got = ps.query_knn(k, xyz.to(DEV), new_xyz.to(DEV), include_self=inc)
    assert got.dtype == torch.int32 and tuple(got.shape) == (B, S, k)
    want = O.knn(xyz.numpy(), new_xyz.numpy(), k, 0 if inc else 1)
    assert np.array_equal(got.cpu().numpy(), want)


def test_knn_golden_torch_cuda():
    """Golden = the reference's torch expression run by torch on a B200 (cuBLAS + torch sort)."""
    z = load_golden("knn")
    for name in ("k16", "dups", "noself", "small", "k40"):
        k, inc = int(z[f"{name}.k"]), bool(z[f"{name}.include_self"])
        got = ps.query_knn(k, t(z[f"{name}.xyz"]), t(z[f"{name}.new_xyz"]), include_self=inc).cpu().numpy()
        want = z[f"{name}.idx"]
        if name == "dups":
            # exactly tied distances (duplicated points): torch.argsort(stable=False) leaves their
            # relative order unspecified; compare as sets per row and exactly where distances differ
            assert np.array_equal(np.sort(got, -1), np.sort(want, -1)), name
        else:
            assert np.array_equal(got, want), name


def test_knn_vs_torch_cuda_live_full_size():
    """C3 shape: our kernel vs query_knn evaluated by torch on this GPU; exact-match rate reported."""
    g = torch.Generator().manual_seed(1234 + 3)
    xyz = make_cloud(g, 32, 2048).to(DEV)
    got = ps.query_knn(16, xyz, xyz)
    want = O.torch_knn(16, xyz, xyz)
    match = (got == want).float().mean().item()
    print(f"kNN exact-match rate vs torch CUDA at C3: {match:.6f}")
    assert match == 1.0


# ---------------------------------------------------------------- error behaviour
def test_errors_raise_runtime_error():
    x = torch.rand(2, 16, 3)
    with pytest.raises(RuntimeError):
        ps.furthest_point_sample(x, 4)  # CPU tensor
    xc = x.to(DEV)
    with pytest.raises(RuntimeError):
        ps.furthest_point_sample(xc.transpose(1, 2), 4)  # non-contiguous / wrong shape
    with pytest.raises(RuntimeError):
        ps.gather_operation(xc, torch.zeros(2, 4, device=DEV, dtype=torch.int64))  # idx must be int32
    with pytest.raises(RuntimeError):
        ps.query_knn(32, xc, xc)  # k > N
    with pytest.raises(RuntimeError):
        ps.chamfer_forward(xc.double(), xc)


def test_streams_and_reentrancy():
    """Ops run on the caller's current stream and are safe from several host threads."""
    import threading
    g = torch.Generator().manual_seed(11)
    x = make_cloud(g, 4, 2048).to(DEV)
    want = ps.furthest_point_sample(x, 128)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = ps.furthest_point_sample(x, 128)
    s.synchronize()
    assert torch.equal(got, want)
    results = [None] * 4

    def work(i):
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            d = ps.chamfer_forward(x, x.flip(1).contiguous())
            results[i] = (d[0].sum().item(), ps.furthest_point_sample(x, 128))
    th = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [t_.start() for t_ in th]
    [t_.join() for t_ in th]
    assert all(torch.equal(r[1], want) for r in results)
    assert len({r[0] for r in results}) == 1


# ---------------------------------------------------------------- robustness
def _misaligned(t):
    """Same values in a contiguous tensor whose data pointer is only 4-byte aligned."""
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    view = flat[1:].view(t.shape)
    view.copy_(t)
    assert view.is_contiguous() and view.data_ptr() % 16 != 0
    return view


def test_misaligned_and_odd_sized_inputs_take_the_scalar_paths():
    g = torch.Generator().manual_seed(21)
    a, b = make_cloud(g, 3, 1031), make_cloud(g, 3, 2050)  # B*N*3 floats not a multiple of 4 either
    A, Bc = _misaligned(a.to(DEV)), _misaligned(b.to(DEV))
    d1, d2, i1, i2 = ps.chamfer_forward(A, Bc)
    od1, od2, oi1, oi2 = O.chamfer_fwd(a.numpy(), b.numpy())
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(i2.cpu().numpy(), oi2)
    assert np.array_equal(d1.cpu().numpy(), od1) and np.array_equal(d2.cpu().numpy(), od2)
    assert np.array_equal(ps.furthest_point_sample(Bc, 77).cpu().numpy(), O.fps(b.numpy(), 77))
    assert np.array_equal(ps.query_knn(9, Bc, A).cpu().numpy(), O.knn(b.numpy(), a.numpy(), 9))
    feat = torch.randn(3, 5, 2050, generator=g)
    idx = torch.randint(0, 2050, (3, 1031, 7), generator=g, dtype=torch.int32)
    F, I = _misaligned(feat.to(DEV)), _misaligned(idx.to(DEV))
    out = pu.group_raw(F, I)
    assert np.array_equal(out.cpu().numpy(), O.group(feat.numpy(), idx.numpy()))
    go = torch.randn(3, 5, 1031, 7, generator=g)
    gr = pu.group_grad_raw(_misaligned(go.to(DEV)), I, 2050)
    assert_close_rel(gr.cpu().numpy(), O.group_grad(go.numpy(), idx.numpy(), 2050), what="misaligned group grad")


def test_cuda_graph_capture_and_replay():
    """The whole path is stream-ordered (no host syncs, stream-ordered scratch), so a step can be
    captured once and replayed: launch-bound inner loops belong in CUDA graphs."""
    g = torch.Generator().manual_seed(31)
    a, b = make_cloud(g, 4, 2048).to(DEV), make_cloud(g, 4, 4096).to(DEV)
    feat = torch.randn(4, 16, 4096, generator=g).to(DEV)
    for _ in range(2):  # warm-up outside capture (function attributes, pools)
        ps.chamfer_forward(a, b); ps.furthest_point_sample(b, 256)
        pu.group_raw(feat, ps.query_knn(8, b, a))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        d1, d2, i1, i2 = ps.chamfer_forward(a, b)
        fidx = ps.furthest_point_sample(b, 256)
        knn = ps.query_knn(8, b, a)
        grp = pu.group_raw(feat, knn)
    a2, b2 = make_cloud(g, 4, 2048), make_cloud(g, 4, 4096)
    a.copy_(a2.to(DEV)); b.copy_(b2.to(DEV))
    graph.replay()
    torch.cuda.synchronize()
    od1, od2, oi1, oi2 = O.chamfer_fwd(a2.numpy(), b2.numpy())
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(d2.cpu().numpy(), od2)
    assert np.array_equal(fidx.cpu().numpy(), O.fps(b2.numpy(), 256))
    want_knn = O.knn(b2.numpy(), a2.numpy(), 8)
    assert np.array_equal(knn.cpu().numpy(), want_knn)
    assert np.array_equal(grp.cpu().numpy(), O.group(feat.cpu().numpy(), want_knn))


def test_repeatability_as_a_race_guard():
    """compute-sanitizer is closed on this GPU pool, so races in the cluster exchange (FPS), the
    shared-memory key merges (Chamfer) and the mbarrier rings (group) are guarded by repetition:
    25 back-to-back runs on two streams must be bit-identical (all three are deterministic by design)."""
    g = torch.Generator().manual_seed(41)
    x = make_cloud(g, 6, 16384, dup=2000, near_origin=6).to(DEV)
    y = make_cloud(g, 6, 3000, dup=500).to(DEV)
    feat = torch.randn(6, 16, 3000, generator=g).to(DEV)
    idx = torch.randint(0, 3000, (6, 2048, 16), generator=g, dtype=torch.int32).to(DEV)
    go = torch.randn(6, 16, 2048, 16, generator=g).to(DEV)
    ref = None
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for it in range(25):
        with torch.cuda.stream(streams[it & 1]):
            out = (ps.furthest_point_sample(x, 512), *ps.chamfer_forward(x, y), pu.group_raw(feat, idx),
                   pu.group_grad_raw(go, idx, 3000))
        streams[it & 1].synchronize()
        if ref is None:
            ref = [o.clone() for o in out]
        else:
            for k, (o, r) in enumerate(zip(out, ref)):
                assert torch.equal(o, r), f"output {k} changed on repetition {it}"


@pytest.mark.parametrize("cluster,threads,exchange", [(c, t, e) for c in (1, 2, 4, 8, 16) for t in (128, 256)
                                                     for e in (("lean", "async", "poll") if 1 < c <= 4 else ("async",))])
def test_fps_exchange_race_guard_over_the_forced_plan_matrix(monkeypatch, cluster, threads, exchange):
    """Every exchange protocol of the FPS kernel (single CTA, st.async + mbarrier all-to-all with 8-byte ("lean") and
    32-byte messages, the two-level variant for 8 / 16 CTAs, and the polling variant on plain remote stores), at both
    thread counts: 12 back-to-back runs on two streams with duplicates (ties on every iteration) must equal the oracle
    bit for bit, every time."""
    monkeypatch.setenv("PS_FPS_CLUSTER", str(cluster))
    monkeypatch.setenv("PS_FPS_THREADS", str(threads))
    monkeypatch.setenv("PS_FPS_LEAN", "1" if exchange == "lean" else "0")
    if exchange == "poll":
        monkeypatch.setenv("PS_FPS_EXCHANGE", "poll")
    N = {1: 2048, 2: 4096, 4: 8192, 8: 16384, 16: 16384}[cluster]
    g = torch.Generator().manual_seed(100 + cluster + threads)
    x = make_cloud(g, 3, N, dup=N // 4, near_origin=5)
    want = O.fps(x.numpy(), 200)
    xc = x.to(DEV)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for it in range(12):
        with torch.cuda.stream(streams[it & 1]):
            got = ps.furthest_point_sample(xc, 200)
        streams[it & 1].synchronize()
        assert np.array_equal(got.cpu().numpy(), want), f"cluster={cluster} threads={threads} {exchange}: run {it} differs"


def test_fused_fps_subsample_matches_unfused_call_site():
    """fps_subsample (models/model_utils.py:489-499): one kernel vs FPS + gather + transposes,
    forward values and the gather gradient."""
    g = torch.Generator().manual_seed(51)
    x = make_cloud(g, 3, 5000, dup=700, near_origin=4)
    xc = x.to(DEV).requires_grad_(True)
    sub = ps.fps_subsample(xc, 333)
    want_idx = O.fps(x.numpy(), 333)
    want = np.take_along_axis(x.numpy(), want_idx[..., None].astype(np.int64), axis=1)
    assert np.array_equal(sub.detach().cpu().numpy(), want)
    go = torch.randn(3, 333, 3, generator=g)
    sub.backward(go.to(DEV))
    want_g = O.gather_grad(go.numpy().transpose(0, 2, 1).copy(), want_idx, 5000).transpose(0, 2, 1)
    assert_close_rel(xc.grad.cpu().numpy(), want_g, what="fps_subsample grad")
    # the unfused composition gives the same tensor
    unf = ps.gather_operation(xc.detach().permute(0, 2, 1).contiguous(), ps.furthest_point_sample(xc.detach(), 333))
    assert torch.equal(unf.permute(0, 2, 1).contiguous(), sub.detach())


@pytest.mark.parametrize("select", ["1", "0"])
def test_knn_heavy_duplication_and_both_kernels(select, monkeypatch):
    """The threshold-selection kernel (N <= 2048, k+skip <= 16) must fall back correctly when far
    more than 32 candidates tie at the threshold; PS_KNN_SELECT=0 exercises the streaming kernel."""
    monkeypatch.setenv("PS_KNN_SELECT", select)
    g = torch.Generator().manual_seed(61)
    xyz = make_cloud(g, 2, 1500)
    xyz[:, 100:400] = xyz[:, 7:8]          # 300 copies of one point
    xyz[:, 900:960] = xyz[:, 800:801]      # 60 copies of another
    q = torch.cat([xyz[:, 5:9], xyz[:, 798:803], make_cloud(g, 2, 40)], 1).contiguous()
    for k, inc in ((16, True), (15, False), (3, True)):
        got = ps.query_knn(k, xyz.to(DEV), q.to(DEV), include_self=inc)
        want = O.knn(xyz.numpy(), q.numpy(), k, 0 if inc else 1)
        assert np.array_equal(got.cpu().numpy(), want), (k, inc)
    for N in (16, 33, 500, 2048):          # short clouds: padding steps, N < 32 lanes
        x = make_cloud(g, 2, N, dup=N // 5)
        got = ps.query_knn(min(16, N), x.to(DEV), x.to(DEV))
        assert np.array_equal(got.cpu().numpy(), O.knn(x.numpy(), x.numpy(), min(16, N))), N


def test_empty_batches_and_zero_sized_requests_are_no_ops():
    """B = 0, npoint = 0, M = 0: the reference's kernels simply do not iterate; ours return
    correctly shaped empty tensors without touching the (null) pointers."""
    e3 = torch.empty(0, 16, 3, device=DEV)
    d1, d2, i1, i2 = ps.chamfer_forward(e3, torch.empty(0, 8, 3, device=DEV))
    assert tuple(d1.shape) == (0, 16) and tuple(i2.shape) == (0, 8) and i1.dtype == torch.int32
    assert tuple(ps.furthest_point_sample(e3, 4).shape) == (0, 4)
    x = make_cloud(torch.Generator().manual_seed(1), 2, 64).to(DEV)
    assert tuple(ps.furthest_point_sample(x, 0).shape) == (2, 0)
    feat = torch.randn(2, 5, 64, device=DEV)
    assert tuple(ps.gather_operation(feat, torch.empty(2, 0, device=DEV, dtype=torch.int32)).shape) == (2, 5, 0)
    assert tuple(ps.grouping_operation(feat, torch.empty(2, 0, 4, device=DEV, dtype=torch.int32)).shape) == (2, 5, 0, 4)
    g = pu.gather_grad_raw(torch.empty(2, 5, 0, device=DEV), torch.empty(2, 0, device=DEV, dtype=torch.int32), 64)
    assert tuple(g.shape) == (2, 5, 64) and torch.count_nonzero(g) == 0
    assert tuple(ps.query_knn(4, x, torch.empty(2, 0, 3, device=DEV)).shape) == (2, 0, 4)
    assert tuple(ps.ball_query(0.1, 4, x, torch.empty(2, 0, 3, device=DEV)).shape) == (2, 0, 4)
    torch.cuda.synchronize()


def test_chamfer_host_step_matches_device_entry_points():
    """ps_chamfer_host_step: host clouds in, loss sums out, gradients left in device buffers — equal to
    forward + sums + backward on resident tensors, for ragged chunk plans and on replay of the captured graph."""
    g = torch.Generator().manual_seed(77)
    B, N, M = 7, 700, 1900
    a, b = make_cloud(g, B, N, dup=100).pin_memory(), make_cloud(g, B, M, dup=300).pin_memory()
    gd1, gd2 = torch.randn(B, N, generator=g).pin_memory(), torch.randn(B, M, generator=g).pin_memory()
    A, Bc = a.to(DEV), b.to(DEV)
    d1, d2, i1, i2 = ps.chamfer_forward(A, Bc)
    want_sums = ps.chamfer_sums(d1, d2).cpu()
    w1, w2 = ps.chamfer_backward(A, Bc, gd1.to(DEV), gd2.to(DEV), i1, i2)
    for chunk in (0, 2, 7, 3):
        for rep in range(2):  # second call replays the CUDA graph
            sums, g1, g2 = ps.chamfer_host_step(a, b, gd1, gd2, chunk=chunk)
            assert torch.allclose(sums, want_sums, rtol=1e-12, atol=0), (chunk, rep)
            assert_close_rel(g1.cpu().numpy(), w1.cpu().numpy(), what="gradxyz1")
            assert_close_rel(g2.cpu().numpy(), w2.cpu().numpy(), what="gradxyz2")
    sums, g1, g2 = ps.chamfer_host_step(a, b)  # forward + sums only
    assert g1 is None and g2 is None and torch.allclose(sums, want_sums, rtol=1e-12, atol=0)
    with pytest.raises(ps.PointSeaError):
        ps.chamfer_host_step(a, b, gd1, None)
    with pytest.raises(ps.PointSeaError):
        ps.chamfer_host_step(A, Bc)
