"""Pins the CPU oracle (oracle/pointsea_oracle.c) to the golden vectors in tests/golden/, which
are outputs of the reference's OWN CUDA kernels run on a B200 (tests/golden/make_golden.py)."""
import numpy as np

from conftest import load_golden
from oracle import oracle as O


def rel(a, b):
    return np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / max(np.abs(b).max(), 1e-30)


def test_chamfer_forward_bit_exact_and_backward_close():
    z = load_golden("chamfer")
    for name in ("small", "tiles", "dups", "tiny"):
        d1, d2, i1, i2 = O.chamfer_fwd(z[f"{name}.xyz1"], z[f"{name}.xyz2"])
        assert np.array_equal(i1, z[f"{name}.idx1"]) and np.array_equal(i2, z[f"{name}.idx2"]), name
        assert np.array_equal(d1, z[f"{name}.dist1"]) and np.array_equal(d2, z[f"{name}.dist2"]), name
        g1, g2 = O.chamfer_bwd(z[f"{name}.xyz1"], z[f"{name}.xyz2"], z[f"{name}.gd1"], z[f"{name}.gd2"], i1, i2)
        assert rel(g1, z[f"{name}.g1"]) < 1e-5 and rel(g2, z[f"{name}.g2"]) < 1e-5, name


def test_chamfer_ties_resolve_to_lowest_index():
    z = load_golden("chamfer")
    # the 'dups' case has duplicated targets: every reported index must be the first of its twins
    xyz2, idx1 = z["dups.xyz2"], z["dups.idx1"]
    for b in range(xyz2.shape[0]):
        for j in np.unique(idx1[b]):
            twins = np.where((xyz2[b] == xyz2[b, j]).all(-1))[0]
            assert j == twins.min()


def test_fps_bit_exact_including_ties_and_origin_skip():
    z = load_golden("fps")
    for name in ("n1000", "dups2048", "bs256", "origin", "n16384", "npow2", "tiny"):
        want = z[f"{name}.idx"]
        got = O.fps(z[f"{name}.xyz"], want.shape[1])
        assert np.array_equal(got, want), name
    # the 'origin' case really exercises the skip rule
    x = z["origin.xyz"]
    mag = (x.astype(np.float64) ** 2).sum(-1)
    skipped = np.where(mag[0] <= 1e-3)[0]
    assert len(skipped) > 0 and not np.isin(z["origin.idx"][0][1:], skipped).any()


def test_gather_group_exact():
    z = load_golden("pointnet2")
    assert np.array_equal(O.gather(z["gather.feat"], z["gather.idx"]), z["gather.out"])
    assert rel(O.gather_grad(z["gather.go"], z["gather.idx"], z["gather.feat"].shape[2]), z["gather.grad"]) < 1e-6
    assert np.array_equal(O.group(z["group.feat"], z["group.idx"]), z["group.out"])
    assert rel(O.group_grad(z["group.go"], z["group.idx"], z["group.feat"].shape[2]), z["group.grad"]) < 1e-6


def test_ball_query_exact():
    z = load_golden("pointnet2")
    for r, ns in ((0.2, 16), (0.05, 8), (0.6, 32)):
        got = O.ball_query(z["ball.new_xyz"], z["ball.xyz"], r, ns)
        assert np.array_equal(got, z[f"ball.r{r}.ns{ns}.idx"]), (r, ns)


def test_three_nn_and_interpolate_exact():
    z = load_golden("pointnet2")
    d2, ix = O.three_nn(z["three.unknown"], z["three.known"])
    assert np.array_equal(ix, z["three.idx"]) and np.array_equal(d2, z["three.dist2"])
    assert np.array_equal(O.three_interpolate(z["three.points"], ix, z["three.weight"]), z["three.out"])
    assert rel(O.three_interpolate_grad(z["three.go"], ix, z["three.weight"], z["three.points"].shape[2]), z["three.grad"]) < 1e-6


def test_knn_matches_torch_cuda_golden():
    """kNN golden = the reference's torch expression run on the GPU (cuBLAS dot + torch sort)."""
    z = load_golden("knn")
    for name in ("k16", "dups", "noself", "small", "k40"):
        k, inc = int(z[f"{name}.k"]), bool(z[f"{name}.include_self"])
        got = O.knn(z[f"{name}.xyz"], z[f"{name}.new_xyz"], k, 0 if inc else 1)
        assert np.array_equal(got, z[f"{name}.idx"]), name


def test_knn_distance_arithmetic_matches_torch_cuda_bits():
    """The stored (S,N) distance rows pin the fp32 arithmetic: dot = fma(z,z',fma(y,y',x*x')),
    |p|^2 = (x^2 + z^2) + y^2, dist = ((-2*dot) + |q|^2) + |p|^2.  'dups' stores a seeded sample of its rows."""
    z = load_golden("knn")
    f = np.float32
    for name in ("small", "dups"):
        rows = z[f"{name}.rows"] if f"{name}.rows" in z.files else slice(None)
        q, p, dist = z[f"{name}.new_xyz"][:, rows], z[f"{name}.xyz"], z[f"{name}.dist"]

        def ss(v):
            a, b, c = [(v[..., i] * v[..., i]).astype(f) for i in range(3)]
            return ((a + c).astype(f) + b).astype(f)

        d = ((f(-2) * z[f"{name}.dot"]).astype(f) + ss(q)[:, :, None]).astype(f) + ss(p)[:, None, :]
        assert np.array_equal(d.astype(f), dist)


def test_oracle_against_pure_torch_reexpression():
    """Independent cross-check on fresh seeded inputs: indices agree wherever the minimum is unique
    enough for torch's unfused arithmetic."""
    import torch
    g = torch.Generator().manual_seed(3)
    a, b = torch.rand(2, 200, 3, generator=g) - 0.5, torch.rand(2, 333, 3, generator=g) - 0.5
    d1, d2, i1, i2 = O.chamfer_fwd(a.numpy(), b.numpy())
    t1, t2, j1, j2 = O.torch_chamfer(a, b)
    assert (i1 == j1.numpy()).mean() > 0.995 and (i2 == j2.numpy()).mean() > 0.995
    assert rel(d1, t1.numpy()) < 1e-5
    fi = O.fps(b.numpy(), 32)
    assert (fi == O.torch_fps(b, 32).numpy()).mean() > 0.9
