import hashlib
import os.path as osp
import sys

import numpy as np
import pytest

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = osp.join(ROOT, "tests", "golden")

from __graft_entry__ import reference_path  # noqa: E402

# checkout of the reference (not part of this repository) for the tests that run its own code
REFERENCE = reference_path()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class Golden(dict):
    """The arrays of one golden .npz file (`files` lists their names, as numpy's NpzFile does)."""

    @property
    def files(self):
        return list(self)


# next.npz leaves out its largest input, edge256.x (0.5 MB of float32 noise): it is redrawn from the seeded generator
# sequence that produced it (tests/golden/make_golden_next.py), and the digest of the array it replaces guards it
EDGE256_X_SHA256 = "d7df3ef47eea38e4f38b1379afbe95039b39bae883a0201a99c88858221057a6"


def _edge256_x():
    import torch
    g = torch.Generator().manual_seed(1234 + 12)
    make_cloud(g, 2, 1024)                 # edge3, edge3dup and edge64 draw first
    make_cloud(g, 2, 700, dup=200)
    torch.randn(2, 64, 512, generator=g)
    x = torch.randn(1, 256, 512, generator=g).numpy()
    assert hashlib.sha256(x.tobytes()).hexdigest() == EDGE256_X_SHA256, "torch's generator no longer redraws edge256.x"
    return x


def load_golden(name):
    path = osp.join(GOLDEN, name + ".npz")
    if not osp.exists(path):
        pytest.skip(f"{path} not generated yet")
    z = Golden(np.load(path))
    if name == "next":
        z["edge256.x"] = _edge256_x()
    return z


def make_cloud(gen, B, N, dup=0, near_origin=0):
    """Seeded rand-0.5 cloud (SURVEY 8d); `dup` duplicates points like UpSamplePoints does."""
    import torch
    x = torch.rand(B, N, 3, generator=gen) - 0.5
    if dup:
        uniq = N - dup
        for b in range(B):
            src = torch.randint(0, uniq, (dup,), generator=gen)
            x[b, uniq:] = x[b, src]
    if near_origin:
        for b in range(B):
            pos = torch.randperm(N, generator=gen)[:near_origin]
            x[b, pos] = (torch.rand(near_origin, 3, generator=gen) - 0.5) * 0.03
    return x.contiguous()
