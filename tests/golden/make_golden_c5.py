"""Generate tests/golden/c5.npz: the CPU oracle's FPS indices for the C5 stress input (2 clouds of 131072 points
with duplicates and points inside the skip ball, 131072 -> 16384), the input's seed recipe being that of
tests/test_gpu_configs.py.  The oracle is the reference kernel restated bit for bit (tests/test_oracle_golden.py
pins it to the reference's own outputs); it needs no GPU, but a few minutes of one core at this size.

    python tests/golden/make_golden_c5.py tests/golden
"""
import hashlib
import os.path as osp
import sys

import numpy as np
import torch

ROOT = osp.dirname(osp.dirname(osp.dirname(osp.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, osp.join(ROOT, "tests"))
from conftest import make_cloud  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main(out_dir):
    g = torch.Generator().manual_seed(1234 + 5)
    xyz = make_cloud(g, 2, 131072, dup=3000, near_origin=40).numpy()
    np.savez_compressed(osp.join(out_dir, "c5.npz"), **{"fps.idx": O.fps(xyz, 16384),
                                                        "fps.xyz_sha256": np.str_(hashlib.sha256(xyz.tobytes()).hexdigest())})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else osp.join(ROOT, "tests", "golden"))
