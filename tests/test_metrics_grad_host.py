"""Host-side checks of the differentiable calc_cd / calc_dcd: the backward entry point validates its arguments before
any device work, and CPU clouds are refused whether or not they require grad (no CPU fallback)."""
import ctypes

import pytest
import torch

import svdformer_pointsea_b200 as ps
from svdformer_pointsea_b200 import _lib as L

FAKE = ctypes.c_void_p(0x1000)  # never dereferenced: validation fails first


def bwd(dist1=FAKE, dist2=FAKE, idx1=FAKE, idx2=FAKE, gcoef5=FAKE, terms=31, graw1=None, graw2=None, gd1=FAKE,
        gd2=FAKE, B=2, n1=8, n2=9):
    lib = L.load()
    rc = lib.ps_chamfer_metrics_bwd(dist1, dist2, idx1, idx2, gcoef5, terms, graw1, graw2, gd1, gd2, B, n1, n2,
                                    1000.0, 1.0, 1.0, 1.0, 0, None)
    return rc, lib.ps_last_error()


@pytest.mark.parametrize("B,n1,n2", [(-1, 8, 9), (2, 0, 9), (2, 8, 0), (2, -4, 9)])
def test_metrics_bwd_rejects_bad_sizes(B, n1, n2):
    rc, msg = bwd(B=B, n1=n1, n2=n2)
    assert rc == -1 and b"bad sizes" in msg


@pytest.mark.parametrize("terms", [32, 64, 1 << 31, 31 | 128])
def test_metrics_bwd_rejects_unknown_term_bits(terms):
    rc, msg = bwd(terms=terms)
    assert rc == -1 and b"unknown terms bits" in msg
    rc, msg = bwd(terms=terms, B=0)  # even when there is no work
    assert rc == -1 and b"unknown terms bits" in msg


@pytest.mark.parametrize("missing,terms", [("dist1", 31), ("dist2", 1), ("gd1", 0), ("gd2", 4), ("gcoef5", 1),
                                           ("gcoef5", 16), ("idx1", 16), ("idx2", 31)])
def test_metrics_bwd_rejects_null_pointers(missing, terms):
    rc, msg = bwd(terms=terms, **{missing: None})
    assert rc == -1 and b"null pointer" in msg


def test_metrics_bwd_empty_batch_is_a_no_op():
    assert bwd(None, None, None, None, None, 31, None, None, None, None, B=0)[0] == 0


@pytest.mark.parametrize("which", ["cd", "dcd"])
@pytest.mark.parametrize("grad", ["x", "gt", "both", "none"])
def test_cpu_clouds_raise_with_or_without_grad(which, grad):
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(2, 16, 3, generator=g) - 0.5).requires_grad_(grad in ("x", "both"))
    gt = (torch.rand(2, 20, 3, generator=g) - 0.5).requires_grad_(grad in ("gt", "both"))
    fn = ps.calc_cd if which == "cd" else ps.calc_dcd
    with pytest.raises(ps.PointSeaError):
        fn(x, gt)
