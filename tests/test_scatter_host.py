"""Host-side checks of the torch_scatter drop-in: ps_scatter_max validates its arguments before any CUDA call, the
Python scatter() refuses what it does not cover without touching a device, and `import torch_scatter` resolves to the
drop-in only where no torch_scatter is installed (checked in subprocesses, so this process's sys.modules stays clean)."""
import ctypes
import json
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT
from svdformer_pointsea_b200 import _lib as L
from svdformer_pointsea_b200 import dropin
from svdformer_pointsea_b200.scatter import scatter

FAKE = ctypes.c_void_p(0x1000)  # never dereferenced: validation fails first or there is nothing to do


def call(src=FAKE, index=FAKE, out=FAKE, arg=None, outer=2, E=5, inner=3, D=4, fresh=0):
    lib = L.load()
    rc = lib.ps_scatter_max(src, index, out, arg, outer, E, inner, D, fresh, 0, None)
    return rc, lib.ps_last_error()


@pytest.mark.parametrize("outer,E,inner,D", [(-1, 5, 3, 4), (2, -5, 3, 4), (2, 5, -3, 4), (2, 5, 3, -4),
                                             (1 << 40, 1 << 40, 1, 4), (2, 5, 1 << 40, 1 << 40)])
def test_scatter_max_rejects_bad_sizes(outer, E, inner, D):
    rc, msg = call(outer=outer, E=E, inner=inner, D=D)
    assert rc == -1 and b"bad sizes" in msg


@pytest.mark.parametrize("missing,fresh", [("src", 0), ("index", 0), ("out", 0), ("out", 1), ("src", 1)])
def test_scatter_max_rejects_null_pointers(missing, fresh):
    rc, msg = call(fresh=fresh, **{missing: None})
    assert rc == -1 and b"null pointer" in msg


def test_scatter_max_fresh_output_without_src_needs_out():
    rc, msg = call(src=None, index=None, out=None, E=0, fresh=1)
    assert rc == -1 and b"null pointer" in msg


@pytest.mark.parametrize("kw", [dict(outer=0), dict(inner=0), dict(D=0), dict(D=0, fresh=1, arg=FAKE), dict(E=0),
                                dict(outer=0, fresh=1, arg=FAKE)])
@pytest.mark.parametrize("pointers", ["null", "given"])
def test_scatter_max_empty_work_is_a_no_op(kw, pointers):
    """Nothing to write (an empty output; with D == 0 every index is out of range) or nothing to read into an `out=`
    output: success without a CUDA call, whatever the pointers."""
    ptrs = dict(src=None, index=None, out=None) if pointers == "null" else {}
    assert call(**ptrs, **kw)[0] == 0


@pytest.fixture
def no_device(monkeypatch):
    """Any attempt to reach the native library or a device fails the test."""
    def boom(*a, **k):
        raise AssertionError("touched the device")
    monkeypatch.setattr(L, "load", boom)
    monkeypatch.setattr(L, "same_device", boom)
    monkeypatch.setattr(torch.cuda, "synchronize", boom)


def test_other_reductions_are_not_implemented(no_device):
    src, idx = torch.rand(2, 8), torch.zeros(2, 8, dtype=torch.int64)
    for reduce in ("sum", "add", "mean", "min", "mul"):
        with pytest.raises(NotImplementedError, match="installed torch_scatter takes precedence"):
            scatter(src, idx, 1, reduce=reduce)
    with pytest.raises(NotImplementedError):
        scatter(src, idx, 1)  # torch_scatter's default reduce is "sum"


def test_refused_dtypes_and_cpu_tensors(no_device):
    src, idx = torch.rand(2, 8), torch.zeros(2, 8, dtype=torch.int64)
    with pytest.raises(L.PointSeaError, match="float32"):
        scatter(src.double(), idx, 1, reduce="max")
    with pytest.raises(L.PointSeaError, match="int64"):
        scatter(src, idx.int(), 1, reduce="max")
    with pytest.raises(L.PointSeaError, match="CUDA"):
        scatter(src, idx, 1, reduce="max")
    with pytest.raises(L.PointSeaError, match="CUDA"):
        scatter(src.requires_grad_(True), idx, 1, out=torch.zeros(2, 3), reduce="max")


def resolve(code, extra_path=None, prologue=""):
    """Runs `code` in a fresh interpreter with the repository importable; returns the JSON it prints."""
    pp = [ROOT] + ([extra_path] if extra_path else [])
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(pp))
    script = "import json, sys\n" + prologue + code
    p = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, env=env, cwd=ROOT,
                       timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


# whether a torch_scatter other than the drop-in is importable before install_dropin() runs
FIND = """import importlib.util
spec = importlib.util.find_spec('torch_scatter')
installed = spec is not None and 'dropin_fallback' not in (spec.origin or '')
"""
IMPORTS = """import svdformer_pointsea_b200 as ps
ps.install_dropin()
import torch_scatter
import metrics.CD.chamfer3D.dist_chamfer_3D as cd
import pointnet2_ops.pointnet2_utils as pu
from svdformer_pointsea_b200.scatter import scatter
print(json.dumps({"installed": installed, "torch_scatter": torch_scatter.__file__,
                  "same_scatter": getattr(torch_scatter, "scatter", None) is scatter,
                  "cd": cd.__file__, "pu": pu.__file__}))
"""


def test_install_dropin_resolves_torch_scatter_to_the_fallback():
    r = resolve(FIND + IMPORTS)
    if r["installed"]:
        pytest.skip("a torch_scatter is installed here; the fallback correctly stays behind it")
    assert r["torch_scatter"].startswith(dropin.DROPIN_FALLBACK_PATH + os.sep) and r["same_scatter"]
    assert r["cd"].startswith(dropin.DROPIN_PATH + os.sep) and r["pu"].startswith(dropin.DROPIN_PATH + os.sep)


def fake_torch_scatter(tmp_path):
    pkg = tmp_path / "site" / "torch_scatter"
    pkg.mkdir(parents=True)
    (pkg / "__init__.py").write_text("def scatter(*a, **k):\n    return 'fake'\n")
    return str(tmp_path / "site")


def test_torch_scatter_on_pythonpath_wins(tmp_path):
    site = fake_torch_scatter(tmp_path)
    r = resolve(FIND + IMPORTS, extra_path=site)
    assert r["torch_scatter"].startswith(site + os.sep) and not r["same_scatter"]
    assert r["cd"].startswith(dropin.DROPIN_PATH + os.sep) and r["pu"].startswith(dropin.DROPIN_PATH + os.sep)


def test_torch_scatter_on_sys_path_before_install_wins(tmp_path):
    """An installed package sits in a sys.path entry (site-packages) that exists before install_dropin() runs."""
    site = fake_torch_scatter(tmp_path)
    r = resolve(FIND + IMPORTS, prologue=f"sys.path.append({site!r})\n")
    assert r["torch_scatter"].startswith(site + os.sep) and not r["same_scatter"]
    assert r["cd"].startswith(dropin.DROPIN_PATH + os.sep) and r["pu"].startswith(dropin.DROPIN_PATH + os.sep)


def test_documented_pythonpath_form_resolves_every_dropin():
    """INTEGRATION.md §1: PYTHONPATH=<repo>:<dropin_pkgs>:...:<dropin_fallback>, no install_dropin() call."""
    code = FIND + """import torch_scatter, metrics.CD.chamfer3D.dist_chamfer_3D as cd, pointnet2_ops.pointnet2_utils as pu
print(json.dumps({"installed": installed, "torch_scatter": torch_scatter.__file__, "cd": cd.__file__,
                  "pu": pu.__file__}))
"""
    r = resolve(code, extra_path=os.pathsep.join([dropin.DROPIN_PATH, dropin.DROPIN_FALLBACK_PATH]))
    assert r["cd"].startswith(dropin.DROPIN_PATH + os.sep) and r["pu"].startswith(dropin.DROPIN_PATH + os.sep)
    if not r["installed"]:
        assert r["torch_scatter"].startswith(dropin.DROPIN_FALLBACK_PATH + os.sep)
