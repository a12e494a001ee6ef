"""CPU tests (no GPU, no compute calls): the C-ABI library loads and exports exactly what
include/geoformer_b200.h declares, and the Python binding table agrees with both."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "geoformer_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return set(re.findall(r"\b(gf_[a-z0-9_]+)\s*\(", src))


def test_header_declares_every_binding_and_vice_versa(cuda_lib):
    from geoformer_b200 import _capi

    declared = _declared()
    assert declared, "no gf_* prototypes found in the header"
    assert declared == set(_capi.SIGNATURES), (declared ^ set(_capi.SIGNATURES))
    for name in declared:
        assert hasattr(cuda_lib, name), "library does not export %s" % name


def test_library_exports_no_torch_or_oracle_symbols(cuda_lib):
    from geoformer_b200 import _capi

    out = subprocess.check_output(["nm", "-D", "--defined-only", _capi.LIB_PATH], text=True)
    exported = [l.split()[-1] for l in out.splitlines() if " T " in l]
    gf = [s for s in exported if s.startswith("gf_")]
    assert set(gf) == _declared()
    assert not [s for s in exported if "orc_" in s], "the product must not contain the oracle"
    needed = subprocess.check_output(["ldd", _capi.LIB_PATH], text=True)
    assert "libtorch" not in needed and "libc10" not in needed and "liboracle" not in needed


def test_library_is_built_for_sm_100a(cuda_lib):
    from geoformer_b200 import _capi

    out = subprocess.run(["cuobjdump", "-lelf", _capi.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:  # cuobjdump not on PATH
        out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", _capi.LIB_PATH], capture_output=True, text=True)
    assert "sm_100a" in out.stdout, out.stdout + out.stderr


def test_version_and_error_plumbing(cuda_lib):
    assert cuda_lib.gf_version() >= 100
    # argument validation happens before any CUDA call: negative sizes are rejected with a message
    rc = cuda_lib.gf_gather_points(None, None, -1, 1, 1, 1, None, None)
    assert rc == 1 and b"negative" in cuda_lib.gf_last_error()
    assert cuda_lib.gf_knn_workspace_bytes(1000, 1000, 16, 1) == 0
    assert cuda_lib.gf_knn_workspace_bytes(1000, 1000, 16, 0) > 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "geoformer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "liboracle" not in text, f


def test_ops_fail_loudly_on_cpu_tensors(cuda_lib):
    import pytest
    import torch

    from geoformer_b200.geodesic_utils import cal_geodesic_vectorize, knn_graph
    from geoformer_b200.pointnet2 import _ext

    with pytest.raises(RuntimeError):
        _ext.furthest_point_sampling(torch.zeros(1, 8, 3), 2)
    with pytest.raises(RuntimeError):
        knn_graph(torch.zeros(8, 3), 2)
    with pytest.raises(RuntimeError):
        cal_geodesic_vectorize(None, torch.zeros(1, 4, dtype=torch.int32), torch.zeros(8, 3),
                               torch.tensor([0, 8], dtype=torch.int32), n_queries=2, neighbor=2)
