"""The C-ABI library builds, loads without a GPU and exports what include/ofc.h declares."""
import ctypes
import os
import re

import pytest

from tests.conftest import ROOT, run_without_gpu


@pytest.fixture(scope="module")
def so_path():
    from opticalflowclustering_b200 import _build
    return _build.build()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "ofc.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ofc_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(so_path):
    lib = ctypes.CDLL(so_path)
    names = declared_symbols()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/ofc.h but not exported"
    assert lib.ofc_version() >= 100


def test_python_binding_covers_header(so_path):
    from opticalflowclustering_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    _lib.lib()                                        # sets argtypes on every symbol


def test_sass_is_sm100a(so_path):
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", so_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_gpu_means_loud_failure():
    """No CPU fallback: without a CUDA device the operators raise."""
    out = run_without_gpu("""
import numpy as np
import torch
assert not torch.cuda.is_available()
from opticalflowclustering_b200 import _lib, flow
try:
    flow.calc_optical_flow_farneback(np.zeros((64, 64), np.uint8), np.zeros((64, 64), np.uint8), None,
                                     0.5, 3, 15, 3, 5, 1.2, 0)
except _lib.OfcError:
    print("raised")
""")
    assert out.split() == ["raised"]


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "opticalflowclustering_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "libofc_emu" not in text, f
