"""The C-ABI library loads on a CPU-only box and exports every symbol include/ogl_b200.h declares
(no compute calls here); the product fails loudly without a device."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "ogl_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ogl_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported():
    import ogl_b200
    lib = ctypes.CDLL(ogl_b200.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), "missing export: " + n


def test_binding_table_covers_header():
    from ogl_b200._lib import SIGNATURES
    assert sorted(SIGNATURES) == declared_symbols()


def test_abi_version():
    """105: ogl_plan_backward takes max |dlogits| (mode OGL_FP16 picks its gradient scale from it)"""
    import ogl_b200
    lib = ctypes.CDLL(ogl_b200.LIB_PATH)
    assert lib.ogl_version() == 105
    from ogl_b200._lib import SIGNATURES
    assert SIGNATURES["ogl_plan_backward"][1][2] is ctypes.c_float


def test_fails_loudly_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ogl_b200
    with pytest.raises(ogl_b200.OglError) as e:
        ogl_b200.native.Graph(16, 16)
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "online-gnn-learning_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
