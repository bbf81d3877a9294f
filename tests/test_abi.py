"""The C-ABI library loads, exports every symbol include/cuba_b200.h declares, and refuses to compute
without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "cuba_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cuba_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(pkg):
    lib = ctypes.CDLL(pkg.library_path())
    names = _declared_functions()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), "libcuba_b200.so lacks %s" % n
    # the binding's list is the same set
    assert sorted(pkg.binding.exported_symbols()) == names


def test_cpp_api_symbols_present(pkg):
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", "-C", pkg.library_path()], capture_output=True, text=True).stdout
    assert "cuba::CudaBundleAdjustment::create()" in out
    assert "cuba::CudaBundleAdjustment::~CudaBundleAdjustment()" in out


def test_only_sm100a_code_is_embedded(pkg):
    import subprocess
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", pkg.library_path()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_no_cpu_fallback(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.CubaError, match="no CPU fallback"):
        pkg.Engine()


def _create_with_reserved(pkg, field, value):
    """cuba_engine_create straight through the C ABI, with cuba_config.reserved[field] = value"""
    b = pkg.binding
    L = b.load_library()
    res = (ctypes.c_int * 7)()
    res[field] = value
    cfg = b._Config(-1, 0, 0, 0.0, 1, res)
    h = ctypes.c_void_p()
    b._check(L.cuba_engine_create(ctypes.byref(cfg), ctypes.byref(h)))
    L.cuba_engine_destroy(h)


@pytest.mark.parametrize("field,value", [(0, 1), (0, 9), (0, -1), (1, 2), (2, 1), (2, 2), (2, 3), (2, 5), (2, 6), (2, 7), (2, 8), (2, 9),
                                         (3, 1), (3, 2), (3, 4), (3, 5), (3, 6)])
def test_engine_refuses_reserved_values_that_select_no_kernel(pkg, field, value):
    """reserved[0..3] select kernels; a value that selects none (a retired kernel, or one that never existed) is refused before
    any device is touched, and the message names the field and the value"""
    with pytest.raises(pkg.CubaError, match=r"reserved\[%d\] = %d selects no kernel" % (field, value)):
        _create_with_reserved(pkg, field, value)


@pytest.mark.parametrize("field,value", [(0, v) for v in (0, 2, 3, 4, 5, 6, 7, 8)] + [(1, 1), (2, 4), (3, 3)])
def test_engine_accepts_reserved_values_that_select_a_kernel(pkg, field, value):
    """validation lets every kept value through: engine creation then succeeds, or, without a GPU, fails for that reason alone"""
    try:
        _create_with_reserved(pkg, field, value)
    except pkg.CubaError as e:
        assert "no CPU fallback" in str(e)


def test_product_does_not_touch_the_oracle():
    """the product package and its native sources never import / link anything under oracle/"""
    pdir = os.path.join(ROOT, "cuda-bundle-adjustment_b200")
    for dirpath, _, files in os.walk(pdir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "ba_oracle" not in text and "libcuba_ref" not in text, f
                assert not re.search(r"^\s*(import|from)\s+oracle", text, flags=re.M), f
