"""CPU tier: the C-ABI library loads without a GPU and exports every symbol include/afe_cuda.h declares;
compute entry points fail loudly (no CPU fallback) when no CUDA device is usable."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import afe_loader

afe = afe_loader.load()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "afe_cuda.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(afe_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    assert header_symbols() == sorted(afe.SYMBOLS)


def header_abi_version():
    return int(re.search(r"#define AFE_ABI_VERSION (\d+)", open(os.path.join(ROOT, "include", "afe_cuda.h")).read()).group(1))


def test_library_abi_version_and_exported_symbols():
    """The library, the header and the binding name the same ABI version (3: the tensor-core phase-2 flag removed, unknown
    batch flags refused), and the library exports every symbol the header declares."""
    L = afe.lib()
    for name in header_symbols():
        assert hasattr(L, name), name
    assert L.afe_abi_version() == afe.ABI_VERSION == header_abi_version() == 3
    assert L.afe_build_flags() == 0, "the product library must not be a -DAFE_DEVTOOLS build"


def test_product_build_has_no_debug_environment_hooks():
    """ADVICE r1 / VERDICT r1 #7: no getenv in the shipped sources outside #ifdef AFE_DEVTOOLS, no library override."""
    pkg = os.path.join(ROOT, "asr-featext-opencl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                continue
            text = open(os.path.join(dirpath, f), errors="ignore").read()
            assert "AFE_LIB_OVERRIDE" not in text and "AFE_TILE_FRAMES" not in text, f
            # every getenv sits inside an AFE_DEVTOOLS block
            stripped = re.sub(r"#ifdef AFE_DEVTOOLS.*?#endif", "", text, flags=re.S)
            assert "getenv" not in stripped and "environ" not in stripped, f


def test_no_cpu_fallback_without_device():
    L = afe.lib()
    if L.afe_device_count() > 0:
        pytest.skip("a CUDA device is present")
    p = afe.make_params()
    for ctor in (lambda: afe.MfccCuda(p), lambda: afe.BatchMfcc(p), lambda: afe.SegmenterCuda(400, 160, 10, 0),
                 lambda: afe.DeltaCuda(13, 10, 3), lambda: afe.NormalizerCuda(1, 13)):
        with pytest.raises(afe.AfeError, match="no usable CUDA device"):
            ctor()


def test_product_does_not_import_the_oracle():
    """The product path must never route through oracle/ (it is test infrastructure)."""
    pkg = os.path.join(ROOT, "asr-featext-opencl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in text.lower() or f == "__init__.py" and "oracle's parameter" in text, os.path.join(dirpath, f)
    ldd = os.popen(f"ldd {afe.LIB_PATH}").read()
    assert "oracle" not in ldd and "libref" not in ldd and "torch" not in ldd
