"""CPU tests: the C-ABI library loads and exports every symbol include/mdf_b200.h declares, and the
product fails loudly (never falls back) when no GPU is present."""
import ctypes
import os
import re

import numpy as np
import pytest

from metagenomic_deepfri_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "mdf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set(re.findall(r"\b(mdf_[a-z0-9_]+)\s*\(", src))
    names.discard("mdf_packed_row_words")          # static inline helper
    return sorted(names)


def test_library_exports_every_declared_symbol():
    L = ctypes.CDLL(_lib.LIB_PATH)
    declared = header_functions()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/mdf_b200.h but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared


def test_no_torch_types_in_abi():
    src = open(os.path.join(ROOT, "include", "mdf_b200.h")).read()
    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)          # comments stripped
    assert "torch" not in code and "at::" not in code and "cudaStream_t" not in code and "#include <cuda" not in code


def test_version_and_row_words():
    assert _lib.lib().mdf_version() >= 100
    assert [_lib.packed_row_words(L) for L in (0, 1, 128, 129, 300)] == [0, 4, 4, 8, 12]


def cuda_device_count():
    """Devices the CUDA driver reports (0 without a driver), as the library's context creation counts them: a GPU's device
    node need not be /dev/nvidia0."""
    try:
        cu = ctypes.CDLL("libcuda.so.1")
    except OSError:
        return 0
    n = ctypes.c_int(0)
    if cu.cuInit(0) != 0 or cu.cuDeviceGetCount(ctypes.byref(n)) != 0:
        return 0
    return n.value


@pytest.mark.skipif(cuda_device_count() > 0, reason="GPU present")
def test_no_cpu_fallback_without_gpu(model_dir):
    from metagenomic_deepfri_b200 import contact_map_utils, predict
    with pytest.raises(RuntimeError, match="no CUDA device|CUDA"):
        contact_map_utils.pairwise_sqeuclidean(np.zeros((3, 3), np.float32))
    with pytest.raises(RuntimeError):
        predict.Predictor(model_dir["small"])


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "metagenomic-deepfri_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "cmap_oracle" not in text and "gcn_oracle" not in text and "oracle/" not in text, f
