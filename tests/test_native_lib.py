"""The C-ABI library: builds for sm_100a, loads, exports every symbol the header declares, and
fails loudly (never computes) when no GPU is present.  CPU only."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "bore_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bore_[a-z0-9_]+)\s*\(", src)))


def test_header_and_library_agree(native_lib):
    from bore_b200 import _lib
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(native_lib, name), f"{name} declared in include/bore_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == declared, "ctypes table and header drifted apart"
    assert native_lib.bore_abi_version() == 1


def test_library_is_sm100a_and_torch_free():
    import subprocess
    from bore_b200 import build
    path = build.build_library()
    out = subprocess.run(["cuobjdump", "--list-elf", path], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    ldd = subprocess.run(["ldd", path], capture_output=True, text=True).stdout
    ldd = re.sub(r"\(0x[0-9a-f]+\)", "", ldd)  # load addresses are random and may contain "c10"
    assert "torch" not in ldd and "c10" not in ldd  # plain C ABI: no torch types or libs


def test_no_cpu_fallback(native_lib):
    """Without a CUDA device every compute entry point must refuse, with a message."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from bore_b200 import _lib
    from bore_b200.engine import NativeMLP
    assert native_lib.bore_device_count() == 0
    with pytest.raises(_lib.BoreNativeError, match="no CPU fallback"):
        NativeMLP([2, 16, 1], ["relu", "sigmoid"])
    h = C.c_void_p()
    dims = (C.c_int * 3)(2, 16, 1); acts = (C.c_int * 2)(1, 3)
    assert native_lib.bore_mlp_create(2, dims, acts, 1, 0, C.byref(h)) != 0
    assert b"no CPU fallback" in native_lib.bore_last_error()
    out = C.c_double()
    assert native_lib.bore_bench_ffma_peak(0, 1, C.byref(out)) != 0
    from bore_b200.models import MaximizableSequential
    from bore_b200.layers import Dense
    m = MaximizableSequential(); m.add(Dense(1, activation="sigmoid", input_dim=2))
    with pytest.raises(_lib.BoreNativeError):
        m.predict([[0.0, 0.0]])


def test_argument_validation(native_lib):
    h = C.c_void_p()
    dims = (C.c_int * 3)(2, 16, 3); acts = (C.c_int * 2)(1, 0)
    assert native_lib.bore_mlp_create(2, dims, acts, 1, 0, C.byref(h)) != 0
    assert b"output dimension must be 1" in native_lib.bore_last_error()
    assert native_lib.bore_lbfgsb_workspace_bytes(1024, 6, 10) > 1024 * (4 * 6 + 6 * 21 + 300) * 8
    assert native_lib.bore_topk_workspace_bytes(1000, 5) == 1024 * 8
