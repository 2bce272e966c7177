"""The C-ABI library loads on a GPU-less host and exports exactly what include/*.h declares.
No compute is launched here (there is no GPU in the dev container)."""
import ctypes
import os
import re

import pytest

from bevformer_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "bevformer_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.findall(r"BEVF_API\s+[\w\s\*]+?\b(bevf_\w+)\s*\(", text)


def test_header_declares_something():
    syms = declared_symbols()
    assert "bevf_msda_forward" in syms and "bevf_msda_backward" in syms and len(syms) >= 5


def test_library_builds_and_exports_every_declared_symbol():
    path = build.build()
    lib = ctypes.CDLL(path)
    for s in declared_symbols():
        assert hasattr(lib, s), f"{s} declared in the header but not exported"


def test_binding_covers_header_exactly():
    assert sorted(_lib.SIGNATURES) == sorted(declared_symbols())


def test_version_and_error_channel():
    lib = _lib.load()
    assert lib.bevf_version() == _lib.ABI_VERSION
    assert lib.bevf_msda_forward(None, 0, None, None, None, None, None, 0, 1, 1, 1, 1, 1, 1, 1,
                                 None) != 0
    assert b"null pointer" in lib.bevf_last_error()
    with pytest.raises(RuntimeError, match="null pointer"):
        _lib.check(1, lib)
    # too many levels is rejected before any launch
    assert lib.bevf_msda_forward(16, 0, 16, 16, 16, 16, 16, 0, 1, 1, 1, 32, 1, 17, 1, None) != 0
    assert b"16 levels" in lib.bevf_last_error()


def test_ops_refuse_cpu_tensors():
    import torch
    from bevformer_b200 import ops
    v = torch.zeros(1, 4, 1, 32)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.msda_forward(v, torch.tensor([[2, 2]]), torch.tensor([0]), torch.zeros(1, 1, 1, 1, 1, 2),
                         torch.zeros(1, 1, 1, 1, 1))


def test_sass_has_vector_reductions():
    """The scatter is built on 16-byte fp32 reductions (REDG.E.ADD.F32x4), not scalar atomics."""
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(build.nvcc_path()), "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", build.build()], capture_output=True,
                          text=True).stdout
    assert "REDG.E.ADD.F32x4" in sass
