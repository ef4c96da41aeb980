"""The C-ABI shared library: it loads, exports every symbol include/pinn_b200.h declares, and fails
loudly (no CPU fallback) when no CUDA device is present.  No compute calls here."""
import ctypes as C
import os
import re

import pytest

import neuralpde_jl_b200 as npde
from conftest import HAS_GPU

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    txt = open(os.path.join(ROOT, "include", "pinn_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(pinn_[a-z_0-9]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    lib = npde.load_library()
    declared = _header_functions()
    assert set(declared) == set(npde.EXPORTS), (declared, npde.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pinn_abi_version() == 2


def test_library_is_in_tree_and_sm100a():
    assert os.path.dirname(npde.LIB_PATH) == os.path.join(ROOT, "neuralpde.jl_b200", "lib")
    import shutil
    import subprocess
    # the toolkit's bin directory need not be on PATH; build.py falls back to the default install for nvcc likewise
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([cuobjdump, "-lelf", npde.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device error path")
def test_create_without_gpu_fails_loudly():
    from neuralpde_jl_b200 import configs
    cfg = configs.config1()
    with pytest.raises(npde.EngineError, match="no CUDA device|no CPU fallback"):
        npde.symbolic_discretize(cfg.pde_system, cfg.discretization())


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "neuralpde.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|oracle/", src, flags=re.M), os.path.join(dirpath, f)
