"""The C-ABI library loads and exports every symbol include/opfg_b200.h declares
(no compute calls: there is no GPU on the builder box)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from opfgym_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "opfg_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return set(re.findall(r"\b(opfg_[a-z0-9_]+)\s*\(", text))


def test_prototypes_cover_header():
    assert header_functions() == set(capi.PROTOTYPES)


def test_cuda_library_exports_every_symbol():
    if not os.path.exists(capi.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(capi.LIB_PATH)
    for name in header_functions():
        assert getattr(lib, name) is not None
    capi.declare(lib)
    assert lib.opfg_version() == 1
    # the launch counter of a freshly loaded library starts at 0: checked in a new process, because earlier
    # tests of this session may have launched kernels through the same (process-wide) library
    code = ("import ctypes, sys; lib = ctypes.CDLL(sys.argv[1]); lib.opfg_launch_count.restype = ctypes.c_int64; "
            "print(lib.opfg_launch_count())")
    res = subprocess.run([sys.executable, "-c", code, capi.LIB_PATH], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    assert int(res.stdout) == 0


def test_no_cpu_fallback_in_product():
    """Constructing the product engine without a CUDA device must fail loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from opfgym_b200.engine import Engine
    from tests import common
    case = common.make_case("1-MV-rural--0-sw", n_profile_steps=96)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Engine(case.program, 4)


def test_product_does_not_import_oracle_or_hostsim():
    pkg = os.path.join(ROOT, "opfgym_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+(oracle|tests)\b", src, flags=re.M), f
