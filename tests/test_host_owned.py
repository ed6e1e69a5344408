"""The CUDA resource owners (hymet_b200/csrc/cuda_owned.h) against a fake runtime.

tests/host_emul/owned_emul.cpp compiles the header with g++ and defines the runtime calls it uses:
live handles per kind, the current device, and a switch that fails the n-th acquisition.  No GPU is
involved; the copy ban is a static_assert, so a header that allowed copies would not compile.
"""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


@pytest.fixture(scope="module")
def owned(tmp_path_factory):
    if not os.path.exists(os.path.join(CUDA_INCLUDE, "cuda_runtime.h")):
        pytest.skip("the CUDA toolkit headers are needed to compile cuda_owned.h")
    so = str(tmp_path_factory.mktemp("owned") / "libowned.so")
    # -Bsymbolic: the fake's runtime calls bind to its own definitions even when another test has put the
    # real runtime in the process's global scope
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-Werror", "-shared", "-fPIC", "-Wl,-Bsymbolic",
                    "-I" + CUDA_INCLUDE, "-o", so,
                    os.path.join(ROOT, "tests", "host_emul", "owned_emul.cpp")], check=True)
    return C.CDLL(so)


@pytest.mark.parametrize("check", ["moves", "grow", "devices", "borrowed_stream"])
def test_owner(owned, check):
    fn = getattr(owned, "check_" + check)
    fn.restype = C.c_int
    line = fn()
    assert line == 0, "expectation at owned_emul.cpp:%d does not hold" % line
