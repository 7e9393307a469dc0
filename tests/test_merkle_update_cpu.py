"""CPU: the statuses of p252_merkle_update_batch that need no device (null context, arity other than 2 or 4), from
Python and from the C++ mirror program tests/cpp/merkle_update_test.cpp."""
import ctypes
import os
import subprocess

import numpy as np

from poseidon252_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "poseidon252_b200", "lib")
EXE = os.path.join(ROOT, "tests", "cpp", "merkle_update_test")


def build_and_run_cpp():
    from poseidon252_b200 import build
    build.build()
    src = os.path.join(ROOT, "tests", "cpp", "merkle_update_test.cpp")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                           "-L", LIBDIR, "-lposeidon252_b200", "-Wl,-rpath," + LIBDIR])
    return subprocess.run([EXE], capture_output=True, text=True, timeout=300)


def test_update_statuses_without_device():
    lib = _native.lib()
    leaves = np.arange(64, dtype=np.uint64).reshape(16, 4)
    nodes = np.zeros((5, 4), dtype=np.uint64)
    idx = np.array([3], dtype=np.uint64)
    vals = np.full((1, 4), 9, dtype=np.uint64)
    before = leaves.copy()
    rej = ctypes.c_size_t(7)
    for arity in (4, 2, 3, 0, 8):
        rc = lib.p252_merkle_update_batch(None, arity, leaves.ctypes.data, 16, nodes.ctypes.data, idx.ctypes.data,
                                          vals.ctypes.data, 1, ctypes.byref(rej), _native.MEM_HOST)
        assert rc == -1                                             # P252_ERR_INVALID_ARGUMENT
    assert np.array_equal(leaves, before) and not nodes.any()


def test_cpp_merkle_update_cpu():
    res = build_and_run_cpp()
    assert res.returncode == 0, (res.returncode, res.stdout, res.stderr)
    assert "merkle update ok" in res.stdout
