"""CPU check of the msb intrinsic used by the fast step body (csrc/b2048_device.cuh), compiled with g++ from
tests/host_check/step_bits_check.cpp, against a bit scan."""
import ctypes as C
import os
import subprocess

import pytest

from helpers import ROOT


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "host_check", "step_bits_check.cpp")
    so = str(tmp_path_factory.mktemp("step_bits") / "libstepbits.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src])
    h = C.CDLL(so)
    h.hc_msb_mismatches.restype = C.c_int64
    h.hc_msb_mismatches.argtypes = [C.c_int64, C.c_uint64]
    return h


def test_msb_matches_bit_scan(lib):
    assert lib.hc_msb_mismatches(1 << 20, 0xB17) == 0
