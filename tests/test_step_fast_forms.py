"""CPU checks of the closed forms in the fast step body (csrc/b2048_step_fast.cuh), compiled with g++ from
tests/host_check/fast_forms_check.cpp: the table-driven auto-reset against reset_board + legal_mask, and the
shift-free canonicalisation against canon_fwd / canon_inv."""
import ctypes as C
import os
import subprocess

import pytest

from helpers import ROOT


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "host_check", "fast_forms_check.cpp")
    so = str(tmp_path_factory.mktemp("fast_forms") / "libfastforms.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src])
    h = C.CDLL(so)
    h.hc_start_board_mismatches.restype = C.c_int64
    h.hc_start_board_mismatches.argtypes = [C.c_int64, C.c_uint64, C.c_uint64, C.c_uint32]
    h.hc_canon_m_mismatches.restype = C.c_int64
    h.hc_canon_m_mismatches.argtypes = [C.c_int64, C.c_uint64]
    return h


@pytest.mark.parametrize("seed,gid0,t", [(0xB200, 0, 0), (0x1234_5678_9ABC_DEF0, 1 << 33, 77)])
def test_start_board_matches_reset_board(lib, seed, gid0, t):
    assert lib.hc_start_board_mismatches(1 << 20, seed, gid0, t) == 0


def test_shift_free_canonicalisation_matches(lib):
    assert lib.hc_canon_m_mismatches(1 << 20, 0x5EED) == 0
