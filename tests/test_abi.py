"""The C-ABI library loads without a GPU and exports exactly the symbols include/b2048.h declares
(no compute calls here)."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b2048.h")
PKG = os.path.join(ROOT, "rl-2048-with-reinforce-and-actor-critic_b200")
LIB = os.path.join(PKG, "libb2048.so")


def header_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b2048_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib_path():
    if not os.path.exists(LIB):
        import __graft_entry__ as g
        g.build()
    return LIB


def test_header_declares_the_expected_surface():
    syms = header_symbols()
    for s in ("b2048_create", "b2048_destroy", "b2048_reset_many", "b2048_step_many", "b2048_move_many",
              "b2048_encode_obs", "b2048_policy_step", "b2048_rollout_many", "b2048_mlp_forward", "b2048_dense_forward", "b2048_reverse_scan",
              "b2048_advantages", "b2048_weighted_stats", "b2048_td_errors", "b2048_mlp_backward", "b2048_apply_update", "b2048_last_error"):
        assert s in syms



def test_inline_ptx_only_in_the_wrapper_header():
    # Each PTX operation, with its operand constraints and clobbers, is written once in b2048_ptx.cuh.  The exception is
    # b2048_device.cuh: its prmt / mul.hi / lop3 intrinsics sit in a header that also compiles with g++ (host_check),
    # and their C forms (__byte_perm, __umulhi, an and-or select) compile the step kernels to different SASS.
    csrc = os.path.join(PKG, "csrc")
    stmt = re.compile(r"asm\s*(volatile)?\s*\(")
    with_asm = sorted(f for f in os.listdir(csrc) if stmt.search(open(os.path.join(csrc, f)).read()))
    assert [f for f in with_asm if f not in ("b2048_ptx.cuh", "b2048_device.cuh")] == []


def test_no_static_pointer_caches():
    # Buffers belong to a handle (b2048_handle in b2048_internal.h), which lives on one device and frees them in
    # b2048_destroy.  A function-level or file-level `static T* p` would be shared by every handle of the process.
    csrc = os.path.join(PKG, "csrc")
    decl = re.compile(r"^\s*static\s+(?:const\s+)?[\w:<>]+(?:\s+[\w:<>]+)*\s*\*+\s*\w+\s*(?:=[^=;]*)?;", re.M)
    found = [(f, m.group(0).strip()) for f in sorted(os.listdir(csrc)) if f.endswith(".cu")
             for m in decl.finditer(open(os.path.join(csrc, f)).read())]
    assert found == []

def test_library_exports_every_declared_symbol(lib_path):
    lib = C.CDLL(lib_path)           # loads without a GPU (CUDA runtime is linked statically)
    for s in header_symbols():
        assert hasattr(lib, s), f"{s} declared in include/b2048.h but not exported by libb2048.so"
    out = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r"\bT (b2048_[a-z0-9_]+)", out)))
    assert exported == header_symbols(), "exported b2048_* symbols and header declarations differ"
    lib.b2048_version.restype = C.c_int
    assert lib.b2048_version() >= 100


def test_python_binding_covers_the_header(lib_path):
    import b2048
    declared = set(header_symbols()) - {"b2048_last_error"}
    assert set(b2048._lib.SIGNATURES) == declared
    b2048._lib.load()
    assert C.sizeof(b2048._lib.EnvCfg) == 96 and C.sizeof(b2048._lib.MlpDesc) == 16 + 36 + 4 + 128


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import b2048
    monkeypatch.setattr(b2048._lib, "_lib", None)
    monkeypatch.setattr(b2048._lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(b2048.B2048Error):
        b2048._lib.load()


def test_host_side_validation_without_gpu():
    import b2048
    with pytest.raises(ValueError):
        b2048.make_env_cfg(b2048.Game2048EnvConfig(size=3))
    with pytest.raises(ValueError):
        b2048.make_env_cfg(b2048.Game2048EnvConfig(reward_mode="nope"))
    with pytest.raises(ValueError):
        b2048.make_env_cfg(b2048.Game2048EnvConfig(bonus_mode="nope"))
    cfg = b2048.make_env_cfg(b2048.Game2048EnvConfig(max_steps=None), "random_legal", True)
    assert cfg.max_steps == 0 and cfg.action_mode == 1 and cfg.auto_reset == 1
    with pytest.raises(b2048.B2048Error):
        b2048.Batched2048Env(4, device="cpu")
