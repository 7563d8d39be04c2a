"""The device-side NumPy streams (csrc/b2048_np_rng.cuh) against the installed NumPy, on the CPU: the header is
compiled with g++ (tests/host_check/np_rng_check.cpp).  np.random.default_rng(seed) is PCG64 seeded through
SeedSequence; the reference draws its spawns with integers / random and its actions with choice(4, p)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_check", "np_rng_check.cpp")
MULT = 0x2360ed051fc65da44385df649fccf645
M128 = (1 << 128) - 1


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("np_rng") / "libnprng.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so, SRC])
    lib = C.CDLL(so)
    vp, i64 = C.c_void_p, C.c_int64
    lib.npc_seed.argtypes = [vp, vp, i64]
    lib.npc_run.argtypes = [vp, vp, vp, vp, vp, i64]
    lib.npc_spawn.argtypes = [vp, vp, i64]
    lib.npc_reset.argtypes = [vp, vp, i64]
    return lib


def P(a):
    return a.ctypes.data_as(C.c_void_p)


def words(bg_state):
    """numpy's PCG64 bit_generator.state -> the six words of b2048_np_rng"""
    s, inc = bg_state["state"]["state"], bg_state["state"]["inc"]
    return [s >> 64, s & (2**64 - 1), inc >> 64, inc & (2**64 - 1), bg_state["has_uint32"], bg_state["uinteger"]]


def set_words(gen, w):
    st = gen.bit_generator.state
    st["state"] = {"state": (int(w[0]) << 64) | int(w[1]), "inc": (int(w[2]) << 64) | int(w[3])}
    st["has_uint32"], st["uinteger"] = int(w[4]), int(w[5])
    gen.bit_generator.state = st


def fixed_seed_iter(base_seed):
    rng = np.random.default_rng(base_seed)
    while True:
        yield int(rng.integers(low=0, high=np.iinfo(np.int64).max, dtype=np.int64))


def test_state_is_48_bytes(lib):
    assert lib.npc_sizeof_rng() == 48


def test_seeding_matches_numpy(lib):
    it = fixed_seed_iter(3)
    edge = [0, 1, 3, 2**32 - 1, 2**32, 2**32 + 1, 2**63 - 1, 2**63, 2**64 - 1]
    seeds = edge + [next(it) for _ in range(1000)] + \
        [int(x) for x in np.random.default_rng(11).integers(0, 2**64 - 1, 5000, dtype=np.uint64, endpoint=True)] + \
        [int(x) for x in np.random.default_rng(12).integers(0, 2**32, 4000, dtype=np.uint64)]
    assert len(seeds) >= 10000
    arr = np.array(seeds, dtype=np.uint64)
    out = np.zeros((len(seeds), 6), dtype=np.uint64)
    lib.npc_seed(P(arr), P(out), len(seeds))
    for s, w in zip(seeds, out):
        assert [int(x) for x in w] == words(np.random.default_rng(s).bit_generator.state), s


def random_probs(rng, k):
    kind = k % 4
    if kind == 0:
        p = np.zeros(4, np.float32)
        p[rng.integers(4)] = 1.0                                  # a single non-zero entry
        return p
    x = rng.random(4).astype(np.float32)
    if kind == 1:
        x[rng.choice(4, size=rng.integers(1, 3), replace=False)] = 0.0   # zero entries
    if kind == 2:
        x = x ** 8                                                # very unequal
    return (x / x.sum(dtype=np.float32)).astype(np.float32)


def test_draws_match_numpy(lib):
    meta = np.random.default_rng(2024)
    for seed in [0, 1, 2**32, 2**64 - 1] + [int(x) for x in meta.integers(0, 2**63, 200)]:
        n_ops = 300
        ops = meta.integers(0, 4, n_ops).astype(np.int32)
        arg = meta.integers(1, 17, n_ops).astype(np.uint32)
        probs = np.stack([random_probs(meta, k) for k in range(n_ops)]).astype(np.float32)
        ref = np.random.default_rng(seed)
        want = []
        for op, a, p in zip(ops, arg, probs):
            if op == 0:
                want.append(float(ref.integers(int(a))))
            elif op == 1:
                want.append(ref.random())
            elif op == 2:
                want.append(float(ref.choice(4, p=p)))
            else:
                k = int(ref.integers(int(a)))
                four = 0 if ref.random() < 0.9 else 1
                want.append(float(k | (four << 4)))
        state = np.zeros(6, np.uint64)
        lib.npc_seed(P(np.array([seed], np.uint64)), P(state), 1)
        out = np.zeros(n_ops, np.float64)
        lib.npc_run(P(state), P(ops), P(arg), P(np.ascontiguousarray(probs)), P(out), n_ops)
        assert out.tolist() == want, seed
        assert [int(x) for x in state] == words(ref.bit_generator.state), seed


def test_lemire_rejection_branch(lib):
    """A state whose next 32-bit output is 0: integers(3) gets leftover 0 < (2^32 - 3) % 3 = 1 and must redraw."""
    inc = (0x5851f42d4c957f2d << 64 | 0x14057b7ef767814f) | 1
    hi = 0x9E3779B97F4A7C15                      # new state's high word; rotation = hi >> 58
    rot = hi >> 58
    x = 0xDEADBEEF << 32                         # the desired 64-bit output: low half 0, high half 0xDEADBEEF
    rotl = ((x << rot) | (x >> (64 - rot))) & (2**64 - 1) if rot else x
    lo = hi ^ rotl
    new_state = (hi << 64) | lo
    state = ((new_state - inc) * pow(MULT, -1, 1 << 128)) & M128    # one LCG step backwards
    w = [state >> 64, state & (2**64 - 1), inc >> 64, inc & (2**64 - 1), 0, 0]
    ref = np.random.default_rng(0)
    set_words(ref, w)
    assert ref.bit_generator.random_raw() == x     # the construction is right (then restore the state)
    set_words(ref, w)
    want = [float(ref.integers(3)), float(ref.integers(3)), ref.random()]
    st = np.array(w, dtype=np.uint64)
    ops = np.array([0, 0, 1], np.int32)
    arg = np.array([3, 3, 0], np.uint32)
    out = np.zeros(3, np.float64)
    lib.npc_run(P(st), P(ops), P(arg), P(np.zeros(12, np.float32)), P(out), 3)
    assert out.tolist() == want
    assert want[0] == float((0xDEADBEEF * 3) >> 32)   # the redraw took the buffered high half
    assert [int(v) for v in st] == words(ref.bit_generator.state)


def pack(board):
    b = 0
    for i, v in enumerate(np.asarray(board, np.int64).reshape(16)):
        if v:
            b |= (int(v).bit_length() - 1) << (4 * i)
    return b


def test_spawn_and_reset_match_game2048(lib):
    from oracle.pyport import PyGame
    meta = np.random.default_rng(7)
    for n_empty in range(1, 17):
        for rep in range(40):
            seed = int(meta.integers(0, 2**63))
            tiles = np.where(np.arange(16) < 16 - n_empty, 2 ** meta.integers(1, 12, 16), 0)
            board = meta.permutation(tiles).reshape(4, 4).astype(np.int64)
            g = PyGame()
            g.board = board.copy()
            g.rng = np.random.default_rng(seed)
            g.spawn()
            st = np.zeros(6, np.uint64)
            lib.npc_seed(P(np.array([seed], np.uint64)), P(st), 1)
            b = np.array([pack(board)], np.uint64)
            lib.npc_spawn(P(st), P(b), 1)
            assert int(b[0]) == pack(g.board), (n_empty, seed)
            assert [int(v) for v in st] == words(g.rng.bit_generator.state)
    it = fixed_seed_iter(3)
    seeds = [0, 1, 5, 2**64 - 1] + [next(it) for _ in range(500)]
    st = np.zeros((len(seeds), 6), np.uint64)
    lib.npc_seed(P(np.array(seeds, np.uint64)), P(st), len(seeds))
    b = np.zeros(len(seeds), np.uint64)
    lib.npc_reset(P(st), P(b), len(seeds))
    for i, s in enumerate(seeds):
        g = PyGame()
        g.reset(s)
        assert int(b[i]) == pack(g.board), s
        assert [int(v) for v in st[i]] == words(g.rng.bit_generator.state)


def test_seed_validation_without_gpu():
    import b2048
    from b2048.batched_env import np_seed_streams
    for bad in (-1, 2**64, 1.0, "3", None, True):
        with pytest.raises(ValueError):
            np_seed_streams([bad], "cpu")
    it = b2048.make_fixed_seed_iter(3)
    ref = fixed_seed_iter(3)
    assert [next(it) for _ in range(50)] == [next(ref) for _ in range(50)]
