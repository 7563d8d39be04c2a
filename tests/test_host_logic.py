"""CPU-side check of the PRODUCT's bit tricks and step body: the kernels' host+device headers
(csrc/b2048_device.cuh, csrc/b2048_step.cuh) are compiled with g++ (tests/host_check) and compared
bit-exactly with the independent cell-by-cell CPU oracle.  No GPU needed."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import oracle
from helpers import ENV_CONFIGS, GOLDEN, P, ROOT, full_env_kwargs, host_check_lib, random_boards


def test_row_tables_match_reference_fixture():
    hc = host_check_lib()
    left = np.zeros(65536, np.uint16)
    merge = np.zeros(65536, np.uint8)
    hc.hc_get_lut(P(left), P(merge))
    g = np.load(os.path.join(GOLDEN, "row_lut.npz"))
    assert (left == g["left"]).all() and (merge == g["merge"]).all()


def test_moves_and_masks_random_boards():
    hc = host_check_lib()
    rng = np.random.default_rng(7)
    n = 200000
    boards = random_boards(rng, n)
    for a in range(4):
        act = np.full(n, a, np.uint8)
        o, ms, _, fl = oracle.move_many(boards, act)
        o2 = np.zeros(n, np.uint64); ms2 = np.zeros(n, np.int32); fl2 = np.zeros(n, np.uint8)
        hc.hc_move_many(P(boards), P(o2), P(act), P(ms2), P(fl2), C.c_int64(n))
        assert (o == o2).all() and (ms == ms2).all() and (fl == fl2).all()
    m, _ = oracle.mask_done(boards)
    m2 = np.zeros(n, np.uint8)
    hc.hc_mask(P(boards), P(m2), C.c_int64(n))
    assert (m == m2).all()


def test_moves_golden_fixture():
    hc = host_check_lib()
    g = np.load(os.path.join(GOLDEN, "moves.npz"))
    boards = g["boards"]
    n = len(boards)
    for a in range(4):
        act = np.full(n, a, np.uint8)
        o2 = np.zeros(n, np.uint64); ms2 = np.zeros(n, np.int32); fl2 = np.zeros(n, np.uint8)
        hc.hc_move_many(P(boards), P(o2), P(act), P(ms2), P(fl2), C.c_int64(n))
        assert (o2 == g["result"][:, a]).all() and (ms2 == g["merge_sum"][:, a]).all()
    m2 = np.zeros(n, np.uint8)
    hc.hc_mask(P(boards), P(m2), C.c_int64(n))
    assert (m2 == g["mask"]).all()


def test_reset_many():
    hc = host_check_lib()
    n = 50000
    for seed, gid0, t in ((0xB200, 0, 0), (2**63 + 5, 2**40, 77)):
        st = oracle.reset_many(n, seed, gid0, t)
        b = np.zeros(n, np.uint64); f = np.zeros(n, np.uint8)
        hc.hc_reset_many(P(b), P(f), C.c_int64(n), C.c_uint64(seed), C.c_uint64(gid0), C.c_uint32(t))
        assert (b == st["board"]).all() and (f == st["flags"]).all()


@pytest.mark.parametrize("name", list(ENV_CONFIGS))
@pytest.mark.parametrize("auto_reset", [False, True])
def test_step_body_vs_oracle(name, auto_reset):
    hc = host_check_lib()
    kw = full_env_kwargs(name)
    kw.pop("size")
    mask_on = kw["use_action_mask"]
    if kw["max_steps"] is None:
        kw["max_steps"] = 0
    n, T, seed, gid0 = 4096, 220, 31337, 10**9
    cfg = oracle.make_cfg(action_mode="random_legal" if mask_on else "random_any", auto_reset=auto_reset, **kw)
    st = oracle.reset_many(n, seed, gid0, 0)
    board = st["board"].copy(); score = st["score"].copy(); step = st["step"].copy(); mx = st["max_exp"].copy()
    flags_prev = st["flags"].copy()
    for t in range(1, T + 1):
        o = oracle.step_many(st, cfg, seed, gid0, t)
        act = np.zeros(n, np.uint8); ms = np.zeros(n, np.int32); rw = np.zeros(n, np.float32)
        rw64 = np.zeros(n, np.float64); fl = np.zeros(n, np.uint8)
        # alternate between supplying the previous mask and letting the step recompute it
        hc.hc_step_many(P(board), P(board), P(score), P(step), P(mx), None, P(act),
                        P(flags_prev) if t % 2 else None, C.byref(cfg), P(ms), P(rw), P(rw64), P(fl),
                        C.c_int64(n), C.c_uint64(seed), C.c_uint64(gid0), C.c_uint32(t))
        assert (act == o["action"]).all()
        assert (board == st["board"]).all()
        assert (ms == o["merge_sum"]).all()
        assert (rw64 == o["reward64"]).all() and (rw == o["reward"]).all()
        assert (fl == o["flags"]).all()
        assert (score == st["score"]).all() and (step == st["step"]).all() and (mx == st["max_exp"]).all()
        flags_prev = fl.copy()


def test_step_buffer_actions_including_illegal():
    hc = host_check_lib()
    rng = np.random.default_rng(3)
    n, T, seed = 2048, 120, 5
    kw = full_env_kwargs("shaped_raw"); kw.pop("size"); kw["max_steps"] = 50
    cfg = oracle.make_cfg(action_mode="buffer", **kw)
    st = oracle.reset_many(n, seed, 0, 0)
    board = st["board"].copy(); score = st["score"].copy(); step = st["step"].copy(); mx = st["max_exp"].copy()
    for t in range(1, T + 1):
        a = rng.integers(0, 4, n).astype(np.uint8)
        o = oracle.step_many(st, cfg, seed, 0, t, action=a)
        ms = np.zeros(n, np.int32); rw64 = np.zeros(n, np.float64); fl = np.zeros(n, np.uint8)
        hc.hc_step_many(P(board), P(board), P(score), P(step), P(mx), P(a), None, None, C.byref(cfg), P(ms), None,
                        P(rw64), P(fl), C.c_int64(n), C.c_uint64(seed), C.c_uint64(0), C.c_uint32(t))
        assert (board == st["board"]).all() and (rw64 == o["reward64"]).all() and (fl == o["flags"]).all()
        assert (score == st["score"]).all() and (step == st["step"]).all() and (mx == st["max_exp"]).all()


@pytest.mark.parametrize("reward_mode", ["log2", "sum"])
@pytest.mark.parametrize("mode", ["random_legal", "random_any", "buffer", "priority"])
@pytest.mark.parametrize("track", [True, False])
def test_fast_step_body_vs_oracle(reward_mode, mode, track):
    """The instruction-lean step body (csrc/b2048_step_fast.cuh) used by the large-batch kernel."""
    hc = host_check_lib()
    n, T, seed, gid0 = 6000, 260, 99, 2**33
    cfg = oracle.make_cfg(reward_mode=reward_mode, base_reward_scale=0.5, step_reward=-0.125, max_steps=100,
                          action_mode=mode, auto_reset=True, action_priority=(0, 1, 3, 2))
    st = oracle.reset_many(n, seed, gid0, 0)
    board = st["board"].copy(); score = st["score"].copy(); step = st["step"].copy(); mx = st["max_exp"].copy()
    flags_prev = st["flags"].copy()
    rng = np.random.default_rng(1)
    for t in range(1, T + 1):
        a = rng.integers(0, 4, n).astype(np.uint8) if mode == "buffer" else None
        o = oracle.step_many(st, cfg, seed, gid0, t, action=a, use_state=track)
        act = np.zeros(n, np.uint8); ms = np.zeros(n, np.int32); rw = np.zeros(n, np.float32); fl = np.zeros(n, np.uint8)
        hc.hc_step_fast_many(P(board), P(board), P(score) if track else None, P(step) if track else None,
                             P(mx) if track else None, P(a), P(act), P(flags_prev) if t % 3 else None, C.byref(cfg),
                             P(ms), P(rw), P(fl), C.c_int64(n), C.c_uint64(seed), C.c_uint64(gid0), C.c_uint32(t))
        assert (act == o["action"]).all(), t
        assert (board == st["board"]).all(), t
        assert (ms == o["merge_sum"]).all() and (rw == o["reward"]).all() and (fl == o["flags"]).all()
        if track:
            assert (score == st["score"]).all() and (step == st["step"]).all() and (mx == st["max_exp"]).all()
        flags_prev = fl.copy()


@pytest.mark.parametrize("name,track", [("shaped_raw", True), ("onehot_log2bonus", True), ("shaped_nobonus", False),
                                        ("shaped_nobonus", True)])
def test_fast_step_body_shaped_rewards_vs_oracle(name, track):
    """Reward shaping in the fast body (empty-tile / merge rewards, new-max-tile bonus, end-game penalty; env.py:226-259):
    bit-equal float32 rewards, boards, flags and counters against the oracle on the reference-test env configurations."""
    hc = host_check_lib()
    n, T, seed, gid0 = 5000, 200, 123, 7 * 2**32
    if name == "shaped_nobonus":
        kw = dict(reward_mode="log2", base_reward_scale=0.5, empty_tile_reward=0.05, merge_reward=0.3, step_reward=-0.01,
                  endgame_penalty=-7.5, max_steps=80)
    else:
        kw = {k: v for k, v in full_env_kwargs(name).items() if k not in ("size", "obs_mode", "obs_log2_scale")}
        kw["max_steps"] = kw["max_steps"] or 150
    cfg = oracle.make_cfg(action_mode="random_legal", auto_reset=True, **kw)
    st = oracle.reset_many(n, seed, gid0, 0)
    board = st["board"].copy(); score = st["score"].copy(); step = st["step"].copy(); mx = st["max_exp"].copy()
    flags_prev = st["flags"].copy()
    seen_bonus = False
    for t in range(1, T + 1):
        mx_before = st["max_exp"].copy()
        o = oracle.step_many(st, cfg, seed, gid0, t, use_state=track)
        act = np.zeros(n, np.uint8); ms = np.zeros(n, np.int32); rw = np.zeros(n, np.float32); fl = np.zeros(n, np.uint8)
        hc.hc_step_fast_many(P(board), P(board), P(score) if track else None, P(step) if track else None,
                             P(mx) if track else None, None, P(act), P(flags_prev), C.byref(cfg),
                             P(ms), P(rw), P(fl), C.c_int64(n), C.c_uint64(seed), C.c_uint64(gid0), C.c_uint32(t))
        assert (act == o["action"]).all() and (board == st["board"]).all(), t
        assert (ms == o["merge_sum"]).all() and (fl == o["flags"]).all(), t
        assert (rw == o["reward"]).all(), (t, np.flatnonzero(rw != o["reward"])[:5])
        if track:
            assert (score == st["score"]).all() and (step == st["step"]).all() and (mx == st["max_exp"]).all()
            seen_bonus |= bool((st["max_exp"] > mx_before).any())
        flags_prev = fl.copy()
    assert not track or seen_bonus


def test_fast_step_overflow_and_dense_boards():
    hc = host_check_lib()
    rng = np.random.default_rng(9)
    n = 100000
    boards = random_boards(rng, n)
    cfg = oracle.make_cfg(reward_mode="sum", action_mode="random_any", auto_reset=False, max_steps=0)
    st = dict(board=boards.copy(), score=np.zeros(n, np.uint32), step=np.zeros(n, np.uint32),
              max_exp=np.full(n, 2, np.uint8), flags=np.zeros(n, np.uint8))
    board = boards.copy(); score = st["score"].copy(); step = st["step"].copy(); mx = st["max_exp"].copy()
    for t in range(1, 4):
        o = oracle.step_many(st, cfg, 5, 0, t)
        act = np.zeros(n, np.uint8); ms = np.zeros(n, np.int32); rw = np.zeros(n, np.float32); fl = np.zeros(n, np.uint8)
        hc.hc_step_fast_many(P(board), P(board), P(score), P(step), P(mx), None, P(act), None, C.byref(cfg), P(ms), P(rw),
                             P(fl), C.c_int64(n), C.c_uint64(5), C.c_uint64(0), C.c_uint32(t))
        assert (board == st["board"]).all() and (fl == o["flags"]).all() and (ms == o["merge_sum"]).all()
        assert (rw == o["reward"]).all() and (mx == st["max_exp"]).all() and (score == st["score"]).all()
        if t == 1:
            assert (fl & 0x80).any()      # the random boards contain 15+15 merges


@pytest.mark.parametrize("prio", [(0, 1, 2, 3), (0, 1, 3, 2), (3, 2, 1, 0)])
def test_generic_step_body_priority_mode_vs_oracle(prio):
    """B2048_ACT_PRIORITY (tools/simple_action_gen.py:16-33) in the generic step body."""
    hc = host_check_lib()
    n, T, seed, gid0 = 3000, 150, 17, 123
    kw = full_env_kwargs("shaped_raw"); kw.pop("size"); kw["max_steps"] = 90
    cfg = oracle.make_cfg(action_mode="priority", action_priority=prio, auto_reset=True, **kw)
    st = oracle.reset_many(n, seed, gid0, 0)
    board = st["board"].copy(); score = st["score"].copy(); step = st["step"].copy(); mx = st["max_exp"].copy()
    flags_prev = st["flags"].copy()
    for t in range(1, T + 1):
        o = oracle.step_many(st, cfg, seed, gid0, t)
        act = np.zeros(n, np.uint8); ms = np.zeros(n, np.int32); rw = np.zeros(n, np.float32)
        rw64 = np.zeros(n, np.float64); fl = np.zeros(n, np.uint8)
        hc.hc_step_many(P(board), P(board), P(score), P(step), P(mx), None, P(act),
                        P(flags_prev) if t % 2 else None, C.byref(cfg), P(ms), P(rw), P(rw64), P(fl),
                        C.c_int64(n), C.c_uint64(seed), C.c_uint64(gid0), C.c_uint32(t))
        assert (act == o["action"]).all() and (board == st["board"]).all() and (rw64 == o["reward64"]).all()
        assert (fl == o["flags"]).all() and (score == st["score"]).all()
        flags_prev = fl.copy()


def test_episode_rank_weights_vs_reference_fixture():
    """dist.episode_rank_weights (torch sort; runs on the GPU in production) vs the reference's
    _compute_episode_rank_weights outputs (tests/golden/rank_weights.npz).  Tie-free inputs: identical per episode.
    Tied inputs: identical multiset, identical for every episode whose reward is unique."""
    import sys
    import torch
    from helpers import GOLDEN, ROOT
    sys.path.insert(0, ROOT)
    from b2048 import dist as bd
    g = np.load(os.path.join(GOLDEN, "rank_weights.npz"))
    for k in range(int(g["n_cases"])):
        r, conf, want = g[f"case{k}/reward"], g[f"case{k}/conf"].tolist(), g[f"case{k}/weights"]
        got = bd.episode_rank_weights(torch.from_numpy(r), conf).numpy()
        if not int(g[f"case{k}/ties"]):
            assert np.allclose(got, want, rtol=1e-6, atol=0), k
        else:
            assert np.allclose(np.sort(got), np.sort(want), rtol=1e-6), k
            vals, counts = np.unique(r, return_counts=True)
            uniq = np.isin(r, vals[counts == 1])
            assert np.allclose(got[uniq], want[uniq], rtol=1e-6), k


def test_bench_reads_roofline_traffic_from_the_committed_ncu_summary():
    """bench.py's roofline.traffic comes from profiles/*.csv (dram__bytes_read + dram__bytes_write per launch), not from a literal."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    t, src = bench.profile_traffic(["r02_ncu_step_fast_kernel.csv", "r01_ncu_step_fast_kernel.csv"], "step_fast")
    assert src is not None and src.startswith("profiles/") and 1.8e7 < t < 2.4e7          # ~19 MB per 1 M-board launch
    assert bench.profile_traffic(["does_not_exist.csv"]) == (None, None)
    # unit handling: the update pipeline's summary mixes Mbyte and Gbyte
    t2, _ = bench.profile_traffic(["r02_ncu_update_pipe_kernel_r288_276k.csv"], "update_pipe")      # 80 MB ring (superseded)
    assert t2 is not None and 1e9 < t2 < 4e9
    t3, _ = bench.profile_traffic(["r02_ncu_update_pipe_kernel.csv"], "update_pipe")                # 59 MB ring: ~0.34 GB per 1 M samples
    assert t3 is not None and 2e8 < t3 < 1e9


@pytest.mark.parametrize("track", [True, False])
def test_bench_dump_outputs_format_and_size_cap(tmp_path, monkeypatch, track):
    """bench.py --dump-outputs: float32 / float64 .npy files that hold the step's outputs exactly (the packed board as
    two 32-bit words); above the size cap, the same fixed seeded sample of boards every time, with its indices."""
    import importlib.util
    import types
    import torch
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(3)
    n = 1000
    board = rng.integers(0, 2**64, n, dtype=np.uint64)
    env = types.SimpleNamespace(
        board=torch.from_numpy(board.view(np.int64)), reward=torch.from_numpy(rng.random(n, np.float32)),
        flags=torch.from_numpy(rng.integers(0, 256, n, dtype=np.uint8)), track_state=track,
        score=torch.from_numpy(rng.integers(0, 2**31, n, dtype=np.int32)) if track else None,
        step_count=torch.from_numpy(rng.integers(0, 1025, n, dtype=np.int32)) if track else None,
        max_exp=torch.from_numpy(rng.integers(0, 16, n, dtype=np.uint8)) if track else None)
    names = ["board", "reward", "flags"] + (["score", "step", "max_exp"] if track else [])

    def load(d):
        got = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        return got

    def check(got, idx):
        w = got["board"].astype(np.uint64)
        assert ((w[:, 1] << np.uint64(32)) | w[:, 0] == board[idx]).all()
        assert (got["reward"] == env.reward.numpy()[idx]).all() and (got["flags"] == env.flags.numpy()[idx]).all()
        if track:
            assert (got["score"] == env.score.numpy()[idx]).all() and (got["step"] == env.step_count.numpy()[idx]).all()
            assert (got["max_exp"] == env.max_exp.numpy()[idx]).all()

    bench.dump_outputs(env, str(tmp_path / "full"))
    got = load(tmp_path / "full")
    assert sorted(got) == sorted(names)
    check(got, np.arange(n))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 20000)
    for d in ("a", "b"):
        bench.dump_outputs(env, str(tmp_path / d))
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(a) == sorted(names + ["index"])
    assert sum(x.nbytes for x in a.values()) <= 20000
    idx = a["index"].astype(np.int64)
    assert 0 < len(idx) < n and (np.diff(idx) > 0).all()
    assert all((a[k] == b[k]).all() for k in a)
    check(a, idx)


def test_debug_options_match_the_header():
    """_lib.DEBUG_OPTIONS mirrors the B2048_DBG_* enum of include/b2048.h."""
    import re
    sys.path.insert(0, ROOT)
    import b2048
    from b2048 import _lib
    hdr = open(os.path.join(ROOT, "include", "b2048.h")).read()
    enum = dict((m.group(1).lower(), int(m.group(2))) for m in re.finditer(r"B2048_DBG_(?:PARAM_)?([A-Z_]+) = (\d+)", hdr))
    for name, val in _lib.DEBUG_OPTIONS.items():
        assert enum[name] == val, (name, val, enum)
    assert enum["count"] == 1 + max(v for k, v in _lib.DEBUG_OPTIONS.items() if k != "pipe_split")


def test_trainer_tile_histogram_is_the_references_list():
    """max_tile_counts is a list over [16, 32, ..., 4096] like runner.py:557, :617-624 (tiles outside the bins are not counted)."""
    import torch
    sys.path.insert(0, ROOT)
    from b2048 import trainer
    exps = torch.tensor([4, 4, 5, 11, 12, 3, 13], dtype=torch.uint8)      # 16, 16, 32, 2048, 4096, 8, 8192
    assert trainer.tile_histogram(exps) == [2, 1, 0, 0, 0, 0, 0, 1, 1]
    assert trainer.TILE_BINS == [16, 32, 64, 128, 256, 512, 1024, 2048, 4096]
