"""CPU checks of bootstrapping at truncation (update_from_horizon / update_from_rollout(bootstrap_truncation=True)): the
pre-reset replay of csrc/b2048_horizon.cuh against the CPU oracle's step, the fold of gamma V(s') followed by the window
recurrence against the NumPy restatement with V(s') at the truncated boundaries, and the configurations that are refused."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from helpers import ROOT, P, random_boards
from test_horizon_targets import CASES, boundary_patterns, restate

F_DONE, F_TRUNC = 0x20, 0x40


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = os.path.join(ROOT, "tests", "host_check")
    so = str(tmp_path_factory.mktemp("bootstrap") / "libbootstrap.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                           os.path.join(d, "bootstrap_check.cpp"), os.path.join(d, "horizon_check.cpp")])
    h = C.CDLL(so)
    for name in ("hc_pre_reset_many", "hc_fold_bootstrap", "hc_segment_targets"):
        getattr(h, name).restype = None
    h.hc_pre_reset_many.argtypes = [C.c_void_p] * 6 + [C.c_int64]
    h.hc_fold_bootstrap.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_float, C.c_void_p]
    h.hc_segment_targets.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_double,
                                     C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return h


def trunc_only(flags):
    """The boundaries that are bootstrapped: TRUNC after step t without DONE ([T, B] from flags [T + 1, B])."""
    return (flags[1:] & (F_DONE | F_TRUNC)) == F_TRUNC


def restate_boot(reward, flags, value, boot, gamma, lam, huber, huber_delta, n_traj):
    """restate() with vn = boot[t] at the TRUNC-only boundaries.  restate uses vn = 0 at every boundary, and its target
    r + gamma 0 is r exactly, so a reward of r + gamma boot (float32, rounded separately) there gives target r + gamma boot."""
    g32 = np.float32(gamma)
    r = np.where(trunc_only(flags), reward + g32 * boot.astype(np.float32), reward).astype(np.float32)
    return restate(r, flags, value, gamma, lam, huber, huber_delta, n_traj)


def test_pre_reset_replay_equals_oracle_step(lib):
    """>= 10,000 boards (random, full, unmovable; every action) with random seeds, global ids and counters: the replayed
    board is the oracle's step with auto-reset off, bit for bit."""
    rng = np.random.default_rng(2048)
    groups, per = 80, 128
    boards = random_boards(rng, groups * per)
    boards[:per] = boards[:per] | np.uint64(0x1111111111111111)       # no empty cell: nothing moves unless tiles merge
    # full boards without a legal move: two exponents on a checkerboard (every move changes nothing, nothing spawns)
    ab = rng.integers(1, 16, (1024, 2))
    ab[:, 1] = np.where(ab[:, 0] == ab[:, 1], ab[:, 0] % 15 + 1, ab[:, 1])
    cells = np.where((np.arange(16) // 4 + np.arange(16) % 4) % 2 == 0, ab[:, :1], ab[:, 1:]).astype(np.uint64)
    boards[per: per + 1024] = (cells << (np.uint64(4) * np.arange(16, dtype=np.uint64))).sum(1, dtype=np.uint64)
    actions = rng.integers(0, 4, groups * per).astype(np.uint8)
    cfg = oracle.make_cfg(action_mode="buffer", auto_reset=False, max_steps=None)
    seeds = np.zeros(groups * per, np.uint64)
    gids = np.zeros(groups * per, np.uint64)
    counters = np.zeros(groups * per, np.uint32)
    want = np.zeros(groups * per, np.uint64)
    changed = np.zeros(groups * per, bool)
    for g in range(groups):
        sl = slice(g * per, (g + 1) * per)
        seed = int(rng.integers(0, 2**63)) * 2 + int(rng.integers(0, 2))
        gid0 = int(rng.integers(0, 2**40))
        t = int(rng.integers(1, 2**32))
        st = dict(board=boards[sl].copy(), score=np.zeros(per, np.uint32), step=np.zeros(per, np.uint32),
                  max_exp=np.full(per, 2, np.uint8), flags=np.zeros(per, np.uint8))
        o = oracle.step_many(st, cfg, seed, gid0, t, action=actions[sl])
        want[sl] = st["board"]
        changed[sl] = (o["flags"] & 0x10) != 0
        seeds[sl], gids[sl], counters[sl] = seed, gid0 + np.arange(per, dtype=np.uint64), t
    got = np.zeros_like(want)
    lib.hc_pre_reset_many(P(boards), P(actions), P(seeds), P(gids), P(counters), P(got), boards.size)
    assert np.array_equal(got, want)
    assert changed.sum() > 1000 and (~changed).sum() > 1000          # spawning moves and moves that change nothing
    assert np.array_equal(got[~changed], boards[~changed])


@pytest.mark.parametrize("critic,gamma,lam,huber", [c for c in CASES if c[0]])
def test_fold_then_segment_lane_equals_restatement(lib, critic, gamma, lam, huber):
    rng = np.random.default_rng(int(gamma * 100) * 11 + int(lam * 100) * 5 + huber)
    T, B, n_traj = 37, 600, 4800.0
    reward = (rng.standard_normal((T, B)) * 3).astype(np.float32)
    flags = boundary_patterns(rng, T, B)
    value = (rng.standard_normal((T + 1, B)) * 5).astype(np.float32)
    boot = (rng.standard_normal((T, B)) * 7).astype(np.float32)       # V(s') of every slot; read at TRUNC-only ones
    slots = np.flatnonzero(trunc_only(flags)).astype(np.int64)
    assert slots.size > 100
    vnext = boot.reshape(-1)[slots].copy()
    folded = np.zeros_like(reward)
    lib.hc_fold_bootstrap(P(reward), P(slots), P(vnext), slots.size, reward.size, gamma, P(folded))
    v = np.zeros((T, B), np.float32); td = np.zeros((T, B), np.float32); gc = np.zeros((T, B), np.float32)
    valid = np.zeros(B, np.int32)
    lib.hc_segment_targets(P(folded), P(flags), P(value), T, B, gamma, lam, huber, 1.5, n_traj, P(v), P(td), P(gc), P(valid))
    rv, rtd, rgc, _ = restate_boot(reward, flags, value, boot, gamma, lam, huber, 1.5, n_traj)
    for a, b in ((v, rv), (td, rtd), (gc, rgc)):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # the definition, slot by slot: delta = (r + gamma V(s')) - V(s) at TRUNC-only boundaries, r - V(s) at the others
    f32 = np.float32
    tr = trunc_only(flags)
    end = (flags[1:] & (F_DONE | F_TRUNC)) != 0
    want_tr = (reward + f32(gamma) * boot) + (-value[:T])
    assert np.array_equal(td[tr].view(np.uint32), want_tr[tr].astype(f32).view(np.uint32))
    assert np.array_equal(td[end & ~tr].view(np.uint32), (reward + (-value[:T]))[end & ~tr].view(np.uint32))
    if gamma > 0:
        plain = restate(reward, flags, value, gamma, lam, huber, 1.5, n_traj)[1]
        assert not np.array_equal(td[tr], plain[tr])


def _bare_agent(b2048, critic=False, **cfg):
    agent = object.__new__(b2048.ReinforceAgent)
    agent.agent_config = b2048.ReinforceAgentConfig(use_critic=critic, **cfg)
    agent._critic = object() if critic else None
    return agent


def _window(b2048, **kw):
    import torch
    T, B = 4, 8
    return b2048.Rollout(torch.zeros((T + 1, B), dtype=torch.int64), torch.zeros((T + 1, B), dtype=torch.uint8),
                         torch.zeros((T, B), dtype=torch.uint8), torch.zeros((T, B)), torch.full((B,), T, dtype=torch.int32),
                         T, **kw)


@pytest.mark.parametrize("critic,kw", [
    (False, dict(seed=1, gid0=0, t0=0)),      # no value function
    (True, dict(gid0=0, t0=0)),               # no env seed
    (True, dict(seed=1, gid0=0)),             # no counter
])
def test_window_bootstrap_refusals(critic, kw):
    import b2048
    with pytest.raises(ValueError, match="bootstrap_truncation"):
        _bare_agent(b2048, critic).update_from_horizon(_window(b2048, auto_reset=True, **kw), bootstrap_truncation=True)


def test_episode_bootstrap_needs_a_critic():
    import b2048
    with pytest.raises(ValueError, match="bootstrap_truncation"):
        _bare_agent(b2048).update_from_rollout(_window(b2048), bootstrap_truncation=True)


def test_rollout_positional_fields_unchanged():
    """seed / gid0 / t0 are appended with default None: positional construction keeps its meaning."""
    import b2048
    ro = _window(b2048)
    assert (ro.ep_weight, ro.n_traj, ro.auto_reset, ro.seed, ro.gid0, ro.t0) == (None, None, False, None, None, None)
