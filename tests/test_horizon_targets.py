"""CPU checks of the fixed-horizon window update (ReinforceAgent.update_from_horizon): the per-lane recurrence of
csrc/b2048_horizon.cuh, compiled with g++ from tests/host_check/horizon_check.cpp, bit for bit against a NumPy float64
restatement with the same operation order; and the configurations the window update rejects."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, P

F_DONE, F_TRUNC = 0x20, 0x40


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "host_check", "horizon_check.cpp")
    so = str(tmp_path_factory.mktemp("horizon") / "libhorizon.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so, src])
    h = C.CDLL(so)
    h.hc_segment_targets.restype = None
    h.hc_segment_targets.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_double,
                                     C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return h


def restate(reward, flags, value, gamma, lam, huber, huber_delta, n_traj):
    """The window's definitions in NumPy: float32 TD arithmetic, float64 recurrence, reverse in t."""
    T, B = reward.shape
    f32 = np.float32
    c = np.float64(gamma) * np.float64(lam) if value is not None else np.float64(gamma)
    inv = f32(1.0) / (f32(T) * f32(n_traj))
    g32, hd = f32(gamma), f32(huber_delta)
    v = np.zeros((T, B), f32); td = np.zeros((T, B), f32); gc = np.zeros((T, B), f32)
    valid = np.full(B, T if value is not None else 0, np.int32)
    G = np.zeros(B, np.float64)
    for t in range(T - 1, -1, -1):
        e = (flags[t + 1] & (F_DONE | F_TRUNC)) != 0
        valid = np.where(e & (valid == 0), t + 1, valid).astype(np.int32)
        x = reward[t].copy()
        if value is not None:
            vc = value[t]
            vn = np.where(e, f32(0.0), value[t + 1]).astype(f32)
            target = x + g32 * vn
            diff = vc + (-target)
            g = diff.copy()
            if huber:
                clip = (diff > hd) | (diff < -hd)
                g = np.where(clip, np.where(diff > f32(0), hd, -hd), diff).astype(f32)
            x = target + (-vc)
            td[t] = x
            gc[t] = g * inv
        G = np.where(e, x.astype(np.float64), x.astype(np.float64) + c * G)
        v[t] = np.where((value is not None) | (t < valid), G.astype(f32), f32(0.0))
    return v, td, gc, valid


def boundary_patterns(rng, T, B):
    """none, every step, only at t = T-1, random DONE, random TRUNC, DONE mixed with TRUNC (+ legal-mask noise)."""
    f = rng.integers(0, 16, (T + 1, B)).astype(np.uint8) | (rng.integers(0, 2, (T + 1, B)).astype(np.uint8) * 0x10)
    k = B // 6
    f[:, k: 2 * k] |= F_DONE
    f[T, 2 * k: 3 * k] |= F_TRUNC
    f[:, 3 * k: 4 * k] |= np.where(rng.random((T + 1, k)) < 0.2, F_DONE, 0).astype(np.uint8)
    f[:, 4 * k: 5 * k] |= np.where(rng.random((T + 1, k)) < 0.2, F_TRUNC, 0).astype(np.uint8)
    r = rng.random((T + 1, B - 5 * k))
    f[:, 5 * k:] |= np.where(r < 0.1, F_DONE, np.where(r < 0.2, F_TRUNC, np.where(r < 0.25, F_DONE | F_TRUNC, 0))).astype(np.uint8)
    return f


# lambda and the critic loss enter only with a critic
CASES = [(False, g, 0.0, 0) for g in (0.0, 0.99, 1.0)] + \
        [(True, g, l, hb) for g in (0.0, 0.99, 1.0) for l in (0.0, 0.95, 1.0) for hb in (0, 1)]


@pytest.mark.parametrize("critic,gamma,lam,huber", CASES)
def test_segment_targets_bit_equal_to_numpy(lib, critic, gamma, lam, huber):
    rng = np.random.default_rng(int(gamma * 100) * 7 + int(lam * 100) * 3 + huber + 2 * critic)
    T, B, n_traj = 37, 600, 4800.0
    reward = (rng.standard_normal((T, B)) * 3).astype(np.float32)
    reward[rng.random((T, B)) < 0.1] = 0.0
    flags = boundary_patterns(rng, T, B)
    value = (rng.standard_normal((T + 1, B)) * 5).astype(np.float32) if critic else None
    v = np.zeros((T, B), np.float32); td = np.zeros((T, B), np.float32); gc = np.zeros((T, B), np.float32)
    valid = np.zeros(B, np.int32)
    lib.hc_segment_targets(P(reward), P(flags), P(value), T, B, gamma, lam, huber, 1.5, n_traj, P(v),
                           P(td) if critic else None, P(gc) if critic else None, P(valid))
    rv, rtd, rgc, rvalid = restate(reward, flags, value, gamma, lam, huber, 1.5, n_traj)
    assert np.array_equal(valid, rvalid)
    assert np.array_equal(v.view(np.uint32), rv.view(np.uint32))
    if critic:
        assert np.array_equal(td.view(np.uint32), rtd.view(np.uint32))
        assert np.array_equal(gc.view(np.uint32), rgc.view(np.uint32))
        assert (valid == T).all()
    else:
        k = B // 6
        assert (valid[:k] == 0).all() and (valid[k: 2 * k] == T).all() and (valid[2 * k: 3 * k] == T).all()
    if huber and critic:
        assert (np.abs(rgc) * (np.float32(T) * np.float32(n_traj)) <= 1.5 * (1 + 1e-6)).all()


def test_segment_targets_definitions(lib):
    """A hand-made lane: the returns restart after a boundary, the tail after the last boundary is not a sample."""
    T = 5
    reward = np.array([[1], [2], [4], [8], [16]], np.float32)
    flags = np.zeros((T + 1, 1), np.uint8)
    flags[2, 0] = F_DONE          # the episode ends with step 1
    flags[4, 0] = F_TRUNC         # the next one is truncated after step 3
    v = np.zeros((T, 1), np.float32); valid = np.zeros(1, np.int32)
    lib.hc_segment_targets(P(reward), P(flags), None, T, 1, 0.5, 0.0, 0, 1.0, 1.0, P(v), None, None, P(valid))
    assert valid[0] == 4
    assert v[:, 0].tolist() == [1 + 0.5 * 2, 2, 4 + 0.5 * 8, 8, 0]


def _bare_agent(b2048, **cfg):
    agent = object.__new__(b2048.ReinforceAgent)
    agent.agent_config = b2048.ReinforceAgentConfig(**cfg)
    return agent


def _window(b2048, auto_reset=True):
    import torch
    T, B = 4, 8
    return b2048.Rollout(torch.zeros((T + 1, B), dtype=torch.int64), torch.zeros((T + 1, B), dtype=torch.uint8),
                         torch.zeros((T, B), dtype=torch.uint8), torch.zeros((T, B)), torch.full((B,), T, dtype=torch.int32),
                         T, auto_reset=auto_reset)


@pytest.mark.parametrize("cfg,kw,auto_reset", [
    (dict(baseline_mode="each"), {}, True),
    (dict(reward_rank_weights=[0.5, 1.0, 1.5]), {}, True),
    (dict(baseline_mode="batch"), dict(exchange="one_message"), True),
    (dict(), {}, False),
])
def test_update_from_horizon_rejects(cfg, kw, auto_reset):
    import b2048
    with pytest.raises(ValueError):
        _bare_agent(b2048, **cfg).update_from_horizon(_window(b2048, auto_reset), **kw)


def test_trainer_rejects_horizon_with_numpy_streams():
    from b2048 import trainer
    cfg = trainer.merge_config({"train": {"horizon": 16, "seed_streams": "numpy", "out_dir": None}})
    with pytest.raises(ValueError, match="horizon"):
        trainer.training(cfg)
