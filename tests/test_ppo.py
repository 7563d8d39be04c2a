"""CPU checks of PPO on fixed-horizon windows (ReinforceAgent.update_ppo): the keyed minibatch permutation and the
per-sample coefficients of csrc/b2048_ppo.cuh, compiled with g++ from tests/host_check/ppo_check.cpp, against NumPy
restatements; and the configurations update_ppo, sharded_update and the trainer refuse."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from helpers import ROOT, P

DOM_PPO = 2
M32 = np.uint64(0xFFFFFFFF)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("ppo") / "libppo.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "host_check", "ppo_check.cpp")])
    h = C.CDLL(so)
    for name in ("hc_ppo_positions", "hc_ppo_minibatches", "hc_ppo_samples"):
        getattr(h, name).restype = None
    h.hc_ppo_positions.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
    h.hc_ppo_minibatches.argtypes = [C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
    h.hc_ppo_samples.argtypes = [C.c_void_p] * 8 + [C.c_int64, C.c_double, C.c_double, C.c_double, C.c_int32, C.c_double,
                                                    C.c_void_p]
    return h


def positions(lib, N, seed, epoch):
    out = np.zeros(N, np.uint64)
    lib.hc_ppo_positions(N, seed, epoch, P(out))
    return out


def minibatches(lib, T, B, n_traj, gid0, M, seed, epoch):
    out = np.zeros((T, B), np.int32)
    lib.hc_ppo_minibatches(T, B, n_traj, gid0, M, seed, epoch, P(out))
    return out


# ---------------------------------------------------------------- NumPy restatement of the permutation
def np_philox_w0(c0, c1, c2, c3, seed):
    """Word 0 of Philox4x32-10 on uint64 arrays holding 32-bit lanes (the counter words may be arrays or scalars)."""
    c = [np.asarray(x, np.uint64) & M32 for x in (c0, c1, c2, c3)]
    c = [np.broadcast_to(x, np.broadcast(*c).shape).copy() for x in c]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return c[0]


def np_positions(g, N, seed, epoch):
    """P_e(g): the 4-round balanced Feistel network on 2h bits with cycle-walking (csrc/b2048_ppo.cuh)."""
    bits = int(np.ceil(np.log2(N))) if N > 1 else 0
    while (1 << bits) < N:
        bits += 1
    h = max(1, (bits + 1) // 2)
    mask = np.uint64((1 << h) - 1)
    x = np.asarray(g, np.uint64).copy()
    todo = np.ones(x.shape, bool)
    while todo.any():
        L, R = x[todo] >> np.uint64(h), x[todo] & mask
        for r in range(4):
            F = np_philox_w0(R, r, epoch, DOM_PPO, seed) & mask
            L, R = R, L ^ F
        x[todo] = (L << np.uint64(h)) | R
        todo = x >= np.uint64(N)
    return x


def test_numpy_philox_matches_oracle():
    rng = np.random.default_rng(1)
    for _ in range(20):
        ctr = [int(v) for v in rng.integers(0, 2**32, 4)]
        seed = int(rng.integers(0, 2**63)) * 2 + 1
        assert int(np_philox_w0(*ctr, seed)) == oracle.philox(ctr, [seed & 0xFFFFFFFF, seed >> 32])[0]


BIJECTION_N = [1, 2, 3, 5, 4095, 4096, 4097, 65536 * 64, 2**22 + 1]


@pytest.mark.parametrize("N", BIJECTION_N)
def test_position_is_a_bijection(lib, N):
    cases = [(0, 0), (0xDEADBEEF12345678, 1), (7, 3)] if N < 2**20 else [(0, 0), (0xDEADBEEF12345678, 3)]
    perms = []
    for seed, epoch in cases:
        p = positions(lib, N, seed, epoch)
        assert np.array_equal(np.sort(p), np.arange(N, dtype=np.uint64))
        perms.append(p)
    if N >= 4095:                                          # seeds and epochs give different permutations
        assert not np.array_equal(perms[0], perms[1]) and (perms[0] != np.arange(N)).mean() > 0.99


@pytest.mark.parametrize("N", [1, 2, 3, 5, 4095, 4096, 4097, 100_003])
def test_position_matches_numpy_restatement(lib, N):
    for seed, epoch in ((0, 0), (0x0123456789ABCDEF, 2), (2**64 - 1, 7)):
        g = np.arange(N, dtype=np.uint64)
        assert np.array_equal(positions(lib, N, seed, epoch), np_positions(g, N, seed, epoch))


@pytest.mark.parametrize("T,n_traj,M", [(1, 1, 1), (3, 5, 2), (48, 4096, 4), (64, 1000, 7), (5, 3, 15), (16, 4097, 4096)])
def test_partition_sizes_match_closed_form(lib, T, n_traj, M):
    N = T * n_traj
    for seed, epoch in ((3, 0), (11, 1)):
        mb = minibatches(lib, T, n_traj, n_traj, 0, M, seed, epoch)
        counts = np.bincount(mb.reshape(-1), minlength=M)
        closed = np.array([-(-(m + 1) * N // M) + (-m * N // M) for m in range(M)])
        assert counts.size == M and np.array_equal(counts, closed)
        assert closed.max() - closed.min() <= 1
        pos = np_positions(np.arange(N, dtype=np.uint64), N, seed, epoch)
        assert np.array_equal(mb.reshape(-1), (pos * np.uint64(M) // np.uint64(N)).astype(np.int32))


def test_shards_equal_the_whole(lib):
    T, n_traj, M, seed = 24, 1000, 5, 99
    for epoch in range(3):
        whole = minibatches(lib, T, n_traj, n_traj, 0, M, seed, epoch)
        for cuts in ((0, 400, 1000), (0, 1, 999, 1000), (0, 333, 666, 1000)):
            parts = [minibatches(lib, T, b - a, n_traj, a, M, seed, epoch) for a, b in zip(cuts[:-1], cuts[1:])]
            assert np.array_equal(np.concatenate(parts, axis=1), whole)


def test_epochs_mix_the_minibatches(lib):
    T, n_traj, M = 64, 4096, 4
    mbs = [minibatches(lib, T, n_traj, n_traj, 0, M, 1234, e).reshape(-1) for e in range(3)]
    rng = np.random.default_rng(0)
    i, j = rng.integers(0, T * n_traj, (2, 200_000))
    keep = i != j
    i, j = i[keep], j[keep]
    for e in range(3):
        assert abs((mbs[e][i] == mbs[e][j]).mean() - 1 / M) < 0.01
    for a, b in ((0, 1), (1, 2)):
        together = mbs[a][i] == mbs[a][j]
        assert abs((mbs[b][i][together] == mbs[b][j][together]).mean() - 1 / M) < 0.015
        assert (mbs[a] != mbs[b]).mean() > 0.7


# ---------------------------------------------------------------- coefficients
def np_samples(z, legal, a, logp_old, adv, ret, v_old, v, mb, eps, veps, huber, hd):
    """The per-sample definitions in NumPy float64."""
    z = z.astype(np.float64)
    bits = ((legal[:, None] >> np.arange(4)) & 1).astype(bool)
    x = np.where(bits, z, -1e9)
    mx = x.max(1)
    logp = (x[np.arange(len(a)), a] - mx) - np.log(np.exp(x - mx[:, None]).sum(1))
    r = np.exp(logp - logp_old)
    A = adv.astype(np.float64)
    clip = ((A > 0) & (r > 1 + eps)) | ((A < 0) & (r < 1 - eps))
    coef = np.where(clip, 0.0, A * r / mb)
    surr = np.minimum(r * A, np.clip(r, 1 - eps, 1 + eps) * A)
    kl = (r - 1) - (logp - logp_old)
    V, R, Vo = v.astype(np.float64), ret.astype(np.float64), v_old.astype(np.float64)
    d = V - R
    e, g = d.copy(), d.copy()
    if veps > 0:
        dv = V - Vo
        dc = Vo + np.clip(dv, -veps, veps) - R
        use_c = dc * dc > d * d
        e = np.where(use_c, dc, d)
        g = np.where(use_c, np.where(np.abs(dv) < veps, dc, 0.0), d)
    if huber:
        g = np.clip(g, -hd, hd)
        loss = np.where(np.abs(e) <= hd, 0.5 * e * e, hd * (np.abs(e) - 0.5 * hd))
    else:
        loss = 0.5 * e * e
    return np.stack([logp, r, coef, g / mb, clip.astype(np.float64), kl, surr, loss], 1)


def sample_inputs(rng, n, eps):
    f32 = np.float32
    z = (rng.standard_normal((n, 4)) * 3).astype(f32)
    z[: n // 8] *= f32(3000)                                    # logit spreads of 1e4
    legal = rng.integers(1, 16, n).astype(np.uint8)
    legal[n // 8: n // 4] = (1 << rng.integers(0, 4, n // 4 - n // 8)).astype(np.uint8)    # one legal action
    a = np.array([rng.choice(np.flatnonzero((l >> np.arange(4)) & 1)) for l in legal], np.uint8)
    # logp_old: the current logp plus a shift that puts r on both sides of 1 +- eps
    cur = np_samples(z, legal, a, np.zeros(n), np.zeros(n, f32), np.zeros(n, f32), np.zeros(n, f32), np.zeros(n, f32),
                     1.0, eps, 0.0, 0, 1.0)[:, 0]
    shift = rng.choice([0.0, 0.05, -0.05, 0.5, -0.5, np.log(1 + eps) * 0.999, np.log(1 + eps) * 1.001,
                        np.log(1 - eps) * 0.999, np.log(1 - eps) * 1.001], n)
    logp_old = cur - shift
    adv = (rng.standard_normal(n) * 2).astype(f32)
    adv[rng.random(n) < 0.1] = 0.0
    v_old = (rng.standard_normal(n) * 4).astype(f32)
    v = (v_old + rng.standard_normal(n) * rng.choice([0.05, 0.5, 3.0], n)).astype(f32)
    ret = (v_old + rng.standard_normal(n) * 2).astype(f32)
    return z, legal, a, logp_old, adv, ret, v_old, v


@pytest.mark.parametrize("huber,veps", [(0, 0.0), (0, 0.2), (1, 0.0), (1, 0.2)])
def test_coefficients_match_numpy(lib, huber, veps):
    rng = np.random.default_rng(7 + huber + int(veps * 10))
    n, eps, mb, hd = 20000, 0.2, 4096.0, 0.7
    ins = sample_inputs(rng, n, eps)
    out = np.zeros((n, 8))
    lib.hc_ppo_samples(*[P(np.ascontiguousarray(x)) for x in ins], n, mb, eps, veps, huber, hd, P(out))
    want = np_samples(*ins, mb, eps, veps, huber, hd)
    scale = np.maximum(np.abs(want), 1e-300)
    # r - 1 - log r cancels near r = 1: relative to the size of its terms
    scale[:, 5] = np.abs(want[:, 1]) + np.abs(want[:, 0] - ins[3])
    assert (np.abs(out - want) <= 1e-12 * scale + 1e-300).all(), np.max(np.abs(out - want) / scale)
    z, legal, a, logp_old, adv, ret, v_old, v = ins
    single = (legal & (legal - 1)) == 0
    assert single.sum() > 1000 and np.all(out[single, 0] == 0.0)     # one legal action: log pi = 0
    assert out[adv == 0, 2].tolist() == [0.0] * int((adv == 0).sum())
    clipped = out[:, 4] == 1
    assert clipped.sum() > 1000 and (~clipped).sum() > 1000
    assert ((out[:, 1] > 1 + eps) & (adv > 0) == (clipped & (adv > 0))).all()
    assert ((out[:, 1] < 1 - eps) & (adv < 0) == (clipped & (adv < 0))).all()
    if veps > 0:
        dv = v.astype(np.float64) - v_old
        assert ((np.abs(dv) >= veps) & (out[:, 3] == 0)).sum() > 100    # the clipped value branch: no gradient
    if huber:
        assert (np.abs(out[:, 3]) * mb <= hd * (1 + 1e-12)).all() and (np.abs(out[:, 3]) * mb == hd).sum() > 100


# ---------------------------------------------------------------- refusals
def _bare_agent(b2048, critic=True, **cfg):
    agent = object.__new__(b2048.ReinforceAgent)
    agent.agent_config = b2048.ReinforceAgentConfig(use_critic=critic, **cfg)
    agent._critic = object() if critic else None
    return agent


def _window(b2048, auto_reset=True, **kw):
    import torch
    T, B = 4, 8
    return b2048.Rollout(torch.zeros((T + 1, B), dtype=torch.int64), torch.zeros((T + 1, B), dtype=torch.uint8),
                         torch.zeros((T, B), dtype=torch.uint8), torch.zeros((T, B)), torch.full((B,), T, dtype=torch.int32),
                         T, auto_reset=auto_reset, **kw)


@pytest.mark.parametrize("case,cfg,rkw,kw", [
    ("no_critic", dict(critic=False), {}, {}),
    ("no_reset_on_done", {}, dict(auto_reset=False), {}),
    ("augmentation", dict(augmentation=True), {}, {}),
    ("rank_weights", dict(reward_rank_weights=[0.5, 1.0, 1.5]), {}, {}),
    ("baseline_each", dict(baseline_mode="each"), {}, {}),
    ("epochs_0", {}, {}, dict(epochs=0)),
    ("minibatches_0", {}, {}, dict(minibatches=0)),
    ("minibatches_over_N", {}, {}, dict(minibatches=33)),          # N = 4 x 8
    ("clip_eps_0", {}, {}, dict(clip_eps=0.0)),
    ("clip_eps_negative", {}, {}, dict(clip_eps=-0.1)),
    ("value_clip_eps_0", {}, {}, dict(value_clip_eps=0.0)),
    ("shard_without_gid0", {}, dict(n_traj=16), {}),
])
def test_update_ppo_refusals(case, cfg, rkw, kw):
    import b2048
    with pytest.raises(ValueError):
        _bare_agent(b2048, **cfg).update_ppo(_window(b2048, **rkw), **kw)


def test_sharded_update_refuses_ppo_with_one_message_or_episodes():
    import b2048
    from b2048 import dist as bd
    for kw in (dict(fixed_horizon=True, exchange="one_message"), dict(fixed_horizon=False)):
        with pytest.raises(ValueError, match="ppo|PPO"):
            bd.sharded_update(_bare_agent(b2048), _window(b2048), bd.DistInfo(), total_episodes=8, ppo=dict(epochs=2), **kw)


@pytest.mark.parametrize("train,extra,match", [
    (dict(ppo={"epochs": 2}), {}, "horizon"),
    (dict(horizon=16, ppo={"epochs": 2}), {}, "value function"),
    (dict(horizon=16, ppo={"epoch": 2}), dict(agent={"use_critic": True}), "unknown"),
])
def test_trainer_refuses_bad_ppo_sections(train, extra, match):
    from b2048 import trainer
    cfg = trainer.merge_config(dict({"train": dict(train, out_dir=None)}, **extra))
    with pytest.raises(ValueError, match=match):
        trainer.training(cfg)
