"""CPU checks of the entropy bonus (b2048_mlp_backward_entropy): the helper of csrc/b2048_entropy.cuh, compiled with g++ from
tests/host_check/entropy_check.cpp, against a NumPy float64 restatement; its exact zeros and bounds; and the configurations
the updates, sharded_update and the trainer refuse."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, P


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("entropy") / "libentropy.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "host_check", "entropy_check.cpp")])
    h = C.CDLL(so)
    h.hc_entropy_rows.restype = None
    h.hc_entropy_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    return h


def rows(lib, logits, legal, use_mask=True, n_out=4):
    n = logits.shape[0]
    p, t, H = np.zeros((n, 4), np.float32), np.zeros((n, 4), np.float32), np.zeros(n, np.float32)
    lib.hc_entropy_rows(P(np.ascontiguousarray(logits, np.float32)), P(np.ascontiguousarray(legal, np.uint8)), int(use_mask),
                        n_out, n, P(p), P(t), P(H))
    return p, t, H


def np_entropy(logits, legal, n_out=4):
    """float64: p over the legal outputs, H = -sum p log p, t_j = p_j (log p_j + H) (0 off the legal set; rows without a
    legal output: 0)."""
    z = logits.astype(np.float64)
    lg = ((legal[:, None] >> np.arange(4)) & 1).astype(bool) & (np.arange(4) < n_out)
    zm = np.where(lg, z, -np.inf)
    mx = np.max(np.where(lg.any(1, keepdims=True), zm, 0.0), axis=1, keepdims=True)
    e = np.where(lg, np.exp(np.where(lg, z - mx, 0.0)), 0.0)
    s = e.sum(1, keepdims=True)
    p = np.divide(e, s, out=np.zeros_like(e), where=s > 0)
    logp = np.where(lg, np.where(lg, z - mx, 0.0) - np.log(np.where(s > 0, s, 1.0)), 0.0)
    H = -(p * logp).sum(1)
    t = np.where(lg, p * (logp + H[:, None]), 0.0)
    return p, t, H


def random_rows(rng, n, scale=3.0):
    logits = (rng.standard_normal((n, 4)) * scale).astype(np.float32)
    legal = rng.integers(1, 16, n).astype(np.uint8)
    return logits, legal


@pytest.mark.parametrize("scale", [0.3, 3.0, 30.0])
def test_helper_matches_numpy(lib, scale):
    rng = np.random.default_rng(int(scale * 10))
    logits, legal = random_rows(rng, 50000, scale)
    p, t, H = rows(lib, logits, legal)
    wp, wt, wH = np_entropy(logits, legal)
    assert np.allclose(p, wp, rtol=1e-6, atol=1e-7)
    # float32 rounding of H = lse - sum p z: relative to the size of its terms, plus the rounding of the softmax sum (~1 when
    # one move dominates) before its log, a few float32 ulps of 1
    lg = ((legal[:, None] >> np.arange(4)) & 1).astype(bool)
    z = np.where(lg, logits.astype(np.float64) - np.max(np.where(lg, logits, -np.inf), 1, keepdims=True), 0.0)
    lse = np.log(np.where(lg, np.exp(z), 0.0).sum(1))
    hscale = lse + (wp * np.abs(z)).sum(1)
    eps = 4 * 2.0 ** -24
    assert (np.abs(H - wH) <= 1e-6 * hscale + eps).all(), np.max(np.abs(H - wH) - 1e-6 * hscale)
    tscale = wp * (np.abs(z) + lse[:, None] + hscale[:, None])
    assert (np.abs(t - wt) <= 1e-6 * tscale + wp * eps + 1e-12).all(), np.max(np.abs(t - wt) - 1e-6 * tscale - wp * eps)


@pytest.mark.parametrize("n_out", [1, 2, 3, 4])
def test_unmasked_and_padded_outputs(lib, n_out):
    rng = np.random.default_rng(n_out)
    logits, _ = random_rows(rng, 10000)
    legal = np.full(10000, 0xF, np.uint8)
    p, t, H = rows(lib, logits, legal, use_mask=False, n_out=n_out)
    wp, wt, wH = np_entropy(logits, legal, n_out)
    assert np.all(t[:, n_out:] == 0.0) and np.all(p[:, n_out:] == 0.0)
    assert np.allclose(H, wH, rtol=1e-5, atol=1e-6) and np.allclose(t, wt, rtol=1e-5, atol=1e-6)
    if n_out == 1:
        assert np.all(H == 0.0) and np.all(t == 0.0)


def test_exact_zeros(lib):
    rng = np.random.default_rng(7)
    logits, legal = random_rows(rng, 40000)
    p, t, H = rows(lib, logits, legal)
    lg = ((legal[:, None] >> np.arange(4)) & 1).astype(bool)
    assert np.all(t[~lg] == 0.0) and np.all(p[~lg] == 0.0)        # illegal outputs: exactly 0, no 0 * inf
    single = (legal & (legal - 1)) == 0
    assert single.sum() > 5000
    assert np.all(H[single] == 0.0) and np.all(t[single] == 0.0)   # one legal move: no entropy, no gradient
    # equally likely legal moves: H = log(k), t = 0 up to rounding
    eq = np.zeros((4, 4), np.float32) + 1.25
    p, t, H = rows(lib, eq, np.array([1, 3, 7, 15], np.uint8))
    assert np.allclose(H, np.log([1, 2, 3, 4]), rtol=1e-6, atol=0) and np.all(np.abs(t) <= 1e-7)


def test_extreme_logits_and_all_masked_rows(lib):
    rng = np.random.default_rng(11)
    n = 20000
    logits = rng.choice(np.array([-1e4, 1e4, 0.0, 1.0], np.float32), size=(n, 4))
    legal = rng.integers(0, 16, n).astype(np.uint8)           # 0: every output masked
    p, t, H = rows(lib, logits, legal)
    assert np.isfinite(p).all() and np.isfinite(t).all() and np.isfinite(H).all()
    assert np.all(H[legal == 0] == 0.0) and np.all(t[legal == 0] == 0.0)
    wp, wt, wH = np_entropy(logits, legal)
    ok = legal != 0
    assert np.allclose(H[ok], wH[ok], rtol=1e-6, atol=1e-6) and np.allclose(t[ok], wt[ok], rtol=1e-6, atol=1e-6)


def test_term_bound(lib):
    """|t_j| <= ln 4, so |d_j| <= |coef| + ln 4 |ecoef| < |coef| + 1.5 |ecoef| (the fp16 loss scale's bound)."""
    rng = np.random.default_rng(3)
    for scale in (0.1, 1.0, 10.0, 1e4):
        logits, legal = random_rows(rng, 50000, scale)
        legal[::7] = 0xF
        _, t, H = rows(lib, logits, legal)
        assert np.abs(t).max() <= math.log(4.0) * (1 + 1e-6)
        assert H.max() <= math.log(4.0) * (1 + 1e-6) and H.min() >= -1e-6


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


BAD = [
    ("negative", dict(entropy_coef=-0.01)),
    ("nan", dict(entropy_coef=float("nan"))),
    ("inf", dict(entropy_coef=float("inf"))),
    ("bf16", dict(entropy_coef=0.01, precision=1)),
]


@pytest.mark.parametrize("case,kw", BAD + [("one_message", dict(entropy_coef=0.01, exchange="one_message"))])
def test_update_from_rollout_refusals(case, kw):
    import b2048
    with pytest.raises(ValueError, match="entropy"):
        _bare_agent(b2048).update_from_rollout(_window(b2048, auto_reset=False), **kw)


@pytest.mark.parametrize("case,kw", BAD + [("one_message", dict(entropy_coef=0.01, exchange="one_message"))])
def test_update_from_horizon_refusals(case, kw):
    import b2048
    with pytest.raises(ValueError, match="entropy"):
        _bare_agent(b2048).update_from_horizon(_window(b2048), **kw)


@pytest.mark.parametrize("case,kw", BAD)
def test_update_ppo_refusals(case, kw):
    import b2048
    with pytest.raises(ValueError, match="entropy"):
        _bare_agent(b2048).update_ppo(_window(b2048), **kw)


def test_sharded_update_refusals():
    import b2048
    from b2048 import dist as bd
    for kw in (dict(entropy_coef=-1.0), dict(entropy_coef=0.01, exchange="one_message"),
               dict(entropy_coef=0.01, exchange="one_message", fixed_horizon=True)):
        with pytest.raises(ValueError, match="entropy"):
            bd.sharded_update(_bare_agent(b2048), _window(b2048), bd.DistInfo(), total_episodes=8, **kw)


@pytest.mark.parametrize("train", [dict(entropy_coef=-0.5), dict(entropy_coef=0.01, exchange="one_message"),
                                   dict(entropy_coef=0.01, exchange="one_message", horizon=16)])
def test_trainer_refuses_bad_entropy_coef(train):
    from b2048 import trainer
    cfg = trainer.merge_config({"train": dict(train, out_dir=None)})
    with pytest.raises(ValueError, match="entropy"):
        trainer.training(cfg)
