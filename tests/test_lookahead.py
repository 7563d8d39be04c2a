"""CPU checks of the one-ply expectimax over the critic (csrc/b2048_lookahead.cuh, compiled with g++ from
tests/host_check/lookahead_check.cpp): the expansion against the cell-by-cell oracle enumeration
(tests/host_check/lookahead_oracle.c on top of oracle/b2048_oracle.c) and against the step body with a replayed spawn; the
Q / argmax fold against a float64 restatement; and the calls that refuse a lookahead."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from helpers import ROOT, P, full_env_kwargs, random_boards

# The five env configurations of the expansion checks.
EXPAND_CONFIGS = {
    "log2": dict(reward_mode="log2", base_reward_scale=0.5),
    "sum": dict(reward_mode="sum"),
    "shaped_log2_bonus": dict(reward_mode="log2", empty_tile_reward=0.05, merge_reward=0.3, bonus_mode="log2",
                              bonus_scale=2.0, endgame_penalty=-7.5, step_reward=-0.01),
    "mask_off": dict(reward_mode="sum", use_action_mask=False, invalid_action_penalty=-2.5, step_reward=0.125),
    "raw_bonus": dict(reward_mode="sum", base_reward_scale=0.25, bonus_mode="raw", bonus_scale=0.125),
}


def build_libs(d):
    """(header check, oracle enumeration) compiled into directory d and bound with ctypes."""
    hc, orc = str(d / "liblookahead_check.so"), str(d / "liblookahead_oracle.so")
    hdir = os.path.join(ROOT, "tests", "host_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", hc,
                           os.path.join(hdir, "lookahead_check.cpp")])
    subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-shared", "-o", orc,
                           os.path.join(hdir, "lookahead_oracle.c"), "-lm"])
    h, o = C.CDLL(hc), C.CDLL(orc)
    h.hc_lookahead_expand.restype = C.c_int64
    h.hc_lookahead_expand.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_int64] + [C.c_void_p] * 5
    h.hc_lookahead_select.restype = None
    h.hc_lookahead_select.argtypes = [C.c_void_p] * 5 + [C.c_double, C.c_int64, C.c_void_p, C.c_void_p]
    h.hc_step_replay.restype = None
    h.hc_step_replay.argtypes = [C.c_void_p] * 5 + [C.c_int64] + [C.c_void_p] * 3
    o.orc_lookahead_expand.restype = C.c_int64
    o.orc_lookahead_expand.argtypes = [C.c_void_p] * 3 + [C.c_int64] + [C.c_void_p] * 5
    o.orc_lookahead_play.restype = C.c_int
    o.orc_lookahead_play.argtypes = [C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_double, C.c_float, C.c_int32,
                                     C.c_int64] + [C.c_void_p] * 6
    return h, o


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    return build_libs(tmp_path_factory.mktemp("lookahead"))


def env_cfg(name):
    kw = {k: v for k, v in full_env_kwargs("dataclass_default").items() if k not in ("size", "obs_mode", "obs_log2_scale")}
    kw.update(EXPAND_CONFIGS[name])
    return oracle.make_cfg(**kw)


def replayed_boards(n, steps, seed):
    """Mid- and late-game boards: random-legal games of the oracle (auto-reset), snapshots after each entry of steps."""
    cfg = oracle.make_cfg(action_mode="random_legal", auto_reset=True, max_steps=None)
    st = oracle.reset_many(n, seed)
    out = []
    for t in range(1, max(steps) + 1):
        oracle.step_many(st, cfg, seed, 0, t)
        if t in steps:
            out.append(st["board"].copy())
    return np.concatenate(out)


def board_set():
    rng = np.random.default_rng(2048)
    b = np.concatenate([random_boards(rng, 6000), replayed_boards(2048, (60, 200, 500), 7)])
    mx = rng.integers(2, 12, b.size).astype(np.uint8)
    return b, mx


def expand(fn, boards, cfg, max_exp, flags=None, header=True):
    n = boards.size
    cap = 120 * n
    cb, cr, cd = np.zeros(cap, np.uint64), np.zeros(cap, np.float64), np.zeros(cap, np.uint8)
    first, count = np.zeros((n, 4), np.int32), np.zeros((n, 4), np.int32)
    if header:
        total = fn(P(boards), P(flags), P(max_exp), C.byref(cfg), n, cap, P(cb), P(cr), P(cd), P(first), P(count))
    else:
        total = fn(P(boards), P(max_exp), C.byref(cfg), n, P(cb), P(cr), P(cd), P(first), P(count))
    return dict(total=total, board=cb[:total], reward=cr[:total], done=cd[:total], first=first, count=count)


@pytest.mark.parametrize("name", list(EXPAND_CONFIGS))
@pytest.mark.parametrize("with_max", [True, False])
def test_expand_matches_oracle_enumeration(libs, name, with_max):
    h, o = libs
    boards, mx = board_set()
    assert boards.size >= 10000
    cfg = env_cfg(name)
    m = mx if with_max else None
    got = expand(h.hc_lookahead_expand, boards, cfg, m)
    want = expand(o.orc_lookahead_expand, boards, cfg, m, header=False)
    assert got["total"] == want["total"] and got["total"] > 10 * boards.size
    for k in ("first", "count", "board", "done"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["reward"].view(np.uint64), want["reward"].view(np.uint64))
    # the candidate set: the legal mask with the action mask on, all four actions with it off
    legal, _ = oracle.mask_done(boards)
    cand = (got["count"] > 0)
    bits = np.stack([(legal >> a) & 1 for a in range(4)], 1).astype(bool)
    assert np.array_equal(cand, bits if cfg.use_action_mask else np.ones_like(bits))
    assert got["count"].sum(1).max() <= 120
    # the flags argument gives the same children as the recomputed mask
    flagged = expand(h.hc_lookahead_expand, boards, cfg, m, flags=legal)
    assert np.array_equal(flagged["board"], got["board"]) and np.array_equal(flagged["count"], got["count"])


@pytest.mark.parametrize("name", list(EXPAND_CONFIGS))
def test_children_equal_the_replayed_step(libs, name):
    """Every child equals the step body (b2048_step_many's step_one) on its (board, action, spawn_replay)."""
    h, _ = libs
    boards, mx = board_set()
    cfg = env_cfg(name)
    got = expand(h.hc_lookahead_expand, boards, cfg, mx)
    src, act, rep = [], [], []
    for a in range(4):
        for i in np.nonzero(got["count"][:, a])[0]:
            c = int(got["count"][i, a])
            src += [i] * c
            act += [a] * c
            rep += [0x80 if c == 1 else 0x80 | (j >> 1) | ((j & 1) << 4) for j in range(c)]
    order = np.argsort(np.concatenate([got["first"][i, a] + np.arange(got["count"][i, a]) for a in range(4)
                                       for i in np.nonzero(got["count"][:, a])[0]]), kind="stable")
    src, act, rep = (np.asarray(x)[order] for x in (src, act, rep))
    n = src.size
    assert n == got["total"]
    ob, orw, ofl = np.zeros(n, np.uint64), np.zeros(n), np.zeros(n, np.uint8)
    h.hc_step_replay(P(np.ascontiguousarray(boards[src])), P(act.astype(np.uint8)), P(rep.astype(np.uint8)),
                     P(np.ascontiguousarray(mx[src])), C.byref(cfg), n, P(ob), P(orw), P(ofl))
    assert np.array_equal(ob, got["board"])
    assert np.array_equal(orw.view(np.uint64), got["reward"].view(np.uint64))
    assert np.array_equal((ofl & oracle.F_DONE) != 0, got["done"] != 0)


# ---------------------------------------------------------------- the Q / argmax fold
def np_select(first, count, reward, done, value, gamma):
    """Q and the action in float64, each multiply and add rounded on its own (NumPy scalars, sequential sums)."""
    n = first.shape[0]
    q = np.full((n, 4), np.nan)
    act = np.zeros(n, np.uint8)
    g = np.float64(gamma)

    def t(j):
        return reward[j] + g * (np.float64(0.0) if done[j] else np.float64(value[j]))

    for i in range(n):
        best = None
        for a in range(4):
            f, c = int(first[i, a]), int(count[i, a])
            if c == 0:
                continue
            if c == 1:
                qa = t(f)
            else:
                s = np.float64(0.0)
                for k in range(c // 2):
                    s = s + (np.float64(0.9) * t(f + 2 * k) + np.float64(0.1) * t(f + 2 * k + 1))
                qa = s / np.float64(c // 2)
            q[i, a] = qa
            if best is None or qa > q[i, best]:
                best = a
        act[i] = 0 if best is None else best
    return act, q


@pytest.mark.parametrize("name", ["log2", "mask_off", "shaped_log2_bonus"])
@pytest.mark.parametrize("gamma", [0.99, 1.0, 0.0])
def test_select_matches_float64_restatement(libs, name, gamma):
    h, o = libs
    rng = np.random.default_rng(5)
    boards = np.concatenate([random_boards(rng, 1500), replayed_boards(256, (300,), 3)])
    boards[:20] = np.uint64(0x1212212112122121)    # a finished checkerboard: no candidate with the mask on
    cfg = env_cfg(name)
    e = expand(h.hc_lookahead_expand, boards, cfg, None)
    total = e["total"]
    # few distinct values: many exact ties between moves
    value = rng.choice(np.array([0.0, 1.5, -2.0, 3.25], np.float32), total) if gamma != 0.99 else \
        rng.normal(0, 3, total).astype(np.float32)
    act = np.zeros(boards.size, np.uint8)
    q = np.zeros((boards.size, 4))
    h.hc_lookahead_select(P(e["first"]), P(e["count"]), P(e["reward"]), P(e["done"]), P(value), gamma, boards.size, P(act),
                          P(q))
    want_act, want_q = np_select(e["first"], e["count"], e["reward"], e["done"], value, gamma)
    assert np.array_equal(act, want_act)
    assert np.array_equal(np.isnan(q), np.isnan(want_q))
    assert np.array_equal(np.nan_to_num(q).view(np.uint64), np.nan_to_num(want_q).view(np.uint64))
    if cfg.use_action_mask:
        assert np.isnan(q[:20]).all() and (act[:20] == 0).all()
    else:
        assert (e["count"] == 1).any()          # unchanged moves of the mask-off configuration
    valid = ~np.isnan(q)
    top = np.where(valid, q, -np.inf)
    assert (np.sum(top == top.max(1, keepdims=True), 1) > 1).sum() > (10 if gamma != 0.99 else -1)   # ties occur


# ---------------------------------------------------------------- refusals
def _bare_agent(b2048, critic=True):
    agent = object.__new__(b2048.ReinforceAgent)
    agent.agent_config = b2048.ReinforceAgentConfig(use_critic=critic)
    agent._critic = object() if critic else None
    return agent


def test_lookahead_refuses_an_agent_without_a_value_function():
    import torch
    import b2048
    agent = _bare_agent(b2048, critic=False)
    with pytest.raises(ValueError, match="value function"):
        agent.lookahead_actions(torch.zeros(4, dtype=torch.int64), None)
    with pytest.raises(ValueError, match="value function"):
        agent.rollout_lookahead(object())


@pytest.mark.parametrize("precision", ["fast", 4, -1, 1.5, True, None])
def test_lookahead_refuses_a_bad_precision(precision):
    import torch
    import b2048
    with pytest.raises(ValueError, match="precision"):
        _bare_agent(b2048).lookahead_actions(torch.zeros(4, dtype=torch.int64), None, precision=precision)
    with pytest.raises(ValueError, match="precision"):
        _bare_agent(b2048).rollout_lookahead(object(), precision=precision)


@pytest.mark.parametrize("ev,extra,match", [
    (dict(lookahead=True), dict(agent={"use_critic": True}), "checkpoint"),
    (dict(lookahead=True, model_path="actor.npz"), dict(agent={"use_critic": True}), "checkpoint"),
    (dict(lookahead=True, checkpoint="ck.npz"), {}, "value function"),
])
def test_trainer_refuses_lookahead_evaluation(ev, extra, match):
    from b2048 import trainer
    cfg = trainer.merge_config(dict({"eval": ev}, **extra))
    with pytest.raises(ValueError, match=match):
        trainer.evaluation(cfg)


def test_trainer_refuses_lookahead_for_an_agent_without_critic():
    import b2048
    from b2048 import trainer
    cfg = trainer.merge_config({"eval": dict(lookahead=True)})
    with pytest.raises(ValueError, match="value function"):
        trainer.evaluation(cfg, agent=_bare_agent(b2048, critic=False))
