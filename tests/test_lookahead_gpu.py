"""The one-ply expectimax over the critic on the device (b2048_lookahead_expand / _select, ReinforceAgent.lookahead_actions /
rollout_lookahead, trainer eval.lookahead): the expansion against the g++ build of csrc/b2048_lookahead.cuh, the fold
against the float64 restatement, whole games against the oracle playing the same rule on the same Philox streams, real
critics against the float64 NumPy forward, the shared-trunk agent, sharded envs and the trainer."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle  # noqa: E402
from helpers import P, full_env_kwargs, random_boards  # noqa: E402
from oracle import learner  # noqa: E402
from test_lookahead import build_libs, expand, np_select, replayed_boards  # noqa: E402


@pytest.fixture(scope="module")
def b2048():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import b2048 as m
    return m


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    return build_libs(tmp_path_factory.mktemp("lookahead_gpu"))


def env_of(b2048, n, name="runner_default", seed=11, gid0=0, obs=None):
    kw = full_env_kwargs(name)
    if obs == "onehot":
        kw.update(obs_mode="onehot", obs_log2_scale=1.0)
    return b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**kw), seed=seed, gid0=gid0)


def agent_of(b2048, env, hidden=(256, 256), shared=False, gamma=0.99):
    mlp = b2048.MLPConfig(hidden_sizes=list(hidden), activation="ReLU", init_distribution="HeNormal")
    cfg = b2048.ReinforceAgentConfig(gamma=gamma, model_seed=3, use_critic=not shared)
    if shared:
        return b2048.SharedTrunkActorCritic(env, mlp, cfg, value_coef=0.5, gae_lambda=0.9)
    return b2048.ReinforceAgent(env, mlp, cfg)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64) if a.dtype == np.uint64 else np.ascontiguousarray(a)).cuda()


def host(t, dtype=None):
    a = t.cpu().numpy()
    return a.view(dtype) if dtype is not None else a


def board_batch(n, seed=1):
    rng = np.random.default_rng(seed)
    b = np.concatenate([random_boards(rng, n // 2), replayed_boards(n // 8, (40, 150, 300, 600), seed)])
    return b[:n], rng.integers(2, 12, n).astype(np.uint8)


def device_expand(b2048, boards_d, flags_d, mx_d, cfg, slot_map=None, n=None):
    lib, h = b2048._lib.load(), b2048.batched_env.get_handle(boards_d.device)
    B = boards_d.numel()
    n = B if n is None else n
    cap = 120 * B
    out = dict(board=torch.zeros(cap, dtype=torch.int64, device="cuda"), reward=torch.zeros(cap, dtype=torch.float64, device="cuda"),
               done=torch.zeros(cap, dtype=torch.uint8, device="cuda"), first=torch.full((B, 4), -7, dtype=torch.int32, device="cuda"),
               count=torch.full((B, 4), -7, dtype=torch.int32, device="cuda"), total=torch.zeros(1, dtype=torch.int32, device="cuda"))
    p = b2048.batched_env._ptr
    b2048._lib.check(lib.b2048_lookahead_expand(h, p(boards_d), p(flags_d), p(mx_d), C.byref(cfg), p(slot_map), n, None, B, cap,
                                                p(out["board"]), p(out["reward"]), p(out["done"]), p(out["first"]), p(out["count"]),
                                                p(out["total"]), None), "expand")
    torch.cuda.synchronize()
    return out


def per_board(first, count, *arrays):
    """The children of every (board, action) in (board, action, j) order, wherever the segments were placed."""
    f, c = first.reshape(-1).astype(np.int64), count.reshape(-1).astype(np.int64)
    c = np.maximum(c, 0)
    start = np.repeat(np.cumsum(c) - c, c)
    idx = np.repeat(f, c) + (np.arange(c.sum()) - start)
    return [a[idx] for a in arrays]


def host_children(d, rows=None):
    first, count = host(d["first"]), host(d["count"])
    if rows is not None:
        first, count = first[rows], count[rows]
    return count, per_board(first, count, host(d["board"], np.uint64), host(d["reward"]).view(np.uint64), host(d["done"]))


@pytest.mark.parametrize("name", ["runner_default", "mask_off", "shaped_raw"])
def test_expand_kernel_equals_host(b2048, libs, name):
    h, _ = libs
    n = 262144
    boards, mx = board_batch(n)
    cfg = b2048.batched_env.make_env_cfg(b2048.Game2048EnvConfig(**full_env_kwargs(name)), "buffer", emit_obs=False)
    legal, _ = oracle.mask_done(boards)
    want = expand(h.hc_lookahead_expand, boards, cfg, mx)
    wc, wch = want["count"], per_board(want["first"], want["count"], want["board"], want["reward"].view(np.uint64), want["done"])
    bd, fd, md = cuda(boards), cuda(legal), cuda(mx)
    got = device_expand(b2048, bd, fd, md, cfg)
    assert int(got["total"]) == want["total"]
    count, ch = host_children(got)
    assert np.array_equal(count, wc)
    for g, w in zip(ch, wch):
        assert np.array_equal(g, w)
    assert (host(got["first"])[wc == 0] == -1).all()
    # a second run, a permuted batch and a batch split into two slot_map halves give the same per-board results
    again = device_expand(b2048, bd, fd, md, cfg)
    c2, ch2 = host_children(again)
    assert np.array_equal(c2, count) and all(np.array_equal(a, b) for a, b in zip(ch2, ch))
    perm = np.random.default_rng(4).permutation(n)
    pg = device_expand(b2048, cuda(boards[perm]), cuda(legal[perm]), cuda(mx[perm]), cfg)
    inv = np.argsort(perm)
    cp, chp = host_children(pg, inv)
    assert np.array_equal(cp, count) and all(np.array_equal(a, b) for a, b in zip(chp, ch))
    halves = np.random.default_rng(5).permutation(n).astype(np.int32)
    parts = [device_expand(b2048, bd, fd, md, cfg, slot_map=cuda(s), n=s.size) for s in (halves[: n // 2], halves[n // 2:])]
    for s, part in zip((halves[: n // 2], halves[n // 2:]), parts):
        rows = np.sort(s)
        cs, chs = host_children(part, rows)
        keep = np.isin(np.repeat(np.arange(n), count.sum(1)), rows)
        assert np.array_equal(cs, count[rows])
        assert all(np.array_equal(a, b[keep]) for a, b in zip(chs, ch))
        others = np.setdiff1d(np.arange(n), rows)
        assert (host(part["count"])[others] == -7).all()           # rows of boards not listed are not written


def test_select_kernel_equals_restatement(b2048, libs):
    h, _ = libs
    n = 262144
    env = env_of(b2048, 4096)
    agent = agent_of(b2048, env)
    boards, mx = board_batch(n, seed=9)
    cfg = b2048.batched_env.make_env_cfg(env.config, "buffer", emit_obs=False)
    d = device_expand(b2048, cuda(boards), None, cuda(mx), cfg)
    total = int(d["total"])
    v = torch.zeros(total, dtype=torch.float32, device="cuda")
    agent._net_forward(agent._critic, d["board"][:total], v, 0)
    act = torch.zeros(n, dtype=torch.uint8, device="cuda")
    q = torch.zeros((n, 4), dtype=torch.float64, device="cuda")
    lib, p = b2048._lib.load(), b2048.batched_env._ptr
    b2048._lib.check(lib.b2048_lookahead_select(agent._h, None, n, None, n, p(d["first"]), p(d["count"]), p(d["reward"]),
                                                p(d["done"]), p(v), 0.99, p(act), p(q), None), "select")
    first, count, reward, done, val = host(d["first"]), host(d["count"]), host(d["reward"]), host(d["done"]), host(v)
    want_act, want_q = np.zeros(n, np.uint8), np.zeros((n, 4))
    h.hc_lookahead_select(P(first), P(count), P(reward), P(done), P(val), 0.99, n, P(want_act), P(want_q))
    ga, gq = host(act), host(q)
    assert np.array_equal(ga, want_act)
    assert np.array_equal(np.nan_to_num(gq).view(np.uint64), np.nan_to_num(want_q).view(np.uint64))
    assert np.array_equal(np.isnan(gq), np.isnan(want_q))
    sub = np.arange(0, n, 64)                        # the NumPy restatement itself on a subset
    na, nq = np_select(first[sub], count[sub], reward, done, val, 0.99)
    assert np.array_equal(ga[sub], na) and np.array_equal(np.nan_to_num(gq[sub]).view(np.uint64), np.nan_to_num(nq).view(np.uint64))


def oracle_games(libs, cfg, seed, n, gamma, v, cap):
    _, o = libs
    acts, rews, fls = (np.zeros((cap, n), dt) for dt in (np.uint8, np.float32, np.uint8))
    length, score, mx = np.zeros(n, np.int32), np.zeros(n, np.uint32), np.zeros(n, np.uint8)
    workers = max(1, min(32, os.cpu_count() or 1))
    step = (n + workers - 1) // workers

    def run(s):
        e = min(n, s + step)
        off = lambda a: C.c_void_p(a.ctypes.data + s * a.itemsize)   # noqa: E731
        o.orc_lookahead_play(seed, s, e - s, C.byref(cfg), gamma, v, cap, n, off(acts), off(rews), off(fls), off(length),
                             off(score), off(mx))

    with ThreadPoolExecutor(workers) as ex:
        list(ex.map(run, range(0, n, step)))
    return acts, rews, fls, length, score, mx


@pytest.mark.parametrize("name", ["runner_default", "mask_off"])
def test_whole_games_against_oracle(b2048, libs, name):
    n, seed, bias = 65536, 0xC0FFEE, 0.75
    env = env_of(b2048, n, name, seed=seed)
    agent = agent_of(b2048, env)
    cp = agent.critic_params
    cp["W"][-1] = np.zeros_like(cp["W"][-1])
    cp["b"][-1] = np.full_like(cp["b"][-1], bias)
    agent.critic_params = cp
    ro = agent.rollout_lookahead(env, precision=0)
    cfg = b2048.batched_env.make_env_cfg(env.config, "buffer", emit_obs=False)
    cap = int(env.config.max_steps or 4096)
    acts, rews, fls, length, score, mx = oracle_games(libs, cfg, seed, n, 0.99, np.float32(bias), cap)
    T = ro.T
    L = host(ro.length)
    assert np.array_equal(L, length) and T == length.max()
    live = np.arange(T)[:, None] < L[None, :]
    assert np.array_equal(host(ro.actions)[live], acts[:T][live])
    assert np.array_equal(host(ro.rewards)[live], rews[:T][live])
    assert np.array_equal(host(ro.flags)[1:][live], fls[:T][live])
    assert np.array_equal(host(env.score).astype(np.uint32), score) and np.array_equal(host(env.max_exp), mx)
    assert live.sum() > 100 * n


def q_reference(libs, agent, boards, mx, cfg, gamma):
    """Q of every board with V from oracle/learner.py's float64 forward of the critic."""
    h, _ = libs
    e = expand(h.hc_lookahead_expand, boards, cfg, mx)
    cp = agent.critic_params
    p64 = {"W": [np.asarray(w, np.float64) for w in cp["W"]], "b": [np.asarray(b, np.float64) for b in cp["b"]]}
    X = learner.encode(e["board"], agent._obs_mode, agent._obs_scale)
    v = np.concatenate([learner.forward(p64, X[i: i + 65536], "ReLU")[0][:, 0] for i in range(0, len(X), 65536)])
    v = np.where(e["done"] != 0, 0.0, v)
    t = e["reward"] + gamma * v
    cnt = e["count"].reshape(-1)
    nsp = np.repeat(np.where(cnt > 1, cnt // 2, 1), cnt)
    kind = np.concatenate([np.arange(c) % 2 if c > 1 else np.full(1, -1) for c in cnt if c > 0])
    w = np.where(kind == 0, 0.9, np.where(kind == 1, 0.1, 1.0)) / nsp
    seg = np.repeat(np.arange(cnt.size), cnt)
    q = np.full(cnt.size, np.nan)
    q[cnt > 0] = np.bincount(seg, weights=w * t, minlength=cnt.size)[cnt > 0]
    return q.reshape(-1, 4)


@pytest.mark.parametrize("obs,hidden", [("log2", (256, 256)), ("onehot", (256, 128, 64))])
def test_real_critic_against_float64_forward(b2048, libs, obs, hidden):
    n = 16384
    env = env_of(b2048, 4096, obs=obs)
    agent = agent_of(b2048, env, hidden=hidden)
    boards, mx = board_batch(n, seed=21)
    legal, _ = oracle.mask_done(boards)
    cfg = b2048.batched_env.make_env_cfg(env.config, "buffer", emit_obs=False)
    qref = q_reference(libs, agent, boards, mx, cfg, 0.99)
    for precision, tol in ((0, 1e-5), ("auto", 1e-3)):
        q = torch.zeros((n, 4), dtype=torch.float64, device="cuda")
        act = host(agent.lookahead_actions(cuda(boards), cuda(legal), cuda(mx), precision=precision, q_out=q))
        gq = host(q)
        assert np.array_equal(np.isnan(gq), np.isnan(qref))
        ok = ~np.isnan(qref)
        scale = np.abs(qref[ok]).max()
        assert (np.abs(gq[ok] - qref[ok]) <= tol * scale).all(), precision          # relative to max |Q|
        srt = np.sort(np.where(np.isnan(qref), -np.inf, qref), 1)
        clear = (srt[:, -1] - srt[:, -2]) > (1e-4 if precision == 0 else 2e-3) * scale
        want = np.nanargmax(np.where(np.isnan(qref), -np.inf, qref), 1)
        assert clear.sum() > n // 2 and np.array_equal(act[clear], want[clear]), precision


def test_shared_trunk_plays_and_shards_reproduce_the_batch(b2048):
    n, seed = 8192, 77
    whole_env = env_of(b2048, n, seed=seed)
    agent = agent_of(b2048, whole_env, shared=True)
    whole = agent.rollout_lookahead(whole_env, precision=0)
    assert host(whole.length).min() > 0 and float(whole.total_reward().mean()) > 0
    # the rollout's buffers are the agent's scratch, which the next rollout reuses: keep host copies
    W_actions, W_rewards, W_mx, L = host(whole.actions), host(whole.rewards), host(whole_env.max_exp), host(whole.length)
    halves = []
    for g in (0, n // 2):
        e = env_of(b2048, n // 2, seed=seed, gid0=g)
        ro = agent.rollout_lookahead(e, precision=0)
        halves.append((type(ro)(*(x.clone() if torch.is_tensor(x) else x for x in (ro.boards, ro.flags, ro.actions, ro.rewards,
                                                                                     ro.length, ro.T))), e))
    for k, (ro, e) in enumerate(halves):
        cols = slice(k * n // 2, (k + 1) * n // 2)
        assert np.array_equal(host(ro.length), L[cols])
        T = ro.T
        live = np.arange(T)[:, None] < L[None, cols]
        assert np.array_equal(host(ro.actions)[live], W_actions[:T, cols][live])
        assert np.array_equal(host(ro.rewards)[live], W_rewards[:T, cols][live])
        assert np.array_equal(host(e.max_exp), W_mx[cols])


def test_trainer_lookahead_evaluation(b2048, tmp_path):
    from b2048 import dist as bd
    from b2048 import trainer
    cfg = trainer.merge_config({"agent": {"use_critic": True}, "eval": {"num_episodes": 4096}})
    info = bd.DistInfo()
    default = trainer.evaluation(cfg, info)
    env = bd.make_sharded_env(4096, b2048.Game2048EnvConfig(**cfg["env"]), info, seed=int(cfg["seed"]) + 12345)
    agent = trainer.make_agent(cfg, env)
    ro = agent.rollout_many(env, greedy=True, precision="auto")
    assert default["avg_reward"] == pytest.approx(float(ro.total_reward().mean()), rel=1e-12)
    assert default["mean_len"] == float(ro.length.float().mean())
    ck = str(tmp_path / "ck.npz")
    agent.save_checkpoint(ck)
    la = trainer.evaluation(trainer.merge_config({"agent": {"use_critic": True},
                                                  "eval": {"num_episodes": 4096, "lookahead": True, "checkpoint": ck}}), info)
    assert set(la) == set(default) and la["mean_len"] > 0 and sum(la["max_tile_counts"]) <= 4096
    env2 = bd.make_sharded_env(4096, b2048.Game2048EnvConfig(**cfg["env"]), info, seed=int(cfg["seed"]) + 12345)
    ro2 = agent.rollout_lookahead(env2)
    assert la["avg_reward"] == pytest.approx(float(ro2.total_reward().mean()), rel=1e-12)
