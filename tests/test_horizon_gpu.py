"""Fixed-horizon window updates on the device (ReinforceAgent.update_from_horizon, b2048_segment_targets,
b2048_advantages_window, b2048_horizon_episodes): the kernel outputs of a fused-kernel rollout against the NumPy restatement,
the update gradient against PyTorch float32 autograd, two emulated ranks against one process, the episode accounting
against the oracle's replay, and the trainer's train.horizon mode."""
import json
import os
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle  # noqa: E402
from helpers import full_env_kwargs, rel_err  # noqa: E402
from test_horizon_targets import restate  # noqa: E402  (the NumPy restatement of the window definitions)

F_END = 0x60


@pytest.fixture(scope="module")
def b2048():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import b2048 as m
    return m


def env_of(b2048, n, seed, max_steps=25, obs="log2"):
    kw = full_env_kwargs("runner_default")
    kw["max_steps"] = max_steps
    if obs == "onehot":
        kw.update(obs_mode="onehot", obs_log2_scale=1.0)
    return b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**kw), seed=seed, gid0=0)


def agent_of(b2048, env, hidden=(256, 256), shared_lambda=None, **cfg):
    base = dict(gamma=0.99, learning_rate=1e-3, baseline_mode="batch", model_seed=5, max_grad_norm=1e9)
    base.update(cfg)
    mlp = b2048.MLPConfig(hidden_sizes=list(hidden), activation="ReLU", init_distribution="HeNormal")
    if shared_lambda is not None:
        return b2048.SharedTrunkActorCritic(env, mlp, b2048.ReinforceAgentConfig(**base), value_coef=0.7,
                                            gae_lambda=shared_lambda)
    return b2048.ReinforceAgent(env, mlp, b2048.ReinforceAgentConfig(**base))


def np_window(ro):
    T = ro.T
    return (ro.rewards[:T].cpu().numpy(), ro.flags[: T + 1].cpu().numpy(), ro.boards[: T + 1].cpu().numpy(),
            ro.actions[:T].cpu().numpy())


def test_segment_kernel_bit_equal_on_fused_rollout(b2048):
    n, H = 65536, 64
    env = env_of(b2048, n, seed=21)
    agent = agent_of(b2048, env)
    assert agent._fused_shape()
    ro = agent.rollout_many(env, horizon=H, precision=1)
    rewards, flags, _, _ = np_window(ro)
    ends = flags[1:] & F_END
    assert (ends == 0x20).sum() > 0 and (ends == 0x40).sum() > 0     # terminations and truncations at max_steps = 25
    values = torch.randn((H + 1, n), device="cuda") * 4
    for critic, lam, huber in ((False, 0.0, 0), (True, 0.0, 1), (True, 0.95, 0)):
        agent.agent_config.critic_loss_type = "huber" if huber else "mse"
        agent.agent_config.huber_delta = 1.5
        v = torch.empty((H, n), device="cuda")
        td = torch.empty((H, n), device="cuda") if critic else None
        gc = torch.empty((H, n), device="cuda") if critic else None
        valid = torch.empty(n, dtype=torch.int32, device="cuda")
        agent._segment_targets(ro.rewards[:H].contiguous(), ro.flags[: H + 1].contiguous(), values if critic else None,
                               lam, float(n), v, td, gc, valid)
        rv, rtd, rgc, rvalid = restate(rewards, flags, values.cpu().numpy() if critic else None, 0.99, lam, huber, 1.5, float(n))
        assert np.array_equal(valid.cpu().numpy(), rvalid)
        assert np.array_equal(v.cpu().numpy().view(np.uint32), rv.view(np.uint32))
        if critic:
            assert np.array_equal(td.cpu().numpy().view(np.uint32), rtd.view(np.uint32))
            assert np.array_equal(gc.cpu().numpy().view(np.uint32), rgc.view(np.uint32))
        else:
            assert (rvalid > 0).all() and (rvalid < H).any()       # every lane ends an episode; some keep a tail


def restate_coef(v, valid, mode, T, n_traj):
    """advantage_window_kernel's coefficients from the restated targets."""
    f32 = np.float32
    mask = np.arange(T)[:, None] < valid[None, :]
    mean, std = f32(0), f32(1)
    if mode != "off":
        x = v[mask].astype(np.float64)
        m = x.sum() / x.size
        mean = f32(m)
        std = f32(np.sqrt(max((x * x).sum() / x.size - m * m, 0.0))) if mode == "batch_norm" else f32(1)
        std = max(std, f32(1e-8))
    a = (v - mean) / std if mode == "batch_norm" else v - mean
    return np.where(mask, a * (f32(1) / (f32(T) * f32(n_traj))), f32(0)).astype(f32)


def mlp_forward(Ws, bs, x):
    h = x
    for W, b in zip(Ws[:-1], bs[:-1]):
        h = torch.relu(h @ W + b)
    return h, h @ Ws[-1] + bs[-1]


def torch_grad(agent, ro, coef, gcoef, onehot, actor_p, critic_p=None, value_head=None, vc=1.0):
    """float32 autograd gradient of J = sum coef log pi(a|s) - vc sum gcoef V(s) (separate critic: [d sum coef log pi |
    d sum gcoef V], the layout of the agent's flat gradient buffer)."""
    T = ro.T
    boards = ro.boards[:T].reshape(-1)
    flags = ro.flags[:T].reshape(-1).long()
    acts = ro.actions[:T].reshape(-1).long()
    e = torch.stack([(boards >> (4 * i)) & 15 for i in range(16)], 1)
    x = torch.nn.functional.one_hot(e, 17).float().reshape(-1, 272) if onehot else e.float() * 0.0625
    cf = torch.from_numpy(coef.reshape(-1)).cuda()
    leaf = lambda a: torch.tensor(np.asarray(a), device="cuda", requires_grad=True)
    Ws, bs = [leaf(W) for W in actor_p["W"]], [leaf(b) for b in actor_p["b"]]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        h, logits = mlp_forward(Ws, bs, x)
        legal = ((flags.unsqueeze(1) >> torch.arange(4, device="cuda")) & 1).bool()
        logp = torch.log_softmax(logits.masked_fill(~legal, float("-inf")), 1).gather(1, acts.unsqueeze(1)).reshape(-1)
        J = (cf * logp).sum()
        extra = []
        if gcoef is not None:
            gc = torch.from_numpy(gcoef.reshape(-1)).cuda()
            if value_head is not None:                                  # shared trunk: value head on the policy trunk
                Wv, bv = leaf(value_head["W"]), leaf(value_head["b"])
                J = J - vc * (gc * (h @ Wv + bv).reshape(-1)).sum()
                extra = [Wv, bv]
                J.backward()
            else:
                Wc, bc = [leaf(W) for W in critic_p["W"]], [leaf(b) for b in critic_p["b"]]
                _, V = mlp_forward(Wc, bc, x)
                J.backward()
                (gc * V.reshape(-1)).sum().backward()
                extra = [t for pair in zip(Wc, bc) for t in pair]
        else:
            J.backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    parts = [t.grad.reshape(-1) for pair in zip(Ws, bs) for t in pair] + [t.grad.reshape(-1) for t in extra]
    return torch.cat(parts).cpu().numpy()


CASES = {
    "reinforce_batch_fp32": dict(prec=0, tol=2e-4, cfg=dict(baseline_mode="batch")),
    "reinforce_batch_norm_tc": dict(prec="auto", tol=1e-2, cfg=dict(baseline_mode="batch_norm")),
    "critic_td0_huber_fp32": dict(prec=0, tol=2e-4, cfg=dict(use_critic=True, critic_loss_type="huber", huber_delta=0.5)),
    "critic_td0_huber_tc": dict(prec="auto", tol=1e-2, cfg=dict(use_critic=True, critic_loss_type="huber", huber_delta=0.5)),
    "shared_trunk_gae_fp32": dict(prec=0, tol=2e-4, shared=0.95, cfg=dict(baseline_mode="batch_norm")),
    "onehot_256_128_64_tc": dict(prec="auto", tol=1e-2, hidden=(256, 128, 64), obs="onehot", cfg=dict(baseline_mode="batch_norm")),
    "augmented_fp32": dict(prec=0, tol=2e-4, cfg=dict(baseline_mode="batch", augmentation=True)),
}


@pytest.mark.parametrize("case", list(CASES))
def test_horizon_gradient_vs_torch_autograd(b2048, case):
    c = CASES[case]
    n, H = 4096, 48
    env = env_of(b2048, n, seed=31, obs=c.get("obs", "log2"))
    agent = agent_of(b2048, env, hidden=c.get("hidden", (256, 256)), shared_lambda=c.get("shared"), **c["cfg"])
    agent.rollout_many(env, horizon=16, precision=0)                  # start the window mid-episode
    ro = agent.rollout_many(env, horizon=H, reset=False, precision=0)
    actor_p = agent.params
    critic_p = agent.critic_params if c["cfg"].get("use_critic") else None
    value_head = agent.value_head if c.get("shared") is not None else None
    info = agent.update_from_horizon(ro, precision=c["prec"])
    got = (agent._shared_net.grad if value_head is not None else agent._grad_all).cpu().numpy().copy()
    wro = b2048.symmetry.augment_rollout(ro) if c["cfg"].get("augmentation") else ro
    T, B = wro.T, wro.B
    rewards, flags, _, _ = np_window(wro)
    critic = critic_p is not None or value_head is not None
    values = agent._scratch["values"][: (T + 1) * B].reshape(T + 1, B).cpu().numpy() if critic else None
    lam = c.get("shared") or 0.0
    cfg = agent.agent_config
    v, _, gc, valid = restate(rewards, flags, values, 0.99, lam, int(cfg.critic_loss_type == "huber"), cfg.huber_delta, float(B))
    coef = restate_coef(v, valid, cfg.baseline_mode, T, B)
    dev_coef = agent._scratch["coef"][: T * B].reshape(T, B).cpu().numpy()
    assert rel_err(dev_coef, coef) < (1e-5 if c["prec"] == 0 else 1e-3)
    assert np.array_equal(info["valid_len"].cpu().numpy(), valid)
    ref = torch_grad(agent, wro, coef, gc if critic else None, c.get("obs") == "onehot", actor_p, critic_p, value_head, vc=0.7)
    err = rel_err(got, ref)
    print(f"{case} ({info['precision']}): window gradient vs torch autograd fp32 {err:.2e}")
    assert got.shape == ref.shape and err < c["tol"]


def test_update_from_rollout_still_refuses_windows(b2048):
    env = env_of(b2048, 512, seed=3)
    agent = agent_of(b2048, env, hidden=(32,))
    ro = agent.rollout_many(env, horizon=8)
    with pytest.raises(ValueError):
        agent.update_from_rollout(ro)


def test_two_emulated_ranks_equal_one_process(b2048):
    n, H = 8192, 40
    cfg = dict(baseline_mode="batch_norm", use_critic=True)
    env = env_of(b2048, n, seed=41)
    single = agent_of(b2048, env, **cfg)
    ro = single.rollout_many(env, horizon=H, precision=0)
    ranks = [agent_of(b2048, env_of(b2048, 1, seed=0), **cfg) for _ in range(2)]

    def part(sl):
        return b2048.Rollout(ro.boards[:, sl].contiguous(), ro.flags[:, sl].contiguous(), ro.actions[:, sl].contiguous(),
                             ro.rewards[:, sl].contiguous(), ro.length[sl].contiguous(), H, n_traj=n, auto_reset=True)

    parts = [part(slice(0, n // 2)), part(slice(n // 2, n))]
    bar, slots, sent, errors = threading.Barrier(2), [None, None], [[], []], []

    def allreduce(r):
        def ar(t):
            torch.cuda.synchronize()
            slots[r] = t.clone()
            bar.wait()
            total = slots[0] + slots[1]
            bar.wait()
            t.copy_(total)
            torch.cuda.synchronize()
            sent[r].append(t.numel() * t.element_size())
        return ar

    def run(r):
        try:
            ranks[r].update_from_horizon(parts[r], allreduce=allreduce(r), precision=0)
        except Exception as e:          # noqa: BLE001  (re-raised below)
            errors.append(e)
            bar.abort()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    single.update_from_horizon(ro, precision=0)
    n_grad = single._grad_all.numel() * 4
    assert sent == [[32, n_grad], [32, n_grad]]                      # the baseline sums, then ONE gradient message
    want = single._grad_all.cpu().numpy()
    for a in ranks:
        assert rel_err(a._grad_all.cpu().numpy(), want) < 1e-6
        assert rel_err(a._actor.theta.cpu().numpy(), single._actor.theta.cpu().numpy()) < 1e-6


def test_episode_accounting_matches_oracle_replay(b2048):
    n, seed, H = 33000, 5, 40
    kw = full_env_kwargs("runner_default")
    kw["max_steps"] = 25
    env = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**kw), seed=seed, gid0=3)
    agent = b2048.ReinforceAgent(env, b2048.MLPConfig(hidden_sizes=[32], activation="Sigmoid", init_distribution="XavierNormal"),
                                 b2048.ReinforceAgentConfig(learning_rate=1e-4))
    windows = []
    for k in range(2):
        ro = agent.rollout_many(env, horizon=H, reset=(k == 0))
        windows.append(np_window(ro))
        agent.update_from_horizon(ro)
    got = agent.horizon_episode_stats()
    okw = dict(kw)
    okw.pop("size")
    cfg = oracle.make_cfg(action_mode="buffer", auto_reset=True, **okw)
    st = oracle.reset_many(n, seed, 3, 0)
    carry = np.zeros(n)
    returns, exps = [], []
    for k, (rewards, flags, boards, actions) in enumerate(windows):
        for t in range(H):
            before = st["board"].copy()
            assert (before == boards[t].view(np.uint64)).all()
            o = oracle.step_many(st, cfg, seed, 3, k * H + t + 1, action=actions[t])
            assert (o["reward"] == rewards[t]).all() and (o["flags"] == flags[t + 1]).all()
            carry += o["reward"].astype(np.float64)
            end = (o["flags"] & F_END) != 0
            if end.any():
                moved, _, _, _ = oracle.move_many(before[end], actions[t][end])
                cells = (moved[:, None] >> (4 * np.arange(16, dtype=np.uint64))) & np.uint64(15)
                exps.append(np.maximum(cells.max(1).astype(np.int64), 2))
                returns.append(carry[end].copy())
                carry[end] = 0.0
    returns, exps = np.concatenate(returns), np.concatenate(exps)
    spanning = int(((windows[0][1][H] & F_END) == 0).sum())
    print(f"{returns.size} episodes ended in 2 x {H} steps; {spanning} lanes carried an episode across the window edge")
    assert got["episodes"] == returns.size and spanning > 0
    assert got["avg_reward"] == pytest.approx(returns.mean(), rel=1e-12)
    assert got["max_reward"] == returns.max() and got["min_reward"] == returns.min()
    assert got["max_tile_counts"] == [int((exps == e).sum()) for e in range(4, 13)]
    empty = agent.horizon_episode_stats()                             # reset by the previous call
    assert empty["episodes"] == 0 and np.isnan(empty["avg_reward"]) and sum(empty["max_tile_counts"]) == 0


def test_trainer_horizon_smoke(b2048, tmp_path):
    from b2048 import trainer
    cfg = trainer.merge_config({"env": {"max_steps": 64}, "mlp": {"hidden_sizes": [32, 32]},
                                "agent": {"optimizer": "adam", "learning_rate": 1e-3, "baseline_mode": "batch_norm"},
                                "train": {"batch_size": 2048, "num_batches": 12, "horizon": 32, "out_dir": str(tmp_path)}})
    rows = trainer.training(cfg)
    assert len(rows) == 12 and all(r["steps"] == 32 * 2048 for r in rows)
    assert all(np.isfinite([r["avg_reward"], r["max_reward"], r["min_reward"]]).all() for r in rows[2:])
    files = os.listdir(tmp_path)
    assert "config.json" in files and "final.npz" in files
    assert json.load(open(os.path.join(tmp_path, "config.json")))["train"]["horizon"] == 32
    lines = open(os.path.join(tmp_path, "training_stats.csv")).read().strip().splitlines()
    assert lines[0] == "batch,avg_reward,max_reward,min_reward,max_tile_counts" and len(lines) == 13
    assert [int(l.split(",")[0]) for l in lines[1:]] == list(range(1, 13))
    assert all(len(json.loads(r["max_tile_counts"])) == 9 for r in rows)


def test_horizon_training_raises_the_return(b2048):
    """Adam updates on 64-step windows of 8192 lanes raise the mean return of the completed episodes."""
    n, H = 8192, 64
    env = env_of(b2048, n, seed=99, max_steps=1024)
    agent = agent_of(b2048, env, baseline_mode="batch_norm", optimizer="adam", learning_rate=1e-3, max_grad_norm=1.0)
    env.reset_many()
    means = []
    for it in range(60):
        ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
        agent.update_from_horizon(ro)
        es = agent.horizon_episode_stats()
        means.append((es["episodes"], es["avg_reward"]))
    first = [m for c, m in means[2:12] if c]
    last = [m for c, m in means[-10:] if c]
    print(f"horizon training, 60 windows of {n} x {H}: completed-episode return {np.mean(first):.1f} -> {np.mean(last):.1f}")
    assert np.mean(last) > 1.05 * np.mean(first)
