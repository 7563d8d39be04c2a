"""PPO on fixed-horizon windows on the device (ReinforceAgent.update_ppo, b2048_ppo_minibatches / _logp / _coefficients):
the device partition against the g++ build of csrc/b2048_ppo.cuh, the reduction to update_from_horizon, eight clipped steps
against a PyTorch float32 autograd restatement, two emulated ranks against one process, bootstrapping at truncation,
the trainer's train.ppo section and a short learning run."""
import json
import os
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from helpers import full_env_kwargs, rel_err  # noqa: E402
from test_horizon_gpu import mlp_forward  # noqa: E402
from test_ppo import lib, minibatches  # noqa: E402,F401  (the g++ build of csrc/b2048_ppo.cuh)


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
    base = dict(gamma=0.99, learning_rate=1e-3, baseline_mode="batch_norm", model_seed=5, max_grad_norm=1e9, use_critic=True)
    base.update(cfg)
    mlp = b2048.MLPConfig(hidden_sizes=list(hidden), activation="ReLU", init_distribution="HeNormal")
    if shared_lambda is not None:
        base["use_critic"] = False
        return b2048.SharedTrunkActorCritic(env, mlp, b2048.ReinforceAgentConfig(**base), value_coef=0.7,
                                            gae_lambda=shared_lambda)
    return b2048.ReinforceAgent(env, mlp, b2048.ReinforceAgentConfig(**base))


def theta(agent):
    if hasattr(agent, "_shared_net"):
        return agent._shared_net.theta.detach().cpu().numpy().copy()
    parts = [agent._actor.theta] + ([agent._critic.theta] if agent._critic is not None else [])
    return torch.cat(parts).cpu().numpy().copy()


def test_device_partition_equals_host(b2048, lib):
    n, H, M = 65536, 64, 4
    env = env_of(b2048, n, seed=1)
    agent = agent_of(b2048, env, hidden=(32,))
    for seed, epoch in ((0, 0), (0xC0FFEE123, 3)):
        order, counts = agent.ppo_minibatch_lists(H, n, n, 0, M, seed, epoch)
        want = minibatches(lib, H, n, n, 0, M, seed, epoch).reshape(-1)
        got = np.empty(H * n, np.int32)
        o = order.cpu().numpy()
        got[o] = np.repeat(np.arange(M, dtype=np.int32), counts)
        assert np.array_equal(got, want)
        starts = np.cumsum([0] + counts[:-1])
        for m in range(M):                                       # each list ascends by slot
            assert (np.diff(o[starts[m]: starts[m] + counts[m]]) > 0).all()
        assert counts == [H * n // M] * M


@pytest.mark.parametrize("loss,prec,tol,rtol", [("mse", 0, 1e-5, 1e-6), ("huber", 0, 1e-5, 1e-6), ("mse", "auto", 1e-3, 1e-5),
                                                 ("huber", "auto", 1e-3, 1e-5)])
def test_one_epoch_one_minibatch_is_update_from_horizon(b2048, loss, prec, tol, rtol):
    n, H = 8192, 32
    env = env_of(b2048, n, seed=7)
    agent = agent_of(b2048, env, critic_loss_type=loss, huber_delta=0.5, learning_rate=0.05, critic_learning_rate=0.05)
    agent.rollout_many(env, horizon=16, precision=0)
    ro = agent.rollout_many(env, horizon=H, reset=False, precision=0)
    st = agent.save_state()
    t0 = theta(agent)
    agent.update_from_horizon(ro, precision=prec)
    want = theta(agent) - t0
    agent.load_state(st)
    info = agent.update_ppo(ro, epochs=1, minibatches=1, precision=prec)
    got = theta(agent) - t0
    err = rel_err(got, want)
    print(f"{loss} {prec}: PPO(1 epoch, 1 minibatch) vs update_from_horizon {err:.2e}, r {info['mean_ratio']}")
    assert err < tol
    assert abs(info["mean_ratio"][0] - 1.0) <= rtol and info["clip_fraction"] == [0.0]


def encode(boards, onehot):
    e = torch.stack([(boards >> (4 * i)) & 15 for i in range(16)], 1)
    return torch.nn.functional.one_hot(e, 17).float().reshape(-1, 272) if onehot else e.float() * 0.0625


def restate_ppo(agent, ro, info, lists, eps, veps, cfg, onehot, actor_p, critic_p=None, value_head=None, vc=0.7):
    """The clipped steps in PyTorch float32 autograd on the agent's minibatch lists, logp_old, A and R = A_raw + V_old:
    loss gradients, the global-norm clip and SGD.  Returns the flat parameters after the last step."""
    T = ro.T
    x = encode(ro.boards[:T].reshape(-1), onehot)
    legal = ((ro.flags[:T].reshape(-1).long().unsqueeze(1) >> torch.arange(4, device="cuda")) & 1).bool()
    acts = ro.actions[:T].reshape(-1).long()
    logp_old = info["logp_old"].clone()
    adv = info["advantages"].reshape(-1).double()
    v_old = info["values_old"][:T].reshape(-1).clone()
    R = (info["gae"].reshape(-1) + v_old).double()
    v_old = v_old.double()
    leaf = lambda a: torch.tensor(np.asarray(a, np.float32), device="cuda", requires_grad=True)
    Wa, ba = [leaf(W) for W in actor_p["W"]], [leaf(b) for b in actor_p["b"]]
    pa = [t for pair in zip(Wa, ba) for t in pair]
    if value_head is not None:
        pc = [leaf(value_head["W"]), leaf(value_head["b"])]
    else:
        Wc, bc = [leaf(W) for W in critic_p["W"]], [leaf(b) for b in critic_p["b"]]
        pc = [t for pair in zip(Wc, bc) for t in pair]

    def huber(e):
        d = cfg.huber_delta
        return torch.where(e.abs() <= d, 0.5 * e * e, d * (e.abs() - 0.5 * d)) if cfg.critic_loss_type == "huber" else 0.5 * e * e

    def clip_step(params, grads, lr, sign):
        norm = float(torch.sqrt(sum((g.double() ** 2).sum() for g in grads)))
        c = min(1.0, cfg.max_grad_norm / max(norm, 1e-8))
        with torch.no_grad():
            for p_, g in zip(params, grads):
                p_ += sign * lr * c * g

    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for idx, size in lists:
            h, logits = mlp_forward(Wa, ba, x[idx])
            logp = torch.log_softmax(logits.double().masked_fill(~legal[idx], -1e9), 1).gather(1, acts[idx].unsqueeze(1)).reshape(-1)
            r = torch.exp(logp - logp_old[idx])
            A = adv[idx]
            surr = torch.minimum(r * A, torch.clamp(r, 1 - eps, 1 + eps) * A).sum() / size
            if value_head is not None:
                V = (h @ pc[0] + pc[1]).reshape(-1).double()
            else:
                V = mlp_forward(pc[0::2], pc[1::2], x[idx])[1].reshape(-1).double()
            e = V - R[idx]
            if veps:
                ec = v_old[idx] + torch.clamp(V - v_old[idx], -veps, veps) - R[idx]
                lv = torch.where(ec * ec > e * e, huber(ec), huber(e))
            else:
                lv = huber(e)
            vloss = lv.sum() / size
            if value_head is not None:
                grads = torch.autograd.grad(surr - vc * vloss, pa + pc)
                clip_step(pa + pc, grads, cfg.learning_rate, +1.0)
            else:
                clip_step(pa, torch.autograd.grad(surr, pa), cfg.learning_rate, +1.0)
                clip_step(pc, torch.autograd.grad(vloss, pc), cfg.critic_learning_rate, -1.0)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return torch.cat([p_.detach().reshape(-1) for p_ in pa + pc]).cpu().numpy()


AUTOGRAD_CASES = {
    "critic_mse_fp32": dict(prec=0, tol=1e-4, cfg={}),
    "critic_mse_tc": dict(prec="auto", tol=1e-2, cfg={}),
    "huber_value_clip_fp32": dict(prec=0, tol=1e-4, veps=0.05, cfg=dict(critic_loss_type="huber", huber_delta=0.5)),
    "huber_value_clip_tc": dict(prec="auto", tol=1e-2, veps=0.05, cfg=dict(critic_loss_type="huber", huber_delta=0.5)),
    "shared_trunk_gae_fp32": dict(prec=0, tol=1e-4, shared=0.95, cfg={}),
    "shared_trunk_gae_tc": dict(prec="auto", tol=1e-2, shared=0.95, cfg={}),
    "onehot_256_128_64_tc": dict(prec="auto", tol=1e-2, hidden=(256, 128, 64), obs="onehot", cfg={}),
}


@pytest.mark.parametrize("case", list(AUTOGRAD_CASES))
def test_clipped_steps_vs_torch_autograd(b2048, case):
    c = AUTOGRAD_CASES[case]
    n, H, E, M, eps, seed = 4096, 48, 2, 4, 0.2, 77
    env = env_of(b2048, n, seed=31, obs=c.get("obs", "log2"))
    agent = agent_of(b2048, env, hidden=c.get("hidden", (256, 256)), shared_lambda=c.get("shared"), optimizer="sgd",
                     max_grad_norm=1.0, **c["cfg"])
    agent.rollout_many(env, horizon=16, precision=0)                  # start the window mid-episode
    ro = agent.rollout_many(env, horizon=H, reset=False, precision=0)
    st = agent.save_state()
    actor_p = agent.params
    critic_p = agent.critic_params if c.get("shared") is None else None
    value_head = agent.value_head if c.get("shared") is not None else None
    # the smallest step size (the norm of each clipped SGD step) that makes epoch 2 clip more than 1 % of the samples
    for lr in (0.05, 0.2, 0.5, 1.0, 2.0):
        agent.load_state(st)
        agent.agent_config.learning_rate = agent.agent_config.critic_learning_rate = lr
        info = agent.update_ppo(ro, epochs=E, minibatches=M, clip_eps=eps, value_clip_eps=c.get("veps"), shuffle_seed=seed,
                                precision=c["prec"])
        if info["clip_fraction"][1] > 0.01:
            break
    got = theta(agent)
    assert info["clip_fraction"][1] > 0.01, info["clip_fraction"]
    lists = []
    for e in range(E):
        order, counts = agent.ppo_minibatch_lists(H, n, n, 0, M, seed, e)
        off = np.cumsum([0] + counts)
        lists += [(order[off[m]: off[m + 1]], -(-(m + 1) * H * n // M) + (-m * H * n // M)) for m in range(M)]
    ref = restate_ppo(agent, ro, info, lists, eps, c.get("veps"), agent.agent_config, c.get("obs") == "onehot", actor_p,
                      critic_p, value_head)
    t0 = np.concatenate([np.concatenate([np.asarray(W).reshape(-1), np.asarray(b).reshape(-1)])
                         for W, b in zip(actor_p["W"], actor_p["b"])] +
                        ([np.concatenate([np.asarray(W).reshape(-1), np.asarray(b).reshape(-1)])
                          for W, b in zip(critic_p["W"], critic_p["b"])] if critic_p is not None else
                         [value_head["W"].reshape(-1), value_head["b"].reshape(-1)]))
    err = rel_err(got - t0, ref - t0)
    print(f"{case} ({info['precision']}), step {lr}: clip fraction {info['clip_fraction']}, approx KL {info['approx_kl']}; "
          f"8 steps vs torch autograd {err:.2e}")
    assert err < c["tol"]


def test_two_emulated_ranks_equal_one_process(b2048):
    n, H, E, M = 8192, 40, 2, 3
    cfg = dict(learning_rate=0.01, critic_learning_rate=0.01, max_grad_norm=1.0)
    env = env_of(b2048, n, seed=41)
    single = agent_of(b2048, env, **cfg)
    ro = single.rollout_many(env, horizon=H, precision=0)
    ranks = [agent_of(b2048, env_of(b2048, 1, seed=0), **cfg) for _ in range(2)]
    cut = 3000                                                         # uneven shards

    def part(sl):
        return b2048.Rollout(ro.boards[:, sl].contiguous(), ro.flags[:, sl].contiguous(), ro.actions[:, sl].contiguous(),
                             ro.rewards[:, sl].contiguous(), ro.length[sl].contiguous(), H, n_traj=n, auto_reset=True,
                             gid0=sl.start)

    parts = [part(slice(0, cut)), part(slice(cut, n))]
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
            ranks[r].update_ppo(parts[r], epochs=E, minibatches=M, shuffle_seed=5, allreduce=allreduce(r), precision=0)
        except Exception as e:          # noqa: BLE001  (re-raised below)
            errors.append(e)
            bar.abort()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    single.update_ppo(ro, epochs=E, minibatches=M, shuffle_seed=5, precision=0)
    n_grad = single._grad_all.numel() * 4
    assert sent == [[32] + [n_grad] * (E * M)] * 2                     # the baseline sums, then one message per step
    want = theta(single)
    for a in ranks:
        assert rel_err(theta(a), want) < 1e-6


def test_bootstrap_truncation_gives_the_horizon_advantages(b2048):
    n, H = 8192, 64
    env = env_of(b2048, n, seed=13, max_steps=25)
    agent = agent_of(b2048, env)
    ro = agent.rollout_many(env, horizon=H, precision="auto")
    assert ((ro.flags[1:] & 0x60) == 0x40).any()
    st = agent.save_state()
    want = agent.update_from_horizon(ro, bootstrap_truncation=True)["advantages"].clone()
    agent.load_state(st)
    got = agent.update_ppo(ro, bootstrap_truncation=True)["advantages"]
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    agent.load_state(st)
    plain = agent.update_ppo(ro)["advantages"]
    assert not torch.equal(plain, want)


def test_trainer_ppo(b2048, tmp_path):
    from b2048 import trainer
    cfg = trainer.merge_config({"env": {"max_steps": 64}, "mlp": {"hidden_sizes": [32, 32]},
                                "agent": {"optimizer": "adam", "learning_rate": 1e-3, "baseline_mode": "batch_norm",
                                          "use_critic": True},
                                "train": {"batch_size": 2048, "num_batches": 6, "horizon": 32, "out_dir": str(tmp_path),
                                          "ppo": {"epochs": 2, "minibatches": 2, "value_clip_eps": 0.5}}})
    rows = trainer.training(cfg)
    assert len(rows) == 6 and all(r["steps"] == 32 * 2048 for r in rows) and all(np.isfinite(r["grad_norm"]) for r in rows)
    files = os.listdir(tmp_path)
    assert "config.json" in files and "final.npz" in files and "final_checkpoint.npz" in files
    assert json.load(open(os.path.join(tmp_path, "config.json")))["train"]["ppo"]["epochs"] == 2
    lines = open(os.path.join(tmp_path, "training_stats.csv")).read().strip().splitlines()
    assert lines[0] == "batch,avg_reward,max_reward,min_reward,max_tile_counts" and len(lines) == 7
    bad = trainer.merge_config({"agent": {"use_critic": True}, "train": {"ppo": {"epochs": 2}, "out_dir": None}})
    with pytest.raises(ValueError, match="horizon"):
        trainer.training(bad)


def test_ppo_training_raises_the_return(b2048):
    """40 PPO windows of 8192 x 64 with Adam raise the mean return of the completed episodes."""
    n, H = 8192, 64
    env = env_of(b2048, n, seed=99, max_steps=1024)
    agent = agent_of(b2048, env, optimizer="adam", learning_rate=3e-4, critic_learning_rate=1e-3, max_grad_norm=1.0)
    env.reset_many()
    means = []
    for it in range(40):
        ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
        agent.update_ppo(ro, epochs=4, minibatches=4, shuffle_seed=it)
        es = agent.horizon_episode_stats()
        means.append((es["episodes"], es["avg_reward"]))
    first = [m for c, m in means[2:10] if c]
    last = [m for c, m in means[-8:] if c]
    print(f"PPO training, 40 windows of {n} x {H}: completed-episode return {np.mean(first):.1f} -> {np.mean(last):.1f}")
    assert np.mean(last) > 1.05 * np.mean(first)
