"""Bootstrapping at truncation on the device (b2048_replay_pre_reset, b2048_fold_bootstrap, update_from_horizon /
update_from_rollout(bootstrap_truncation=True)): the replayed boards against the step kernel and the oracle, the targets
against the NumPy restatement with V(s') at the truncated boundaries, the no-op cases, the gradient against PyTorch float32
autograd, two emulated ranks, augmentation, whole episodes, the refusals and the trainer key."""
import json
import os
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle  # noqa: E402
from helpers import full_env_kwargs, rel_err  # noqa: E402
from test_horizon_gpu import mlp_forward, np_window, restate_coef, torch_grad  # noqa: E402
from test_truncation_bootstrap import restate_boot, trunc_only  # noqa: E402
from test_horizon_targets import restate  # noqa: E402

F_DONE, F_TRUNC = 0x20, 0x40
GAMMA = 0.99


@pytest.fixture(scope="module")
def b2048():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import b2048 as m
    return m


def env_kw(max_steps):
    kw = full_env_kwargs("runner_default")
    kw["max_steps"] = max_steps
    return kw


def env_of(b2048, n, seed, max_steps=25, gid0=7):
    return b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**env_kw(max_steps)), seed=seed, gid0=gid0)


def agent_of(b2048, env, shared_lambda=None, **cfg):
    base = dict(gamma=GAMMA, learning_rate=1e-3, baseline_mode="batch", model_seed=5, max_grad_norm=1e9, use_critic=True)
    base.update(cfg)
    mlp = b2048.MLPConfig(hidden_sizes=[256, 256], activation="ReLU", init_distribution="HeNormal")
    if shared_lambda is not None:
        return b2048.SharedTrunkActorCritic(env, mlp, b2048.ReinforceAgentConfig(**base), value_coef=0.7,
                                            gae_lambda=shared_lambda)
    return b2048.ReinforceAgent(env, mlp, b2048.ReinforceAgentConfig(**base))


def boot_grid(info, T, B):
    """V(s') at the bootstrapped slots of a [T, B] window, zero elsewhere."""
    g = np.zeros(T * B, np.float32)
    g[info["bootstrap_slots"].cpu().numpy()] = info["bootstrap_values"].cpu().numpy()
    return g.reshape(T, B)


@pytest.mark.parametrize("precision", [1, 0])
def test_replay_equals_step_kernel_and_oracle(b2048, precision):
    """65,536 lanes x 64 steps with max_steps = 25, on the fused tensor-core rollout (1) and the loop (0): the replayed
    boards are b2048_step_many with auto-reset off on (boards[t], actions[t]) at counter t0 + t + 1, and the oracle's step."""
    n, H = 65536, 64
    env = env_of(b2048, n, seed=21)
    agent = agent_of(b2048, env, use_critic=False)
    agent.rollout_many(env, horizon=8, precision=precision)           # the window starts at t0 = 8, mid-episode
    ro = agent.rollout_many(env, horizon=H, reset=False, precision=precision)
    assert (ro.seed, ro.gid0, ro.t0) == (env.seed, 7, 8)
    rewards, flags, boards, actions = np_window(ro)
    ends = flags[1:] & (F_DONE | F_TRUNC)
    assert (ends == F_DONE).sum() > 0 and (ends == F_TRUNC).sum() > 0
    slots, nxt = agent._truncated_window_steps(ro)
    slots, nxt = slots.cpu().numpy(), nxt.cpu().numpy().view(np.uint64)
    assert np.array_equal(slots, np.flatnonzero(ends == F_TRUNC))
    ts, bs = slots // n, slots % n
    step_env = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**env_kw(None)), seed=ro.seed, gid0=ro.gid0, track_state=False)
    cfg = oracle.make_cfg(action_mode="buffer", auto_reset=False, max_steps=None)
    want_dev = np.zeros(slots.size, np.uint64)
    want_orc = np.zeros(slots.size, np.uint64)
    for t in range(H):
        sel = ts == t
        step_env.board = ro.boards[t].clone()
        step_env.t = ro.t0 + t
        step_env.step_many(ro.actions[t].contiguous(), action_mode="buffer", auto_reset=False)
        want_dev[sel] = step_env.board.cpu().numpy().view(np.uint64)[bs[sel]]
        st = dict(board=boards[t].view(np.uint64).copy(), score=np.zeros(n, np.uint32), step=np.zeros(n, np.uint32),
                  max_exp=np.full(n, 2, np.uint8), flags=np.zeros(n, np.uint8))
        oracle.step_many(st, cfg, ro.seed, ro.gid0, ro.t0 + t + 1, action=actions[t])
        want_orc[sel] = st["board"][bs[sel]]
    assert np.array_equal(nxt, want_dev) and np.array_equal(nxt, want_orc)
    after = boards[ts + 1, bs].view(np.uint64)                        # the reset boards that replaced s'
    assert (nxt != after).mean() > 0.99


@pytest.mark.parametrize("lam,huber", [(0.0, 0), (0.0, 1), (0.95, 0)])
def test_window_targets_equal_restatement(b2048, lam, huber):
    n, H = 16384, 64
    env = env_of(b2048, n, seed=23)
    agent = agent_of(b2048, env, critic_loss_type="huber" if huber else "mse", huber_delta=1.5)
    agent.gae_lambda = lam
    ro = agent.rollout_many(env, horizon=H, precision=0)
    cp = agent.critic_params
    info = agent.update_from_horizon(ro, precision=0, bootstrap_truncation=True)
    rewards, flags, _, _ = np_window(ro)
    values = agent._scratch["values"][: (H + 1) * n].reshape(H + 1, n).cpu().numpy()
    boot = boot_grid(info, H, n)
    assert np.array_equal(info["bootstrap_slots"].cpu().numpy(), np.flatnonzero(trunc_only(flags)))
    rv, rtd, rgc, _ = restate_boot(rewards, flags, values, boot, GAMMA, lam, huber, 1.5, float(n))
    got = {"td": info["td"], "gae": agent._scratch["gae"][: H * n], "gcoef": agent._scratch["gcoef"][: H * n]}
    for name, want in (("td", rtd), ("gae", rv), ("gcoef", rgc)):
        assert np.array_equal(got[name].reshape(H, n).cpu().numpy().view(np.uint32), want.view(np.uint32)), name
    # V(s') is the critic's value of the replayed boards
    bb = info["bootstrap_boards"]
    x = torch.stack([(bb >> (4 * i)) & 15 for i in range(16)], 1).float() * 0.0625
    _, V = mlp_forward([torch.tensor(W, device="cuda") for W in cp["W"]], [torch.tensor(b, device="cuda") for b in cp["b"]], x)
    assert rel_err(info["bootstrap_values"].cpu().numpy(), V.reshape(-1).cpu().numpy()) < 1e-5


def test_no_truncation_and_flag_off_are_unchanged(b2048):
    """Without truncations (max_steps=None) bootstrap on gives bit-identical parameters; with the flag off the update is the
    default update and its TD errors are the unbootstrapped restatement.  128 lanes x 16 steps = 2048 samples on the fp32
    kernels with no baseline statistics: every gradient element is then accumulated once, so two updates agree bit for bit."""
    n, H = 128, 16
    for max_steps in (None, 25):
        env = env_of(b2048, n, seed=25, max_steps=max_steps)
        agent = agent_of(b2048, env, baseline_mode="off", optimizer="adam")
        agent.rollout_many(env, horizon=16, precision=0)              # the window holds step 25 of most episodes
        ro = agent.rollout_many(env, horizon=H, reset=False, precision=0)
        has_trunc = bool(trunc_only(ro.flags[: H + 1].cpu().numpy()).any())
        assert has_trunc == (max_steps is not None)
        st = agent.save_state()
        results = []
        for kw in ({}, dict(bootstrap_truncation=False), dict(bootstrap_truncation=True)):
            agent.load_state(st)
            info = agent.update_from_horizon(ro, precision=0, **kw)
            results.append((agent._actor.theta.clone(), agent._critic.theta.clone(), info["td"].clone()))
            if not kw.get("bootstrap_truncation") and max_steps is not None:
                rewards, flags, _, _ = np_window(ro)
                values = agent._scratch["values"][: (H + 1) * n].reshape(H + 1, n).cpu().numpy()
                assert np.array_equal(info["td"].cpu().numpy().view(np.uint32),
                                      restate(rewards, flags, values, GAMMA, 0.0, 0, 1.0, float(n))[1].view(np.uint32))
        for a, b in zip(results[0], results[1]):
            assert torch.equal(a, b)
        same = all(torch.equal(a, b) for a, b in zip(results[0], results[2]))
        assert same == (max_steps is None)


GRAD_CASES = {
    "critic_fp32": dict(prec=0, tol=1e-3, cfg=dict(critic_loss_type="huber", huber_delta=0.5)),
    "critic_tc": dict(prec="auto", tol=1e-2, cfg=dict(baseline_mode="batch_norm")),
    "shared_trunk_fp32": dict(prec=0, tol=1e-3, shared=0.95, cfg=dict(baseline_mode="batch_norm")),
    "shared_trunk_tc": dict(prec="auto", tol=1e-2, shared=0.0, cfg=dict()),
}


@pytest.mark.parametrize("case", list(GRAD_CASES))
def test_bootstrapped_gradient_vs_torch_autograd(b2048, case):
    c = GRAD_CASES[case]
    n, H = 4096, 48
    env = env_of(b2048, n, seed=31)
    agent = agent_of(b2048, env, shared_lambda=c.get("shared"), **c["cfg"])
    agent.rollout_many(env, horizon=16, precision=0)
    ro = agent.rollout_many(env, horizon=H, reset=False, precision=0)
    actor_p = agent.params
    shared = c.get("shared") is not None
    critic_p = None if shared else agent.critic_params
    value_head = agent.value_head if shared else None
    info = agent.update_from_horizon(ro, precision=c["prec"], bootstrap_truncation=True)
    assert info["bootstrap_slots"].numel() > 0
    got = (agent._shared_net.grad if shared else agent._grad_all).cpu().numpy().copy()
    rewards, flags, _, _ = np_window(ro)
    values = agent._scratch["values"][: (H + 1) * n].reshape(H + 1, n).cpu().numpy()
    cfg = agent.agent_config
    v, _, gc, valid = restate_boot(rewards, flags, values, boot_grid(info, H, n), GAMMA, c.get("shared") or 0.0,
                                   int(cfg.critic_loss_type == "huber"), cfg.huber_delta, float(n))
    coef = restate_coef(v, valid, cfg.baseline_mode, H, n)
    dev_coef = agent._scratch["coef"][: H * n].reshape(H, n).cpu().numpy()
    assert rel_err(dev_coef, coef) < (1e-5 if c["prec"] == 0 else 1e-3)
    ref = torch_grad(agent, ro, coef, gc, False, actor_p, critic_p, value_head, vc=0.7)
    err = rel_err(got, ref)
    print(f"{case} ({info['precision']}): bootstrapped window gradient vs torch autograd fp32 {err:.2e}")
    assert got.shape == ref.shape and err < c["tol"]


def test_two_emulated_ranks_equal_one_process(b2048):
    n, H = 8192, 40
    cfg = dict(baseline_mode="batch_norm")
    env = env_of(b2048, n, seed=41)
    single = agent_of(b2048, env, **cfg)
    ro = single.rollout_many(env, horizon=H, precision=0)
    ranks = [agent_of(b2048, env_of(b2048, 1, seed=0), **cfg) for _ in range(2)]

    def part(lo, hi):
        sl = slice(lo, hi)
        return b2048.Rollout(ro.boards[:, sl].contiguous(), ro.flags[:, sl].contiguous(), ro.actions[:, sl].contiguous(),
                             ro.rewards[:, sl].contiguous(), ro.length[sl].contiguous(), H, n_traj=n, auto_reset=True,
                             seed=ro.seed, gid0=ro.gid0 + lo, t0=ro.t0)

    parts = [part(0, n // 2), part(n // 2, n)]
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
            ranks[r].update_from_horizon(parts[r], allreduce=allreduce(r), precision=0, bootstrap_truncation=True)
        except Exception as e:          # noqa: BLE001  (re-raised below)
            errors.append(e)
            bar.abort()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    info = single.update_from_horizon(ro, precision=0, bootstrap_truncation=True)
    assert info["bootstrap_slots"].numel() > 0
    n_grad = single._grad_all.numel() * 4
    assert sent == [[32, n_grad], [32, n_grad]]                      # no message added by the bootstrap
    want = single._grad_all.cpu().numpy()
    for a in ranks:
        assert rel_err(a._grad_all.cpu().numpy(), want) < 1e-6
        assert rel_err(a._actor.theta.cpu().numpy(), single._actor.theta.cpu().numpy()) < 1e-6
        assert rel_err(a._critic.theta.cpu().numpy(), single._critic.theta.cpu().numpy()) < 1e-6


def test_augmented_columns_fold_the_variant_value(b2048):
    from b2048 import symmetry
    n, H = 4096, 40
    env = env_of(b2048, n, seed=43)
    agent = agent_of(b2048, env, augmentation=True)
    ro = agent.rollout_many(env, horizon=H, precision=0)
    slots0, nxt0 = agent._truncated_window_steps(ro)
    K = slots0.numel()
    assert K > 0
    variants = [symmetry.transform_boards(nxt0, v) for v in range(8)]
    Vs = [torch.empty(K, dtype=torch.float32, device="cuda") for _ in range(8)]
    for sv, V in zip(variants, Vs):                                   # the critic before the update takes its step
        agent._values(sv, V, 0)
    info = agent.update_from_horizon(ro, precision=0, bootstrap_truncation=True)
    wro = symmetry.augment_rollout(ro)
    B8 = 8 * n
    t, b = slots0 // n, slots0 % n
    values = agent._scratch["values"][: (H + 1) * B8].reshape(H + 1, B8)
    td = info["td"].reshape(H, B8)
    g = torch.tensor(GAMMA, dtype=torch.float32, device="cuda")
    for v, (sv, V) in enumerate(zip(variants, Vs)):
        col = v * n + b
        assert torch.equal(info["bootstrap_slots"][v * K: (v + 1) * K], t * B8 + col)
        assert torch.equal(info["bootstrap_boards"][v * K: (v + 1) * K], sv)
        assert torch.equal(info["bootstrap_values"][v * K: (v + 1) * K], V)
        want = (wro.rewards[t, col] + g * V) - values[t, col]
        assert torch.equal(td[t, col], want)


@pytest.mark.parametrize("max_steps", [25, 100])
@pytest.mark.parametrize("precision", [1, 0])
def test_whole_episode_bootstrap(b2048, precision, max_steps):
    """update_from_rollout on run-to-termination episodes (the compact fused rollout and the loop): the last delta of a
    truncated lane is r + gamma V(boards[len]) - V(s_{len-1}); every other delta, among them the last one of a lane whose
    game ended, is unchanged.  With max_steps = 25 every lane is truncated; with 100 some games end first."""
    n = 8192
    env = env_of(b2048, n, seed=47, max_steps=max_steps)
    agent = agent_of(b2048, env)
    ro = agent.rollout_many(env, precision=precision)
    T = ro.T
    L = ro.length.long()
    fin = ro.flags[: T + 1].gather(0, L.unsqueeze(0)).reshape(-1) & (F_DONE | F_TRUNC)
    trunc = fin == F_TRUNC
    assert trunc.any() and (max_steps == 25 or (fin == F_DONE).any())
    st = agent.save_state()
    off = agent.update_from_rollout(ro, precision=0)
    td_off = off["td"].clone()
    agent.load_state(st)
    on = agent.update_from_rollout(ro, precision=0, bootstrap_truncation=True)
    values = agent._scratch["values"][: T * n].reshape(T, n)
    lanes = torch.nonzero(trunc).reshape(-1)
    assert torch.equal(on["bootstrap_slots"], (L[lanes] - 1) * n + lanes)
    assert torch.equal(on["bootstrap_boards"], ro.boards[: T + 1].gather(0, L.unsqueeze(0)).reshape(-1)[lanes])
    td_on = on["td"].reshape(T, n)
    last = L[lanes] - 1
    g = torch.tensor(GAMMA, dtype=torch.float32, device="cuda")
    want = (ro.rewards[last, lanes] + g * on["bootstrap_values"]) - values[last, lanes]
    assert torch.equal(td_on[last, lanes], want)
    mask = torch.ones((T, n), dtype=torch.bool, device="cuda")
    mask[last, lanes] = False
    assert torch.equal(td_on[mask], td_off.reshape(T, n)[mask])

    # lanes cut by rollout_many's own cap carry no TRUNC flag: nothing is bootstrapped
    env2 = env_of(b2048, n, seed=48, max_steps=max_steps)
    ro2 = agent.rollout_many(env2, max_steps=20, precision=precision)
    assert (ro2.length == 20).any()
    st = agent.save_state()
    td_off = agent.update_from_rollout(ro2, precision=0)["td"].clone()
    agent.load_state(st)
    on = agent.update_from_rollout(ro2, precision=0, bootstrap_truncation=True)
    assert "bootstrap_slots" not in on and torch.equal(on["td"], td_off)


def test_refusals_on_real_agents(b2048):
    env = env_of(b2048, 512, seed=3)
    no_critic = agent_of(b2048, env, use_critic=False)
    ro = no_critic.rollout_many(env, horizon=8)
    with pytest.raises(ValueError, match="bootstrap_truncation"):
        no_critic.update_from_horizon(ro, bootstrap_truncation=True)
    with pytest.raises(ValueError, match="bootstrap_truncation"):
        no_critic.update_from_rollout(no_critic.rollout_many(env), bootstrap_truncation=True)
    critic = agent_of(b2048, env)
    ro = critic.rollout_many(env, horizon=8)
    ro.seed = None
    with pytest.raises(ValueError, match="bootstrap_truncation"):
        critic.update_from_horizon(ro, bootstrap_truncation=True)


@pytest.mark.parametrize("horizon", [32, None])
def test_trainer_bootstrap_truncation(b2048, tmp_path, horizon):
    from b2048 import trainer
    train = {"batch_size": 2048, "num_batches": 12 if horizon else 4, "horizon": horizon, "out_dir": str(tmp_path),
             "bootstrap_truncation": True, "checkpoint_every": 4}
    cfg = trainer.merge_config({"env": {"max_steps": 64}, "mlp": {"hidden_sizes": [32, 32]},
                                "agent": {"optimizer": "adam", "learning_rate": 1e-3, "baseline_mode": "batch_norm",
                                          "use_critic": True, "critic_learning_rate": 1e-3},
                                "train": train})
    rows = trainer.training(cfg)
    assert len(rows) == train["num_batches"] and all(np.isfinite(r["grad_norm"]) for r in rows)
    files = os.listdir(tmp_path)
    assert {"config.json", "final.npz", "final_checkpoint.npz", "checkpoint.npz", "training_stats.csv"} <= set(files)
    assert json.load(open(os.path.join(tmp_path, "config.json")))["train"]["bootstrap_truncation"] is True
    lines = open(os.path.join(tmp_path, "training_stats.csv")).read().strip().splitlines()
    assert lines[0] == "batch,avg_reward,max_reward,min_reward,max_tile_counts" and len(lines) == train["num_batches"] + 1
    if horizon:
        assert all(r["steps"] == 32 * 2048 for r in rows)
