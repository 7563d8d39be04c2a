"""The entropy bonus on the device (b2048_mlp_backward_entropy and the entropy_coef of the updates): ecoef = 0 against
b2048_mlp_backward on every kernel family, the entropy term and both terms against a PyTorch float32 autograd restatement,
whole updates against the restatement of their entropy part, two emulated ranks against one process, the trainer key and
the direction of the bonus."""
import ctypes as C
import sys
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from helpers import full_env_kwargs, rel_err  # noqa: E402

NO_UPDATE_PIPE = 5
PIPE_N = 1 << 17                     # >= 4 x 148 tiles of 128 samples: the persistent update pipeline


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
    base = dict(gamma=0.99, learning_rate=1e-2, critic_learning_rate=1e-2, baseline_mode="batch_norm", model_seed=5,
                max_grad_norm=1e9, use_critic=True)
    base.update(cfg)
    mlp = b2048.MLPConfig(hidden_sizes=list(hidden), activation="ReLU", init_distribution="HeNormal")
    if shared_lambda is not None:
        base["use_critic"] = False
        return b2048.SharedTrunkActorCritic(env, mlp, b2048.ReinforceAgentConfig(**base), value_coef=0.7,
                                            gae_lambda=shared_lambda)
    return b2048.ReinforceAgent(env, mlp, b2048.ReinforceAgentConfig(**base))


def b2048_agent_module(agent):
    for k in type(agent).__mro__:
        if k.__name__ == "ReinforceAgent":
            return k.__module__
    raise AssertionError


def backward(agent, boards, flags, acts, cf, ecf, prec, entropy=True, chunk=1 << 20):
    """(policy gradient, sum H) of one b2048_mlp_backward[_entropy] call on the actor."""
    ra = sys.modules[b2048_agent_module(agent)]
    lib, net, n = agent._lib, agent._actor, boards.numel()
    wsf = int(lib.b2048_backward_workspace_floats(C.byref(net.desc), min(chunk, n)))
    ws = torch.empty(wsf, dtype=torch.float32, device="cuda")
    es = torch.zeros(1, dtype=torch.float64, device="cuda")
    net.grad.zero_()
    if entropy:
        st = lib.b2048_mlp_backward_entropy(agent._h, ra._ptr(boards), ra._ptr(flags), ra._ptr(acts), ra._ptr(cf), ra._ptr(ecf),
                                            C.byref(net.desc), ra._ptr(net.grad), n, ra._ptr(ws), wsf, min(chunk, n), prec,
                                            ra._ptr(es), ra._stream())
    else:
        st = lib.b2048_mlp_backward(agent._h, ra._ptr(boards), ra._ptr(flags), ra._ptr(acts), ra._ptr(cf), C.byref(net.desc),
                                    ra._ptr(net.grad), n, 0, ra._ptr(ws), wsf, min(chunk, n), prec, ra._stream())
    assert st == 0, lib.b2048_last_error()
    torch.cuda.synchronize()
    return net.grad.double().cpu().numpy(), float(es[0])


def encode(boards, onehot):
    e = torch.stack([(boards >> (4 * i)) & 15 for i in range(16)], 1)
    return torch.nn.functional.one_hot(e, 17).float().reshape(-1, 272) if onehot else e.float() * 0.0625


def torch_objective_grad(params, boards, flags, acts, cf, ecf, onehot):
    """float32 autograd of J = sum cf log pi(a|s) + sum ecf H over the legal actions; (flat gradient W_0, b_0, ..., sum H)."""
    leaf = lambda a: torch.tensor(np.asarray(a, np.float32), device="cuda", requires_grad=True)
    Ws, bs = [leaf(W) for W in params["W"]], [leaf(b) for b in params["b"]]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        h = encode(boards, onehot)
        for W, b in zip(Ws[:-1], bs[:-1]):
            h = torch.relu(h @ W + b)
        logits = h @ Ws[-1] + bs[-1]
        legal = ((flags.long().unsqueeze(1) >> torch.arange(4, device="cuda")) & 1).bool()
        logp = torch.log_softmax(logits.masked_fill(~legal, -1e9), 1)
        p = logp.exp()
        H = -(torch.where(legal, p * logp, torch.zeros_like(p))).sum(1)
        J = (cf * logp.gather(1, acts.long().unsqueeze(1)).reshape(-1)).sum() + (ecf * H).sum()
        gs = torch.autograd.grad(J, [t for pair in zip(Ws, bs) for t in pair])
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return torch.cat([g.reshape(-1) for g in gs]).double().cpu().numpy(), float(H.double().sum())


def batch(b2048, n, seed, obs="log2", hidden=(256, 256)):
    """A rollout-derived batch (fp32 policy, masks with 1-4 legal moves) and an agent."""
    H = 32
    env = env_of(b2048, max(n // H, 1), seed, obs=obs)
    agent = agent_of(b2048, env, hidden=hidden)
    ro = agent.rollout_many(env, horizon=H, precision=0)
    boards = ro.boards[:H].reshape(-1)[:n].contiguous()
    flags = ro.flags[:H].reshape(-1)[:n].contiguous()
    acts = ro.actions[:H].reshape(-1)[:n].contiguous()
    legal = (flags.long() & 15)
    assert bool((legal != 0).all())
    return agent, boards, flags, acts


def coefs(n, seed, zero_mean=True):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cf = torch.randn(n, generator=g, device="cuda") * (1.0 / n)
    if zero_mean:
        cf -= cf.mean()
    ecf = torch.full((n,), 0.01 / n, device="cuda")
    return cf, ecf


PATHS = {   # name: (n, obs, hidden, precision, chunked)
    "fp32": (65536, "log2", (256, 256), 0, False),
    "hp_pipeline": (PIPE_N, "log2", (256, 256), 3, False),
    "hp_chunked": (65536, "log2", (256, 256), 3, True),
    "generic_onehot": (65536, "onehot", (256, 128, 64), 3, False),
}


@pytest.mark.parametrize("path", list(PATHS))
def test_zero_ecoef_equals_mlp_backward(b2048, path):
    n, obs, hidden, prec, chunked = PATHS[path]
    agent, boards, flags, acts = batch(b2048, n, seed=3, obs=obs, hidden=hidden)
    if chunked:
        agent._lib.b2048_debug_set(agent._h, NO_UPDATE_PIPE, 1)
    cf, _ = coefs(n, 1)
    zero = torch.zeros(n, device="cuda")
    want, _ = backward(agent, boards, flags, acts, cf, zero, prec, entropy=False)
    got, hs = backward(agent, boards, flags, acts, cf, zero, prec)
    assert hs > 0.0
    err = rel_err(got, want)
    print(f"{path}: ecoef = 0 vs b2048_mlp_backward {err:.2e}")
    assert err <= 1e-6
    if path == "hp_pipeline":
        # the pipeline's dW partials meet in float atomics, whose order varies run to run for both entry points
        again, _ = backward(agent, boards, flags, acts, cf, zero, prec)
        plain_again, _ = backward(agent, boards, flags, acts, cf, zero, prec, entropy=False)
        print(f"run to run: entropy {rel_err(again, got):.2e}, b2048_mlp_backward {rel_err(plain_again, want):.2e}")
        assert rel_err(again, got) <= 1e-6 and rel_err(plain_again, want) <= 1e-6


@pytest.mark.parametrize("path,tol", [("fp32", 1e-5), ("hp_pipeline", 1e-3), ("hp_chunked", 1e-3), ("generic_onehot", 3e-3)])
@pytest.mark.parametrize("terms", ["entropy", "both"])
def test_against_torch_autograd(b2048, path, tol, terms):
    n, obs, hidden, prec, chunked = PATHS[path]
    agent, boards, flags, acts = batch(b2048, n, seed=5, obs=obs, hidden=hidden)
    if chunked:
        agent._lib.b2048_debug_set(agent._h, NO_UPDATE_PIPE, 1)
    cf, ecf = coefs(n, 2)
    if terms == "entropy":
        cf = torch.zeros(n, device="cuda")
    got, hs = backward(agent, boards, flags, acts, cf, ecf, prec)
    want, hw = torch_objective_grad(agent.params, boards, flags, acts, cf, ecf, obs == "onehot")
    err = rel_err(got, want)
    print(f"{path} {terms}: vs autograd {err:.2e}, sum H {hs:.6e} vs {hw:.6e}")
    assert err <= tol
    assert abs(hs - hw) <= 1e-5 * abs(hw)


def test_precision_1_is_refused(b2048):
    agent, boards, flags, acts = batch(b2048, 8192, seed=1)
    cf, ecf = coefs(8192, 1)
    ra = sys.modules[b2048_agent_module(agent)]
    net = agent._actor
    wsf = int(agent._lib.b2048_backward_workspace_floats(C.byref(net.desc), 8192))
    ws = torch.empty(wsf, dtype=torch.float32, device="cuda")
    st = agent._lib.b2048_mlp_backward_entropy(agent._h, ra._ptr(boards), ra._ptr(flags), ra._ptr(acts), ra._ptr(cf), ra._ptr(ecf),
                                               C.byref(net.desc), ra._ptr(net.grad), 8192, ra._ptr(ws), wsf, 8192, 1, None,
                                               ra._stream())
    assert st != 0


# ---------------------------------------------------------------- whole updates
def flat_theta(agent):
    if hasattr(agent, "_shared_net"):
        return agent._shared_net.theta.double().cpu().numpy().copy()
    return agent._actor.theta.double().cpu().numpy().copy()


def samples_of(ro, length=None):
    T = ro.T
    b, f, a = (x[:T].reshape(-1) for x in (ro.boards, ro.flags, ro.actions))
    if length is None:
        return b, f, a
    live = torch.nonzero((torch.arange(T, device="cuda").unsqueeze(1) < length.unsqueeze(0)).reshape(-1)).reshape(-1)
    return b[live], f[live], a[live]


@pytest.mark.parametrize("case", ["horizon_critic", "horizon_onehot", "horizon_reinforce", "rollout_critic", "ppo_critic",
                                  "horizon_augmented"])
def test_update_entropy_part_vs_autograd(b2048, case):
    """The actor gradient of the update is linear in its terms: g(beta) - g(0) = the restated entropy gradient of the update's
    samples with their weights ecoef (the policy term is the same in both runs)."""
    beta, lr = 0.05, 1e-2
    obs, hidden = ("onehot", (256, 128, 64)) if case == "horizon_onehot" else ("log2", (256, 256))
    n, T = 8192, 32
    env = env_of(b2048, n, seed=17, obs=obs)
    agent = agent_of(b2048, env, hidden=hidden, use_critic=case != "horizon_reinforce", learning_rate=lr,
                     augmentation=case == "horizon_augmented", baseline_mode="batch" if case == "rollout_critic" else "batch_norm")
    if case == "rollout_critic":
        ro = agent.rollout_many(env, max_steps=64, precision=0)
    else:
        agent.rollout_many(env, horizon=8, precision=0)
        ro = agent.rollout_many(env, horizon=T, reset=False, precision=0)
    st = agent.save_state()
    params0 = agent.params

    def run(b):
        agent.load_state(st)
        if case == "rollout_critic":
            info = agent.update_from_rollout(ro, precision=0, entropy_coef=b)
        elif case == "ppo_critic":
            info = agent.update_ppo(ro, epochs=1, minibatches=1, precision=0, entropy_coef=b)
        else:
            info = agent.update_from_horizon(ro, precision=0, entropy_coef=b)
        return agent._actor.grad.double().cpu().numpy().copy(), info      # the update's (unclipped) actor gradient

    d0, info0 = run(0.0)
    d1, info1 = run(beta)
    assert "entropy" not in info0
    aug = agent.agent_config.augmentation
    src = agent._augment_rollout(ro) if aug else ro
    n_traj = src.B
    if case == "rollout_critic":
        b, f, a = samples_of(src, src.length)
        L = src.length.long().unsqueeze(0).expand(src.T, -1).reshape(-1)
        live = torch.nonzero((torch.arange(src.T, device="cuda").unsqueeze(1) < src.length.unsqueeze(0)).reshape(-1)).reshape(-1)
        ecf = (beta * (1.0 / (L[live].float() * n_traj))).float()
    elif case == "horizon_reinforce":
        valid = info1["valid_len"]
        b, f, a = samples_of(src, valid)
        ecf = torch.full((b.numel(),), beta / (src.T * n_traj), device="cuda")
    else:
        b, f, a = samples_of(src)
        ecf = torch.full((b.numel(),), beta / (src.T * n_traj), device="cuda")
    g, hsum = torch_objective_grad(params0, b, f, a, torch.zeros(b.numel(), device="cuda"), ecf, obs == "onehot")
    na = g.size
    assert d1.size == na
    err = rel_err(d1 - d0, g)
    mean_h = info1["entropy"][0] if case == "ppo_critic" else info1["entropy"]
    print(f"{case}: entropy part vs autograd {err:.2e}; mean H {mean_h:.6f} vs {hsum / b.numel():.6f}")
    assert err <= 1e-3
    assert abs(mean_h - hsum / b.numel()) <= 1e-5 * hsum / b.numel()


def test_shared_trunk_update_runs_and_is_world_size_invariant(b2048):
    """Shared trunk (lambda = 0.95), horizon update and PPO: two emulated ranks equal one process with the bonus on."""
    n, T, beta = 8192, 32, 0.02
    env = env_of(b2048, n, seed=23)
    single = agent_of(b2048, env, shared_lambda=0.95, max_grad_norm=1.0)
    ro = single.rollout_many(env, horizon=T, precision=0)
    for mode in ("horizon", "ppo"):
        st = single.save_state()
        ranks = [agent_of(b2048, env_of(b2048, 1, seed=0), shared_lambda=0.95, max_grad_norm=1.0) for _ in range(2)]
        for r in ranks:
            r.load_state(st)
        cut = 3000

        def part(sl):
            return b2048.Rollout(ro.boards[:, sl].contiguous(), ro.flags[:, sl].contiguous(), ro.actions[:, sl].contiguous(),
                                 ro.rewards[:, sl].contiguous(), ro.length[sl].contiguous(), T, n_traj=n, auto_reset=True,
                                 gid0=sl.start)

        parts = [part(slice(0, cut)), part(slice(cut, n))]
        bar, slots, errors = threading.Barrier(2), [None, None], []

        def allreduce(r):
            def ar(t):
                torch.cuda.synchronize()
                slots[r] = t.clone()
                bar.wait()
                total = slots[0] + slots[1]
                bar.wait()
                t.copy_(total)
                torch.cuda.synchronize()
            return ar

        def run(r):
            try:
                if mode == "horizon":
                    ranks[r].update_from_horizon(parts[r], allreduce=allreduce(r), precision=0, entropy_coef=beta)
                else:
                    ranks[r].update_ppo(parts[r], epochs=2, minibatches=2, shuffle_seed=3, allreduce=allreduce(r), precision=0,
                                        entropy_coef=beta)
            except Exception as e:      # noqa: BLE001  (re-raised below)
                errors.append(e)
                bar.abort()

        threads = [threading.Thread(target=run, args=(r,)) for r in range(2)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert not errors, errors
        if mode == "horizon":
            info = single.update_from_horizon(ro, precision=0, entropy_coef=beta)
        else:
            info = single.update_ppo(ro, epochs=2, minibatches=2, shuffle_seed=3, precision=0, entropy_coef=beta)
        assert "entropy" in info
        want = flat_theta(single)
        for a in ranks:
            assert rel_err(flat_theta(a), want) < 1e-6, mode


def test_bonus_raises_the_entropy(b2048):
    """Ten SGD steps on sum ecoef H alone (coef = 0) raise the mean H of a fixed 65,536-board batch at every step."""
    n = 65536
    agent, boards, flags, acts = batch(b2048, n, seed=9)
    cf = torch.zeros(n, device="cuda")
    ecf = torch.full((n,), 1.0 / n, device="cuda")
    hs = []
    for _ in range(11):
        g, h = backward(agent, boards, flags, acts, cf, ecf, 2)
        hs.append(h / n)
        with torch.no_grad():
            agent._actor.theta += 0.5 * agent._actor.grad
    print("mean H per step", hs)
    assert all(b > a for a, b in zip(hs, hs[1:]))


def test_trainer_entropy_coef(b2048, tmp_path):
    from b2048 import trainer
    for extra in ({}, {"ppo": {"epochs": 2, "minibatches": 2}}):
        cfg = trainer.merge_config({"env": {"max_steps": 64}, "mlp": {"hidden_sizes": [32, 32]},
                                    "agent": {"optimizer": "adam", "learning_rate": 1e-3, "use_critic": True},
                                    "train": dict({"batch_size": 2048, "num_batches": 3, "horizon": 32, "entropy_coef": 0.01,
                                                   "out_dir": str(tmp_path)}, **extra)})
        rows = trainer.training(cfg)
        assert len(rows) == 3 and all(np.isfinite(r["grad_norm"]) for r in rows)
