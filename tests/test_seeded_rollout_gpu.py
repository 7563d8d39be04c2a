"""Reference-seeded batched episodes (ReinforceAgent.run_episodes): per-board NumPy PCG64 streams on the device give
every board exactly the episode the single-env drop-in's run_episode(env_seed, policy_seed) plays — and therefore the
reference's own (tests/golden/seeded.json)."""
import json
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from helpers import GOLDEN, full_env_kwargs, rel_err  # noqa: E402


@pytest.fixture(scope="module")
def b2048():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import b2048 as m
    return m


def seeds(base, n, skip=0):
    from b2048 import make_fixed_seed_iter
    it = make_fixed_seed_iter(base)
    out = [next(it) for _ in range(skip + n)]
    return out[skip:]


def words(st):
    s, inc = st["state"]["state"], st["state"]["inc"]
    return [s >> 64, s & (2**64 - 1), inc >> 64, inc & (2**64 - 1), st["has_uint32"], st["uinteger"]]


def dev_words(t):
    """b2048_np_rng rows (int64 [n, 6]: four uint64, has_uint32 | uinteger << 32, reserved) -> words() layout"""
    out = []
    for row in t.cpu().numpy().view(np.uint64):
        w = [int(x) for x in row]
        assert w[5] == 0
        out.append(w[:4] + [w[4] & 0xFFFFFFFF, w[4] >> 32])
    return out


RUNNER_MLP = dict(hidden_sizes=[256, 256], activation="ReLU", init_distribution="HeNormal")
RUNNER_AGENT = dict(gamma=0.99, learning_rate=1e-4, baseline_mode="batch", model_seed=0)
NETS = [("runner_default", full_env_kwargs("runner_default"), RUNNER_MLP),
        ("onehot", dict(full_env_kwargs("runner_default"), obs_mode="onehot", obs_log2_scale=1.0, empty_tile_reward=0.05),
         dict(hidden_sizes=[256, 128, 64], activation="ReLU", init_distribution="HeNormal")),
        ("sigmoid", dict(full_env_kwargs("runner_default"), obs_log2_scale=1.0),
         dict(hidden_sizes=[48], activation="Sigmoid", init_distribution="XavierNormal"))]


def make(b2048, env_kw, mlp_kw, n):
    env = b2048.Game2048Env(b2048.Game2048EnvConfig(**env_kw))
    agent = b2048.ReinforceAgent(env, b2048.MLPConfig(**mlp_kw), b2048.ReinforceAgentConfig(**RUNNER_AGENT))
    benv = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**env_kw))
    return agent, benv


def test_seeding_kernel_matches_numpy(b2048):
    from b2048.batched_env import np_seed_streams
    s = seeds(3, 65536 - 6) + [0, 1, 2**32 - 1, 2**32, 2**63 - 1, 2**64 - 1]
    got = dev_words(np_seed_streams(s, torch.device("cuda", 0)))
    for k in range(len(s)):
        assert got[k] == words(np.random.default_rng(s[k]).bit_generator.state), s[k]


def test_runner_default_first_episodes(b2048):
    """The fixture episodes test_reference_config1_first_episodes pins, from a batch of 8."""
    with open(os.path.join(GOLDEN, "seeded.json")) as f:
        facts = json.load(f)
    agent, benv = make(b2048, full_env_kwargs("runner_default"), RUNNER_MLP, 8)
    ro = agent.run_episodes(benv, seeds(3, 8), seeds(7, 8))
    tot = ro.total_reward().cpu().numpy()
    got = [[int(ro.length[b]), float(tot[b]), int(1 << int(benv.max_exp[b]))] for b in range(8)]
    ref = facts["runner_default_first8"]
    assert got[:3] == ref[:3]
    n_match = sum(g == r for g, r in zip(got, ref))
    print(f"runner_default_first8: {n_match} of {len(ref)} episodes match")


@pytest.mark.parametrize("greedy", [False, True])
@pytest.mark.parametrize("tag,env_kw,mlp_kw", NETS)
def test_batched_equals_single_env_episodes(b2048, tag, env_kw, mlp_kw, greedy):
    n = 256
    es, ps = seeds(3, n, skip=100), seeds(7, n, skip=100)
    agent, benv = make(b2048, env_kw, mlp_kw, n)
    ro = agent.run_episodes(benv, es, ps, use_greedy=greedy)
    lens = ro.length.cpu().numpy()
    acts, rews = ro.actions.cpu().numpy(), ro.rewards.cpu().numpy()
    max_exp = benv.max_exp.cpu().numpy()
    env_rng = dev_words(benv.env_rng)
    for b in range(n):
        tr = agent.run_episode(es[b], ps[b], use_greedy=greedy)
        T = len(tr["actions"])
        assert int(lens[b]) == T, (tag, b)
        assert acts[:T, b].tolist() == tr["actions"], (tag, b)
        assert rews[:T, b].view(np.uint32).tolist() == np.asarray(tr["rewards"], np.float32).view(np.uint32).tolist(), (tag, b)
        assert int(1 << int(max_exp[b])) == tr["max_tile"], (tag, b)
        assert env_rng[b] == words(agent.env.game._rng.bit_generator.state), (tag, b)


def clone(ro):
    return {k: getattr(ro, k).clone() for k in ("boards", "flags", "actions", "rewards", "length")}


def test_live_list_and_batch_split_do_not_change_episodes(b2048):
    n = 65536
    es, ps = seeds(3, n), seeds(7, n)
    agent, benv = make(b2048, full_env_kwargs("runner_default"), RUNNER_MLP, n)
    a = clone(agent.run_episodes(benv, es, ps))
    rng_a = benv.env_rng.clone()
    b = clone(agent.run_episodes(benv, es, ps, live_list=False))
    assert torch.equal(a["length"], b["length"]) and a["boards"].shape == b["boards"].shape
    for k in ("boards", "flags", "rewards"):
        assert torch.equal(a[k], b[k]), k
    T = a["actions"].shape[0]
    live = torch.arange(T, device="cuda").unsqueeze(1) < a["length"].unsqueeze(0)
    assert torch.equal(a["actions"][live], b["actions"][live])
    assert torch.equal(rng_a, benv.env_rng)
    h = n // 2
    half_env = b2048.Batched2048Env(h, b2048.Game2048EnvConfig(**full_env_kwargs("runner_default")))
    for part in (slice(0, h), slice(h, n)):
        c = clone(agent.run_episodes(half_env, es[part], ps[part]))
        assert torch.equal(c["length"], a["length"][part])
        Tc = c["actions"].shape[0]
        livec = live[:Tc, part]
        assert torch.equal(c["actions"][livec], a["actions"][:Tc, part][livec])
        assert torch.equal(c["rewards"], a["rewards"][:Tc, part])
        assert torch.equal(c["boards"], a["boards"][: Tc + 1, part])
    with pytest.raises(ValueError):
        agent.run_episodes(half_env, [-1] * h, ps[:h])
    with pytest.raises(ValueError):
        agent.run_episodes(half_env, es[:h], ps[: h - 1])


def test_trainer_numpy_streams(b2048, tmp_path):
    from b2048 import trainer
    user = {"train": {"batch_size": 8, "num_batches": 2, "out_dir": str(tmp_path), "seed_streams": "numpy"}}
    rows = trainer.training(trainer.merge_config(user))
    assert [r["batch"] for r in rows] == [1, 2]
    lines = open(os.path.join(tmp_path, "training_stats.csv")).read().strip().splitlines()
    assert len(lines) == 3 and lines[0].startswith("batch,")

    def direct(skip):
        agent, benv = make(b2048, full_env_kwargs("runner_default"), RUNNER_MLP, 8)
        tot = agent.run_episodes(benv, seeds(3, 8, skip), seeds(7, 8, skip)).total_reward().cpu().numpy()
        return [float(tot.mean()), float(tot.max()), float(tot.min())]

    assert [rows[0]["avg_reward"], rows[0]["max_reward"], rows[0]["min_reward"]] == pytest.approx(direct(0), rel=1e-12)
    user["train"].update(start_batch=1, out_dir=str(tmp_path / "resumed"))
    more = trainer.training(trainer.merge_config(user))
    assert [r["batch"] for r in more] == [2]
    assert [more[0]["avg_reward"], more[0]["max_reward"], more[0]["min_reward"]] == pytest.approx(direct(8), rel=1e-12)
    with pytest.raises(ValueError):
        trainer.training(trainer.merge_config({"train": {"batch_size": 8, "num_batches": 1, "out_dir": None,
                                                         "seed_streams": "mt19937"}}))


def test_update_from_seeded_rollout_equals_update_batch(b2048):
    agent, benv = make(b2048, full_env_kwargs("runner_default"), RUNNER_MLP, 3)
    other, _ = make(b2048, full_env_kwargs("runner_default"), RUNNER_MLP, 3)
    es, ps = seeds(3, 3), seeds(7, 3)
    before = agent.params
    trajs = [other.run_episode(e, p) for e, p in zip(es, ps)]
    other.update_batch(trajs)
    agent.update_from_rollout(agent.run_episodes(benv, es, ps))
    a, o = agent.params, other.params
    assert abs(agent.last_update_info["actor_grad_norm"] - other.last_update_info["actor_grad_norm"]) < \
        1e-3 * other.last_update_info["actor_grad_norm"]
    for l in range(3):
        assert rel_err(a["W"][l] - before["W"][l], o["W"][l] - before["W"][l]) < 1e-3
        assert rel_err(a["b"][l] - before["b"][l], o["b"][l] - before["b"][l]) < 1e-3
