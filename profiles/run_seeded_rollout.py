"""Rate of reference-seeded batched episodes (ReinforceAgent.run_episodes) next to the single-env drop-in's run_episode.

Runner defaults (16-256-256-4 ReLU, log2 observations, model_seed 0, seeds from make_fixed_seed_iter(3) / (7)):
65,536 episodes in one run_episodes call, timed with device events around the call and a final synchronise (the call
is warmed up once on the first 4,096 seeds), then 32 episodes of the drop-in on the same seeds.  A rollout step is one
board stepping once; steps are counted up to each episode's end.  Prints the GPU name and power limit and writes
profiles/seeded_rollout.json.

    python profiles/run_seeded_rollout.py
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import b2048  # noqa: E402

N, N_DROPIN = 65536, 32


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    env_kw = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5, max_steps=1024)
    mlp = b2048.MLPConfig(hidden_sizes=[256, 256], activation="ReLU", init_distribution="HeNormal")
    acfg = b2048.ReinforceAgentConfig(gamma=0.99, learning_rate=1e-4, baseline_mode="batch", model_seed=0)
    it_e, it_p = b2048.make_fixed_seed_iter(3), b2048.make_fixed_seed_iter(7)
    es = [next(it_e) for _ in range(N)]
    ps = [next(it_p) for _ in range(N)]

    benv = b2048.Batched2048Env(N, b2048.Game2048EnvConfig(**env_kw))
    agent = b2048.ReinforceAgent(benv, mlp, acfg)
    warm = b2048.Batched2048Env(4096, b2048.Game2048EnvConfig(**env_kw))
    agent.run_episodes(warm, es[:4096], ps[:4096])
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    ro = agent.run_episodes(benv, es, ps)
    ev1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    dev_s = ev0.elapsed_time(ev1) / 1e3
    steps = int(ro.length.sum())

    denv = b2048.Game2048Env(b2048.Game2048EnvConfig(**env_kw))
    dagent = b2048.ReinforceAgent(denv, mlp, acfg)
    t0 = time.perf_counter()
    dsteps = sum(len(dagent.run_episode(es[k], ps[k])["actions"]) for k in range(N_DROPIN))
    dwall = time.perf_counter() - t0

    name, power = gpu_info()
    res = {"gpu": name, "power_limit": power, "episodes": N, "rollout_steps": steps, "horizon_T": ro.T,
           "device_seconds": dev_s, "wall_seconds": wall, "steps_per_s": steps / dev_s,
           "dropin_episodes": N_DROPIN, "dropin_steps": dsteps, "dropin_seconds": dwall, "dropin_steps_per_s": dsteps / dwall}
    print(json.dumps(res, indent=1))
    with open(os.path.join(ROOT, "profiles", "seeded_rollout.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
