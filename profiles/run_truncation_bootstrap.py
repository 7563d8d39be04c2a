"""Cost and effect of bootstrapping truncated episodes in fixed-horizon training (update_from_horizon(bootstrap_truncation=True)).

1. Timing: CUDA-event time of the bootstrap alone (truncated-slot list, pre-reset replay, V(s') and the fold, with the
   host waits they contain) next to the whole update_from_horizon with and without it, on windows of H = 64 steps of
   65,536 and 262,144 lanes of the runner-default env and network, with max_steps 25 (about one truncation per lane every
   25 steps) and 1024 (almost none).
2. Critic bias: a critic trained on windows with the actor frozen (learning_rate = 0) learns V = r on the last step
   before the step limit when a truncation is treated as a game over.  After N critic updates the mean V of the boards one
   step before the limit is compared with that of mid-episode boards, with and without the bootstrap.

The card's name and power limit are read in the same call.

    python profiles/run_truncation_bootstrap.py [--out profiles/truncation_bootstrap.json] [--bias-updates 300]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import b2048  # noqa: E402

RUNNER_ENV = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5)
F_END, F_TRUNC = 0x60, 0x40


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make(n, max_steps, seed=1, lr=1e-4, critic_lr=1e-4):
    env = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(max_steps=max_steps, **RUNNER_ENV), seed=seed)
    agent = b2048.ReinforceAgent(env, b2048.MLPConfig(hidden_sizes=[256, 256], activation="ReLU", init_distribution="HeNormal"),
                                 b2048.ReinforceAgentConfig(gamma=0.99, learning_rate=lr, baseline_mode="batch", use_critic=True,
                                                            critic_learning_rate=critic_lr, optimizer="adam"))
    return env, agent


def timed(fn, reps, setup):
    ts = []
    for _ in range(reps):
        setup()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return float(np.median(ts)), ts


def bootstrap_only(agent, ro):
    """The work bootstrap_truncation adds to update_from_horizon: the slot list and replay, V(s'), the fold."""
    slots, nxt = agent._truncated_window_steps(ro)
    update = agent._update
    agent._update = lambda *a, **k: {}                  # everything of _update_bootstrapped but the unchanged update body
    try:
        agent._update_bootstrapped(ro, (slots, nxt), 1 << 20, None, "auto", "default", window=True)
    finally:
        agent._update = update
    return int(slots.numel())


def timing(n, max_steps, H, reps):
    env, agent = make(n, max_steps)
    env.reset_many()
    for _ in range(3):                                  # reach the steady mix of episode ages
        agent.rollout_many(env, horizon=H, reset=False, precision="auto")
    ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
    st = agent.save_state()
    out = {"lanes": n, "horizon": H, "max_steps": max_steps}
    out["truncations"] = bootstrap_only(agent, ro)
    for name, fn in (("bootstrap_s", lambda: bootstrap_only(agent, ro)),
                     ("update_s", lambda: agent.update_from_horizon(ro)),
                     ("update_bootstrap_s", lambda: agent.update_from_horizon(ro, bootstrap_truncation=True))):
        fn()                                            # warm-up of this shape
        agent.load_state(st)
        med, ts = timed(fn, reps, lambda: agent.load_state(st))
        out[name] = med
        out[name + "_all"] = ts
    out["bootstrap_share_of_update"] = out["bootstrap_s"] / out["update_bootstrap_s"]
    return out


def episode_steps(step0, flags, H):
    """Steps already played in its episode by every board of the window, [H, B] (0 right after a reset)."""
    c = step0.clone().long()
    out = []
    for t in range(H):
        out.append(c.clone())
        c = torch.where((flags[t + 1] & F_END) != 0, torch.zeros_like(c), c + 1)
    return torch.stack(out)


def critic_bias(boot, n, H, max_steps, updates):
    env, agent = make(n, max_steps, seed=7, lr=0.0, critic_lr=1e-3)    # the actor is frozen: a fixed policy's values
    env.reset_many()
    pre, mid = [], []
    for k in range(updates):
        step0 = env.step_count.clone()
        ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
        if k >= updates - 20:                           # the critic's values of the last 20 windows' boards
            steps = episode_steps(step0, ro.flags, H)
            values = torch.empty((H, n), dtype=torch.float32, device=agent.device)
            agent._values(ro.boards[:H].reshape(-1), values.view(-1), 0)
            pre.append(values[steps == max_steps - 1])
            mid.append(values[steps == max_steps // 2])
        agent.update_from_horizon(ro, bootstrap_truncation=boot)
    pre, mid = torch.cat(pre), torch.cat(mid)
    return {"bootstrap": boot, "critic_updates": updates, "lanes": n, "horizon": H, "max_steps": max_steps,
            "mean_V_one_step_before_limit": float(pre.mean()), "n_before_limit": int(pre.numel()),
            "mean_V_mid_episode": float(mid.mean()), "n_mid_episode": int(mid.numel())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "truncation_bootstrap.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--bias-updates", type=int, default=300)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"gpu": card(), "timing": [], "critic_bias": []}
    for n in (65536, 262144):
        for max_steps in (25, 1024):
            r = timing(n, max_steps, 64, args.reps)
            print(json.dumps({k: v for k, v in r.items() if not k.endswith("_all")}), flush=True)
            res["timing"].append(r)
    for boot in (False, True):
        r = critic_bias(boot, 8192, 64, 64, args.bias_updates)
        print(json.dumps(r), flush=True)
        res["critic_bias"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
