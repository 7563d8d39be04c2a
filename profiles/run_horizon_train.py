"""Times training on fixed-horizon windows (rollout_many(horizon=H, reset=False) + update_from_horizon) per iteration,
next to the run-to-termination train_iter (rollout_many + update_from_rollout), and runs a short learning comparison of
the two modes (mean completed-episode return against wall time, same network and learning rate).  The card's name and
power limit are read in the same call.

    python profiles/run_horizon_train.py [--out profiles/horizon_train.json] [--learn-seconds 60]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import b2048  # noqa: E402

RUNNER_ENV = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5, max_steps=1024)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make(n, hidden, obs="log2", seed=1, lr=1e-4, optimizer="sgd"):
    kw = dict(RUNNER_ENV)
    if obs == "onehot":
        kw.update(obs_mode="onehot", obs_log2_scale=1.0)
    env = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**kw), seed=seed)
    agent = b2048.ReinforceAgent(env, b2048.MLPConfig(hidden_sizes=list(hidden), activation="ReLU", init_distribution="HeNormal"),
                                 b2048.ReinforceAgentConfig(gamma=0.99, learning_rate=lr, baseline_mode="batch",
                                                            optimizer=optimizer))
    return env, agent


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def horizon_rate(name, n, H, hidden, obs="log2", iters=5, warmup=2):
    env, agent = make(n, hidden, obs)
    env.reset_many()
    rows = []
    for it in range(warmup + iters):
        ro, ms_r = timed(lambda: agent.rollout_many(env, horizon=H, reset=False, precision="auto"))
        info, ms_u = timed(lambda: agent.update_from_horizon(ro, precision="auto"))
        if it >= warmup:
            rows.append((ms_r, ms_u))
    r = np.array(rows)
    res = {"name": name, "lanes": n, "horizon": H, "network": [16 if obs == "log2" else 272] + list(hidden) + [4],
           "obs": obs, "rollout_ms": r[:, 0].tolist(), "update_ms": r[:, 1].tolist(),
           "samples_per_s": (n * H / (r.sum(1) / 1e3)).tolist(), "update_precision": info["precision"],
           "fused_rollout": agent._fused_shape()}
    print(json.dumps(res), flush=True)
    return res


def episode_rate(n, hidden, iters=3, warmup=1):
    env, agent = make(n, hidden)
    rows = []
    for it in range(warmup + iters):
        env.seed = 1000 + it
        ro, ms_r = timed(lambda: agent.rollout_many(env, precision="auto"))
        info, ms_u = timed(lambda: agent.update_from_rollout(ro))
        if it >= warmup:
            rows.append((ms_r, ms_u, int(ro.length.sum())))
    r = np.array(rows, dtype=np.float64)
    res = {"name": "train_iter run-to-termination", "episodes": n, "network": [16] + list(hidden) + [4],
           "rollout_ms": r[:, 0].tolist(), "update_ms": r[:, 1].tolist(), "samples": r[:, 2].astype(int).tolist(),
           "samples_per_s": (r[:, 2] / ((r[:, 0] + r[:, 1]) / 1e3)).tolist(), "update_precision": info["precision"]}
    print(json.dumps(res), flush=True)
    return res


def learning(seconds, n=8192, H=128, lr=1e-3):
    """Mean completed-episode return against wall time, horizon mode against episode mode, same network and lr."""
    out = {"lanes_or_episodes": n, "horizon": H, "learning_rate": lr, "optimizer": "adam", "baseline": "batch",
           "network": [16, 256, 256, 4]}
    for mode in ("horizon", "episode"):
        env, agent = make(n, (256, 256), lr=lr, optimizer="adam", seed=7)
        if mode == "horizon":
            env.reset_many()
        curve, t0, it = [], time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds:
            if mode == "horizon":
                ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
                agent.update_from_horizon(ro)
                es = agent.horizon_episode_stats()
                count, ret = es["episodes"], es["avg_reward"]
            else:
                env.seed = 5000 + it
                ro = agent.rollout_many(env, precision="auto")
                count, ret = n, float(ro.total_reward().mean())
                agent.update_from_rollout(ro)
            torch.cuda.synchronize()
            curve.append([round(time.perf_counter() - t0, 3), count, ret])
            it += 1
        out[mode] = curve
        print(mode, curve[:2], curve[-2:], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "horizon_train.json"))
    ap.add_argument("--learn-seconds", type=float, default=60.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(), "torch": torch.__version__,
           "timing": "host clock around each call, ending in a device synchronise; 2 warm-up iterations"}
    res["horizon"] = [horizon_rate("runner-default 65536 x 128", 65536, 128, (256, 256)),
                      horizon_rate("runner-default 1M x 32", 1 << 20, 32, (256, 256)),
                      horizon_rate("one-hot 262144 x 64", 262144, 64, (256, 128, 64), obs="onehot")]
    res["episode_reference"] = episode_rate(65536, (256, 256))
    res["learning"] = learning(args.learn_seconds)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
