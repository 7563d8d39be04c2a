"""Cost and effect of playing with the one-ply expectimax over the critic (ReinforceAgent.lookahead_actions /
rollout_lookahead, DESIGN.md K7).

1. Timing: one search step (b2048_lookahead_expand, the 4-byte read of the child count, the critic forward on the children
   at "auto" precision, b2048_lookahead_select) on 65,536 and 262,144 boards of mid-game positions (random-legal play with
   reset-on-done, 150 steps), for the runner-default critic (log2, 16-256-256-1) and the one-hot critic
   (272-256-128-64-1): search steps per second (host clock around whole steps), mean children per board, CUDA-event device
   time of expand, forward and select, and the forward's achieved FLOP/s (2 x sum of the layer products per child over
   its event time).
2. Effect: an actor-critic (runner-default env and network, separate critic, Adam) trained by this script with
   60 horizon-PPO batches of 16,384 lanes x 64 steps, then evaluated on the same 65,536 seeded games with the greedy actor
   (rollout_many(greedy=True)) and with the lookahead (rollout_lookahead): average score and max-tile histogram.

The card's name and power limit are read in the same call.

    python profiles/run_lookahead.py [--out profiles/lookahead.json] [--batches 60]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import b2048  # noqa: E402
from b2048 import _lib  # noqa: E402
from b2048.batched_env import _ptr, _stream, make_env_cfg  # noqa: E402
from b2048.trainer import TILE_BINS, tile_histogram  # noqa: E402

RUNNER_ENV = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5)
CRITICS = {"runner_default_16_256_256_1": ("log2", [256, 256]), "onehot_272_256_128_64_1": ("onehot", [256, 128, 64])}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def env_cfg(obs):
    kw = dict(RUNNER_ENV)
    if obs == "onehot":
        kw.update(obs_mode="onehot", obs_log2_scale=1.0)
    return b2048.Game2048EnvConfig(max_steps=1024, **kw)


def make_agent(env, hidden, **cfg):
    base = dict(gamma=0.99, use_critic=True, model_seed=1)
    base.update(cfg)
    return b2048.ReinforceAgent(env, b2048.MLPConfig(hidden_sizes=hidden, activation="ReLU", init_distribution="HeNormal"),
                                b2048.ReinforceAgentConfig(**base))


def flops_per_child(dims):
    return 2 * sum(dims[l] * dims[l + 1] for l in range(len(dims) - 1))


def timing(n, name, reps=20):
    obs, hidden = CRITICS[name]
    env = b2048.Batched2048Env(n, env_cfg(obs), seed=5)
    agent = make_agent(env, hidden)
    env.reset_many()
    for _ in range(150):
        env.step_many(action_mode="random_legal", auto_reset=True)
    boards, flags, mx = env.board.clone(), env.flags.clone(), env.max_exp.clone()
    cfg = make_env_cfg(env.config, "buffer", emit_obs=False)
    actions = torch.zeros(n, dtype=torch.uint8, device="cuda")
    for _ in range(3):                                   # warm-up: module loads, tensor-core weight images, buffers
        agent._lookahead(boards, flags, mx, cfg, 2, actions, None)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    totals = [agent._lookahead(boards, flags, mx, cfg, 2, actions, None) for _ in range(reps)]
    torch.cuda.synchronize()
    step_s = (time.perf_counter() - t0) / reps
    # the same calls one by one between CUDA events
    B, cap = n, 120 * n
    sc = agent._scratch
    cb, cr, cd, cv = sc["la_child_board"], sc["la_child_reward"], sc["la_child_done"], sc["la_child_value"]
    first, count, tot = sc["la_first"], sc["la_count"], sc["la_total"]
    lib, h = agent._lib, agent._h
    ex, fw, se = [], [], []
    for _ in range(reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        _lib.check(lib.b2048_lookahead_expand(h, _ptr(boards), _ptr(flags), _ptr(mx), C.byref(cfg), None, B, None, B, cap, _ptr(cb),
                                              _ptr(cr), _ptr(cd), _ptr(first), _ptr(count), _ptr(tot), _stream()), "expand")
        ev[1].record()
        total = int(tot.item())
        ev[2].record()
        agent._net_forward(agent._critic, cb[:total], cv[:total], 2)
        ev[3].record()
        _lib.check(lib.b2048_lookahead_select(h, None, B, None, B, _ptr(first), _ptr(count), _ptr(cr), _ptr(cd), _ptr(cv),
                                              0.99, _ptr(actions), None, _stream()), "select")
        ev[4].record()
        ev[4].synchronize()
        ex.append(ev[0].elapsed_time(ev[1]) / 1e3)
        fw.append(ev[2].elapsed_time(ev[3]) / 1e3)
        se.append(ev[3].elapsed_time(ev[4]) / 1e3)
    total = int(np.median(totals))
    f_med = float(np.median(fw))
    dims = agent._critic.dims
    return {"boards": n, "critic": name, "critic_dims": dims, "forward_precision": "auto (split-fp16 tcgen05 where it applies)",
            "search_steps_per_s": 1.0 / step_s, "boards_searched_per_s": n / step_s, "step_ms_host_clock": step_s * 1e3,
            "children": total, "children_per_board": total / n,
            "expand_ms": float(np.median(ex)) * 1e3, "forward_ms": f_med * 1e3, "select_ms": float(np.median(se)) * 1e3,
            "forward_flop_per_child": flops_per_child(dims),
            "forward_tflops": flops_per_child(dims) * total / f_med / 1e12,
            "expand_bytes_per_child_written": 17, "reps": reps}


def effect(batches, lanes=16384, horizon=64, games=65536):
    env = b2048.Batched2048Env(lanes, env_cfg("log2"), seed=3)
    agent = make_agent(env, [256, 256], learning_rate=3e-4, critic_learning_rate=1e-3, optimizer="adam",
                       baseline_mode="batch_norm", max_grad_norm=1.0)
    env.reset_many()
    t0 = time.perf_counter()
    for k in range(batches):
        ro = agent.rollout_many(env, horizon=horizon, reset=False, precision="auto")
        agent.update_ppo(ro, epochs=4, minibatches=4, shuffle_seed=1000 + k)
    torch.cuda.synchronize()
    train_s = time.perf_counter() - t0
    out = {"training": {"batches": batches, "lanes": lanes, "horizon": horizon, "update": "update_ppo(epochs=4, minibatches=4)",
                        "optimizer": "adam lr 3e-4 / critic 1e-3", "seconds": train_s}, "games": games, "tile_bins": TILE_BINS}
    for mode in ("greedy_actor", "lookahead"):
        ev = b2048.Batched2048Env(games, env_cfg("log2"), seed=0xE7A1)
        t0 = time.perf_counter()
        ro = agent.rollout_many(ev, greedy=True, precision="auto") if mode == "greedy_actor" else agent.rollout_lookahead(ev)
        torch.cuda.synchronize()
        tot = ro.total_reward()
        out[mode] = {"avg_reward": float(tot.mean()), "avg_score": float(ev.score.double().mean()),
                     "max_tile_counts": tile_histogram(ev.max_exp), "mean_len": float(ro.length.float().mean()),
                     "seconds": time.perf_counter() - t0}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "lookahead.json"))
    ap.add_argument("--batches", type=int, default=60)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_lookahead.py measures on the GPU; no CUDA device found")
    res = {"card": card(), "timing": [timing(n, name) for name in CRITICS for n in (65536, 262144)],
           "effect": effect(args.batches)}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
