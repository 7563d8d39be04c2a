"""Cost and effect of PPO on fixed-horizon windows (ReinforceAgent.update_ppo) next to the one-step window update
(update_from_horizon).

1. Timing: CUDA-event time of update_ppo(epochs=4, minibatches=4) and of update_from_horizon on windows of H = 64 steps of
   65,536 and 262,144 lanes of the runner-default env and network (separate critic, Adam, "auto" precision), and the
   PPO time broken down by phase: the once-per-window pass at theta_old (V_old on all slices, GAE, advantages, the actor
   forward and logp_old), the partition of one epoch (b2048_ppo_minibatches and the grouping), and for one minibatch the
   gathers and forwards, the coefficient kernel, the two backward passes and the optimizer step.  The phases run the
   same calls as update_ppo, one phase at a time.
2. Learning: the completed-episode return per window of two agents with the same initial parameters, one trained with
   update_from_horizon (A2C) and one with update_ppo, each on its own env of the same seed (the windows differ once the
   policies do).

The card's name and power limit are read in the same call.

    python profiles/run_ppo.py [--out profiles/ppo.json] [--windows 150]
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
from b2048 import _lib  # noqa: E402
from b2048.batched_env import _ptr, _stream  # noqa: E402

RUNNER_ENV = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make(n, max_steps=1024, seed=1, lr=3e-4, critic_lr=1e-3):
    env = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(max_steps=max_steps, **RUNNER_ENV), seed=seed)
    agent = b2048.ReinforceAgent(env, b2048.MLPConfig(hidden_sizes=[256, 256], activation="ReLU", init_distribution="HeNormal"),
                                 b2048.ReinforceAgentConfig(gamma=0.99, learning_rate=lr, baseline_mode="batch_norm",
                                                            use_critic=True, critic_learning_rate=critic_lr, optimizer="adam",
                                                            max_grad_norm=1.0))
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


def phases(agent, ro, M):
    """One function per phase of update_ppo (the same library calls, in the same order)."""
    T, B = ro.T, ro.B
    n = T * B
    boards, mflags, acts = ro.boards[:T].reshape(-1), ro.flags[:T].reshape(-1), ro.actions[:T].reshape(-1)
    lib, h = agent._lib, agent._h
    values = torch.empty((T + 1, B), dtype=torch.float32, device="cuda")
    gae, td, gcoef, adv, coef = (torch.empty((T, B), dtype=torch.float32, device="cuda") for _ in range(5))
    valid = torch.empty(B, dtype=torch.int32, device="cuda")
    stats = torch.zeros(4, dtype=torch.float64, device="cuda")
    logits = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    logp_old = torch.empty(n, dtype=torch.float64, device="cuda")
    st5 = torch.zeros(5, dtype=torch.float64, device="cuda")
    state = {}

    def old_pass():
        agent._forward_checked(agent._critic, ro.boards[: T + 1].reshape(-1), values.view(-1), 2, [], 1)
        agent._segment_targets(ro.rewards[:T].contiguous(), ro.flags[: T + 1].contiguous(), values, 0.0, float(B), gae, td,
                               gcoef, valid)
        _lib.check(lib.b2048_advantages_window(h, _ptr(gae), _ptr(valid), 3, float(B), T, B, _ptr(adv), _ptr(coef), _ptr(stats),
                                               0, _stream()))
        agent._forward_checked(agent._actor, boards, logits, 2, [], 0)
        _lib.check(lib.b2048_ppo_logp(h, _ptr(logits), _ptr(mflags), _ptr(acts), n, _ptr(logp_old), _stream()))

    def partition():
        order, counts = agent.ppo_minibatch_lists(T, B, B, 0, M, 1, 0)
        state.update(idx=order[: counts[0]], k=counts[0])

    def forward():
        idx, k = state["idx"], state["k"]
        state.update(bx=boards.index_select(0, idx), fx=mflags.index_select(0, idx), ax=acts.index_select(0, idx),
                     z=torch.empty((k, 4), dtype=torch.float32, device="cuda"), v=torch.empty(k, dtype=torch.float32, device="cuda"))
        agent._forward_checked(agent._actor, state["bx"], state["z"], 2, [], 0)
        agent._forward_checked(agent._critic, state["bx"], state["v"], 2, [], 1)

    def coefficients():
        k = state["k"]
        state.update(cf=torch.empty(k, dtype=torch.float32, device="cuda"), gc=torch.empty(k, dtype=torch.float32, device="cuda"))
        _lib.check(lib.b2048_ppo_coefficients(h, _ptr(state["idx"]), k, _ptr(state["z"]), _ptr(state["v"]), _ptr(mflags),
                                              _ptr(acts), _ptr(logp_old), _ptr(adv), _ptr(gae), _ptr(values), float(n // M), 0.2,
                                              0.0, 0, 1.0, _ptr(state["cf"]), _ptr(state["gc"]), _ptr(st5), _stream()))

    def backward():
        k = state["k"]
        agent._backward(agent._actor, state["bx"], state["fx"], state["ax"], state["cf"], k, 0, 2, 1 << 20, [])
        agent._backward(agent._critic, state["bx"], state["fx"], state["ax"], state["gc"], k, 1, 2, 1 << 20, [])

    def apply():
        agent._optimizer_step()

    return [("old_pass_s", old_pass), ("partition_per_epoch_s", partition), ("minibatch_forward_s", forward),
            ("minibatch_coefficients_s", coefficients), ("minibatch_backward_s", backward), ("minibatch_apply_s", apply)]


def timing(n, H, reps, epochs=4, M=4):
    env, agent = make(n)
    env.reset_many()
    for _ in range(3):                                  # reach the steady mix of episode ages
        agent.rollout_many(env, horizon=H, reset=False, precision="auto")
    ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
    st = agent.save_state()
    out = {"lanes": n, "horizon": H, "epochs": epochs, "minibatches": M, "samples": n * H}
    for name, fn in (("update_from_horizon_s", lambda: agent.update_from_horizon(ro)),
                     ("update_ppo_s", lambda: agent.update_ppo(ro, epochs=epochs, minibatches=M, shuffle_seed=3))):
        fn()                                            # warm-up of this shape
        agent.load_state(st)
        med, ts = timed(fn, reps, lambda: agent.load_state(st))
        out[name] = med
        out[name + "_all"] = ts
    out["ppo_over_a2c"] = out["update_ppo_s"] / out["update_from_horizon_s"]
    for name, fn in phases(agent, ro, M):
        fn()
        med, ts = timed(fn, reps, lambda: agent.load_state(st))
        out[name] = med
    agent.load_state(st)
    mb = out["minibatch_forward_s"] + out["minibatch_coefficients_s"] + out["minibatch_backward_s"] + out["minibatch_apply_s"]
    out["phases_sum_s"] = out["old_pass_s"] + epochs * out["partition_per_epoch_s"] + epochs * M * mb
    return out


def learning(windows, n=8192, H=64, seed=99):
    res = {"lanes": n, "horizon": H, "windows": windows}
    for mode in ("a2c", "ppo"):
        env, agent = make(n, seed=seed)
        env.reset_many()
        curve = []
        for k in range(windows):
            ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
            if mode == "ppo":
                agent.update_ppo(ro, epochs=4, minibatches=4, shuffle_seed=k)
            else:
                agent.update_from_horizon(ro)
            es = agent.horizon_episode_stats()
            curve.append(es["avg_reward"] if es["episodes"] else None)
        res[mode + "_return_per_window"] = curve
        tail = [c for c in curve[-20:] if c is not None]
        res[mode + "_mean_return_last_20"] = float(np.mean(tail)) if tail else None
        print(mode, res[mode + "_mean_return_last_20"], flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "ppo.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--windows", type=int, default=150)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"gpu": card(), "timing": []}
    for n in (65536, 262144):
        r = timing(n, 64, args.reps)
        print(json.dumps({k: v for k, v in r.items() if not k.endswith("_all")}), flush=True)
        res["timing"].append(r)
    res["learning"] = learning(args.windows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
