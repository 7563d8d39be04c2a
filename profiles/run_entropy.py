"""Cost and effect of the entropy bonus (b2048_mlp_backward_entropy, entropy_coef of the updates).

1. Kernels: CUDA-event time of b2048_mlp_backward against b2048_mlp_backward_entropy on the same rollout-derived inputs:
   the 16-256-256 persistent update pipeline at 1 M samples, the chunked float32-grade kernels (B2048_DBG_NO_UPDATE_PIPE) at
   1 M, the shape-generic kernels of the one-hot 272-256-128-64 network at 1 M, and the fp32 CUDA-core kernels at 65,536.
2. Update: update_ppo (4 epochs x 4 minibatches) on a window of 65,536 lanes x 64 steps, with and without the bonus.
3. Learning: two PPO agents from the same parameters and env seed, 8,192 lanes, 150 windows of 64 steps, beta = 0 and 0.01;
   per window the mean entropy of the updated policy on the window's samples and the mean return of the completed episodes.

The card's name and power limit are read in the same call.

    python profiles/run_entropy.py [--out profiles/entropy.json] [--windows 150]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import b2048  # noqa: E402
from b2048.batched_env import _ptr, _stream  # noqa: E402

RUNNER_ENV = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5)
NO_UPDATE_PIPE = 5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make(n, hidden=(256, 256), obs="log2", max_steps=1024, seed=1, lr=3e-4, critic_lr=1e-3):
    env_kw = dict(RUNNER_ENV) if obs == "log2" else dict(RUNNER_ENV, obs_mode="onehot", obs_log2_scale=1.0)
    env = b2048.Batched2048Env(n, b2048.Game2048EnvConfig(max_steps=max_steps, **env_kw), seed=seed)
    agent = b2048.ReinforceAgent(env, b2048.MLPConfig(hidden_sizes=list(hidden), activation="ReLU", init_distribution="HeNormal"),
                                 b2048.ReinforceAgentConfig(gamma=0.99, learning_rate=lr, baseline_mode="batch_norm",
                                                            use_critic=True, critic_learning_rate=critic_lr, optimizer="adam",
                                                            max_grad_norm=1.0))
    return env, agent


def event_ms(fn, reps, setup=lambda: None):
    ts = []
    for _ in range(reps):
        setup()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return ts


def kernel_times(n, hidden, obs, prec, chunked, reps=20):
    H = 64
    env, agent = make(n // H, hidden, obs)
    ro = agent.rollout_many(env, horizon=H, precision=0)
    boards, flags, acts = (x[:H].reshape(-1).contiguous() for x in (ro.boards, ro.flags, ro.actions))
    g = torch.Generator(device="cuda").manual_seed(0)
    cf = torch.randn(n, generator=g, device="cuda") / n
    cf -= cf.mean()
    ecf = torch.full((n,), 0.01 / n, device="cuda")
    lib, h, net = agent._lib, agent._h, agent._actor
    if chunked:
        lib.b2048_debug_set(h, NO_UPDATE_PIPE, 1)
    wsf = int(lib.b2048_backward_workspace_floats(C.byref(net.desc), n))
    ws = torch.empty(wsf, dtype=torch.float32, device="cuda")
    es = torch.zeros(1, dtype=torch.float64, device="cuda")

    def plain():
        assert lib.b2048_mlp_backward(h, _ptr(boards), _ptr(flags), _ptr(acts), _ptr(cf), C.byref(net.desc), _ptr(net.grad), n, 0,
                                      _ptr(ws), wsf, n, prec, _stream()) == 0

    def ent():
        assert lib.b2048_mlp_backward_entropy(h, _ptr(boards), _ptr(flags), _ptr(acts), _ptr(cf), _ptr(ecf), C.byref(net.desc),
                                              _ptr(net.grad), n, _ptr(ws), wsf, n, prec, _ptr(es), _stream()) == 0

    zero = lambda: net.grad.zero_()
    for f in (plain, ent):                                    # warm-up
        event_ms(f, 3, zero)
    tp, te = [], []
    for _ in range(reps):                                     # alternate the two calls
        tp += event_ms(plain, 1, zero)
        te += event_ms(ent, 1, zero)
    return dict(n=n, hidden=list(hidden), obs=obs, precision=prec, chunked=chunked, plain_ms=float(np.median(tp)),
                entropy_ms=float(np.median(te)), plain_ms_range=[float(min(tp)), float(max(tp))],
                entropy_ms_range=[float(min(te)), float(max(te))],
                overhead_pct=float(100.0 * (np.median(te) / np.median(tp) - 1.0)))


def ppo_times(n=65536, H=64, reps=5):
    env, agent = make(n)
    ro = agent.rollout_many(env, horizon=H, precision="auto")
    st = agent.save_state()
    restore = lambda: agent.load_state(st)
    out = {}
    for beta in (0.0, 0.01):
        fn = lambda: agent.update_ppo(ro, epochs=4, minibatches=4, entropy_coef=beta)
        event_ms(fn, 1, restore)
        out[str(beta)] = event_ms(fn, reps, restore)
    return dict(lanes=n, steps=H, epochs=4, minibatches=4, ms={k: float(np.median(v)) for k, v in out.items()},
                ms_all=out, overhead_pct=float(100.0 * (np.median(out["0.01"]) / np.median(out["0.0"]) - 1.0)))


def mean_entropy(agent, ro):
    """Mean H of the policy over a window's samples (ent_sum of b2048_mlp_backward_entropy with zero coefficients)."""
    T = ro.T
    b, f, a = (x[:T].reshape(-1).contiguous() for x in (ro.boards, ro.flags, ro.actions))
    m = b.numel()
    lib, net = agent._lib, agent._actor
    wsf = int(lib.b2048_backward_workspace_floats(C.byref(net.desc), m))
    ws = torch.empty(wsf, dtype=torch.float32, device="cuda")
    es = torch.zeros(1, dtype=torch.float64, device="cuda")
    z = torch.zeros(m, device="cuda")
    g = torch.empty_like(net.grad)
    assert lib.b2048_mlp_backward_entropy(agent._h, _ptr(b), _ptr(f), _ptr(a), _ptr(z), _ptr(z), C.byref(net.desc), _ptr(g), m,
                                          _ptr(ws), wsf, m, 2, _ptr(es), _stream()) == 0
    return float(es[0]) / m


def learning(windows, n=8192, H=64):
    res = {}
    for beta in (0.0, 0.01):
        env, agent = make(n, seed=77)
        env.reset_many()
        ent, ret, eps = [], [], []
        for w in range(windows):
            ro = agent.rollout_many(env, horizon=H, reset=False, precision="auto")
            info = agent.update_ppo(ro, epochs=4, minibatches=4, shuffle_seed=w, entropy_coef=beta)
            ent.append(mean_entropy(agent, ro))      # the same diagnostic for both: mean H of the window after the update
            st = agent.horizon_episode_stats()
            ret.append(st["avg_reward"])
            eps.append(st["episodes"])
        res[str(beta)] = dict(entropy=ent, avg_return=ret, episodes=eps)
        tail = [r for r in ret[-20:] if np.isfinite(r)]
        print(f"beta {beta}: entropy first/last {ent[0]:.4f}/{ent[-1]:.4f}, mean return of the last 20 windows "
              f"{np.mean(tail) if tail else float('nan'):.1f}", flush=True)
    return dict(lanes=n, steps=H, windows=windows, epochs=4, minibatches=4, optimizer="adam", per_beta=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "entropy.json"))
    ap.add_argument("--windows", type=int, default=150)
    args = ap.parse_args()
    res = {"card": card(), "torch": torch.__version__}
    print(res["card"], flush=True)
    M = 1 << 20
    res["kernels"] = {}
    for name, (n, hidden, obs, prec, chunked) in {
            "hp_pipeline_16_256_256": (M, (256, 256), "log2", 3, False),
            "hp_chunked_16_256_256": (M, (256, 256), "log2", 3, True),
            "generic_onehot_272_256_128_64": (M, (256, 128, 64), "onehot", 3, False),
            "fp32_16_256_256": (65536, (256, 256), "log2", 0, False)}.items():
        r = kernel_times(n, hidden, obs, prec, chunked)
        res["kernels"][name] = r
        print(name, json.dumps({k: v for k, v in r.items() if "range" not in k}), flush=True)
    res["update_ppo"] = ppo_times()
    print("update_ppo", json.dumps(res["update_ppo"]["ms"]), f"{res['update_ppo']['overhead_pct']:.1f} %", flush=True)
    res["learning"] = learning(args.windows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
