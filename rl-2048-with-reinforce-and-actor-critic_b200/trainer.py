"""Batched trainer / evaluator — the `runner.py` equivalent for the batched engine (SURVEY.md section 8f, item 1).

Accepts the reference's JSON schema (sections ``env`` / ``mlp`` / ``agent`` / ``train`` / ``eval`` / ``run_mode``,
runner.py:10-63, defaults runner.py:116-173) and writes the same artefacts (``config.json``,
``training_stats.csv`` with columns ``batch,avg_reward,max_reward,min_reward,max_tile_counts``, best-average
``.npz`` checkpoints taken BEFORE the update once the 1-based ``global_step > 30``, runner.py:526-673; ``checkpoint.npz``
with the full optimiser state every ``train.checkpoint_every`` batches).  One training batch =
``train.batch_size`` episodes played in parallel on the GPU (``rollout_many``) followed by one
``update_from_rollout``; evaluation = greedy rollouts with the max-tile histogram (runner.py:737-828).
Extra keys: ``train.seed_streams`` ("philox", the default: fresh counter-based streams per batch | "numpy": the reference's
own seeded episodes — episode i of batch k plays run_episode(env_seed, policy_seed) with the (k * batch_size + i)-th seed
of make_fixed_seed_iter(``train.env_base_seed``) / make_fixed_seed_iter(``train.policy_base_seed``), the order
runner.py:587-608 draws them, on the fp32 policy kernel; evaluation keeps the Philox streams), ``train.precision`` ("auto" | 0 | 1), ``train.exchange`` ("default" | "one_message": one all-reduce per update),
``seed``, and an optional section ``shared_trunk`` ({"value_coef", "gae_lambda"}: one network with a policy and a value head).  Under torchrun the episodes are sharded over ranks.
``train.horizon`` (default None: the batches above): an integer H trains on fixed-horizon windows instead — the
``train.batch_size`` envs are reset once and keep playing (reset-on-done); each batch is ``rollout_many(horizon=H,
reset=False)`` followed by one ``update_from_horizon`` (segment-aware returns / TD / GAE, the cut-off tail bootstrapped by
the critic when there is one).  The CSV rows then describe the episodes that ended inside the batch's window (NaN stats
and zero counts when none did); a resumed run starts from fresh resets.  Not combinable with ``seed_streams="numpy"``.
``train.bootstrap_truncation`` (default false; needs ``agent.use_critic`` or a ``shared_trunk`` section): in both modes, an
episode truncated by ``env.max_steps`` gets the target r + gamma V(s') at its last step, s' being the board it was cut on,
instead of r (``update_from_rollout`` / ``update_from_horizon(bootstrap_truncation=True)``).

    python -m torch.distributed.run ... b2048_runner.py -conf cfg.json      (or: python b2048_runner.py -conf cfg.json)
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import time
from typing import Any

import numpy as np
import torch

from . import dist as bd
from .MLP import MLPConfig
from .batched_env import Batched2048Env, Game2048EnvConfig, make_fixed_seed_iter
from .reinforce_agent import ReinforceAgent, ReinforceAgentConfig

DEFAULTS: dict[str, Any] = {
    "run_mode": "Training",
    "seed": 3,
    "env": dict(size=4, obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5,
                bonus_mode="off", bonus_scale=1.0, step_reward=0.0, endgame_penalty=0.0, use_action_mask=True,
                invalid_action_penalty=-1.0, max_steps=1024, empty_tile_reward=0.0, merge_reward=0.0),
    "mlp": dict(hidden_sizes=[256, 256], activation="ReLU", init_distribution="HeNormal", last_init_normal=True),
    "agent": dict(gamma=0.99, learning_rate=1e-4, baseline_mode="batch", model_seed=0, reward_rank_weights=None,
                  optimizer="sgd", adam_beta1=0.9, adam_beta2=0.999, augmentation=False, use_critic=False,
                  critic_learning_rate=1e-5, critic_loss_type="mse", huber_delta=1.0),
    "train": dict(batch_size=256, num_batches=256, precision="auto", out_dir="training_history", seed_streams="philox",
                  env_base_seed=3, policy_base_seed=7),
    "eval": dict(num_episodes=2048, model_path=None, use_greedy=True),
}
TILE_BINS = [16, 32, 64, 128, 256, 512, 1024, 2048, 4096]      # runner.py:557


def merge_config(user: dict[str, Any] | None) -> dict[str, Any]:
    cfg = json.loads(json.dumps(DEFAULTS))
    for k, v in (user or {}).items():
        if isinstance(v, dict) and isinstance(cfg.get(k), dict):
            cfg[k].update(v)
        else:
            cfg[k] = v
    return cfg


def tile_histogram(max_exp: torch.Tensor, info: bd.DistInfo | None = None) -> list[int]:
    """Episodes per max tile, a list in TILE_BINS order like the reference's CSV column (runner.py:557, :617-624, :669);
    summed over ranks when the episodes are sharded."""
    tiles = 1 << max_exp.to(torch.int64)
    bins = torch.as_tensor(TILE_BINS, dtype=torch.int64, device=tiles.device)
    counts = (tiles.unsqueeze(1) == bins.unsqueeze(0)).sum(0)
    if info is not None and info.is_distributed:
        bd.allreduce_sum_(counts)
    return [int(c) for c in counts.tolist()]


def make_agent(cfg: dict[str, Any], env):
    """ReinforceAgent, or — with the extra section {"shared_trunk": {"value_coef": .., "gae_lambda": ..}} — the shared-trunk
    actor-critic of shared_trunk.py (one network, policy + value heads)."""
    st = cfg.get("shared_trunk")
    if st is not None:
        from .shared_trunk import SharedTrunkActorCritic
        return SharedTrunkActorCritic(env, MLPConfig(**cfg["mlp"]), ReinforceAgentConfig(**cfg["agent"]),
                                      value_coef=float(st.get("value_coef", 0.5)), gae_lambda=float(st.get("gae_lambda", 0.0)))
    return ReinforceAgent(env, MLPConfig(**cfg["mlp"]), ReinforceAgentConfig(**cfg["agent"]))


def build(cfg: dict[str, Any], num_envs: int, info: bd.DistInfo, device=None):
    env = bd.make_sharded_env(num_envs, Game2048EnvConfig(**cfg["env"]), info, seed=int(cfg["seed"]), device=device)
    return env, make_agent(cfg, env)


def _global_stats(values: torch.Tensor, info: bd.DistInfo):
    s = torch.stack([values.sum(), torch.tensor(float(values.numel()), device=values.device, dtype=values.dtype)])
    mx, mn = values.max().reshape(1).clone(), (-values.min()).reshape(1).clone()
    bd.allreduce_sum_(s)
    bd.allreduce_max_(mx)
    bd.allreduce_max_(mn)
    return float(s[0] / s[1]), float(mx), float(-mn)


def training(cfg: dict[str, Any], info: bd.DistInfo | None = None, device=None, log=print) -> list[dict[str, Any]]:
    info = info or bd.DistInfo()
    tr = cfg["train"]
    horizon = tr.get("horizon")
    if horizon is not None:
        horizon = int(horizon)
        if horizon < 1:
            raise ValueError(f"train.horizon must be a positive number of steps, got {horizon}")
        if tr.get("seed_streams", "philox") == "numpy":
            raise ValueError("train.horizon needs seed_streams='philox': the reference-seeded episodes play to termination")
    env, agent = build(cfg, int(tr["batch_size"]), info, device)
    out_dir = tr.get("out_dir")
    rows: list[dict[str, Any]] = []
    writer = None
    # resume: ``train.resume`` = path of a checkpoint written by an earlier run (actor, critic, Adam moments, step
    # counters — everything the reference's actor-only save_model loses); ``train.start_batch`` continues the seeds
    # and the CSV (rows are appended, like the reference's safe_append_csv_row, runner.py:662-671)
    start = int(tr.get("start_batch", 0))
    resuming = bool(tr.get("resume")) or start > 0
    if info.rank == 0 and out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "config.json"), "w") as f:
            json.dump(cfg, f, indent=1)
        csv_path = os.path.join(out_dir, "training_stats.csv")
        append = resuming and os.path.exists(csv_path)
        fcsv = open(csv_path, "a" if append else "w", newline="")
        writer = csv.DictWriter(fcsv, fieldnames=["batch", "avg_reward", "max_reward", "min_reward", "max_tile_counts"])
        if not append:
            writer.writeheader()
    best = -float("inf")
    if tr.get("resume"):
        agent.load_checkpoint(tr["resume"])
    ckpt_every = int(tr.get("checkpoint_every", 50))
    streams = tr.get("seed_streams", "philox")
    if streams not in ("philox", "numpy"):
        raise ValueError(f"Unknown train.seed_streams: {streams}")
    if horizon is not None:
        env.reset_many(seed=(int(cfg["seed"]) + 0x9E3779B97F4A7C15 * (start + 1)) & (2**64 - 1))
    if streams == "numpy":
        # the runner's seed iterators, advanced past the batches already played; this rank plays its contiguous slice
        # [gid0, gid0 + num_envs) of every batch's global seed list, so the episodes do not depend on the world size
        bs = int(tr["batch_size"])
        env_it = make_fixed_seed_iter(int(tr.get("env_base_seed", 3)))
        pol_it = make_fixed_seed_iter(int(tr.get("policy_base_seed", 7)))
        for _ in range(start * bs):
            next(env_it), next(pol_it)
    for step in range(start, int(tr["num_batches"])):
        t0 = time.perf_counter()
        global_step = step + 1                                                             # 1-based like runner.py:610
        if horizon is not None:
            row, ro, upd = _horizon_batch(agent, env, info, tr, horizon, global_step, best, out_dir)
            avg, mx, mn = row["avg_reward"], row["max_reward"], row["min_reward"]
            if avg > best:
                best = avg
            rows.append(dict(row, steps=ro.T * ro.B, seconds=time.perf_counter() - t0, grad_norm=upd.get("actor_grad_norm")))
        elif streams == "numpy":
            pairs = [(next(env_it), next(pol_it)) for _ in range(bs)][env.gid0: env.gid0 + env.num_envs]
            ro = agent.run_episodes(env, [e for e, _ in pairs], [p for _, p in pairs])
        else:
            env.seed = (int(cfg["seed"]) + 0x9E3779B97F4A7C15 * (step + 1)) & (2**64 - 1)  # fresh episodes every batch
            ro = agent.rollout_many(env, precision=tr.get("precision", "auto"))
        if horizon is None:
            total = ro.total_reward()
            avg, mx, mn = _global_stats(total, info)
            hist = tile_histogram(env.max_exp, info)
            is_record = avg > best                                                         # runner.py:643-660
            if is_record:
                best = avg
            if global_step > 30 and is_record and info.rank == 0 and out_dir:
                agent.save_model(os.path.join(out_dir, f"best_avg_{avg:.2f}_step_{global_step}.npz"))
            upd = bd.sharded_update(agent, ro, info, total_episodes=int(tr["batch_size"]), exchange=tr.get("exchange", "default"),
                                    bootstrap_truncation=bool(tr.get("bootstrap_truncation", False)))
            row = {"batch": global_step, "avg_reward": avg, "max_reward": mx, "min_reward": mn, "max_tile_counts": json.dumps(hist)}
            rows.append(dict(row, steps=int(ro.length.sum().item()), seconds=time.perf_counter() - t0,
                             grad_norm=upd.get("actor_grad_norm")))
        if writer:
            writer.writerow(row)
            fcsv.flush()
        if info.rank == 0 and out_dir and ckpt_every > 0 and global_step % ckpt_every == 0:
            # a crashed run resumes from here: train.resume = this file, train.start_batch = global_step
            agent.save_checkpoint(os.path.join(out_dir, "checkpoint.npz"))
        if info.rank == 0 and (step % max(1, int(tr["num_batches"]) // 20) == 0 or step == int(tr["num_batches"]) - 1):
            log(f"batch {global_step}: avg_reward={avg:.2f} max={mx:.1f} min={mn:.1f} steps={rows[-1]['steps']} "
                f"sec={rows[-1]['seconds']:.3f}")
    if writer:
        fcsv.close()
    if info.rank == 0 and out_dir:
        agent.save_model(os.path.join(out_dir, "final.npz"))
        agent.save_checkpoint(os.path.join(out_dir, "final_checkpoint.npz"))
    return rows


def _horizon_batch(agent, env, info: bd.DistInfo, tr: dict[str, Any], horizon: int, global_step: int, best: float,
                   out_dir: str | None):
    """One fixed-horizon batch: the window, its update, and the CSV row of the episodes that ended inside it (over all
    ranks).  A record average is checkpointed with the parameters that played the window, as the episode batches are."""
    ro = agent.rollout_many(env, horizon=horizon, reset=False, precision=tr.get("precision", "auto"))
    saving = global_step > 30 and info.rank == 0 and bool(out_dir)
    before = agent.save_state() if saving else None
    upd = bd.sharded_update(agent, ro, info, total_episodes=int(tr["batch_size"]), exchange=tr.get("exchange", "default"),
                            fixed_horizon=True, bootstrap_truncation=bool(tr.get("bootstrap_truncation", False)))
    es = agent.horizon_episode_stats(reset=True, info=info)
    avg = es["avg_reward"]
    if saving and avg > best:                                                              # runner.py:643-660
        after = agent.save_state()
        agent.load_state(before)
        agent.save_model(os.path.join(out_dir, f"best_avg_{avg:.2f}_step_{global_step}.npz"))
        agent.load_state(after)
    row = {"batch": global_step, "avg_reward": avg, "max_reward": es["max_reward"], "min_reward": es["min_reward"],
           "max_tile_counts": json.dumps(es["max_tile_counts"])}
    return row, ro, upd


def evaluation(cfg: dict[str, Any], info: bd.DistInfo | None = None, device=None, agent=None) -> dict[str, Any]:
    info = info or bd.DistInfo()
    ev = cfg["eval"]
    env = bd.make_sharded_env(int(ev["num_episodes"]), Game2048EnvConfig(**cfg["env"]), info, seed=int(cfg["seed"]) + 12345,
                              device=device)
    if agent is None:
        agent = make_agent(cfg, env)
        if ev.get("model_path"):
            agent.load_model(ev["model_path"])
    ro = agent.rollout_many(env, greedy=bool(ev.get("use_greedy", True)), precision=cfg["train"].get("precision", "auto"))
    avg, mx, mn = _global_stats(ro.total_reward(), info)
    return {"avg_reward": avg, "max_reward": mx, "min_reward": mn, "max_tile_counts": tile_histogram(env.max_exp, info),
            "mean_len": float(ro.length.float().mean())}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("-conf", "--config", default=None)
    args = ap.parse_args(argv)
    user = json.load(open(args.config)) if args.config else {}
    cfg = merge_config(user)
    info = bd.init_distributed()
    if cfg["run_mode"].lower().startswith("train"):
        training(cfg, info)
    else:
        res = evaluation(cfg, info)
        if info.rank == 0:
            print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
