"""b2048 — B200-native batched 2048 environment and REINFORCE / actor-critic rollout engine.

Drop-in for the hot path of pqpeqr/RL-2048-with-Reinforce-and-Actor-Critic: the reference's own class
API (Game2048, Game2048Env, MLP free functions, ReinforceAgent) plus batched ``reset_many`` /
``step_many`` / ``rollout_many``.  All arithmetic runs in hand-written sm_100a CUDA kernels reached
through the C ABI in include/b2048.h (libb2048.so, bound with ctypes in ``_lib``).  There is no CPU fallback.
"""
from . import _lib
from ._lib import B2048Error
from .batched_env import Batched2048Env, Game2048EnvConfig, debug_set, get_handle, make_env_cfg, make_fixed_seed_iter
from .game2048 import Game2048
from .env import Game2048Env
from .MLP import (MLPConfig, DeviceMLP, encode_observation, init_model_params, load_model_params, save_model_params,
                  forward_logits, logits_to_probs)
from .reinforce_agent import ReinforceAgent, ReinforceAgentConfig, Rollout
from .shared_trunk import SharedTrunkActorCritic
from .rollout_bench import bench_env_trained_boards, bench_rollout, bench_sharded_sweep, bench_train_iter
from . import dist

__all__ = ["B2048Error", "Batched2048Env", "Game2048EnvConfig", "debug_set", "get_handle", "make_env_cfg", "Game2048",
           "Game2048Env", "MLPConfig", "DeviceMLP", "encode_observation", "init_model_params", "load_model_params",
           "save_model_params", "forward_logits", "logits_to_probs", "ReinforceAgent", "ReinforceAgentConfig",
           "Rollout", "SharedTrunkActorCritic", "make_fixed_seed_iter"]
