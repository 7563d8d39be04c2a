"""Batched2048Env — the batched surface added on top of the reference API (reset_many / step_many).

Holds N boards as packed uint64 in HBM (structure of arrays) and advances all of them with ONE fused
CUDA kernel per step through the C ABI (include/b2048.h).  Semantics per board are exactly those of
the reference's ``Game2048Env.reset/step`` (src/env.py:174-194, :264-302) on ``Game2048``
(src/game2048.py); spawns come from a counter-based Philox stream keyed on the GLOBAL board id so
results do not depend on how boards are sharded over GPUs and can be replayed into the reference.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any

import numpy as np
import torch

from . import _lib
from ._lib import ACT, BONUS, OBS, REWARD, EnvCfg


@dataclass
class Game2048EnvConfig:
    """Same 14 fields, names and defaults as the reference's Game2048EnvConfig (src/env.py:19-40)."""
    size: int = 4
    obs_mode: str = "raw"               # raw / log2 / onehot
    obs_log2_scale: float = 1.0
    reward_mode: str = "sum"            # sum / log2
    base_reward_scale: float = 1.0
    empty_tile_reward: float = 0.0
    merge_reward: float = 0.0
    bonus_mode: str = "off"             # off / raw / log2
    bonus_scale: float = 1.0
    step_reward: float = 0.0
    endgame_penalty: float = 0.0
    use_action_mask: bool = True
    invalid_action_penalty: float = -1.0
    max_steps: int | None = 1024


def make_env_cfg(config: Game2048EnvConfig, action_mode: str = "buffer", auto_reset: bool = False,
                 emit_obs: bool = True, action_priority=(0, 1, 2, 3)) -> EnvCfg:
    if config.size != 4:
        raise ValueError(f"only size=4 boards are packable into 16 x 4-bit exponents (got size={config.size})")
    if config.obs_mode not in ("raw", "log2", "onehot"):
        raise ValueError(f"Unsupported obs_mode: {config.obs_mode}")          # src/env.py:110
    if config.reward_mode not in REWARD:
        raise ValueError(f"Unsupported reward mode: {config.reward_mode}")    # src/env.py:223
    if config.bonus_mode not in BONUS:
        raise ValueError(f"Unsupported bonus mode: {config.bonus_mode}")      # src/env.py:249
    return EnvCfg(REWARD[config.reward_mode], BONUS[config.bonus_mode], OBS[config.obs_mode] if emit_obs else 0,
                  int(bool(config.use_action_mask)), int(config.max_steps) if config.max_steps else 0,
                  ACT[action_mode], int(bool(auto_reset)),
                  sum(int(a) << (4 * k) for k, a in enumerate(action_priority)) if action_mode == "priority" else 0,
                  float(config.base_reward_scale),
                  float(config.empty_tile_reward), float(config.merge_reward), float(config.bonus_scale),
                  float(config.step_reward), float(config.endgame_penalty), float(config.invalid_action_penalty),
                  float(config.obs_log2_scale), 0.0)


_handles: dict[int, Any] = {}


def get_handle(device: torch.device) -> C.c_void_p:
    """One library handle (row tables in HBM) per device."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _handles:
        lib = _lib.load()
        with torch.cuda.device(idx):
            h = C.c_void_p()
            _lib.check(lib.b2048_create(C.byref(h)), "b2048_create")
        _handles[idx] = h
    return _handles[idx]


_debug: dict[str, bool] = {}


def debug_set(option: str, value: bool = True, device: torch.device | str | None = None) -> None:
    """Test / profiling switch of the library handle of `device` (b2048_debug_set, include/b2048.h): "no_fused_rollout",
    "no_fast_step", "tc_clocks", "step_clocks", "no_pdl", "no_update_pipe", the integer "pipe_split"; plus the host-side "no_compact_rollout" (rollout_many plays all
    boards of every chunk instead of the live list).  All off by default."""
    if option == "no_compact_rollout":
        _debug[option] = bool(value)
        return
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(dev):
        v = int(value) if option == "pipe_split" else int(bool(value))
        _lib.check(_lib.load().b2048_debug_set(get_handle(dev), _lib.DEBUG_OPTIONS[option], v), "b2048_debug_set")
    _debug[option] = bool(value)


def debug_get(option: str) -> bool:
    return _debug.get(option, False)


def make_fixed_seed_iter(base_seed: int):
    """The reference runner's per-episode seed iterator (runner.py:244-261): an endless stream of int64 seeds drawn
    from np.random.default_rng(base_seed).  runner.py draws env seeds from make_fixed_seed_iter(env base seed) and
    policy seeds from make_fixed_seed_iter(policy base seed), one of each per episode."""
    rng = np.random.default_rng(base_seed)
    while True:
        yield int(rng.integers(low=0, high=np.iinfo(np.int64).max, dtype=np.int64))


def np_seed_streams(seeds, device: torch.device) -> torch.Tensor:
    """One np.random.default_rng(seed) state per seed on `device` (b2048_np_rng_seed): int64 [n, 6].
    Seeds must be integers in [0, 2^64); anything else raises ValueError, as default_rng does for negative seeds."""
    vals = []
    for s in seeds:
        if isinstance(s, (bool, np.bool_)) or not isinstance(s, (int, np.integer)):
            raise ValueError(f"seed {s!r} is not an integer")
        s = int(s)
        if not 0 <= s < 2**64:
            raise ValueError(f"seed {s} is outside [0, 2^64)")
        vals.append(s)
    n = len(vals)
    host = torch.from_numpy(np.array(vals, dtype=np.uint64).view(np.int64))
    rng = torch.empty((n, _lib.NP_RNG_WORDS), dtype=torch.int64, device=device)
    with torch.cuda.device(device):
        _lib.check(_lib.load().b2048_np_rng_seed(_ptr(host.to(device)), _ptr(rng), n, _stream()), "b2048_np_rng_seed")
    return rng


def _ptr(t: torch.Tensor | None):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Batched2048Env:
    """N independent 2048 games on one GPU.

    State tensors (all on ``device``): ``board`` uint64 [N] (stored as int64), ``score`` int32, ``step`` int32,
    ``max_exp`` uint8, ``flags`` uint8 (see B2048_F_* in include/b2048.h; low 4 bits = legal mask).
    """

    def __init__(self, num_envs: int, config: Game2048EnvConfig | None = None, device: str | torch.device = "cuda",
                 seed: int = 0, gid0: int = 0, track_state: bool = True):
        self.config = config or Game2048EnvConfig()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.B2048Error("Batched2048Env runs on CUDA only; there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs = int(num_envs)
        self.seed = int(seed) & (2**64 - 1)
        self.gid0 = int(gid0)
        self.t = 0
        self.track_state = track_state
        make_env_cfg(self.config)  # validate early, like the reference's constructor (src/env.py:79-110)
        self._lib = _lib.load()
        self._h = get_handle(self.device)
        n, dev = self.num_envs, self.device
        self.board = torch.zeros(n, dtype=torch.int64, device=dev)
        self.flags = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.score = torch.zeros(n, dtype=torch.int32, device=dev) if track_state else None
        self.step_count = torch.zeros(n, dtype=torch.int32, device=dev) if track_state else None
        self.max_exp = torch.full((n,), 2, dtype=torch.uint8, device=dev) if track_state else None
        self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.obs_width = 272 if self.config.obs_mode == "onehot" else 16
        self.env_rng: torch.Tensor | None = None   # per-board NumPy env streams (reset_many(env_seeds=...))

    # ------------------------------------------------------------------ reset
    def reset_many(self, seed: int | None = None, spawn_replay: torch.Tensor | None = None, env_seeds=None
                   ) -> tuple[torch.Tensor, torch.Tensor]:
        """Game2048Env.reset for every board; returns (packed boards, flags).
        env_seeds (one integer per board): board i is reset from np.random.default_rng(env_seeds[i]) exactly like
        Game2048Env.reset(seed=env_seeds[i]), and that generator is kept on the device in ``env_rng`` (int64
        [num_envs, 6]) for the spawns of ReinforceAgent.run_episodes."""
        if seed is not None:
            self.seed = int(seed) & (2**64 - 1)
        self.t = 0
        if env_seeds is not None:
            if len(env_seeds) != self.num_envs:
                raise ValueError(f"{len(env_seeds)} env seeds for {self.num_envs} boards")
            self.env_rng = np_seed_streams(env_seeds, self.device)
            with torch.cuda.device(self.device):
                _lib.check(self._lib.b2048_reset_many_np(self._h, _ptr(self.board), _ptr(self.score), _ptr(self.step_count),
                                                         _ptr(self.max_exp), _ptr(self.flags), _ptr(self.env_rng), self.num_envs,
                                                         _stream()), "b2048_reset_many_np")
            return self.board, self.flags
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_reset_many(self._h, _ptr(self.board), _ptr(self.score), _ptr(self.step_count),
                                                  _ptr(self.max_exp), _ptr(self.flags), _ptr(spawn_replay), self.num_envs, self.seed,
                                                  self.gid0, self.t, _stream()), "b2048_reset_many")
        return self.board, self.flags

    # ------------------------------------------------------------------ step
    def step_many(self, actions: torch.Tensor | None = None, *, action_mode: str | None = None,
                  auto_reset: bool = False, obs_out: torch.Tensor | None = None,
                  action_out: torch.Tensor | None = None, merge_sum_out: torch.Tensor | None = None,
                  reward64_out: torch.Tensor | None = None, board_out: torch.Tensor | None = None,
                  reward_out: torch.Tensor | None = None, flags_out: torch.Tensor | None = None,
                  use_prev_mask: bool = True, spawn_replay: torch.Tensor | None = None,
                  ep_len: torch.Tensor | None = None, ep_t: int = 0, flags_in: torch.Tensor | None = None,
                  action_priority=(0, 1, 2, 3)):
        """One env step for every board.  ``actions`` uint8 [N] on the device, or None with
        ``action_mode`` 'random_legal' / 'random_any' (device-side Philox actions) or 'priority' (the first legal
        action in the order ``action_priority`` — the reference's scripted baselines, tools/simple_action_gen.py:16-33:
        (0, 1, 2, 3) = up, right, down, left; (0, 1, 3, 2) = up, right, left, down).

        Returns (reward float32 [N], flags uint8 [N]); boards are updated in place (or written to
        ``board_out``, e.g. the next slice of a rollout buffer)."""
        mode = action_mode or ("buffer" if actions is not None else "random_legal")
        if mode == "buffer":
            if actions is None:
                raise ValueError("actions required for action_mode='buffer'")
            if actions.dtype != torch.uint8 or actions.device != self.device or actions.numel() != self.num_envs:
                raise ValueError("actions must be a uint8 tensor of shape [num_envs] on the env's device")
        cfg = make_env_cfg(self.config, mode, auto_reset, emit_obs=obs_out is not None, action_priority=action_priority)
        self.t += 1
        reward = reward_out if reward_out is not None else self.reward
        if flags_in is None:
            flags_in = self.flags if (use_prev_mask and (mode in ("random_legal", "priority") or ep_len is not None)) else None
        flags = flags_out if flags_out is not None else self.flags
        b_out = board_out if board_out is not None else self.board
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_step_many(
                self._h, _ptr(self.board), _ptr(b_out), _ptr(self.score), _ptr(self.step_count), _ptr(self.max_exp),
                _ptr(actions) if mode == "buffer" else None, _ptr(action_out), _ptr(flags_in), _ptr(spawn_replay),
                C.byref(cfg),
                _ptr(merge_sum_out), _ptr(reward), _ptr(reward64_out), _ptr(flags), _ptr(obs_out),
                _ptr(ep_len), int(ep_t), self.num_envs, self.seed, self.gid0, self.t, _stream()), "b2048_step_many")
        if board_out is not None:
            self.board = board_out
        if flags_out is not None:
            self.flags = flags_out
        return reward, flags

    def step_many_n(self, n_steps: int, *, action_mode: str = "random_legal", auto_reset: bool = False,
                    action_priority=(0, 1, 2, 3), reward_sum_out: torch.Tensor | None = None,
                    episodes_out: torch.Tensor | None = None):
        """`n_steps` consecutive env steps of a device-side action mode ('random_legal', 'random_any', 'priority') in
        ONE kernel launch: boards, counters and legal masks stay in registers across the steps (b2048_step_many_n).
        Identical to calling step_many n_steps times.  Returns (reward of the last step, flags of the last step);
        ``reward_sum_out`` (float32 [N]) and ``episodes_out`` (int32 [N]) are accumulated into when given."""
        if action_mode not in ("random_legal", "random_any", "priority"):
            raise ValueError("step_many_n needs a device-side action mode")
        cfg = make_env_cfg(self.config, action_mode, auto_reset, emit_obs=False, action_priority=action_priority)
        track = self.score is not None
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_step_many_n(
                self._h, _ptr(self.board), _ptr(self.score), _ptr(self.step_count), _ptr(self.max_exp), _ptr(self.flags), 1,
                C.byref(cfg), _ptr(self.reward), _ptr(reward_sum_out), _ptr(episodes_out), self.num_envs, int(n_steps),
                self.seed, self.gid0, self.t + 1, _stream()), "b2048_step_many_n")
        self.t += int(n_steps)
        return self.reward, self.flags

    # ------------------------------------------------------------------ views
    def encode_obs(self, board: torch.Tensor | None = None) -> torch.Tensor:
        """Game2048Env._preprocess_board (src/env.py:131-150) for every board -> float32 [N,16] / [N,16*17]."""
        b = self.board if board is None else board
        n = b.numel()
        obs = torch.empty((n, self.obs_width), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_encode_obs(_ptr(b), _ptr(obs), OBS[self.config.obs_mode],
                                                  float(self.config.obs_log2_scale), n, _stream()), "b2048_encode_obs")
        return obs

    def action_mask(self) -> torch.Tensor:
        """int8 [N,4] legal-move mask in action order up,right,down,left (src/env.py:154-156)."""
        f = self.flags
        return torch.stack([(f >> a) & 1 for a in range(4)], dim=1).to(torch.int8)

    @property
    def terminated(self) -> torch.Tensor:
        return (self.flags & _lib.F_DONE) != 0

    @property
    def truncated(self) -> torch.Tensor:
        return (self.flags & _lib.F_TRUNC) != 0
