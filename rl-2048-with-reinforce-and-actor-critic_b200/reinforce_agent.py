"""Drop-in for the reference's ``src/reinforce_agent.py`` plus the batched rollout / update engine.

``ReinforceAgent`` keeps the reference's constructor, attributes and methods (``select_action``,
``run_episode``, ``compute_returns``, ``update_batch``, ``save_model`` / ``load_model``; reference
src/reinforce_agent.py:50-252, :357-620).  Parameters live on the GPU as flat float32 vectors; every
numeric step — policy forward + masked softmax + sampling, env step, returns scan, advantages, TD
errors, back-propagation, global-norm clip, SGD / Adam — is a CUDA kernel reached through the C ABI.

Added surface: ``rollout_many`` (run-to-termination or fixed-horizon rollouts of a whole
``Batched2048Env``) and ``update_from_rollout``; ``update_batch`` packs reference-style trajectories
into the same rollout buffers and calls the same kernels.  ``update_from_horizon`` trains on fixed-horizon
windows with reset-on-done (segment-aware returns / TD / GAE, ``horizon_episode_stats`` for logging); ``update_ppo`` runs
several epochs of clipped-ratio minibatch steps on such a window.  The window updates and ``update_from_rollout`` can
bootstrap truncated episodes from the critic (``bootstrap_truncation=True``).  ``lookahead_actions`` and
``rollout_lookahead`` play with the critic: a one-ply expectimax over every move and spawn, expanded on the device.
"""
from __future__ import annotations

import ctypes as C
import logging
import math
import os
from collections.abc import Callable
from dataclasses import dataclass, replace
from typing import Any

import numpy as np
import torch

from . import _lib
from .MLP import (DeviceMLP, MLPConfig, encode_observation, init_model_params, load_model_params,  # noqa: F401
                  save_model_params, forward_logits, logits_to_probs)
from .batched_env import Batched2048Env, _ptr, _stream, debug_get, get_handle
from .env import Game2048Env

if not hasattr(logging, "VERBOSE"):  # the reference's custom level (src/utils/logging_ext.py)
    logging.addLevelName(15, "VERBOSE")
    logging.VERBOSE = 15
if not hasattr(logging.Logger, "verbose"):
    def _verbose(self, message, *args, **kwargs):
        if self.isEnabledFor(15):
            self._log(15, message, args, **kwargs)
    logging.Logger.verbose = _verbose

BASELINE = {"off": 0, "each": 1, "batch": 2, "batch_norm": 3}
OPTIMIZER = {"sgd": 0, "adam": 1}


@dataclass
class ReinforceAgentConfig:
    """Same 15 fields / defaults as the reference (src/reinforce_agent.py:24-46)."""
    gamma: float = 1
    learning_rate: float = 1e-3
    baseline_mode: str = "off"                  # "off" / "each" / "batch" / "batch_norm"
    model_seed: int = 0
    reward_rank_weights: list[float] | None = None
    optimizer: str = "sgd"
    adam_beta1: float = 0.9
    adam_beta2: float = 0.999
    augmentation: bool = False
    use_critic: bool = False
    critic_learning_rate: float = 1e-3
    max_grad_norm: float = 1.0
    critic_loss_type: str = "mse"
    huber_delta: float = 1.0


@dataclass
class Rollout:
    """Time-major rollout buffers on the device.  boards/flags have T+1 slices (state before each step and
    the final state); flags[t] low nibble is the legal mask of boards[t]."""
    boards: torch.Tensor      # int64  [T+1, B]
    flags: torch.Tensor       # uint8  [T+1, B]
    actions: torch.Tensor     # uint8  [T, B]
    rewards: torch.Tensor     # float32 [T, B]
    length: torch.Tensor      # int32  [B]  episode length (steps); == T for fixed-horizon rollouts
    T: int
    ep_weight: torch.Tensor | None = None   # float32 [B] episode rank weights (None = 1)
    n_traj: int | None = None               # divisor of the per-episode weight (defaults to B)
    auto_reset: bool = False                # fixed-horizon rollout with reset-on-done: a lane holds SEVERAL episodes
    # The Philox env streams the rollout played on (rollout_many): the env seed, the global id of lane 0 and the env
    # counter before the first step (step t of lane b spawned from counter t0 + t + 1).  A window needs them to replay
    # the boards its truncated episodes were cut on (update_from_horizon(bootstrap_truncation=True)).
    seed: int | None = None
    gid0: int | None = None
    t0: int | None = None

    @property
    def B(self) -> int:
        return int(self.length.numel())

    def total_reward(self) -> torch.Tensor:
        t = torch.arange(self.T, device=self.rewards.device).unsqueeze(1)
        return (self.rewards[: self.T].double() * (t < self.length.unsqueeze(0))).sum(0)


class ReinforceAgent:
    gae_lambda = 0.0                # set by SharedTrunkActorCritic; 0 = the reference's TD(0) advantages
    _adam_t_c = 0                   # Adam step counter of a separate critic

    def __init__(self, env, mlp_config: MLPConfig, agent_config: ReinforceAgentConfig | None = None,
                 initial_params_path: str | None = None):
        self.env = env
        self.mlp_config = mlp_config
        self.agent_config = agent_config or ReinforceAgentConfig()
        self.rng = np.random.default_rng(self.agent_config.model_seed)
        self._logger = logging.getLogger(__name__ + ".ReinforceAgent")
        if not self._logger.handlers:
            self._logger.addHandler(logging.NullHandler())

        ecfg = env.config
        self.device = env.device if isinstance(env, Batched2048Env) else env._benv.device
        self._obs_mode = ecfg.obs_mode
        self._obs_scale = float(ecfg.obs_log2_scale) if ecfg.obs_mode == "log2" else 1.0
        self._use_mask = bool(ecfg.use_action_mask)
        input_dim = 272 if ecfg.obs_mode == "onehot" else 16
        n_actions = 4
        if not isinstance(env, Batched2048Env):
            obs, _ = env.reset(seed=0)                                    # reinforce_agent.py:70-73
            x, _ = encode_observation(obs)
            input_dim = x.shape[0]
            n_actions = env.action_space.n
        self._lib = _lib.load()
        self._h = get_handle(self.device)

        if initial_params_path is None:
            params = init_model_params(input_dim, self.mlp_config.hidden_sizes, n_actions, self.rng,
                                       self.mlp_config.init_distribution, self.mlp_config.last_init_normal)
        else:
            params = load_model_params(initial_params_path)
        self._actor = self._make_net(params)
        self._adam_t = 0
        self._critic: DeviceMLP | None = None
        if self.agent_config.use_critic:                                  # separate critic network, :94-105
            cparams = init_model_params(input_dim, self.mlp_config.hidden_sizes, 1, self.rng,
                                        self.mlp_config.init_distribution, self.mlp_config.last_init_normal)
            self._critic = self._make_net(cparams)
        self._bind_grads()
        self._scratch: dict[str, torch.Tensor] = {}
        self.last_update_info: dict[str, Any] = {}

    # ------------------------------------------------------------------ parameters
    def _make_net(self, params) -> DeviceMLP:
        net = DeviceMLP(params, self.mlp_config.activation, self._obs_mode, self._obs_scale, self.device)
        net.adam_m = torch.zeros_like(net.theta)
        net.adam_v = torch.zeros_like(net.theta)
        net.grad = torch.zeros_like(net.theta)
        return net

    def _bind_grads(self) -> None:
        """The gradients of the actor and (when present) the critic are views into ONE flat float32 buffer
        [actor | critic], so a sharded update exchanges them with a single all-reduce (SURVEY.md section 8e)."""
        nets = [self._actor] + ([self._critic] if self._critic is not None else [])
        self._grad_all = torch.zeros(sum(n.n_params for n in nets), dtype=torch.float32, device=self.device)
        off = 0
        for n in nets:
            n.grad = self._grad_all[off: off + n.n_params]
            off += n.n_params

    @property
    def params(self) -> dict[str, Any]:
        """Reference layout {"W": [...], "b": [...]} (host copies of the device parameters)."""
        return self._actor.to_params()

    @params.setter
    def params(self, value: dict[str, Any]) -> None:
        dims = [np.asarray(value["W"][0]).shape[0]] + [np.asarray(W).shape[1] for W in value["W"]]
        if dims == self._actor.dims:
            self._actor.load_params(value)
        else:
            self._actor = self._make_net(value)
            self._bind_grads()

    @property
    def critic_params(self):
        return None if self._critic is None else self._critic.to_params()

    @critic_params.setter
    def critic_params(self, value) -> None:
        if value is None:
            self._critic = None
            self._bind_grads()
        elif self._critic is not None and [np.asarray(W).shape for W in value["W"]] == \
                [(self._critic.dims[l], self._critic.dims[l + 1]) for l in range(self._critic.n_layers)]:
            self._critic.load_params(value)
        else:
            self._critic = self._make_net(value)
            self._bind_grads()

    def load_model(self, file_path: str | None = "params.npz") -> None:
        self.params = load_model_params(file_path)
        self.mlp_config.hidden_sizes = [int(d) for d in self._actor.dims[1:-1]]   # reinforce_agent.py:114
        self._logger.info(f"Model parameters loaded from {file_path}")

    def save_model(self, file_path: str | None = "params.npz") -> None:
        save_model_params(self.params, file_path)                                 # actor only, like the reference

    # The reference's save_model keeps the actor alone (reinforce_agent.py:119-123), so a run cannot be resumed: the
    # critic, the Adam moments and the step counters are lost.  save_checkpoint / load_checkpoint keep all of it.
    def save_checkpoint(self, file_path: str) -> None:
        """Everything update_batch mutates: actor, critic, Adam moments and step counters (one .npz)."""
        out = {"actor_theta": self._actor.theta.cpu().numpy(), "actor_dims": np.asarray(self._actor.dims, np.int64),
               "actor_adam_m": self._actor.adam_m.cpu().numpy(), "actor_adam_v": self._actor.adam_v.cpu().numpy(),
               "adam_t": np.int64(self._adam_t), "adam_t_c": np.int64(self._adam_t_c),
               "has_critic": np.int64(self._critic is not None)}
        if self._critic is not None:
            out.update(critic_theta=self._critic.theta.cpu().numpy(), critic_dims=np.asarray(self._critic.dims, np.int64),
                       critic_adam_m=self._critic.adam_m.cpu().numpy(), critic_adam_v=self._critic.adam_v.cpu().numpy())
        np.savez(file_path, **out)

    def save_state(self) -> dict[str, Any]:
        """Device-side snapshot of everything an update mutates (see save_checkpoint), for load_state."""
        st = {"adam_t": self._adam_t, "adam_t_c": self._adam_t_c}
        for name, net in (("actor", self._actor), ("critic", self._critic)):
            if net is not None:
                st[name] = (net.theta.clone(), net.adam_m.clone(), net.adam_v.clone())
        return st

    def load_state(self, st: dict[str, Any]) -> None:
        self._adam_t = st["adam_t"]
        if self._critic is not None:
            self._adam_t_c = st["adam_t_c"]
        for name, net in (("actor", self._actor), ("critic", self._critic)):
            if net is not None:
                for dst, src in zip((net.theta, net.adam_m, net.adam_v), st[name]):
                    dst.copy_(src)

    def load_checkpoint(self, file_path: str) -> None:
        ck = np.load(file_path if str(file_path).endswith(".npz") else str(file_path) + ".npz")

        def restore(net, prefix):
            if [int(d) for d in ck[prefix + "_dims"]] != [int(d) for d in net.dims]:
                raise ValueError(f"checkpoint {prefix} shape {ck[prefix + '_dims'].tolist()} != network {net.dims}")
            net.theta.copy_(torch.from_numpy(ck[prefix + "_theta"]).to(self.device))
            net.adam_m.copy_(torch.from_numpy(ck[prefix + "_adam_m"]).to(self.device))
            net.adam_v.copy_(torch.from_numpy(ck[prefix + "_adam_v"]).to(self.device))

        if bool(int(ck["has_critic"])) != (self._critic is not None):
            raise ValueError(f"checkpoint has_critic={int(ck['has_critic'])} but the agent was built with "
                             f"use_critic={self._critic is not None}")
        restore(self._actor, "actor")
        if self._critic is not None:
            restore(self._critic, "critic")
            self._adam_t_c = int(ck["adam_t_c"])
        self._adam_t = int(ck["adam_t"])

    # ------------------------------------------------------------------ kernels
    def _buf(self, name: str, shape, dtype) -> torch.Tensor:
        t = self._scratch.get(name)
        n = int(np.prod(shape))
        if t is None or t.dtype != dtype or t.numel() < n:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._scratch[name] = t
        return t[:n].view(*shape) if n else t[:0]

    def policy_step(self, boards: torch.Tensor, flags: torch.Tensor | None, actions_out: torch.Tensor | None,
                    seed: int, gid0: int, t: int, greedy: bool = False, probs_out: torch.Tensor | None = None,
                    logits_out: torch.Tensor | None = None, precision: int | str = 0) -> None:
        """encode_observation -> forward_logits -> logits_to_probs -> sample/greedy for a batch of packed boards.
        precision: 0 = fp32 CUDA cores (parity path), 1 = bf16 tcgen05 tensor cores, "auto" = 1 when the batch has
        at least 4096 boards and the network is the 16-256-256-4 ReLU shape the tensor-core kernel implements."""
        if precision == "auto":
            precision = 1 if (boards.numel() >= 4096 and self.tc_supported()) else 0
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_policy_step(
                self._h, _ptr(boards), _ptr(flags) if self._use_mask else None, C.byref(self._actor.desc),
                _ptr(actions_out), _ptr(probs_out), _ptr(logits_out), boards.numel(), seed & (2**64 - 1), gid0, t,
                int(greedy), precision, _stream()), "b2048_policy_step")

    def _update_mode_name(self, prec: int, n: int) -> str:
        """Which arithmetic b2048_mlp_backward ran for `prec` on n samples (include/b2048.h)."""
        big = n >= 4096
        if prec in (2, 3) and big and self._fused_shape() and self._actor.obs_mode == "log2":
            return "fp16 split tcgen05 (float32-grade forward, fp16 backward with loss scale)"
        if prec in (2, 3) and big and self._generic_tc_shape():
            return "fp16 split tcgen05, shape-generic kernels (float32-grade forward, fp16 backward with loss scale)"
        if prec == 1 and big and self._fused_shape():
            return "bf16 tcgen05"
        return "fp32 CUDA cores"

    def _fused_shape(self) -> bool:
        """The runner-default 16-256-256-4 ReLU network: hand-specialised kernels (fused persistent rollout, update pipeline)."""
        a = self._actor
        return (a.dims == [16, 256, 256, 4] and a.activation == "ReLU" and a.obs_mode in ("raw", "log2"))

    def _generic_tc_shape(self) -> bool:
        """Shapes of the shape-generic tcgen05 kernels (csrc/b2048_mlp_gen.cu): ReLU or Sigmoid, 1-4 hidden layers of 64 / 128 /
        192 / 256 units, log2 or one-hot observations — e.g. the reference's documented one-hot [256, 128, 64] network (runner.py:27-47)."""
        a = self._actor
        hidden = a.dims[1:-1]
        return (a.activation in ("ReLU", "Sigmoid") and a.obs_mode in ("log2", "onehot") and 1 <= len(hidden) <= 4 and
                all(h % 64 == 0 and 64 <= h <= 256 for h in hidden) and 1 <= a.dims[-1] <= 4)

    def tc_supported(self) -> bool:
        """True when batches of >= 4096 boards run on the tensor cores (policy steps at precision 1, updates at "auto")."""
        return self._fused_shape() or self._generic_tc_shape()

    def _values(self, boards: torch.Tensor, out: torch.Tensor, precision: int = 0) -> None:
        self._net_forward(self._critic, boards, out, precision)

    def _net_forward(self, net: DeviceMLP, boards: torch.Tensor, out: torch.Tensor, precision: int = 0) -> None:
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_mlp_forward(self._h, _ptr(boards), C.byref(net.desc), _ptr(out), boards.numel(),
                                                   int(precision), _stream()), "b2048_mlp_forward")

    def _forward_checked(self, net: DeviceMLP, boards: torch.Tensor, out: torch.Tensor, prec: int, fell_back: list,
                         head_mode: int) -> None:
        """b2048_mlp_forward at prec.  The split-fp16 path keeps activations in fp16: a network whose activations leave the
        fp16 range gives non-finite outputs, which are recomputed on the fp32 kernels; head_mode is then appended to
        fell_back."""
        self._net_forward(net, boards, out, prec)
        if prec in (2, 3) and not bool(torch.isfinite(out).all()):
            self._net_forward(net, boards, out, 0)
            fell_back.append(head_mode)

    @staticmethod
    def _update_precision(precision: int | str) -> int:
        """The precision code of the learner's forward / backward passes for an update's `precision` argument."""
        return 2 if precision == "auto" else int(precision)

    def _precision_info(self, prec: int, n: int, fell_back: list) -> str:
        """info["precision"] of an update of n samples at prec."""
        return self._update_mode_name(prec, n) + (" [fell back to fp32: non-finite fp16 intermediates]" if fell_back else "")

    @staticmethod
    def _small_batch_precision(prec: int, n: int) -> int:
        """The tensor-core kernels take 4096 boards or more; a shorter batch runs where "auto" (2) would put it."""
        return prec if (n >= 4096 or prec in (0, 2)) else (2 if prec == 3 else 0)

    def _backward(self, net: DeviceMLP, boards, mflags, acts, cf: torch.Tensor, n: int, head_mode: int, prec: int, chunk: int,
                  fell_back: list, ent_cf: torch.Tensor | None = None, ent_acc: torch.Tensor | None = None) -> None:
        """net.grad = b2048_mlp_backward of the n samples (head 0: sum cf log pi(a|s), head 1: sum cf V(s)) at prec.  A
        non-finite split-fp16 gradient (fp16 range exceeded) is never applied: the pass is redone in fp32 and head_mode is
        appended to fell_back.  ent_cf (policy head): b2048_mlp_backward_entropy, + sum ent_cf H(pi(.|s)), and the pass's
        sum of H is added to ent_acc (device double[1])."""
        lib, h = self._lib, self._h
        ws_floats = int(lib.b2048_backward_workspace_floats(C.byref(net.desc), min(chunk, n)))
        ws = self._buf("bwd_ws", (ws_floats,), torch.float32)
        es = self._buf("ent_sum_pass", (1,), torch.float64) if ent_cf is not None else None
        for p_try in ((prec, 0) if prec in (2, 3) else (prec,)):
            net.grad.zero_()
            with torch.cuda.device(self.device):
                if ent_cf is None:
                    _lib.check(lib.b2048_mlp_backward(h, _ptr(boards), _ptr(mflags) if self._use_mask else None, _ptr(acts),
                                                      _ptr(cf), C.byref(net.desc), _ptr(net.grad), n, head_mode, _ptr(ws),
                                                      ws_floats, min(chunk, n), p_try, _stream()), "b2048_mlp_backward")
                else:
                    es.zero_()
                    _lib.check(lib.b2048_mlp_backward_entropy(
                        h, _ptr(boards), _ptr(mflags) if self._use_mask else None, _ptr(acts), _ptr(cf), _ptr(ent_cf),
                        C.byref(net.desc), _ptr(net.grad), n, _ptr(ws), ws_floats, min(chunk, n), p_try, _ptr(es), _stream()),
                        "b2048_mlp_backward_entropy")
            if p_try == 0 or bool(torch.isfinite(net.grad).all()):
                break
            fell_back.append(head_mode)
            self._logger.warning("tensor-core gradient not finite (fp16 range exceeded); recomputing on the fp32 kernels")
        if es is not None and ent_acc is not None:
            ent_acc += es

    @staticmethod
    def _check_entropy(entropy_coef: float, exchange: str = "default", precision: int | str = "auto") -> float:
        """entropy_coef (beta of the bonus beta H(pi(.|s))) as a float; the configurations without an entropy kernel raise."""
        beta = float(entropy_coef)
        if not (math.isfinite(beta) and beta >= 0.0):
            raise ValueError(f"entropy_coef must be finite and >= 0, got {entropy_coef}")
        if beta > 0.0 and exchange == "one_message":
            raise ValueError("entropy_coef > 0 is not implemented with exchange='one_message' (the actor gradient is formed "
                             "as (g_A - mean g_B) / std there; the bonus would need a third backward pass)")
        if beta > 0.0 and precision != "auto" and int(precision) == 1:
            raise ValueError("entropy_coef > 0 is not implemented on the single-bf16 path (precision=1)")
        return beta

    def _apply(self, net, lr: float, sign: float, t_adam: int) -> torch.Tensor:
        """b2048_apply_update (global-norm clip, SGD / Adam) of net.grad; returns the device double[1] squared norm."""
        cfg = self.agent_config
        sumsq = self._buf("sumsq_" + str(sign), (1,), torch.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_apply_update(self._h, _ptr(net.theta), _ptr(net.grad), _ptr(net.adam_m), _ptr(net.adam_v),
                                                    net.n_params, OPTIMIZER[cfg.optimizer], float(lr), float(sign),
                                                    float(cfg.max_grad_norm), float(cfg.adam_beta1), float(cfg.adam_beta2),
                                                    int(t_adam), _ptr(sumsq), _stream()), "b2048_apply_update")
        return sumsq

    def _optimizer_step(self) -> tuple[torch.Tensor, torch.Tensor | None]:
        """One optimizer step of the actor and of a separate critic, each Adam counter advanced once; returns their squared
        gradient norms (device double[1]; None without a critic)."""
        cfg = self.agent_config
        if cfg.optimizer == "adam":
            self._adam_t += 1
        ss_a = self._apply(self._actor, cfg.learning_rate, +1.0, self._adam_t)
        ss_c = None
        if self._has_value_function():
            if cfg.optimizer == "adam":
                self._adam_t_c += 1
            ss_c = self._apply(self._critic, cfg.critic_learning_rate, -1.0, self._adam_t_c)
        return ss_a, ss_c

    def _step(self, allreduce) -> tuple[torch.Tensor, torch.Tensor | None]:
        """What follows the backward passes of an update step: ONE all-reduce of [actor gradient | critic gradient] when
        sharded, then _optimizer_step."""
        if allreduce is not None:
            allreduce(self._grad_all)
        return self._optimizer_step()

    def _has_value_function(self) -> bool:
        """A separate critic (use_critic=True) or SharedTrunkActorCritic's value head."""
        return bool(self.agent_config.use_critic) and self._critic is not None

    # ------------------------------------------------------------------ reference API: acting
    def _obs_to_packed(self, obs) -> tuple[int, int]:
        board = obs["board"] if isinstance(obs, dict) else obs
        b = np.asarray(board)
        if self._obs_mode == "onehot":
            e = b.reshape(16, -1).argmax(1)
        elif self._obs_mode == "log2":
            e = np.rint(b.reshape(16) / np.float32(self._obs_scale)).astype(np.int64)
        else:
            e = np.array([0 if v == 0 else int(v).bit_length() - 1 for v in b.reshape(16).astype(np.int64)])
        packed = 0
        for i, x in enumerate(e):
            packed |= int(x) << (4 * i)
        mask = 0xF
        if isinstance(obs, dict) and obs.get("action_mask") is not None:
            mask = sum(int(v) << a for a, v in enumerate(obs["action_mask"]))
        return packed, mask

    def _forward_cache(self, obs) -> tuple[list[np.ndarray], list[np.ndarray]]:
        """forward_logits' cached activations [a_0 .. a_L] and pre-activations [z_0 .. z_{L-1}] of the actor for one
        observation (src/MLP.py:159-196), computed by b2048_dense_forward on the device parameters."""
        x, _ = encode_observation(obs)
        net = self._actor
        L = net.n_layers
        xd = torch.from_numpy(np.ascontiguousarray(x.reshape(1, -1), dtype=np.float32)).to(self.device)
        acts = [torch.empty((1, net.dims[l + 1]), dtype=torch.float32, device=self.device) for l in range(L)]
        pres = [torch.empty((1, net.dims[l + 1]), dtype=torch.float32, device=self.device) for l in range(L)]
        act_ptrs = (C.c_void_p * (L + 1))(None, *[a.data_ptr() for a in acts])
        pre_ptrs = (C.c_void_p * L)(*[p.data_ptr() for p in pres])
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_dense_forward(self._h, _ptr(xd), C.byref(net.desc), act_ptrs, pre_ptrs, 1, _stream()),
                       "b2048_dense_forward")
        return [x] + [a.cpu().numpy()[0] for a in acts], [p.cpu().numpy()[0] for p in pres]

    def select_action(self, obs, rng: np.random.Generator, action_fn: Callable[[Any, np.ndarray | None], int] | None = None,
                      use_greedy: bool = False, return_cache: bool = True):
        """Same contract as reinforce_agent.py:126-192.  Probabilities come from the fused policy kernel; the
        final draw uses the caller's NumPy generator (``rng.choice``) exactly like the reference, so a given
        ``policy_seed`` reproduces the reference's episode.  Returns (action, probs, activations, pre_activations)
        with the reference's cached layer outputs (forward_logits' second / third return values); ``return_cache=False``
        (what run_episode passes: it discards them, reinforce_agent.py:222-227) skips that extra forward and returns
        two empty lists."""
        packed, mask = self._obs_to_packed(obs)
        action_mask = obs["action_mask"] if isinstance(obs, dict) else None
        # one pinned-host -> device copy carries the board and its mask (single-env path: every copy is a round trip)
        if getattr(self, "_sa_dev", None) is None:
            self._sa_host = torch.zeros(16, dtype=torch.uint8).pin_memory()
            self._sa_dev = torch.zeros(16, dtype=torch.uint8, device=self.device)
        self._sa_host[0:8] = torch.from_numpy(np.array([packed], dtype=np.uint64).view(np.uint8))
        self._sa_host[8] = mask
        self._sa_dev.copy_(self._sa_host, non_blocking=True)
        b = self._sa_dev[0:8].view(torch.int64)
        f = self._sa_dev[8:9]
        probs_d = self._buf("sa_probs", (1, 4), torch.float32)
        self.policy_step(b, f if action_mask is not None else None, None, 0, 0, 0, probs_out=probs_d)
        probs = probs_d.cpu().numpy()[0].copy()
        action = None
        if action_fn is not None:
            try:
                candidate = int(action_fn(self.env.state, action_mask))
            except Exception as e:
                self._logger.exception(f"action_fn raised an exception: {e}. Falling back to policy.")
            else:
                if not (0 <= candidate < len(probs)):
                    self._logger.warning(f"action_fn returned out-of-range action {candidate}, falling back to policy.")
                elif action_mask is not None and not bool(action_mask[candidate]):
                    self._logger.warning(f"action_fn returned masked-out action {candidate}, falling back to policy.")
                else:
                    action = candidate
        if action is None:
            if use_greedy:
                p = probs * action_mask if action_mask is not None else probs
                action = int(np.argmax(p))
            else:
                action = int(rng.choice(len(probs), p=probs))
        if not return_cache:
            return action, probs, [], []
        activations, pre_activations = self._forward_cache(obs)
        return action, probs, activations, pre_activations

    def run_episode(self, env_seed: int, policy_seed: int, action_gen=None, use_greedy: bool = False) -> dict[str, Any]:
        """One episode on the single-env drop-in (reinforce_agent.py:195-252); same trajectory dict."""
        obs, info = self.env.reset(seed=env_seed)
        state = self.env.render(mode="ansi")
        policy_rng = np.random.default_rng(policy_seed)
        obs_list, action_list, reward_list, states_list = [], [], [], []
        done, total_reward = False, 0.0
        while not done:
            action, _, _, _ = self.select_action(obs, policy_rng, action_gen, use_greedy=use_greedy, return_cache=False)
            next_obs, reward, terminated, truncated, info = self.env.step(action)
            reward = float(reward)
            obs_list.append(obs); action_list.append(action); reward_list.append(reward); states_list.append(state)
            total_reward += reward
            obs = next_obs
            done = terminated or truncated
            state = self.env.render(mode="ansi")
        return {"obs": obs_list, "actions": action_list, "rewards": reward_list, "total_reward": total_reward,
                "states": states_list, "max_tile": self.env.max_tile_seen}

    # ------------------------------------------------------------------ batched rollouts
    def rollout_many(self, benv: Batched2048Env, max_steps: int | None = None, horizon: int | None = None,
                     greedy: bool = False, precision: int | str = 0, reset: bool = True, check_every: int = 48) -> Rollout:
        """Rolls the whole batch with the current policy.
        horizon=None: every board plays to termination / truncation like run_episode (finished boards are
        frozen by the step kernel); horizon=H: fixed H steps with reset-on-done (all lanes always live)."""
        B = benv.num_envs
        if reset:
            benv.reset_many()
        fixed = horizon is not None
        cap = int(horizon) if fixed else int(max_steps or benv.config.max_steps or 4096)
        boards, flags, actions, rewards, length = self._rollout_buffers(benv, cap)
        if precision == "auto":
            precision = 1 if (B >= 4096 and self.tc_supported()) else 0
        from .batched_env import make_env_cfg
        cfg = make_env_cfg(benv.config, "buffer", auto_reset=fixed, emit_obs=False)
        t0 = benv.t
        T = 0
        # Run-to-termination on the fused tensor-core kernel: every chunk plays only the boards that are still alive
        # (slot_map), so finished episodes cost nothing.  Slices beyond an episode's end are then never written: the
        # rewards buffer is zeroed first (total_reward sums whole columns) and the final state is gathered below.
        compact = (not fixed) and int(precision) == 1 and B >= 4096 and not debug_get("no_compact_rollout") and \
            ((self._fused_shape() and not debug_get("no_fused_rollout")) or (not self._fused_shape() and self._generic_tc_shape()))
        if compact:
            rewards.zero_()

            def launch(T, chunk, slot_map, upper, count):
                _lib.check(self._lib.b2048_rollout_many(
                    self._h, _ptr(boards), _ptr(flags), _ptr(actions), _ptr(rewards), _ptr(benv.score),
                    _ptr(benv.step_count), _ptr(benv.max_exp), _ptr(length), C.byref(cfg), C.byref(self._actor.desc), B, T,
                    chunk, benv.seed, benv.gid0, t0, int(self._use_mask), int(greedy), 1, slot_map, upper, count, _stream()),
                    "b2048_rollout_many")

            T = self._live_chunks(launch, length, cap, check_every)
        while not compact and T < cap:
            chunk = min(check_every if not fixed else 256, cap - T)
            with torch.cuda.device(self.device):
                _lib.check(self._lib.b2048_rollout_many(
                    self._h, _ptr(boards), _ptr(flags), _ptr(actions), _ptr(rewards), _ptr(benv.score), _ptr(benv.step_count),
                    _ptr(benv.max_exp), None if fixed else _ptr(length), C.byref(cfg), C.byref(self._actor.desc), B, T,
                    chunk, benv.seed, benv.gid0, t0, int(self._use_mask), int(greedy), int(precision),
                    None, 0, None, _stream()), "b2048_rollout_many")
            T += chunk
            if not fixed and bool((length != 0).all()):
                break
        benv.t = t0 + T
        if fixed:
            length.fill_(T)
        else:
            length = torch.where(length == 0, torch.full_like(length, T), length)  # cut off by the cap
        if compact:
            # the last written slice of board b is length[b]
            idx = length.long().unsqueeze(0)
            benv.board = boards[: T + 1].gather(0, idx).reshape(-1)
            fl = flags[: T + 1].gather(0, idx).reshape(-1)
            # like the frozen pass-through of the step kernel: an episode that ended before T no longer reports "changed"
            benv.flags = torch.where(length < T, fl & 0xEF, fl)
            return Rollout(boards[: T + 1], flags[: T + 1], actions[:T], rewards[:T], length, T, seed=benv.seed, gid0=benv.gid0,
                           t0=t0)
        benv.board = boards[T]
        benv.flags = flags[T]
        return Rollout(boards[: T + 1], flags[: T + 1], actions[:T], rewards[:T], length, T, auto_reset=fixed, seed=benv.seed,
                       gid0=benv.gid0, t0=t0)

    def _rollout_buffers(self, benv: Batched2048Env, cap: int):
        """(boards, flags, actions, rewards, length) scratch buffers for up to cap steps of benv's boards, slice 0 holding
        the current boards and flags, and zeroed lengths."""
        B = benv.num_envs
        boards = self._buf("ro_boards", (cap + 1, B), torch.int64)
        flags = self._buf("ro_flags", (cap + 1, B), torch.uint8)
        actions = self._buf("ro_actions", (cap, B), torch.uint8)
        rewards = self._buf("ro_rewards", (cap, B), torch.float32)
        length = torch.zeros(B, dtype=torch.int32, device=self.device)
        boards[0].copy_(benv.board)
        flags[0].copy_(benv.flags)
        return boards, flags, actions, rewards, length

    def _live_chunks(self, launch, length: torch.Tensor, cap: int, check_every: int) -> int:
        """Run-to-termination chunks on the live-board list: launch(T, chunk, slot_map, upper, count) enqueues steps
        [T, T + chunk) for the listed boards (every board for the first chunk).  Live-board bookkeeping stays on the
        device: after every chunk b2048_compact_live rebuilds the list and its count, the next chunk's kernels read the
        count from device memory, and the host only looks at the count of the chunk BEFORE the one it has just enqueued
        (pinned copy + event) — the GPU never waits for the host.  Returns the number of steps played."""
        B = int(length.numel())
        slot_buf = self._buf("ro_slot_map", (B,), torch.int32)
        count_dev = self._buf("ro_live_count", (1,), torch.int32)
        n_max = (cap + check_every - 1) // check_every + 1
        count_host = getattr(self, "_ro_count_host", None)
        if count_host is None or count_host.numel() < n_max:
            count_host = self._ro_count_host = torch.zeros(n_max, dtype=torch.int32).pin_memory()
        events: list[torch.cuda.Event] = []
        T, upper, k = 0, B, 0
        while T < cap:
            chunk = min(check_every, cap - T)
            with torch.cuda.device(self.device):
                launch(T, chunk, _ptr(slot_buf) if k > 0 else None, upper, _ptr(count_dev) if k > 0 else None)
                _lib.check(self._lib.b2048_compact_live(self._h, _ptr(length), B, _ptr(slot_buf), _ptr(count_dev), _stream()),
                           "b2048_compact_live")
            count_host[k: k + 1].copy_(count_dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            events.append(ev)
            T += chunk
            if k >= 1:                      # boards alive after chunk k - 1 (that copy finished before chunk k started)
                events[k - 1].synchronize()
                alive = int(count_host[k - 1])
                if alive == 0:              # chunk k found nothing to play
                    T -= chunk
                    break
                upper = alive
            k += 1
        return T

    def run_episodes(self, benv: Batched2048Env, env_seeds, policy_seeds, use_greedy: bool = False,
                     max_steps: int | None = None, check_every: int = 48, live_list: bool = True) -> Rollout:
        """The batched run_episode(env_seed, policy_seed) (reinforce_agent.py:195-252): board b plays exactly the episode
        run_episode(env_seeds[b], policy_seeds[b]) plays — its spawns come from np.random.default_rng(env_seeds[b]) and
        its sampled actions from rng.choice(4, p=probs) on np.random.default_rng(policy_seeds[b]), both kept on the
        device (b2048_rollout_many_np).  The policy runs on the fp32 kernel, the one run_episode uses: a tensor-core
        policy computes other probabilities and would sample other actions.  len(env_seeds) == len(policy_seeds) ==
        benv.num_envs; seeds are integers in [0, 2^64).  Every board plays to termination / truncation (max_steps caps
        the length like rollout_many); after the first chunk the policy visits only the boards still playing
        (live_list=False: every board every step — the same episodes, for testing).  Returns a run-to-termination
        Rollout for update_from_rollout; the episodes' max tiles are 2 ** benv.max_exp."""
        B = benv.num_envs
        if len(env_seeds) != B or len(policy_seeds) != B:
            raise ValueError(f"{len(env_seeds)} env seeds and {len(policy_seeds)} policy seeds for {B} boards")
        from .batched_env import make_env_cfg, np_seed_streams
        policy_rng = np_seed_streams(policy_seeds, self.device)
        benv.reset_many(env_seeds=env_seeds)
        cap = int(max_steps or benv.config.max_steps or 4096)
        boards, flags, actions, rewards, length = self._rollout_buffers(benv, cap)
        actions.zero_()                 # the policy writes no action for a finished board
        rewards.zero_()
        cfg = make_env_cfg(benv.config, "buffer", auto_reset=False, emit_obs=False)

        def launch(T, chunk, slot_map, upper, count):
            _lib.check(self._lib.b2048_rollout_many_np(
                self._h, _ptr(boards), _ptr(flags), _ptr(actions), _ptr(rewards), _ptr(benv.score), _ptr(benv.step_count),
                _ptr(benv.max_exp), _ptr(length), C.byref(cfg), C.byref(self._actor.desc), B, T, chunk, _ptr(benv.env_rng),
                _ptr(policy_rng), int(self._use_mask), int(use_greedy), slot_map if live_list else None, upper, count,
                _stream()), "b2048_rollout_many_np")

        T = self._live_chunks(launch, length, cap, check_every)
        benv.t = T
        length = torch.where(length == 0, torch.full_like(length, T), length)   # cut off by the cap
        benv.board = boards[T]          # the step kernel passes finished boards through: slice T is every final state
        benv.flags = flags[T]
        return Rollout(boards[: T + 1], flags[: T + 1], actions[:T], rewards[:T], length, T)

    # ------------------------------------------------------------------ playing with the critic
    def _lookahead_precision(self, precision: int | str) -> int:
        """The critic forward's precision code of a lookahead call; refuses a play without a value function.  Both checks
        run before any device work."""
        if not self._has_value_function():
            raise ValueError("lookahead play needs a value function: agent.use_critic or a SharedTrunkActorCritic")
        if precision == "auto":
            return 2
        if isinstance(precision, bool) or precision not in (0, 1, 2, 3):
            raise ValueError(f"precision must be 'auto', 0, 1, 2 or 3, got {precision!r}")
        return int(precision)

    def _lookahead(self, boards: torch.Tensor, flags: torch.Tensor | None, max_exp: torch.Tensor | None, cfg, prec: int,
                   actions: torch.Tensor, q_out: torch.Tensor | None, slot_map: torch.Tensor | None = None,
                   count_dev: torch.Tensor | None = None) -> int:
        """b2048_lookahead_expand of boards (the boards listed in slot_map[:*count_dev] when given), one 4-byte read of the
        child count, the critic forward on the children, b2048_lookahead_select into actions (and q_out).  Returns the
        number of children; 0 means no listed board (nothing is selected)."""
        B = boards.numel()
        cap = B * 120
        cb = self._buf("la_child_board", (cap,), torch.int64)
        cr = self._buf("la_child_reward", (cap,), torch.float64)
        cd = self._buf("la_child_done", (cap,), torch.uint8)
        cv = self._buf("la_child_value", (cap,), torch.float32)
        first = self._buf("la_first", (B, 4), torch.int32)
        count = self._buf("la_count", (B, 4), torch.int32)
        total_dev = self._buf("la_total", (1,), torch.int32)
        total_host = getattr(self, "_la_total_host", None)
        if total_host is None:
            total_host = self._la_total_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        lib, h = self._lib, self._h
        sm, nd = _ptr(slot_map), _ptr(count_dev)
        with torch.cuda.device(self.device):
            _lib.check(lib.b2048_lookahead_expand(h, _ptr(boards), _ptr(flags), _ptr(max_exp), C.byref(cfg), sm, B, nd, B, cap,
                                                  _ptr(cb), _ptr(cr), _ptr(cd), _ptr(first), _ptr(count), _ptr(total_dev),
                                                  _stream()), "b2048_lookahead_expand")
            total_host.copy_(total_dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            ev.synchronize()
            total = int(total_host[0])
            if total == 0:
                return 0
            self._forward_checked(self._critic, cb[:total], cv[:total], self._small_batch_precision(prec, total), [], 1)
            _lib.check(lib.b2048_lookahead_select(h, sm, B, nd, B, _ptr(first), _ptr(count), _ptr(cr), _ptr(cd), _ptr(cv),
                                                  float(self.agent_config.gamma), _ptr(actions), _ptr(q_out), _stream()),
                       "b2048_lookahead_select")
        return total

    def lookahead_actions(self, boards: torch.Tensor, flags: torch.Tensor | None, max_exp: torch.Tensor | None = None,
                          precision: int | str = "auto", q_out: torch.Tensor | None = None) -> torch.Tensor:
        """One-ply expectimax over the critic for a batch of packed boards (include/b2048.h, DESIGN.md K7): every candidate
        move and every spawn is expanded on the device, the critic values the children, and the action is the first argmax
        of Q(s, a) = sum p (r + gamma V(s')).  flags: the boards' flags (low nibble = legal mask; None = recomputed);
        max_exp: the per-board new-max-tile state of the bonus (None = no bonus).  q_out (float64 [n, 4], optional)
        receives Q, NaN for a non-candidate.  precision: that of the critic forward ("auto" = the split-fp16 tensor cores
        where they apply, with the fp32 fall-back of the update passes; batches under 4096 children run as "auto" would).
        Returns the actions (uint8 [n])."""
        prec = self._lookahead_precision(precision)
        from .batched_env import make_env_cfg
        cfg = make_env_cfg(self.env.config, "buffer", auto_reset=False, emit_obs=False)
        boards = boards.reshape(-1)
        actions = torch.zeros(boards.numel(), dtype=torch.uint8, device=self.device)
        if q_out is not None:
            q_out.fill_(float("nan"))
        if boards.numel():
            self._lookahead(boards, flags, max_exp, cfg, prec, actions, q_out)
        return actions

    def rollout_lookahead(self, benv: Batched2048Env, max_steps: int | None = None, precision: int | str = "auto") -> Rollout:
        """rollout_many(greedy=True) with the lookahead actions of lookahead_actions instead of the actor's argmax: every
        board plays to termination (or max_steps, like rollout_many) on the env's Philox streams.  Each step is
        b2048_compact_live, the lookahead on the boards still playing, and b2048_step_many; the host reads the 4-byte child
        count once per step.  Returns a run-to-termination Rollout (total_reward(), max tiles 2 ** benv.max_exp)."""
        prec = self._lookahead_precision(precision)
        B = benv.num_envs
        benv.reset_many()
        cap = int(max_steps or benv.config.max_steps or 4096)
        boards, flags, actions, rewards, length = self._rollout_buffers(benv, cap)
        actions.zero_()                 # finished boards get no action
        from .batched_env import make_env_cfg
        cfg = make_env_cfg(benv.config, "buffer", auto_reset=False, emit_obs=False)
        slot = self._buf("ro_slot_map", (B,), torch.int32)
        count_dev = self._buf("ro_live_count", (1,), torch.int32)
        t0 = benv.t
        T = 0
        while T < cap:
            with torch.cuda.device(self.device):
                _lib.check(self._lib.b2048_compact_live(self._h, _ptr(length), B, _ptr(slot), _ptr(count_dev), _stream()),
                           "b2048_compact_live")
            if self._lookahead(boards[T], flags[T], benv.max_exp, cfg, prec, actions[T], None, slot, count_dev) == 0:
                break                   # no board is still playing
            with torch.cuda.device(self.device):
                _lib.check(self._lib.b2048_step_many(
                    self._h, _ptr(boards[T]), _ptr(boards[T + 1]), _ptr(benv.score), _ptr(benv.step_count), _ptr(benv.max_exp),
                    _ptr(actions[T]), None, _ptr(flags[T]), None, C.byref(cfg), None, _ptr(rewards[T]), None, _ptr(flags[T + 1]),
                    None, _ptr(length), T + 1, B, benv.seed, benv.gid0, t0 + T + 1, _stream()), "b2048_step_many")
            T += 1
        benv.t = t0 + T
        length = torch.where(length == 0, torch.full_like(length, T), length)   # cut off by the cap
        benv.board = boards[T]          # the step kernel passes finished boards through: slice T is every final state
        benv.flags = flags[T]
        return Rollout(boards[: T + 1], flags[: T + 1], actions[:T], rewards[:T], length, T, seed=benv.seed, gid0=benv.gid0,
                       t0=t0)

    # ------------------------------------------------------------------ reference API: learning
    def compute_returns(self, rewards: list[float]) -> np.ndarray:
        """G_t = r_t + gamma G_{t+1} (reinforce_agent.py:255-273) with the float64 recurrence on the device."""
        T = len(rewards)
        if T == 0:
            return np.zeros(0, dtype=np.float32)
        x = torch.tensor(np.asarray(rewards, dtype=np.float32).reshape(T, 1), device=self.device)
        y = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_reverse_scan_f64(_ptr(x), _ptr(y), None, float(self.agent_config.gamma), T, 1,
                                                        _stream()), "b2048_reverse_scan_f64")
        return y.cpu().numpy().reshape(T)

    def _compute_episode_rank_weights(self, total_reward_list) -> np.ndarray:
        """CVaR-style episode weights by reward rank (reinforce_agent.py:681-716).  Host-side: it is a sort of
        n_traj scalars, not per-step arithmetic."""
        conf = self.agent_config.reward_rank_weights
        n = len(total_reward_list)
        if n == 0:
            return np.array([], dtype=np.float32)
        if conf is None or len(conf) == 0:
            return np.ones(n, dtype=np.float32)
        conf = np.asarray(conf, dtype=np.float32)
        order = np.argsort(total_reward_list)
        w = np.zeros(n, dtype=np.float32)
        bins = np.minimum(((np.arange(n) + 0.5) / n * len(conf)).astype(np.int64), len(conf) - 1)
        w[order] = conf[bins]
        m = np.mean(w)
        return w / m if m > 1e-8 else w

    def _trajectories_to_rollout(self, trajectories: list[dict[str, Any]]) -> Rollout:
        B = len(trajectories)
        lens = np.array([len(t["actions"]) for t in trajectories], dtype=np.int32)
        T = int(lens.max()) if B else 0
        boards = np.zeros((T + 1, B), dtype=np.uint64)
        flags = np.zeros((T + 1, B), dtype=np.uint8)
        actions = np.zeros((T, B), dtype=np.uint8)
        rewards = np.zeros((T, B), dtype=np.float32)
        for b, tr in enumerate(trajectories):
            for t, o in enumerate(tr["obs"]):
                boards[t, b], flags[t, b] = self._obs_to_packed(o)
            actions[: lens[b], b] = np.asarray(tr["actions"], dtype=np.uint8)
            rewards[: lens[b], b] = np.asarray(tr["rewards"], dtype=np.float32)
        dev = self.device
        return Rollout(torch.from_numpy(boards.view(np.int64)).to(dev), torch.from_numpy(flags).to(dev),
                       torch.from_numpy(actions).to(dev), torch.from_numpy(rewards).to(dev),
                       torch.from_numpy(lens).to(dev), T)

    def _augment_rollout(self, ro: Rollout) -> Rollout:
        """x8 dihedral augmentation of a rollout on packed boards (reinforce_agent.py:773-808, env.py:317-397)."""
        from .symmetry import augment_rollout
        return augment_rollout(ro)

    def _one_message_exchange(self, values, ro, n_traj, adv, coef, stats, ep_mean, backward, allreduce) -> None:
        """The sharded update's exchange as exactly one all-reduce (SURVEY.md 8e; north_star: "a single NCCL allreduce ... for
        the policy gradient only").  With a 'batch' / 'batch_norm' baseline the per-sample coefficient is
        (v - mean) / std * w / (T n) with GLOBAL mean / std (reinforce_agent.py:303-322, :864-881); the backward pass is
        linear in it, so g = (g_A - mean g_B) / std with g_A from the coefficients v w / (T n) and g_B from w / (T n).  Both
        are local sums; they travel with the critic gradient and the four float64 baseline sums in one float64 buffer.
        Ends with adv / coef as the default exchange reports them (global statistics)."""
        lib, h, dev, T, B = self._lib, self._h, self.device, ro.T, ro.B
        mode = BASELINE[self.agent_config.baseline_mode]
        na = self._actor.n_params
        msg = self._buf("one_msg", (na + self._grad_all.numel() + 4,), torch.float64)
        ones = self._buf("one_msg_ones", (T, B), torch.float32)
        ones.fill_(1.0)
        with torch.cuda.device(dev):
            stats.zero_()
            _lib.check(lib.b2048_weighted_stats(h, _ptr(values), _ptr(ro.length), _ptr(ro.ep_weight), T, B, _ptr(stats),
                                                _stream()), "b2048_weighted_stats")
        for k, v in enumerate((values, ones)):                       # g_A, then g_B
            self._advantages(v, ro.length, ro.ep_weight, 0, n_traj, None, coef, stats, ep_mean, window=False, pre=1)
            backward(self._actor, coef.reshape(-1), 0)
            if k == 0:
                msg[:na].copy_(self._actor.grad)
        msg[na: na + self._grad_all.numel()].copy_(self._grad_all)   # [g_B | critic gradient]
        msg[-4:].copy_(stats)
        allreduce(msg)                                               # THE message of this update
        stats.copy_(msg[-4:])
        sw = msg[-4]
        m = torch.where(sw < 1e-8, torch.zeros_like(sw), msg[-3] / sw.clamp_min(1e-300))          # advantage_kernel
        var = torch.where(sw < 1e-8, torch.ones_like(sw), msg[-2] / sw.clamp_min(1e-300) - m * m)
        mean32 = m.to(torch.float32)
        std32 = var.clamp_min(0.0).sqrt().to(torch.float32).clamp_min(1e-8) if mode == 3 else torch.ones_like(mean32)
        g_a, g_b = msg[:na], msg[na: 2 * na]
        self._grad_all.copy_(msg[na: na + self._grad_all.numel()])   # critic part (and g_B, overwritten next)
        self._actor.grad.copy_((g_a - mean32.to(torch.float64) * g_b) / std32.to(torch.float64))
        self._advantages(values, ro.length, ro.ep_weight, mode, n_traj, adv, coef, stats, ep_mean, window=False, pre=1)

    def _advantages(self, values: torch.Tensor, length: torch.Tensor, ep_weight: torch.Tensor | None, mode: int,
                    n_traj: float, adv: torch.Tensor | None, coef: torch.Tensor, stats: torch.Tensor,
                    ep_mean: torch.Tensor | None, window: bool, pre: int = 0, allreduce=None) -> None:
        """adv / coef of the baseline `mode` on the [T, B] values (the raw advantages, or a constant for the entropy
        coefficients): b2048_advantages with the weight w_b / (len_b n_traj) on episodes, b2048_advantages_window with
        1 / (T n_traj) on a window (length = valid_len).  pre=1: stats already holds the baseline sums.  Sharded (allreduce
        given) with a 'batch' / 'batch_norm' baseline, the local sums are all-reduced first (the 32-byte message)."""
        lib, h = self._lib, self._h
        T, B = values.shape
        with torch.cuda.device(self.device):
            if allreduce is not None and mode >= 2 and not pre:
                stats.zero_()
                _lib.check(lib.b2048_weighted_stats(h, _ptr(values), _ptr(length), _ptr(ep_weight), T, B, _ptr(stats),
                                                    _stream()), "b2048_weighted_stats")
                allreduce(stats)
                pre = 1
            if window:
                _lib.check(lib.b2048_advantages_window(h, _ptr(values), _ptr(length), mode, n_traj, T, B, _ptr(adv),
                                                       _ptr(coef), _ptr(stats), pre, _stream()), "b2048_advantages_window")
            else:
                _lib.check(lib.b2048_advantages(h, _ptr(values), _ptr(length), _ptr(ep_weight), mode, n_traj, T, B,
                                                _ptr(adv), _ptr(coef), _ptr(stats), pre, _ptr(ep_mean), _stream()),
                           "b2048_advantages")

    def update_batch(self, trajectories: list[dict[str, Any]]) -> None:
        """reinforce_agent.py:357-620 on reference-style trajectories (list of dicts from run_episode)."""
        if len(trajectories) == 0:
            return
        ro = self._trajectories_to_rollout(trajectories)
        w = self._compute_episode_rank_weights([t["total_reward"] for t in trajectories])
        ro.ep_weight = torch.from_numpy(w).to(self.device)
        self.update_from_rollout(ro)

    def update_from_rollout(self, ro: Rollout, chunk: int = 1 << 20, allreduce=None,
                            precision: int | str = "auto", exchange: str = "default",
                            bootstrap_truncation: bool = False, entropy_coef: float = 0.0) -> dict[str, Any]:
        """One policy-gradient update from device-resident rollout buffers.  `allreduce(tensor)` (optional) sums
        a tensor over ranks in place: the flat gradients and the advantage statistics are the only exchange.
        precision: 0 = fp32 CUDA cores, "auto" (default) = the float32-grade tensor-core path (split-fp16 forward, fp16
        backward; within 1e-2 of the reference's float32 gradient) whenever the network shape / batch allow it, else fp32;
        3 = that path or an error; 1 = single-bf16 tensor cores, an explicit opt-in (its forward flips ReLU units near zero:
        3-30 % error on cancelling gradients; b2048_mlp_backward, include/b2048.h).
        exchange (sharded updates with a 'batch' / 'batch_norm' baseline): "default" = a 32-byte all-reduce of the four
        float64 baseline sums, then ONE all-reduce of the flat gradient buffer [actor | critic]; "one_message" = exactly
        one all-reduce per update (SURVEY.md 8e): the backward deltas are linear in the per-sample coefficient, so each rank
        accumulates g_A (coefficient w v / (T n)) and g_B (coefficient w / (T n)) locally, one float64 message
        [g_A | g_B | critic gradient | sums] is summed over ranks and g = (g_A - mean g_B) / std is formed afterwards.
        It costs a second actor backward pass, which is why it is an opt-in.
        bootstrap_truncation (needs a critic or a value head): an episode truncated by the env's max_steps (flags[len[b], b]
        has TRUNC) gets the target r + gamma V(boards[len[b], b]) at its last step instead of r, like Gymnasium's `truncated`
        (see _update_bootstrapped).  Episodes cut by rollout_many's own max_steps cap carry no TRUNC flag and are not
        bootstrapped.  The default keeps update_batch's targets.
        entropy_coef (beta >= 0): the actor ascends sum_s coef_s log pi(a_s|s) + ecoef_s H(pi(.|s_s)) with ecoef_s = beta w_b /
        (len_b n_traj), i.e. beta times the sample's weight in the policy term (b2048_mlp_backward_entropy); info["entropy"] is
        then the rank-local mean H over the update's samples.  0 (default) runs exactly the calls without the bonus.  Refused
        with exchange='one_message' and precision=1."""
        cfg = self._check_update_config(exchange)
        beta = self._check_entropy(entropy_coef, exchange, precision)
        if bootstrap_truncation:
            self._check_bootstrap(ro, window=False)
        if ro.B == 0 or ro.T == 0:
            return {}
        if ro.auto_reset:
            # The learner kernels see one episode per lane (returns scan, TD shift and the 1/(T_ep n_traj) weight mask on
            # len[b] only, like update_batch's per-episode arrays, reinforce_agent.py:403-555).  A reset-on-done lane
            # holds several episodes: returns would run across the resets and TD targets would bootstrap from the
            # reset board.  Roll out to termination / truncation instead (horizon=None; max_steps bounds the length).
            raise ValueError("update_from_rollout: fixed-horizon rollouts with reset-on-done hold several episodes per "
                             "lane and are not a reference-equivalent update batch; use rollout_many(horizon=None), or "
                             "update_from_horizon for the segment-aware update")
        if ro.ep_weight is None and cfg.reward_rank_weights:
            # global reward ranks on the device (all-gathered over ranks when the episodes are sharded), computed on
            # the ORIGINAL episodes and repeated by the augmentation like the reference (reinforce_agent.py:369-384, :806)
            from . import dist as bd
            dinfo = bd.DistInfo(int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")),
                                int(os.environ.get("LOCAL_RANK", "0"))) if allreduce is not None else None
            ro.ep_weight = bd.episode_rank_weights(ro.total_reward(), cfg.reward_rank_weights, dinfo)
        boot = self._truncated_episode_ends(ro) if bootstrap_truncation else None
        if cfg.augmentation:
            ro = self._augment_rollout(ro)
        return self._update_bootstrapped(ro, boot, chunk, allreduce, precision, exchange, beta)

    def update_from_horizon(self, ro: Rollout, allreduce=None, precision: int | str = "auto", chunk: int = 1 << 20,
                            exchange: str = "default", bootstrap_truncation: bool = False,
                            entropy_coef: float = 0.0) -> dict[str, Any]:
        """One policy-gradient update from a fixed-horizon window: a rollout_many(horizon=H) rollout with reset-on-done,
        whose lanes keep playing across updates (synchronous A2C / REINFORCE on segments).  Episode boundaries inside a lane
        (flags DONE | TRUNC after step t) restart the returns, TD targets and advantages (b2048_segment_targets; a truncated
        episode is not bootstrapped, like update_batch's last step):
          REINFORCE     G_t = r_t + gamma (1 - e_t) G_{t+1}; only the slots of episodes that end inside the window are samples
                        (the tail after a lane's last boundary is not used);
          actor-critic  V on all T + 1 slices, delta_t = r_t + gamma (1 - e_t) V(s_{t+1}) - V(s_t), the cut-off tail
                        bootstrapped from V(boards[T]); A_t = delta_t + gamma lambda (1 - e_t) A_{t+1} (lambda = gae_lambda,
                        0 = TD(0)); every slot is a sample.
        Baselines off / batch / batch_norm over the samples; per-sample weight adv / (T n_traj) with n_traj = ro.n_traj (the
        global lane count under sharding; x8 with augmentation), i.e. the mean over all slots of the window.  Baseline
        'each', reward_rank_weights (both need whole episodes), exchange='one_message' and rollouts without reset-on-done
        raise ValueError.  The episodes the window completes are added to horizon_episode_stats().
        allreduce / precision / chunk as in update_from_rollout.
        bootstrap_truncation (needs a critic or a value head, and ro.seed / ro.t0 from rollout_many): a TRUNC boundary
        after step t (the env's max_steps ran out, the game was not over) uses V(s') instead of 0, s' being the board the
        episode was cut on: delta_t = r_t + gamma V(s') - V(s_t).  boards[t + 1] already holds the reset board; s' is replayed
        on the device from boards[t], actions[t] and the env streams (b2048_replay_pre_reset).
        entropy_coef as in update_from_rollout, with ecoef = beta / (T n_traj) on the samples (every slot with a value
        function; with REINFORCE the slots t < valid_len[b])."""
        cfg = self._check_update_config(exchange)
        beta = self._check_entropy(entropy_coef, exchange, precision)
        self._check_window(ro, exchange, "update_from_horizon")
        if bootstrap_truncation:
            self._check_bootstrap(ro, window=True)
        if ro.B == 0 or ro.T == 0:
            return {}
        self._horizon_account(ro)                                   # the episode returns are the undiscounted env rewards
        boot = self._truncated_window_steps(ro) if bootstrap_truncation else None
        if cfg.augmentation:
            ro = self._augment_rollout(ro)
        return self._update_bootstrapped(ro, boot, chunk, allreduce, precision, exchange, beta)

    def _check_window(self, ro: Rollout, exchange: str, what: str) -> None:
        """The configurations a window update refuses (ValueError): a rollout without reset-on-done, and what needs whole
        episodes or the one-message exchange."""
        cfg = self.agent_config
        if not ro.auto_reset:
            raise ValueError(f"{what} needs a fixed-horizon rollout with reset-on-done (rollout_many(horizon=H))")
        if cfg.baseline_mode == "each":
            raise ValueError("baseline 'each' needs whole episodes: not available on fixed-horizon windows")
        if cfg.reward_rank_weights or ro.ep_weight is not None:
            raise ValueError("reward rank weights need whole episodes: not available on fixed-horizon windows")
        if exchange == "one_message":
            raise ValueError("exchange='one_message' is not implemented for fixed-horizon windows")

    # ------------------------------------------------------------------ PPO on windows
    def update_ppo(self, ro: Rollout, epochs: int = 4, minibatches: int = 4, clip_eps: float = 0.2,
                   value_clip_eps: float | None = None, shuffle_seed: int = 0, allreduce=None, precision: int | str = "auto",
                   bootstrap_truncation: bool = False, entropy_coef: float = 0.0) -> dict[str, Any]:
        """PPO on a fixed-horizon window (rollout_many(horizon=H), reset-on-done): `epochs` passes over the window's
        N = T n_traj samples, each split into `minibatches` minibatches, one clipped-surrogate step per minibatch
        (epochs x minibatches optimizer steps).  Needs a value function (use_critic=True or SharedTrunkActorCritic).
        Once, at the window's parameters theta_old: V_old on all T + 1 slices, the segment-aware GAE A_raw
        (b2048_segment_targets; lambda = gae_lambda, 0 = TD(0)), the advantages A of the configured baseline (off / batch /
        batch_norm, per window), the value target R = A_raw + V_old, and logp_old = log pi_theta_old(a|s) from the learner's
        own forward at the update's precision (not the rollout's probabilities).
        Minibatches: b2048_ppo_minibatches, a keyed permutation of the global sample index t n_traj + gid0 + b per epoch
        (shuffle_seed, epoch); it depends on neither the world size nor the shard, and every rank knows each minibatch's
        global size.  Per minibatch: forward of actor and critic, r = exp(logp - logp_old), the clipped-surrogate coefficient
        A r / |mb| (0 where clipped), the value coefficient (V - R) / |mb| (value_clip_eps: PPO's clipped value loss; mse or
        Huber as configured), b2048_mlp_backward for both heads, ONE all-reduce of the flat gradient when sharded, the
        global-norm clip and SGD / Adam (the Adam counters advance once per minibatch).
        The window's episodes are added to horizon_episode_stats() as update_from_horizon does.
        Returns per-epoch lists (rank-local): clip_fraction, approx_kl (mean r - 1 - log r), mean_ratio, surrogate
        (mean min(r A, clip(r) A)) and value_loss; per-step actor_grad_norms / critic_grad_norms; advantages (A), gae
        (A_raw), values_old ([T + 1, B]) and logp_old ([T B], float64) of the window; precision.  The tensors are scratch
        buffers, valid until the next update.
        allreduce / precision / bootstrap_truncation as in update_from_horizon.  Refused (ValueError): no value function,
        a rollout without reset-on-done, augmentation, reward rank weights, baseline 'each', epochs < 1, minibatches
        outside [1, N], clip_eps <= 0, value_clip_eps <= 0, and a shard (n_traj > B) without ro.gid0.
        entropy_coef (beta >= 0): each minibatch step adds beta H(pi(.|s)) / |mb| per sample to the surrogate's gradient
        (b2048_mlp_backward_entropy, |mb| the global minibatch size as for the surrogate); info["entropy"] is then the per-epoch
        rank-local mean H at the step's parameters.  Refused with precision=1."""
        cfg = self._check_update_config("default")
        beta = self._check_entropy(entropy_coef, "default", precision)
        if not self._has_value_function():
            raise ValueError("update_ppo needs a value function: use_critic=True or SharedTrunkActorCritic")
        self._check_window(ro, "default", "update_ppo")
        if cfg.augmentation:
            raise ValueError("update_ppo does not implement augmentation")
        n_traj = int(ro.n_traj if ro.n_traj is not None else ro.B)
        N = ro.T * n_traj
        if int(epochs) < 1:
            raise ValueError(f"update_ppo: epochs must be >= 1, got {epochs}")
        if not 1 <= int(minibatches) <= max(N, 1):
            raise ValueError(f"update_ppo: minibatches must be in [1, {N}] (the window's samples), got {minibatches}")
        if not clip_eps > 0:
            raise ValueError(f"update_ppo: clip_eps must be positive, got {clip_eps}")
        if value_clip_eps is not None and not value_clip_eps > 0:
            raise ValueError(f"update_ppo: value_clip_eps must be positive or None, got {value_clip_eps}")
        if n_traj > ro.B and ro.gid0 is None:
            raise ValueError("update_ppo on a shard (n_traj > B) needs Rollout.gid0, the global id of its lane 0, to place "
                             "its samples in the global minibatches")
        if bootstrap_truncation:
            self._check_bootstrap(ro, window=True)
        if ro.B == 0 or ro.T == 0:
            return {}
        self._horizon_account(ro)
        if bootstrap_truncation:
            boot = self._truncated_window_steps(ro)
            if boot[0].numel():
                ro = self._fold_truncation(ro, boot, precision)[0]
        return self._ppo(ro, int(epochs), int(minibatches), float(clip_eps), value_clip_eps, int(shuffle_seed), allreduce,
                         self._update_precision(precision), n_traj, beta)

    def ppo_minibatch_lists(self, T: int, B: int, n_traj: int, gid0: int, minibatches: int, shuffle_seed: int,
                            epoch: int) -> tuple[torch.Tensor, list[int]]:
        """The local slots t B + b of a [T, B] window grouped by minibatch for one epoch of update_ppo: (order, counts) with
        the slots of minibatch m at order[sum(counts[:m]) : sum(counts[:m + 1])], ascending.  gid0 = the global id of lane 0
        (0 for a whole window)."""
        mb = self._buf("ppo_mb", (T, B), torch.int32)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_ppo_minibatches(self._h, T, B, n_traj, gid0, minibatches, shuffle_seed & (2**64 - 1),
                                                       epoch, _ptr(mb), _stream()), "b2048_ppo_minibatches")
        mb = mb.reshape(-1)
        order = torch.sort(mb, stable=True).indices           # grouping only: the order inside a minibatch is by slot
        counts = torch.bincount(mb, minlength=minibatches).cpu().tolist()
        return order, counts

    def _ppo(self, ro: Rollout, epochs: int, M: int, clip_eps: float, value_clip_eps, shuffle_seed: int, allreduce, prec: int,
             n_traj: int, beta: float = 0.0) -> dict[str, Any]:
        cfg = self.agent_config
        lib, h, dev = self._lib, self._h, self.device
        T, B = ro.T, ro.B
        n, N = T * B, T * n_traj
        gid0 = int(ro.gid0) if n_traj > B else 0
        boards = ro.boards[:T].reshape(-1)
        mflags = ro.flags[:T].reshape(-1)
        acts = ro.actions[:T].reshape(-1)
        fell_back: list = []
        # ---- once per window, at theta_old
        tg = self._window_targets(ro, prec, float(n_traj), allreduce, fell_back)
        values, gae, adv = tg["values"], tg["raw"], tg["advantages"]
        logits = self._buf("ppo_logits", (n, 4), torch.float32)
        self._forward_checked(self._actor, boards, logits, prec, fell_back, 0)
        logp_old = self._buf("ppo_logp_old", (n,), torch.float64)
        with torch.cuda.device(dev):
            _lib.check(lib.b2048_ppo_logp(h, _ptr(logits), _ptr(mflags) if self._use_mask else None, _ptr(acts), n,
                                          _ptr(logp_old), _stream()), "b2048_ppo_logp")
        # ---- epochs x minibatches clipped steps
        ep_stats = torch.zeros((epochs, 5), dtype=torch.float64, device=dev)
        norms = torch.zeros((epochs * M, 2), dtype=torch.float64, device=dev)
        ent = torch.zeros(epochs, dtype=torch.float64, device=dev) if beta > 0.0 else None
        vclip = float(value_clip_eps) if value_clip_eps is not None else 0.0
        huber = int(cfg.critic_loss_type == "huber")
        chunk = 1 << 20
        for e in range(epochs):
            order, counts = self.ppo_minibatch_lists(T, B, n_traj, gid0, M, shuffle_seed, e)
            off = 0
            for m in range(M):
                k = counts[m]
                idx = order[off: off + k]
                off += k
                size = (-(-(m + 1) * N // M)) - (-(-m * N // M))   # the minibatch's global size, ceil((m+1)N/M) - ceil(mN/M)
                if k > 0:
                    p = self._small_batch_precision(prec, k)
                    bx, fx, ax = boards.index_select(0, idx), mflags.index_select(0, idx), acts.index_select(0, idx)
                    z = self._buf("ppo_z", (k, 4), torch.float32)
                    v = self._buf("ppo_v", (k,), torch.float32)
                    self._forward_checked(self._actor, bx, z, p, fell_back, 0)
                    self._forward_checked(self._critic, bx, v, p, fell_back, 1)
                    cf, gc = self._buf("ppo_coef", (k,), torch.float32), self._buf("ppo_gcoef", (k,), torch.float32)
                    with torch.cuda.device(dev):
                        _lib.check(lib.b2048_ppo_coefficients(
                            h, _ptr(idx), k, _ptr(z), _ptr(v), _ptr(mflags) if self._use_mask else None, _ptr(acts),
                            _ptr(logp_old), _ptr(adv), _ptr(gae), _ptr(values), float(size), clip_eps, vclip, huber,
                            float(cfg.huber_delta), _ptr(cf), _ptr(gc), _ptr(ep_stats[e]), _stream()), "b2048_ppo_coefficients")
                    if ent is None:
                        self._backward(self._actor, bx, fx, ax, cf, k, 0, p, chunk, fell_back)
                    else:                                      # the bonus beta H / |mb| per sample, like the surrogate's 1 / |mb|
                        ecf = self._buf("ppo_ent_coef", (k,), torch.float32).fill_(beta / size)
                        self._backward(self._actor, bx, fx, ax, cf, k, 0, p, chunk, fell_back, ecf, ent[e: e + 1])
                    self._backward(self._critic, bx, fx, ax, gc, k, 1, p, chunk, fell_back)
                else:                                          # this shard holds none of the minibatch's samples
                    self._actor.grad.zero_()
                    self._critic.grad.zero_()
                ss_a, ss_c = self._step(allreduce)             # ONE message per minibatch step
                norms[e * M + m, 0] = ss_a[0]
                if ss_c is not None:
                    norms[e * M + m, 1] = ss_c[0]
        st = ep_stats.cpu().numpy() / n
        nr = norms.sqrt().cpu().numpy()
        info: dict[str, Any] = {
            "clip_fraction": st[:, 0].tolist(), "mean_ratio": st[:, 1].tolist(), "approx_kl": st[:, 2].tolist(),
            "surrogate": st[:, 3].tolist(), "value_loss": st[:, 4].tolist(), "actor_grad_norms": nr[:, 0].tolist(),
            "advantages": adv, "gae": gae, "values_old": values, "logp_old": logp_old,
            "precision": self._precision_info(prec, n, fell_back)}
        info["actor_grad_norm"] = info["actor_grad_norms"][-1]
        if ent is not None:
            info["entropy"] = (ent.cpu().numpy() / n).tolist()
        if ss_c is not None:                                   # a separate critic (not a value head on the shared trunk)
            info["critic_grad_norms"] = nr[:, 1].tolist()
            info["critic_grad_norm"] = info["critic_grad_norms"][-1]
        self.last_update_info = info
        if self._logger.isEnabledFor(logging.INFO):
            self._logger.info(f"PPO: clip fraction {info['clip_fraction']}, approx KL {info['approx_kl']}")
        return info

    # ------------------------------------------------------------------ bootstrapping at truncation
    def _check_bootstrap(self, ro: Rollout, window: bool) -> None:
        if not self._has_value_function():
            raise ValueError("bootstrap_truncation needs a value function: use_critic=True or SharedTrunkActorCritic")
        if window and (ro.seed is None or ro.t0 is None):
            raise ValueError("bootstrap_truncation on a window needs its env streams (Rollout.seed and Rollout.t0, which "
                             "rollout_many(horizon=H) sets) to replay the boards truncated episodes were cut on")

    def _truncated_window_steps(self, ro: Rollout) -> tuple[torch.Tensor, torch.Tensor]:
        """(slots, s'): the steps t * B + b of a window after which an episode was truncated (TRUNC without DONE), in
        row-major [T, B] order, and the boards those episodes were cut on, replayed on the device."""
        T, B = ro.T, ro.B
        ends = ro.flags[1: T + 1] & (_lib.F_DONE | _lib.F_TRUNC)
        slots = torch.nonzero((ends == _lib.F_TRUNC).reshape(-1)).reshape(-1)
        nxt = torch.empty(slots.numel(), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_replay_pre_reset(
                self._h, _ptr(ro.boards[: T + 1].contiguous()), _ptr(ro.actions[:T].contiguous()), _ptr(slots), slots.numel(), B,
                int(ro.seed) & (2**64 - 1), int(ro.gid0 or 0), int(ro.t0), _ptr(nxt), _stream()), "b2048_replay_pre_reset")
        return slots, nxt

    def _truncated_episode_ends(self, ro: Rollout) -> tuple[torch.Tensor, torch.Tensor]:
        """(slots, s') of a run-to-termination rollout: the last step (len[b] - 1) * B + b of every lane whose episode was
        truncated (flags[len[b], b] has TRUNC, not DONE), and its final board boards[len[b], b]."""
        T, B = ro.T, ro.B
        L = ro.length.long().clamp(0, T)
        last = L.unsqueeze(0)
        fin = ro.flags[: T + 1].gather(0, last).reshape(-1) & (_lib.F_DONE | _lib.F_TRUNC)
        lanes = torch.nonzero((fin == _lib.F_TRUNC) & (L > 0)).reshape(-1)
        slots = (L[lanes] - 1) * B + lanes
        return slots, ro.boards[: T + 1].gather(0, last).reshape(-1)[lanes]

    def _update_bootstrapped(self, ro: Rollout, boot, chunk: int, allreduce, precision: int | str, exchange: str,
                             beta: float = 0.0) -> dict[str, Any]:
        """_update on a copy of the rewards with gamma V(s') folded in at the truncated steps (boot = (slots, s') of the
        rollout before augmentation; None: no bootstrap).  The target kernels use V = 0 after an episode's last step, so
        r' = r + gamma V(s') (each operation rounded separately, b2048_fold_bootstrap) makes every target, TD error,
        advantage and critic coefficient the bootstrapped one.  With augmentation variant v of step (t, b) is column
        v B + b, and it folds the value of variant v of s'."""
        if boot is None or boot[0].numel() == 0:
            return self._update(ro, chunk, allreduce, precision, exchange, beta)
        folded, slots, nxt, values = self._fold_truncation(ro, boot, precision)
        info = self._update(folded, chunk, allreduce, precision, exchange, beta)
        info.update(bootstrap_slots=slots, bootstrap_boards=nxt, bootstrap_values=values)
        return info

    def _fold_truncation(self, ro: Rollout, boot, precision: int | str):
        """(ro with the rewards r + gamma V(s') at the truncated steps, slots, s', V(s')); see _update_bootstrapped."""
        slots, nxt = boot
        lib, h, dev = self._lib, self._h, self.device
        T, B = ro.T, ro.B
        if self.agent_config.augmentation:                         # ro is the augmented rollout: B = 8 x the original
            K, B0 = slots.numel(), B // 8
            nxt8 = torch.empty(8 * K, dtype=torch.int64, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.b2048_symmetries(h, _ptr(nxt), None, None, _ptr(nxt8), None, None, 1, K, _stream()),
                           "b2048_symmetries")                      # variant v of board k at v K + k
            t, b = slots // B0, slots % B0
            slots = ((t * B + b).unsqueeze(0) + B0 * torch.arange(8, device=dev).unsqueeze(1)).reshape(-1)
            nxt = nxt8
        K = slots.numel()
        values = torch.empty(K, dtype=torch.float32, device=dev)
        # a fall-back of this forward is not reported in info["precision"]
        self._forward_checked(self._critic, nxt, values, self._small_batch_precision(self._update_precision(precision), K), [], 1)
        rewards = torch.empty((T, B), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.b2048_fold_bootstrap(h, _ptr(ro.rewards[:T].contiguous()), _ptr(slots), _ptr(values), K, T * B,
                                                float(self.agent_config.gamma), _ptr(rewards), _stream()),
                       "b2048_fold_bootstrap")
        return replace(ro, rewards=rewards), slots, nxt, values

    def _segment_targets(self, rewards, flags, values, lam, n_traj, v, td, gcoef, valid_len) -> None:
        cfg = self.agent_config
        T, B = rewards.shape
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_segment_targets(
                self._h, _ptr(rewards), _ptr(flags), _ptr(values), float(cfg.gamma), float(lam),
                int(cfg.critic_loss_type == "huber"), float(cfg.huber_delta), float(n_traj), T, B, _ptr(v), _ptr(td),
                _ptr(gcoef), _ptr(valid_len), _stream()), "b2048_segment_targets")

    def _horizon_account(self, ro: Rollout) -> None:
        """Adds the episodes that end inside the window to the device sums behind horizon_episode_stats; each lane's
        running return is carried to the next window (windows of one set of envs follow each other: a different lane
        count starts the carries from zero)."""
        carry = getattr(self, "_hz_carry", None)
        if carry is None or carry.numel() != ro.B:
            self._hz_carry = carry = torch.zeros(ro.B, dtype=torch.float64, device=self.device)
        if getattr(self, "_hz_stats", None) is None:
            self._hz_stats = torch.zeros(21, dtype=torch.float64, device=self.device)
            self._hz_stats[2:4] = torch.tensor([-np.inf, np.inf], dtype=torch.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b2048_horizon_episodes(
                self._h, _ptr(ro.rewards[: ro.T].contiguous()), _ptr(ro.flags[: ro.T + 1].contiguous()),
                _ptr(ro.boards[: ro.T + 1].contiguous()), _ptr(ro.actions[: ro.T].contiguous()), ro.T, ro.B, _ptr(carry),
                _ptr(self._hz_stats), _stream()), "b2048_horizon_episodes")

    def horizon_episode_stats(self, reset: bool = True, info=None) -> dict[str, Any]:
        """The episodes completed by the windows update_from_horizon consumed since the last reset:
        {episodes, avg_reward, max_reward, min_reward, max_tile_counts} with the undiscounted episode returns and the
        episodes per max tile in trainer.TILE_BINS order (16 .. 4096).  Stats of no episode are NaN.  info (a dist.DistInfo
        with world_size > 1): summed / maxed over ranks."""
        st = getattr(self, "_hz_stats", None)
        if st is None:
            st = torch.tensor([0.0, 0.0, -np.inf, np.inf] + [0.0] * 17, dtype=torch.float64, device=self.device)
        st = st.clone()
        if info is not None and info.is_distributed:
            from . import dist as bd
            sums = torch.cat([st[:2], st[4:]])
            ext = torch.stack([st[2], -st[3]])
            bd.allreduce_sum_(sums)
            bd.allreduce_max_(ext)
            st = torch.cat([sums[:2], ext[:1], -ext[1:], sums[2:]])
        h = st.cpu().numpy()
        n = int(h[0])
        if reset and getattr(self, "_hz_stats", None) is not None:
            self._hz_stats.zero_()
            self._hz_stats[2:4] = torch.tensor([-np.inf, np.inf], dtype=torch.float64)
        nan = float("nan")
        return {"episodes": n, "avg_reward": float(h[1] / n) if n else nan, "max_reward": float(h[2]) if n else nan,
                "min_reward": float(h[3]) if n else nan, "max_tile_counts": [int(c) for c in h[4 + 4: 4 + 13]]}

    def _check_update_config(self, exchange: str) -> ReinforceAgentConfig:
        if exchange not in ("default", "one_message"):
            raise ValueError(f"Unknown exchange: {exchange}")
        cfg = self.agent_config
        if cfg.baseline_mode not in BASELINE:
            raise ValueError(f"Unknown baseline mode: {cfg.baseline_mode}")          # reinforce_agent.py:325
        if cfg.optimizer not in OPTIMIZER:
            raise ValueError(f"Unknown optimizer: {cfg.optimizer}")                  # reinforce_agent.py:582
        if cfg.use_critic and cfg.critic_loss_type not in ("mse", "huber"):
            raise ValueError(f"Unknown critic loss type: {cfg.critic_loss_type}")    # reinforce_agent.py:908
        return cfg

    def _window_targets(self, ro: Rollout, prec: int, n_traj: float, allreduce, fell_back: list) -> dict[str, torch.Tensor]:
        """The targets of a fixed-horizon window at the current parameters (b2048_segment_targets), then adv / coef of the
        configured baseline over the window's samples, the slots t < valid_len[b].  With a value function: V on all T + 1
        slices (V(boards[T]) bootstraps the cut-off tail), the TD errors td, the critic coefficients gcoef and
        raw = A_t = delta_t + gamma lambda A_{t+1}; every slot is a sample (valid_len = T: the window is never compacted).
        Without: raw = the segment returns, and the samples are the slots of the episodes that end inside the window.
        Returns {valid_len, raw, advantages, coef} and, with a value function, {values, td, gcoef}."""
        T, B = ro.T, ro.B
        rewards, flags = ro.rewards[:T].contiguous(), ro.flags[: T + 1].contiguous()
        valid = self._buf("valid_len", (B,), torch.int32)
        tg: dict[str, torch.Tensor] = {"valid_len": valid}
        if self._has_value_function():
            values = self._buf("values", (T + 1, B), torch.float32)
            self._forward_checked(self._critic, ro.boards[: T + 1].reshape(-1), values.view(-1), prec, fell_back, 1)
            raw, td, gcoef = (self._buf(k, (T, B), torch.float32) for k in ("gae", "td", "gcoef"))
            self._segment_targets(rewards, flags, values, self.gae_lambda, n_traj, raw, td, gcoef, valid)
            tg.update(values=values, td=td, gcoef=gcoef)
        else:
            raw = self._buf("returns", (T, B), torch.float32)
            self._segment_targets(rewards, flags, None, self.gae_lambda, n_traj, raw, None, None, valid)
        adv, coef = self._buf("adv", (T, B), torch.float32), self._buf("coef", (T, B), torch.float32)
        self._advantages(raw, valid, None, BASELINE[self.agent_config.baseline_mode], n_traj, adv, coef,
                         self._buf("stats", (4,), torch.float64), None, window=True, allreduce=allreduce)
        tg.update(raw=raw, advantages=adv, coef=coef)
        return tg

    def _live_samples(self, ro: Rollout, length: torch.Tensor):
        """(live, boards, flags, actions) of the samples t < length[b] of the [T, B] grid, flattened.  Run-to-termination
        rollouts are ragged: slots with t >= len[b] carry no sample.  The per-sample work (forward / backward GEMMs) then runs
        on the compacted list of live slots (ONE stream compaction of the live mask; live = their grid indices, None when
        nothing is compacted); the [T, B] grid is kept for the per-episode time recurrences.  Pure index plumbing (torch)."""
        T = ro.T
        boards, mflags, acts = ro.boards[:T].reshape(-1), ro.flags[:T].reshape(-1), ro.actions[:T].reshape(-1)
        if int(length.sum().item()) >= int(0.9 * T * ro.B):
            return None, boards, mflags, acts
        tgrid = torch.arange(T, device=self.device, dtype=torch.int32).unsqueeze(1)
        live = torch.nonzero((tgrid < length.unsqueeze(0)).reshape(-1)).reshape(-1)
        return live, boards.index_select(0, live), mflags.index_select(0, live), acts.index_select(0, live)

    def _update(self, ro: Rollout, chunk: int, allreduce, precision: int | str, exchange: str,
                beta: float = 0.0) -> dict[str, Any]:
        """The body of update_from_rollout (one episode per lane, t < length) and update_from_horizon (ro.auto_reset: a
        fixed-horizon window, _window_targets).  beta > 0: the entropy bonus."""
        prec = self._update_precision(precision)
        cfg = self.agent_config
        T, B = ro.T, ro.B
        n_traj = float(ro.n_traj if ro.n_traj is not None else B)
        lib, h, dev = self._lib, self._h, self.device
        critic = self._has_value_function()
        mode = BASELINE[cfg.baseline_mode]
        one_msg = exchange == "one_message" and allreduce is not None and mode >= 2
        stats = self._buf("stats", (4,), torch.float64)
        ep_mean = self._buf("ep_mean", (B,), torch.float32)
        fell_back: list = []
        if ro.auto_reset:
            tg = self._window_targets(ro, prec, n_traj, allreduce, fell_back)
            length = tg["valid_len"]
            info: dict[str, Any] = {"td": tg["td"]} if critic else {"returns": tg["raw"]}
            info["valid_len"] = length
            live, boards, mflags, acts = self._live_samples(ro, length)
        else:
            length = ro.length
            live, boards, mflags, acts = self._live_samples(ro, length)
            rewards = ro.rewards[:T].contiguous()
            tg = {"advantages": self._buf("adv", (T, B), torch.float32), "coef": self._buf("coef", (T, B), torch.float32)}
            if critic:
                # critic block (reinforce_agent.py:403-498): V(s_t) for every stored state, TD(0) errors, critic coefficients
                values = self._buf("values", (T, B), torch.float32)
                vc = values.view(-1) if live is None else self._buf("values_c", (boards.numel(),), torch.float32)
                self._forward_checked(self._critic, boards, vc, prec, fell_back, 1)
                if live is not None:
                    values.zero_()
                    values.view(-1)[live] = vc
                td = self._buf("td", (T, B), torch.float32)
                tg["gcoef"] = self._buf("gcoef", (T, B), torch.float32)
                with torch.cuda.device(dev):
                    _lib.check(lib.b2048_td_errors(h, _ptr(rewards), _ptr(values), _ptr(length), _ptr(ro.ep_weight),
                                                   float(cfg.gamma), int(cfg.critic_loss_type == "huber"),
                                                   float(cfg.huber_delta), n_traj, T, B, _ptr(td), _ptr(tg["gcoef"]), _stream()),
                               "b2048_td_errors")
                raw = td                                             # advantages := baseline-processed TD errors (:495-498)
                lam = float(self.gae_lambda)
                if lam > 0.0:
                    raw = self._buf("gae", (T, B), torch.float32)    # A_t = delta_t + gamma lambda A_{t+1}: the returns scan
                    with torch.cuda.device(dev):
                        _lib.check(lib.b2048_reverse_scan_f64(_ptr(td), _ptr(raw), _ptr(length), float(cfg.gamma) * lam, T, B,
                                                              _stream()), "b2048_reverse_scan_f64")
                info = {"td": td}
            else:
                raw = self._buf("returns", (T, B), torch.float32)
                with torch.cuda.device(dev):
                    _lib.check(lib.b2048_reverse_scan_f64(_ptr(rewards), _ptr(raw), _ptr(length), float(cfg.gamma), T, B,
                                                          _stream()), "b2048_reverse_scan_f64")
                info = {"returns": raw}
            tg["raw"] = raw
            if not one_msg:                                          # the one-message exchange forms them after its message
                self._advantages(raw, length, ro.ep_weight, mode, n_traj, tg["advantages"], tg["coef"], stats, ep_mean,
                                 window=False, allreduce=allreduce)
        n = boards.numel()

        ent_cf = ent_acc = None
        if beta > 0.0:
            # ecoef = beta x the sample's weight in the policy term: the advantage kernels in mode 0 on a constant beta give
            # beta w_b / (len_b n_traj) (episodes) or beta / (T n_traj) (windows), masked and rounded like coef
            bvals = self._buf("ent_beta", (T, B), torch.float32).fill_(beta)
            ent_cf = self._buf("ent_coef", (T, B), torch.float32)
            ent_adv = self._buf("ent_adv", (T, B), torch.float32)
            ent_acc = self._buf("ent_acc", (1,), torch.float64).zero_()
            self._advantages(bvals, length, ro.ep_weight, 0, n_traj, ent_adv, ent_cf, stats, ep_mean, window=ro.auto_reset,
                             pre=1)
            ent_cf = ent_cf.reshape(-1)
            if live is not None:
                ent_cf = ent_cf.index_select(0, live)

        def backward(net: DeviceMLP, cf: torch.Tensor, head_mode: int, with_entropy: bool = False):
            if live is not None:
                cf = cf.index_select(0, live)
            self._backward(net, boards, mflags, acts, cf, n, head_mode, prec, chunk, fell_back,
                           ent_cf if with_entropy else None, ent_acc)

        if critic:
            backward(self._critic, tg["gcoef"].reshape(-1), 1)
        if one_msg:
            self._one_message_exchange(tg["raw"], ro, n_traj, tg["advantages"], tg["coef"], stats, ep_mean, backward, allreduce)
            ss_a, ss_c = self._optimizer_step()
        else:
            backward(self._actor, tg["coef"].reshape(-1), 0, with_entropy=True)
            ss_a, ss_c = self._step(allreduce)
        info["advantages"] = tg["advantages"]
        if ent_acc is not None:
            info["entropy"] = float(ent_acc.cpu()[0]) / max(n, 1)
        info["precision"] = self._precision_info(prec, n, fell_back)
        info["actor_grad_norm"] = float(ss_a.cpu()[0]) ** 0.5
        if ss_c is not None:
            info["critic_grad_norm"] = float(ss_c.cpu()[0]) ** 0.5
        self.last_update_info = info
        if self._logger.isEnabledFor(logging.INFO):
            self._logger.info(f"Global Grad Norms: Actor: {info['actor_grad_norm']:.4f}")
            if ss_c is not None:
                self._logger.info(f"Global Grad Norms: Critic: {info['critic_grad_norm']:.4f}")
        return info
