"""Actor-critic with a SHARED trunk and two heads (policy logits + state value) and a generic lambda advantage scan —
BASELINE.json configs[3]'s wording ("shared MLP trunk + value head with advantage scan").  An addition: the reference itself
trains a separate critic network (src/reinforce_agent.py:94-105, :403-498; SURVEY.md Appendix B), which is what
``ReinforceAgent(use_critic=True)`` reproduces.  With ``gae_lambda = 0`` the advantages are the reference's TD(0) errors.

No new kernel: the flat parameter vector is [trunk | W_pi b_pi | W_v b_v]; the policy "view" (trunk + policy head, 4 outputs)
and the value "view" (trunk + value head, 1 output) are two ``b2048_mlp_desc`` whose layer pointers alias the same trunk
storage, so rollouts, the float32-grade value forward and both backward passes run on the kernels of the separate-network
path (tcgen05 included).  Back-propagation is linear in the head delta, so the gradient of
J = sum coef_t log pi(a_t | s_t) - value_coef sum w/(T n) L_v(V(s_t), r_t + gamma V(s_{t+1})) (semi-gradient, target held
constant like reinforce_agent.py:439-447) is  g_policy_view - value_coef g_value_view  on the trunk; one global-norm clip and
one optimizer step (SGD / Adam, learning_rate) act on the whole vector, and a sharded update still exchanges ONE flat buffer.
Advantages: A_t = delta_t + gamma lambda A_{t+1} (the float64 returns-scan kernel with c = gamma lambda) followed by the
configured baseline mode."""
from __future__ import annotations

import copy
from typing import Any

import numpy as np
import torch

from .MLP import ACTV, OBS, DeviceMLP, MlpDesc, init_model_params
from .reinforce_agent import ReinforceAgent, ReinforceAgentConfig


class _FlatNet:
    """theta / grad / Adam moments of the whole shared vector: what b2048_apply_update consumes."""

    def __init__(self, theta: torch.Tensor):
        self.theta = theta
        self.n_params = int(theta.numel())
        self.adam_m = torch.zeros_like(theta)
        self.adam_v = torch.zeros_like(theta)
        self.grad = torch.zeros_like(theta)


def _view(template: DeviceMLP, dims: list[int], layer_ptrs: list[tuple[int, int]]) -> DeviceMLP:
    """A DeviceMLP whose descriptor points at the given (W, b) device addresses instead of into a flat vector of its own."""
    net = object.__new__(DeviceMLP)
    net.device, net.activation = template.device, template.activation
    net.obs_mode, net.obs_log2_scale = template.obs_mode, template.obs_log2_scale
    net.dims, net.n_layers = list(dims), len(dims) - 1
    net.n_params = sum(dims[l] * dims[l + 1] + dims[l + 1] for l in range(net.n_layers))
    d = MlpDesc()
    d.n_layers, d.activation, d.obs_mode, d.obs_log2_scale = net.n_layers, ACTV[net.activation], OBS[net.obs_mode], net.obs_log2_scale
    for l, (pw, pb) in enumerate(layer_ptrs):
        d.dims[l], d.W[l], d.b[l] = dims[l], pw, pb
    d.dims[net.n_layers] = dims[-1]
    net.desc = d
    net.theta = None          # no flat vector of its own
    return net


class SharedTrunkActorCritic(ReinforceAgent):
    """ReinforceAgent API (select_action / run_episode / rollout_many / update_from_rollout / update_batch) on one network
    with a policy head and a value head.  value_coef weighs the value loss in the joint objective; gae_lambda in [0, 1]."""
    _shared_net: _FlatNet | None = None                         # set by _install, after the base constructor

    def __init__(self, env, mlp_config, agent_config: ReinforceAgentConfig | None = None, value_coef: float = 0.5,
                 gae_lambda: float = 0.0, initial_params_path: str | None = None):
        if not 0.0 <= gae_lambda <= 1.0:
            raise ValueError(f"gae_lambda must be in [0, 1], got {gae_lambda}")
        cfg = copy.copy(agent_config or ReinforceAgentConfig())
        cfg.use_critic = False                       # the base constructor builds the policy view only
        super().__init__(env, mlp_config, cfg, initial_params_path)
        self.value_coef, self.gae_lambda = float(value_coef), float(gae_lambda)
        a = self._actor
        head = init_model_params(a.dims[0], self.mlp_config.hidden_sizes, 1, self.rng, self.mlp_config.init_distribution,
                                 self.mlp_config.last_init_normal)
        self._install(a.to_params(), {"W": head["W"][-1], "b": head["b"][-1]})
        self.agent_config.use_critic = True          # update_from_rollout takes the critic branch (TD errors, value gradient)

    # ------------------------------------------------------------------ parameters
    def _install(self, policy_params: dict[str, Any], value_head: dict[str, Any]) -> None:
        tmpl = DeviceMLP(policy_params, self.mlp_config.activation, self._obs_mode, self._obs_scale, self.device)
        wv = torch.from_numpy(np.ascontiguousarray(value_head["W"], np.float32).reshape(-1)).to(self.device)
        bv = torch.from_numpy(np.ascontiguousarray(value_head["b"], np.float32).reshape(-1)).to(self.device)
        H = tmpl.dims[-2]
        assert wv.numel() == H and bv.numel() == 1, "value head must be [hidden, 1]"
        theta = torch.cat([tmpl.theta, wv, bv]).contiguous()
        self._shared_net = _FlatNet(theta)
        na = tmpl.n_params
        self._n_policy = na
        self._n_trunk = tmpl.offsets[-1][0]                     # everything before the policy head
        actor = tmpl
        actor.theta = theta[:na]                                # same storage: the policy view is a prefix of the vector
        actor._build_desc()
        base = theta.data_ptr()
        ptrs = [(int(actor.desc.W[l]), int(actor.desc.b[l])) for l in range(actor.n_layers - 1)]
        ptrs.append((base + 4 * na, base + 4 * (na + H)))
        self._actor = actor
        self._critic = _view(actor, actor.dims[:-1] + [1], ptrs)
        self._bind_grads()

    def _bind_grads(self) -> None:
        sn = self._shared_net
        if sn is None:                                          # during the base constructor
            return super()._bind_grads()
        self._grad_all = sn.grad                                # the one buffer a sharded update all-reduces
        self._actor.grad = sn.grad[: self._n_policy]
        self._critic.grad = torch.zeros(self._critic.n_params, dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ learning
    def _step(self, allreduce):
        """Merges the value view's gradient into the one vector (trunk gradient = policy part - value_coef x value part),
        then the base step: one all-reduce of that vector when sharded and _optimizer_step."""
        g, gc, nt, na = self._shared_net.grad, self._critic.grad, self._n_trunk, self._n_policy
        g[:nt].add_(gc[:nt], alpha=-self.value_coef)            # critic gradients are dL_v/dtheta (descent): minus sign
        g[na:].copy_(gc[nt:]).mul_(-self.value_coef)
        return super()._step(allreduce)

    def _optimizer_step(self):
        """One global-norm clip and SGD / Adam step (learning_rate) of the whole vector; no separate critic norm."""
        cfg = self.agent_config
        if cfg.optimizer == "adam":
            self._adam_t += 1
        return self._apply(self._shared_net, cfg.learning_rate, +1.0, self._adam_t), None

    def _one_message_exchange(self, *args, **kwargs):
        raise ValueError("exchange='one_message' is implemented for separate actor / critic networks")

    @property
    def params(self) -> dict[str, Any]:
        return self._actor.to_params()

    @params.setter
    def params(self, value: dict[str, Any]) -> None:
        """Policy view (trunk + policy head) in the reference layout; the value head is kept."""
        vh = self.value_head if self._shared_net is not None else None
        if vh is None:                                          # base constructor / load_model before _install
            return ReinforceAgent.params.fset(self, value)
        if np.asarray(value["W"][-1]).shape[0] != vh["W"].shape[0]:
            raise ValueError("policy parameters do not match the value head's input width")
        self._install(value, vh)

    @property
    def value_head(self) -> dict[str, Any]:
        t = self._shared_net.theta[self._n_policy:].cpu().numpy()
        return {"W": t[:-1].reshape(-1, 1).copy(), "b": t[-1:].copy()}

    @property
    def critic_params(self):
        """Value view (trunk + value head) in the reference layout {"W": [...], "b": [...]}."""
        p = self._actor.to_params()
        vh = self.value_head
        return {"W": p["W"][:-1] + [vh["W"]], "b": p["b"][:-1] + [vh["b"]]}

    @critic_params.setter
    def critic_params(self, value) -> None:
        raise AttributeError("the value function shares the policy's trunk: set .params and the value head via _install")

    # ------------------------------------------------------------------ state
    def save_state(self) -> dict[str, Any]:
        sn = self._shared_net
        return {"adam_t": self._adam_t, "shared": (sn.theta.clone(), sn.adam_m.clone(), sn.adam_v.clone())}

    def load_state(self, st: dict[str, Any]) -> None:
        self._adam_t = st["adam_t"]
        for dst, src in zip((self._shared_net.theta, self._shared_net.adam_m, self._shared_net.adam_v), st["shared"]):
            dst.copy_(src)

    def save_checkpoint(self, file_path: str) -> None:
        sn = self._shared_net
        np.savez(file_path, shared_theta=sn.theta.cpu().numpy(), shared_adam_m=sn.adam_m.cpu().numpy(),
                 shared_adam_v=sn.adam_v.cpu().numpy(), actor_dims=np.asarray(self._actor.dims, np.int64),
                 adam_t=np.int64(self._adam_t), value_coef=np.float64(self.value_coef), gae_lambda=np.float64(self.gae_lambda))

    def load_checkpoint(self, file_path: str) -> None:
        ck = np.load(file_path if str(file_path).endswith(".npz") else str(file_path) + ".npz")
        if "shared_theta" not in ck or [int(d) for d in ck["actor_dims"]] != [int(d) for d in self._actor.dims]:
            raise ValueError("not a shared-trunk checkpoint of this network shape")
        sn = self._shared_net
        sn.theta.copy_(torch.from_numpy(ck["shared_theta"]).to(self.device))
        sn.adam_m.copy_(torch.from_numpy(ck["shared_adam_m"]).to(self.device))
        sn.adam_v.copy_(torch.from_numpy(ck["shared_adam_v"]).to(self.device))
        self._adam_t = int(ck["adam_t"])
