"""Multi-GPU plumbing: one process per GPU (torch.distributed, NCCL over NVLink on the GPU box, gloo in
the CPU tests).  The path shards by construction — every board / episode is independent (reference
src/reinforce_agent.py:195-252 touches no cross-environment state) — so ranks own contiguous ranges of the
GLOBAL board id, the Philox streams are keyed on that id (results are independent of the world size) and
nothing is exchanged during rollouts.  Per update the only exchange is ONE all-reduce(SUM) of the flat
gradient buffer [actor | critic] (285 KB per network for the runner-default MLP), preceded by a 32-byte
all-reduce of the four float64 baseline sums when the baseline is "batch" / "batch_norm" (the global mean / std
enter every sample's coefficient, so they have to exist before the gradient).  exchange="one_message" (opt-in) folds
both into exactly ONE float64 all-reduce [g_A | g_B | critic gradient | sums] and forms g = (g_A - mean g_B) / std
afterwards; it runs the actor's backward pass twice (+40 % of the update), which is why it is not the default."""
from __future__ import annotations

import os
from dataclasses import dataclass

import torch
import torch.distributed as dist


@dataclass
class DistInfo:
    rank: int = 0
    world_size: int = 1
    local_rank: int = 0

    @property
    def is_distributed(self) -> bool:
        return self.world_size > 1


def init_distributed(backend: str | None = None) -> DistInfo:
    """Reads RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* (torchrun); no-op for a single process."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return DistInfo(rank, world, local)


def _parse_cpulist(text: str) -> set[int]:
    cpus: set[int] = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(device_index: int, sysfs: str = "/sys") -> dict:
    """Pins this process (and therefore its pinned host buffers, which Linux places on the allocating thread's node) to the
    CPUs of the NUMA node the GPU's PCIe root hangs off.  The host-buffer path (step_many with pinned buffers: 14 B per board
    per step over PCIe) is bound by host memory once several ranks stream at once; a rank whose staging buffers sit on the
    other socket sends every byte over the inter-socket link as well.  Call it BEFORE allocating pinned memory.  No-op (and
    says why) when sysfs gives no node, e.g. in a single-node VM.  Returns what it found for the bench line."""
    out = {"numa_node": None, "bound": False}
    try:
        p = torch.cuda.get_device_properties(device_index)
        if hasattr(p, "pci_bus_id"):
            bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        else:                           # older torch: ask NVML for the device with this UUID
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(p.uuid)).encode())
            bus = pynvml.nvmlDeviceGetPciInfo(h).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            bdf = bus.lower()[-12:]     # NVML pads the domain to 8 hex digits, sysfs uses 4
        base = os.path.join(sysfs, "bus", "pci", "devices", bdf)
        with open(os.path.join(base, "numa_node")) as f:
            node = int(f.read().strip())
        out["numa_node"] = node
        out["pci"] = bdf
        if node < 0:
            out["why"] = "sysfs reports no NUMA node for the GPU"
            return out
        with open(os.path.join(sysfs, "devices", "system", "node", f"node{node}", "cpulist")) as f:
            local = _parse_cpulist(f.read())
        allowed = os.sched_getaffinity(0)
        pick = local & allowed
        out["cpus_allowed"], out["cpus_local"] = len(allowed), len(pick)
        if not pick:
            out["why"] = "none of the node's CPUs is in this process's affinity mask"
            return out
        if pick != allowed:
            os.sched_setaffinity(0, pick)
        out["bound"] = True
    except Exception as e:      # never fatal: binding is an optimisation
        out["why"] = f"{type(e).__name__}: {e}"
    return out


def shard_range(total: int, rank: int, world_size: int) -> tuple[int, int]:
    """Contiguous [start, stop) range of global board ids owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(int(total), int(world_size))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def allreduce_sum_(t: torch.Tensor) -> torch.Tensor:
    """In-place SUM over ranks (identity for a single process)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def allreduce_max_(t: torch.Tensor) -> torch.Tensor:
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t


def make_sharded_env(total_boards: int, config, info: DistInfo, seed: int = 0, device=None, **kw):
    """This rank's shard of a `total_boards`-board environment: gid0 = first global id of the shard."""
    from .batched_env import Batched2048Env
    start, stop = shard_range(total_boards, info.rank, info.world_size)
    dev = device if device is not None else torch.device("cuda", info.local_rank)
    return Batched2048Env(stop - start, config, device=dev, seed=seed, gid0=start, **kw)


def sharded_update(agent, rollout, info: DistInfo, total_episodes: int | None = None, precision="auto",
                   exchange: str = "default", fixed_horizon: bool = False, bootstrap_truncation: bool = False,
                   ppo: dict | None = None, entropy_coef: float = 0.0):
    """update_from_rollout with gradients / baseline sums all-reduced over ranks; n_traj = global episode count
    so that every rank applies exactly the update a single process holding all episodes would apply.
    exchange="one_message": exactly one all-reduce per update (see ReinforceAgent.update_from_rollout); pass
    total_episodes as well, otherwise the episode count is one more (8-byte) collective.
    fixed_horizon=True: update_from_horizon on a fixed-horizon window; total_episodes is then the global lane count, the
    per-sample weight 1 / (T n_traj) needs no further exchange (the 32-byte baseline sums, then one gradient all-reduce).
    bootstrap_truncation: passed to the update; it adds no message (the boards are replayed from global ids, V(s') is local).
    ppo (with fixed_horizon=True): keyword arguments of ReinforceAgent.update_ppo (epochs, minibatches, clip_eps,
    value_clip_eps, shuffle_seed); the window is trained with PPO instead, one gradient all-reduce per minibatch step (the
    minibatches are keyed on global sample ids: no message places them).  exchange="one_message" is refused.
    entropy_coef: the entropy bonus of the three updates; its per-sample weight is beta times the policy term's, so it adds
    no message."""
    if ppo is not None and not fixed_horizon:
        raise ValueError("sharded_update: ppo needs fixed_horizon=True (PPO trains on fixed-horizon windows)")
    if ppo is not None and exchange != "default":
        raise ValueError("sharded_update: exchange='one_message' is not implemented for PPO")
    if entropy_coef != 0.0:      # refused configurations raise before the episode-count collective
        type(agent)._check_entropy(entropy_coef, exchange, precision)
    if total_episodes is None:
        n = torch.tensor([rollout.B], dtype=torch.int64, device=rollout.length.device)
        allreduce_sum_(n)
        total_episodes = int(n.item())
    rollout.n_traj = total_episodes
    if ppo is not None:
        return agent.update_ppo(rollout, allreduce=allreduce_sum_ if info.is_distributed else None, precision=precision,
                                bootstrap_truncation=bootstrap_truncation, entropy_coef=entropy_coef, **ppo)
    if fixed_horizon:
        return agent.update_from_horizon(rollout, allreduce=allreduce_sum_ if info.is_distributed else None,
                                         precision=precision, exchange=exchange, bootstrap_truncation=bootstrap_truncation,
                                         entropy_coef=entropy_coef)
    return agent.update_from_rollout(rollout, allreduce=allreduce_sum_ if info.is_distributed else None, precision=precision,
                                     exchange=exchange, bootstrap_truncation=bootstrap_truncation, entropy_coef=entropy_coef)


def episode_rank_weights(total_reward: torch.Tensor, weights_conf, info: DistInfo | None = None) -> torch.Tensor:
    """CVaR-style episode weights by GLOBAL reward rank (reference src/reinforce_agent.py:681-716) computed on the
    device: sort the episode rewards, give the episode of rank r the configured weight of bin
    int((r + 0.5) / n * num_bins), normalise to mean 1.  With `info.world_size > 1` the rewards of every rank are
    all-gathered first (4 bytes per episode), so each rank gets the weights a single process holding all episodes
    would compute, and returns those of its own episodes.

    Ties: the reference sorts with NumPy's default (unstable) argsort, so which of two equal-reward episodes falls
    on the far side of a bin boundary is an accident of introsort there; here the sort is stable by global episode
    index.  The multiset of weights and every episode not sharing its reward with a boundary neighbour agree."""
    n_local = int(total_reward.numel())
    if weights_conf is None or len(weights_conf) == 0:
        return torch.ones(n_local, dtype=torch.float32, device=total_reward.device)
    conf = torch.as_tensor(list(weights_conf), dtype=torch.float32, device=total_reward.device)
    r = total_reward.to(torch.float64).reshape(-1)
    lo = 0
    if info is not None and info.is_distributed:
        sizes = torch.zeros(info.world_size, dtype=torch.int64, device=r.device)
        sizes[info.rank] = n_local
        allreduce_sum_(sizes)
        sizes = [int(x) for x in sizes.tolist()]
        full = torch.zeros(sum(sizes), dtype=torch.float64, device=r.device)
        lo = sum(sizes[: info.rank])
        full[lo: lo + n_local] = r
        allreduce_sum_(full)          # disjoint slices: the sum is the concatenation (works on NCCL and gloo alike)
        r = full
    n = int(r.numel())
    if n == 0:
        return torch.zeros(0, dtype=torch.float32, device=total_reward.device)
    order = torch.argsort(r, stable=True)
    pct = (torch.arange(n, dtype=torch.float64, device=r.device) + 0.5) / n
    bins = torch.clamp((pct * len(conf)).to(torch.int64), max=len(conf) - 1)
    w = torch.zeros(n, dtype=torch.float32, device=r.device)
    w[order] = conf[bins]
    m = w.mean()
    if float(m) > 1e-8:
        w = w / m
    return w[lo: lo + n_local].contiguous()
