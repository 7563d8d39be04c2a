"""D4 symmetry augmentation on packed boards (reference src/env.py:317-397 ``get_symmetries`` and
src/reinforce_agent.py:773-808 ``_augment_trajectories``): the 8 (board, action, mask) variants are
nibble permutations of the packed board, a relabelling of the action and a permutation of the 4 mask
bits.  ``augment_rollout`` runs the CUDA kernel behind ``b2048_symmetries`` (include/b2048.h); the
``transform_*`` helpers restate the same permutations with torch indexing (used by the tests)."""
from __future__ import annotations

import numpy as np
import torch


def _variant_tables():
    """cell permutation / action map / mask-bit permutation of the 8 variants, in the reference's order."""
    base = np.arange(16).reshape(4, 4)
    perms, amaps, mperms = [], [], []
    for flipped in (False, True):
        b = np.fliplr(base.copy()) if flipped else base.copy()
        amap = np.array([0, 3, 2, 1]) if flipped else np.arange(4)        # action a -> amap[a]
        mperm = np.array([0, 3, 2, 1]) if flipped else np.arange(4)       # new_mask[i] = mask[mperm[i]]
        for _ in range(4):
            perms.append(b.reshape(16).copy())       # new_cells[i] = cells[perm[i]]
            amaps.append(amap.copy())
            mperms.append(mperm.copy())
            b = np.rot90(b, k=1)
            amap = (amap - 1) % 4
            mperm = np.roll(mperm, -1)
    return perms, amaps, mperms


_PERMS, _AMAPS, _MPERMS = _variant_tables()


def transform_boards(boards: torch.Tensor, variant: int) -> torch.Tensor:
    shifts = torch.arange(16, device=boards.device, dtype=torch.int64) * 4
    cells = (boards.unsqueeze(-1) >> shifts) & 15
    perm = torch.as_tensor(_PERMS[variant], device=boards.device)
    return (cells[..., perm] << shifts).sum(-1)


def transform_actions(actions: torch.Tensor, variant: int) -> torch.Tensor:
    amap = torch.as_tensor(_AMAPS[variant], device=actions.device, dtype=torch.uint8)
    return amap[actions.long()]


def transform_flags(flags: torch.Tensor, variant: int) -> torch.Tensor:
    mperm = _MPERMS[variant]
    out = flags & 0xF0
    for i in range(4):
        out = out | (((flags >> int(mperm[i])) & 1) << i)
    return out


def augment_rollout(ro):
    """Rollout with 8x the episodes (every dihedral variant), weights repeated, n_traj = 8 x the caller's n_traj (the
    GLOBAL episode count when the episodes are sharded over ranks; B when it was not set).  A fixed-horizon window stays
    one (auto_reset is kept: the DONE / TRUNC flag bits travel with the boards)."""
    import ctypes as C
    from . import _lib
    from .batched_env import get_handle
    from .reinforce_agent import Rollout
    T, B = ro.T, ro.B
    dev = ro.boards.device
    boards = torch.empty((T + 1, 8 * B), dtype=torch.int64, device=dev)
    flags = torch.empty((T + 1, 8 * B), dtype=torch.uint8, device=dev)
    actions = torch.empty((T, 8 * B), dtype=torch.uint8, device=dev)
    lib, h = _lib.load(), get_handle(dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    src_b, src_f, src_a = ro.boards[: T + 1].contiguous(), ro.flags[: T + 1].contiguous(), ro.actions[:T].contiguous()
    with torch.cuda.device(dev):
        _lib.check(lib.b2048_symmetries(h, p(src_b), p(src_f), None, p(boards), p(flags), None, T + 1, B, stream),
                   "b2048_symmetries")
        if T > 0:
            _lib.check(lib.b2048_symmetries(h, None, None, p(src_a), None, None, p(actions), T, B, stream), "b2048_symmetries")
    rewards = ro.rewards.repeat(1, 8)
    length = ro.length.repeat(8)
    w = None if ro.ep_weight is None else ro.ep_weight.repeat(8)
    return Rollout(boards, flags, actions, rewards.contiguous(), length, T, w, 8 * (ro.n_traj if ro.n_traj is not None else B),
                   ro.auto_reset)
