"""Pins the CPU oracle against the fixtures generated from the live reference
(tests/golden/gen_golden.py)."""
import json
import os

import numpy as np
import pytest

import oracle
from helpers import ENV_CONFIGS, GOLDEN, full_env_kwargs


def cfg_for(name, **over):
    kw = full_env_kwargs(name)
    kw.pop("size")
    kw.update(over)
    return oracle.make_cfg(**kw)


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 10 rounds
    assert oracle.philox([0] * 4, [0] * 2) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert oracle.philox([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert oracle.philox([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]) == \
        [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_row_table_all_65536_rows():
    g = np.load(os.path.join(GOLDEN, "row_lut.npz"))
    left, merge, score = oracle.row_lut()
    assert (left == g["left"]).all() and (merge == g["merge"]).all() and (score == g["score"]).all()
    # facts measured on the reference (SURVEY.md section 4)
    assert int((left != np.arange(65536)).sum()) == 21210
    assert int((merge != 0).sum()) == 11295
    assert int(((merge & 0xF0) != 0).sum()) == 225
    assert int(score.sum()) == 100660224 and int(score.max()) == 131072
    assert int(((merge & 0x0F) == 1).sum() + ((merge >> 4) == 1).sum()) >= 767
    assert left[0x1111] == 0x0022 and score[0x1111] == 8
    assert left[0x2110] == 0x0022 and score[0x2110] == 4
    assert left[0x0012] == 0x0012


def test_moves_mask_done():
    g = np.load(os.path.join(GOLDEN, "moves.npz"))
    boards = g["boards"]
    n = len(boards)
    for a in range(4):
        out, msum, minfo, fl = oracle.move_many(boards, np.full(n, a, np.uint8))
        assert (out == g["result"][:, a]).all()
        assert (msum == g["merge_sum"][:, a]).all()
        assert (((fl & oracle.F_CHANGED) != 0) == (g["changed"][:, a] != 0)).all()
        nm = ((minfo & 0x0F) != 0).sum(1) + ((minfo >> 4) != 0).sum(1)
        assert (nm == g["n_merge"][:, a]).all()
        mx = np.maximum(minfo & 0x0F, minfo >> 4).max(1).astype(np.int64)
        assert (np.where(mx > 0, 1 << mx, 0) == g["merge_max"][:, a]).all()
    mask, done = oracle.mask_done(boards)
    assert (mask == g["mask"]).all() and (done == g["done"]).all()
    assert done[0] == 0 and mask[0] == 0  # the empty board: no legal move but not "done" (game2048.py:173-174)


@pytest.mark.parametrize("name", list(ENV_CONFIGS))
def test_replayed_episodes(name):
    g = np.load(os.path.join(GOLDEN, "episodes.npz"))
    seed, gid0 = int(g["seed"]), int(g["gid0"])
    board = g[f"{name}/board"]
    T, n = board.shape
    mask_on = full_env_kwargs(name)["use_action_mask"]
    cfg = cfg_for(name, action_mode="random_legal" if mask_on else "random_any")
    st = oracle.reset_many(n, seed, gid0, 0)
    assert (st["board"] == g[f"{name}/board0"]).all() and (st["flags"] == g[f"{name}/flags0"]).all()
    prev_alive = np.ones(n, bool)
    for t in range(1, T + 1):
        o = oracle.step_many(st, cfg, seed, gid0, t, want_obs=True)
        live = prev_alive
        assert (o["action"][live] == g[f"{name}/action"][t - 1][live]).all()
        assert (st["board"][live] == board[t - 1][live]).all()
        assert (o["reward64"][live] == g[f"{name}/reward"][t - 1][live]).all()
        assert (o["reward"][live] == g[f"{name}/reward"][t - 1][live].astype(np.float32)).all()
        assert (o["flags"][live] == g[f"{name}/flags"][t - 1][live]).all()
        assert (st["score"][live] == g[f"{name}/score"][t - 1][live]).all()
        assert (st["step"][live] == g[f"{name}/step"][t - 1][live]).all()
        assert ((1 << st["max_exp"][live].astype(np.int64)) == g[f"{name}/max_tile"][t - 1][live]).all()
        if t <= g[f"{name}/obs"].shape[0]:
            assert (o["obs"][live] == g[f"{name}/obs"][t - 1][live]).all()
        prev_alive = g[f"{name}/alive"][t - 1]


def test_autoreset_replay():
    g = np.load(os.path.join(GOLDEN, "autoreset.npz"))
    seed, gid0 = int(g["seed"]), int(g["gid0"])
    T, n = g["board"].shape
    cfg = cfg_for("runner_default", action_mode="random_legal", auto_reset=True, max_steps=int(g["max_steps"]))
    st = oracle.reset_many(n, seed, gid0, 0)
    n_reset = 0
    for t in range(1, T + 1):
        o = oracle.step_many(st, cfg, seed, gid0, t)
        assert (st["board"] == g["board"][t - 1]).all()
        assert (o["reward64"] == g["reward"][t - 1]).all()
        assert (o["flags"] == g["flags"][t - 1]).all()
        assert (o["action"] == g["action"][t - 1]).all()
        n_reset += int(((o["flags"] & (oracle.F_DONE | oracle.F_TRUNC)) != 0).sum())
    assert n_reset == 64


def test_seeded_known_answers_pack():
    with open(os.path.join(GOLDEN, "seeded.json")) as f:
        facts = json.load(f)
    # SURVEY.md section 8c
    assert facts["reset_seed"]["0"] == [[0, 0, 0, 0], [0, 0, 0, 0], [0, 2, 0, 0], [0, 2, 0, 0]]
    assert facts["reset_seed"]["1"] == [[0, 0, 0, 0], [0, 0, 0, 4], [2, 0, 0, 0], [0, 0, 0, 0]]
    assert facts["runner_default_first8"][0] == [167, 227.0, 256]
    assert facts["seed_iter_3"][0] == 789974133212406139
    # replay reset(1) + actions 0,1,2,3 through the oracle's move (spawns taken from the recorded states)
    state = np.array(facts["reset_seed"]["1"])
    for s in facts["reset1_steps"]:
        b = np.array([oracle.pack_board(state)], np.uint64)
        out, msum, _, fl = oracle.move_many(b, np.array([s["action"]], np.uint8))
        assert int(msum[0]) == sum(s["merged"])
        after = np.array(s["state"])
        moved = oracle.unpack_board(out[0])
        diff = (after != moved)
        assert diff.sum() == 1 and moved[diff][0] == 0 and after[diff][0] in (2, 4)  # exactly the spawned tile
        state = after
    assert facts["reset1_score"] == 4


def test_reverse_scan_matches_reference_returns():
    g = np.load(os.path.join(GOLDEN, "mlp.npz"))
    lens = g["ret/lens"]
    rewards = g["ret/rewards"]
    T, B = int(lens.max()), len(lens)
    x = np.zeros((T, B), np.float32)
    off = 0
    for b, L in enumerate(lens):
        x[:L, b] = rewards[off:off + L]
        off += L
    for gamma in (0.99, 1.0, 0.5):
        y = oracle.reverse_scan(x, lens, gamma)
        ref = g[f"ret/{gamma}/off/returns"]
        got = np.concatenate([y[:L, b] for b, L in enumerate(lens)])
        assert (got == ref).all()


def test_symmetries_oracle_vs_reference_fixture():
    """oracle/learner.symmetries vs Game2048Env.get_symmetries outputs (tests/golden/symmetries.npz)."""
    from oracle import learner
    g = np.load(os.path.join(GOLDEN, "symmetries.npz"))
    ob, om, oa = learner.symmetries(g["boards"], g["masks"], g["actions"])
    assert (ob == g["out_boards"]).all() and (om == g["out_masks"]).all() and (oa == g["out_actions"]).all()


def test_symmetry_kernel_tables_match_reference_fixture():
    """The permutation constants compiled into symmetries_kernel (csrc/b2048_env.cu), applied on the CPU, reproduce
    the reference's 8 variants — so the GPU kernel is pinned to the reference even without a GPU."""
    import re
    from helpers import ROOT
    src = open(os.path.join(ROOT, "rl-2048-with-reinforce-and-actor-critic_b200", "csrc", "b2048_env.cu")).read()
    body = src[src.index("__constant__ SymVariant kSym[8]"):]
    body = body[:body.index("};")]
    ent = re.findall(r"\{0x([0-9A-F]{16})ull, 0x([0-9A-F]{2})u, 0x([0-9A-F]{2})u\}", body)
    assert len(ent) == 8
    g = np.load(os.path.join(GOLDEN, "symmetries.npz"))
    b, m, a = g["boards"], g["masks"].astype(np.uint32), g["actions"].astype(np.uint32)
    for v, (perm, amap, mperm) in enumerate(ent):
        perm, amap, mperm = int(perm, 16), int(amap, 16), int(mperm, 16)
        nb = np.zeros_like(b)
        for c in range(16):
            src_cell = (perm >> (4 * c)) & 15
            nb |= ((b >> np.uint64(4 * src_cell)) & np.uint64(15)) << np.uint64(4 * c)
        nm = np.zeros_like(m)
        for k in range(4):
            nm |= ((m >> ((mperm >> (2 * k)) & 3)) & 1) << k
        na = (amap >> (2 * a)) & 3
        assert (nb == g["out_boards"][v]).all(), v
        assert (nm == g["out_masks"][v]).all(), v
        assert (na == g["out_actions"][v]).all(), v


@pytest.mark.parametrize("name,prio", [("urdl", (0, 1, 2, 3)), ("urld", (0, 1, 3, 2))])
def test_priority_policies_oracle_vs_reference_fixture(name, prio):
    """Episodes played by the reference's own action_gen_1 / action_gen_2 (tools/simple_action_gen.py:16-33) on the
    reference env (tests/golden/priority.npz) vs the oracle in B2048_ACT_PRIORITY mode."""
    g = np.load(os.path.join(GOLDEN, "priority.npz"))
    seed, gid0 = int(g["seed"]), int(g["gid0"])
    n = len(g[f"{name}/board0"])
    cfg = oracle.make_cfg(reward_mode="sum", obs_mode="none", max_steps=0, action_mode="priority", action_priority=prio)
    st = oracle.reset_many(n, seed, gid0, 0)
    assert (st["board"] == g[f"{name}/board0"]).all() and (st["flags"] == g[f"{name}/flags0"]).all()
    alive = np.ones(n, bool)
    for t in range(len(g[f"{name}/board"])):
        o = oracle.step_many(st, cfg, seed, gid0, t + 1)
        assert (o["action"][alive] == g[f"{name}/action"][t][alive]).all()
        assert (st["board"][alive] == g[f"{name}/board"][t][alive]).all()
        assert (o["reward64"][alive] == g[f"{name}/reward"][t][alive]).all()
        assert (o["flags"][alive] == g[f"{name}/flags"][t][alive]).all()
        assert (st["score"][alive] == g[f"{name}/score"][t][alive]).all()
        alive = g[f"{name}/alive"][t]
