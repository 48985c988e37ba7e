"""Generates the committed golden fixtures from the REAL reference (the original gym-narde, which is not part of
this repository; oracle/ref_loader.py finds it through NARDE_REFERENCE_ROOT or baseline/_ref):
    NARDE_REFERENCE_ROOT=<gym-narde checkout> python tests/golden/gen_golden.py
Outputs (small JSON files next to this script):
  ref_valid_moves.json   Narde.get_valid_moves(roll, player) ordered lists (narde.py:58-92)
  ref_step_traces.json   NardeEnv.reset/step traces with an injected dice stream (narde_env.py:27-120)
  ref_seeded_env.json    NardeEnv driven by the real global numpy RNG (np.random.seed) -- pins the
                         facade's RNG-consumption compatibility
  tier_n_kat.json        full-turn afterstate sets composed from the reference's own primitives
                         (per-ply Narde.get_valid_moves([die]) on a scratch game + per-turn head budget)
"""
import json
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_loader as R  # noqa: E402

narde, narde_env = R.load()


def mv_json(m):
    return [int(m[0]), -1 if m[1] == 'off' else int(m[1])]


def game_json(g):
    return {"board": [int(x) for x in g.board], "off_w": int(g.borne_off_white), "off_b": int(g.borne_off_black),
            "first_w": bool(g.first_turn_white), "first_b": bool(g.first_turn_black)}


def code_of(m):
    return m[0] * 24 + (0 if m[1] == 'off' else m[1])


def valid_random_action(env, dice, rng):
    """A (code1, code2) that the reference will usually accept (evaluate_model.RandomAgent pattern)."""
    import copy
    valid = env.game.get_valid_moves(dice, env.current_player)
    if not valid:
        return (rng.randrange(576), rng.randrange(576))
    m1 = rng.choice(valid)
    c2 = rng.randrange(576)
    if len(valid) > 1:
        g2 = copy.deepcopy(env.game)
        g2.execute_rotated_move(m1, env.current_player)
        dist = m1[0] + 1 if m1[1] == 'off' else abs(m1[0] - m1[1])
        td = list(dice)
        if dist in td:
            td.remove(dist)
        else:
            td.pop(0)
        v2 = g2.get_valid_moves(td, env.current_player)
        if v2:
            c2 = code_of(rng.choice(v2))
    return (code_of(m1), c2)


def gen_step_traces(rng, n_episodes=24, max_steps=400):
    traces = []
    vm_cases = []
    for ep in range(n_episodes):
        env = narde_env.NardeEnv()
        rolls = [rng.randint(1, 6) for _ in range(8)]
        while all(rolls[2 * i] == rolls[2 * i + 1] for i in range(4)):
            rolls = [rng.randint(1, 6) for _ in range(8)]
        with R.injected_dice(rolls):
            obs, _ = env.reset()
        used = 2
        while rolls[used - 2] == rolls[used - 1]:
            used += 2
        tr = {"reset_rolls": rolls[:used], "reset_obs": [int(x) for x in obs], "player0": int(env.current_player),
              "steps": []}
        mode = ep % 3
        for t in range(max_steps):
            dice = [rng.randint(1, 6), rng.randint(1, 6)]
            if rng.random() < 0.1:
                dice[1] = dice[0]
            if rng.random() < 0.08:  # harvest get_valid_moves cases, 1/2/4-dice rolls
                for roll in (dice, [dice[0]], [dice[1]] * 4, dice[::-1]):
                    vm_cases.append({**game_json(env.game), "player": int(env.current_player), "roll": roll,
                                     "moves": [mv_json(m) for m in env.game.get_valid_moves(list(roll), env.current_player)]})
            if mode == 0:
                act = (rng.randrange(576), rng.randrange(576))
            else:
                act = valid_random_action(env, dice, rng)
            with R.injected_dice(dice):
                obs, rew, done, trunc, info = env.step(act)
            tr["steps"].append({"dice": dice, "action": [int(act[0]), int(act[1])], "obs": [int(x) for x in obs],
                                "reward": int(rew), "done": bool(done), "player": int(env.current_player),
                                **game_json(env.game)})
            if done:
                break
        traces.append(tr)
    return traces, vm_cases


def appendix_a_cases():
    """SURVEY.md Appendix A.1 boards, re-evaluated with the reference (not hand-copied answers)."""
    def sparse(d):
        b = [0] * 24
        for k, v in d.items():
            b[k] = v
        return b
    specs = [
        ({23: 15, 11: -15}, True, [3, 5], 1), ({23: 15, 11: -15}, True, [3, 5], -1),
        ({23: 15, 11: -15}, True, [6, 6], 1), ({23: 15, 11: -15}, True, [6, 6, 6, 6], 1),
        ({23: 15, 11: -15}, True, [1, 1], 1), ({23: 15, 11: -15}, True, [2, 1], -1),
        ({23: 13, 20: 1, 18: 1, 11: -15}, False, [3, 5], 1), ({23: 13, 20: 1, 18: 1, 11: -15}, False, [5, 3], 1),
        ({23: 13, 20: 1, 18: 1, 11: -15}, False, [2, 2], 1), ({23: 13, 20: 1, 18: 1, 11: -15}, False, [2, 2, 2, 2], 1),
        ({0: 2, 2: 3, 5: 10, 12: -15}, False, [6, 1], 1), ({0: 2, 2: 3, 5: 10, 12: -15}, False, [3, 4], 1),
        ({0: 2, 2: 3, 5: 9, 6: 1, 12: -15}, False, [6, 1], 1),
        ({8: 2, 9: 2, 10: 2, 11: 2, 12: 2, 14: 5, 20: -15}, False, [1, 2], 1),
        ({8: 2, 9: 2, 10: 2, 11: 2, 12: 2, 14: 5, 3: -1, 20: -14}, False, [1, 2], 1),
        ({23: 15, 17: -15}, False, [6, 5], 1),
        # boards of tests/test_doubles_sequence.py:29-154
        ({23: 14, 17: 1, 10: -15}, False, [6, 6, 6, 6], 1), ({23: 14, 17: 1, 10: -15}, False, [6], 1),
        ({23: 14, 17: 1, 11: -15}, False, [5], 1), ({23: 14, 13: 1, 11: -15}, False, [5, 5], 1),
    ]
    out = []
    for d, ft, roll, player in specs:
        g = narde.Narde()
        g.board = np.array(sparse(d), dtype=np.int32)
        g.first_turn_white = g.first_turn_black = ft
        out.append({**game_json(g), "player": player, "roll": roll,
                    "moves": [mv_json(m) for m in g.get_valid_moves(list(roll), player)]})
    return out


def gen_seeded(n_seeds=6, steps=120):
    out = []
    for s in range(n_seeds):
        arng = random.Random(1000 + s)
        env = narde_env.NardeEnv()
        obs, _ = env.reset(seed=s)
        tr = {"seed": s, "reset_obs": [int(x) for x in obs], "player0": int(env.current_player), "steps": []}
        for t in range(steps):
            # actions that do not consume the numpy RNG: half random codes, half "plausible" codes
            if t % 2 == 0:
                act = (arng.randrange(576), arng.randrange(576))
            else:
                pts = [i for i in range(24) if env._get_obs()[i] > 0]
                f1, f2 = arng.choice(pts), arng.choice(pts)
                act = (f1 * 24 + max(0, f1 - arng.randint(1, 6)), f2 * 24 + max(0, f2 - arng.randint(1, 6)))
            obs, rew, done, trunc, info = env.step(act)
            tr["steps"].append({"action": [int(act[0]), int(act[1])], "obs": [int(x) for x in obs], "reward": int(rew),
                                "done": bool(done), "player": int(env.current_player), **game_json(env.game)})
            if done:
                break
        out.append(tr)
    return out


def ref_turn_afterstates(board_mover, d1, d2, first_turn):
    """Tier-N afterstate set composed from the reference Narde primitives (SURVEY.md 8c N1)."""
    hi, lo = max(d1, d2), min(d1, d2)
    doubles = d1 == d2
    max_head = 2 if (first_turn and doubles and hi in (3, 4, 6)) else 1
    orders = [[hi] * 4] if doubles else [[hi, lo], [lo, hi]]
    nodes = []

    def dfs(board, dice, depth, head_used, oi):
        if depth == len(dice):
            return
        g = narde.Narde()
        g.board = board.copy()
        g.first_turn_white = False
        for mv in g.get_valid_moves([dice[depth]], 1):
            if mv[0] == 23 and head_used >= max_head:
                continue
            g2 = narde.Narde()
            g2.board = board.copy()
            g2.execute_rotated_move(mv, 1)
            nodes.append((depth + 1, oi, tuple(int(x) for x in g2.board)))
            dfs(g2.board, dice, depth + 1, head_used + (mv[0] == 23), oi)

    for oi, dice in enumerate(orders):
        dfs(np.array(board_mover, dtype=np.int32), dice, 0, 0, oi)
    if not nodes:
        return []
    ml = max(n[0] for n in nodes)
    keep = [n for n in nodes if n[0] == ml]
    if not doubles and ml == 1 and any(n[1] == 0 for n in keep):
        keep = [n for n in keep if n[1] == 0]
    return sorted(set(n[2] for n in keep))


def gen_tier_n(rng, n_games=12):
    """Positions from full-rules random self-play (driven by the composition itself)."""
    cases = []
    for g in range(n_games):
        board = np.zeros(24, dtype=np.int32)
        board[23], board[11] = 15, -15
        off = {1: 0, -1: 0}
        first = {1: True, -1: True}
        player = rng.choice([1, -1])
        for t in range(300):
            d1, d2 = rng.randint(1, 6), rng.randint(1, 6)
            if rng.random() < 0.12:
                d2 = d1
            mover = board.copy() if player == 1 else np.concatenate((-board[12:], -board[:12]))
            after = ref_turn_afterstates(mover, d1, d2, first[player])
            if rng.random() < 0.3 and len(after) <= 220:
                cases.append({"board_mover": [int(x) for x in mover], "off": off[player], "dice": [d1, d2],
                              "first_turn": first[player], "afterstates": [list(a) for a in after]})
            if after:
                nb = np.array(rng.choice(after), dtype=np.int32)
                off[player] = 15 - int(nb[nb > 0].sum())
                board = nb if player == 1 else np.concatenate((-nb[12:], -nb[:12]))
                first[player] = False
            if off[player] == 15:
                break
            player = -player
    # head-rule KATs (tests/test_narde_game_manager.py:77-129): per-turn head budget
    start = [0] * 24
    start[23], start[11] = 15, -15
    for dice, ft in (([6, 5], True), ([6, 6], True), ([5, 5], True), ([3, 3], True), ([4, 4], True), ([6, 6], False),
                     ([2, 1], True)):
        cases.append({"board_mover": start, "off": 0, "dice": dice, "first_turn": ft,
                      "afterstates": [list(a) for a in ref_turn_afterstates(start, dice[0], dice[1], ft)]})
    return cases


def main():
    rng = random.Random(20261018)
    traces, vm_cases = gen_step_traces(rng)
    vm_cases = appendix_a_cases() + vm_cases
    seeded = gen_seeded()
    tier_n = gen_tier_n(rng)
    for name, obj in (("ref_valid_moves.json", vm_cases), ("ref_step_traces.json", traces),
                      ("ref_seeded_env.json", seeded), ("tier_n_kat.json", tier_n)):
        p = os.path.join(HERE, name)
        with open(p, "w") as f:
            json.dump(obj, f, separators=(",", ":"))
        print(name, len(obj), os.path.getsize(p), "bytes")


if __name__ == "__main__":
    main()
