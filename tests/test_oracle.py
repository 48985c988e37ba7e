"""CPU: the oracle against the reference's golden vectors / KATs (no GPU, no /root/reference needed)."""
import numpy as np
import pytest

import parity as P
from gym_narde_b200 import state as S
from oracle import oracle as O
from oracle import ref_loader as R


def test_philox_known_answers():
    # Random123 kat_vectors for philox4x32-10 (Salmon et al., SC'11)
    assert O.philox4x32_10([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert O.philox4x32_10([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert O.philox4x32_10([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == [
        0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_dice_are_uniform_and_in_range():
    d = [O.turn_dice(7, e, 3)[:2] for e in range(6000)]
    arr = np.array(d)
    assert arr.min() == 1 and arr.max() == 6
    hist = np.bincount(arr.ravel(), minlength=7)[1:]
    assert hist.min() > 1700 and hist.max() < 2300


def test_oracle_valid_moves_golden():
    cases = P.load_golden("ref_valid_moves.json")
    og = O.OracleNarde()
    for c in cases:
        for k in range(24):
            og.g.board[k] = c["board"][k]
        og.g.first_turn_white, og.g.first_turn_black = int(c["first_w"]), int(c["first_b"])
        got = [(f, -1 if t == 'off' else t) for f, t in og.get_valid_moves(c["roll"], c["player"])]
        assert got == [tuple(m) for m in c["moves"]]


def test_oracle_step_traces_golden():
    for tr in P.load_golden("ref_step_traces.json"):
        e = O.OracleEnv()
        obs, used = e.reset(tr["reset_rolls"])
        assert used == len(tr["reset_rolls"]) and obs.tolist() == tr["reset_obs"] and e.e.current_player == tr["player0"]
        for s in tr["steps"]:
            obs, rew, done = e.step(s["dice"], s["action"])
            assert obs.tolist() == s["obs"] and rew == s["reward"] and done == s["done"]
            assert e.state_tuple() == (tuple(s["board"]), s["off_w"], s["off_b"], int(s["first_w"]), int(s["first_b"]),
                                       s["player"])


def test_oracle_tier_n_kat():
    for c in P.load_golden("tier_n_kat.json"):
        acts, n = O.turn_enumerate(c["board_mover"], c["off"], c["dice"][0], c["dice"][1], c["first_turn"])
        assert n == len(c["afterstates"])
        assert sorted(a["after"] for a in acts) == sorted(tuple(a) for a in c["afterstates"])
        keys = [a["key"] for a in acts]
        assert keys == sorted(set(keys))


def test_oracle_known_answers_from_reference_tests():
    # tests/test_move_validation.py:13-29: start, roll [3,5] -> non-empty, first move validates
    g = O.OracleNarde()
    v = g.get_valid_moves([3, 5], 1)
    assert v == [(23, 18)]
    # tests/test_doubles_sequence.py:29-73: 17->11 with a 6 is offered when idx 11 is empty
    b = np.zeros(24, int)
    b[23], b[17], b[10] = 14, 1, -15
    g.board = b
    g.g.first_turn_white = 0
    assert (17, 11) in g.get_valid_moves([6, 6, 6, 6], 1)
    # tests/test_narde_game_manager.py:77-129: per-turn head rule (Tier N)
    start = [0] * 24
    start[23], start[11] = 15, -15
    acts, _ = O.turn_enumerate(start, 0, 6, 5, True)
    assert all(sum(1 for f, t in a["moves"] if f == 23) == 1 for a in acts)
    acts, _ = O.turn_enumerate(start, 0, 6, 6, True)
    assert max(sum(1 for f, t in a["moves"] if f == 23) for a in acts) == 2
    acts, _ = O.turn_enumerate(start, 0, 5, 5, True)
    assert max(sum(1 for f, t in a["moves"] if f == 23) for a in acts) == 1


def test_obs198_layout_and_bounds():
    # README.md:44-102 and the bounds of tests/test_observation_space.py:5-202
    b = np.zeros(24, int)
    b[23], b[11], b[0], b[5] = 9, -15, 1, 2
    o = O.obs198(b, 3, 0, 1)
    assert o.shape == (198,) and o.dtype == np.float32
    assert o[0:4].tolist() == [1, 0, 0, 0] and o[20:24].tolist() == [1, 1, 0, 0]
    assert o[92:96].tolist() == [1, 1, 1, 3.0] and o[96] == 0 and o[97] == np.float32(3 / 15.0)
    assert o[98 + 44:98 + 48].tolist() == [1, 1, 1, 6.0] and o[196:].tolist() == [1, 0]
    assert O.obs198(b, 3, 0, -1)[196:].tolist() == [0, 1]


@pytest.mark.skipif(not R.available(), reason="the original gym-narde is not in the repository: set NARDE_REFERENCE_ROOT "
                                              "or vendor it with baseline/fetch_ref.py")
def test_oracle_vs_live_reference_short():
    """Re-runs a short lock-step comparison against the real Python reference (build container only)."""
    import random
    narde, narde_env = R.load()
    rng = random.Random(5)
    for game in range(6):
        env, oe = narde_env.NardeEnv(), O.OracleEnv()
        rolls = [rng.randint(1, 6) for _ in range(40)]
        with R.injected_dice(rolls):
            obs, _ = env.reset()
        oobs, _ = oe.reset(rolls)
        assert (obs == oobs).all()
        for t in range(150):
            d = [rng.randint(1, 6), rng.randint(1, 6)]
            a = env.game.get_valid_moves(d, env.current_player)
            og = O.OracleNarde()
            og.g = oe.e.game
            assert [tuple(x) for x in a] == og.get_valid_moves(d, env.current_player)
            act = (rng.randrange(576), rng.randrange(576))
            if a and game % 2:
                m = rng.choice(a)
                act = (m[0] * 24 + (0 if m[1] == 'off' else m[1]), rng.randrange(576))
            with R.injected_dice(d):
                obs, rew, done, _, _ = env.step(act)
            oobs, orew, odone = oe.step(d, act)
            assert (obs == oobs).all() and rew == orew and done == odone
            if done:
                break


def _afterstate_positions():
    """Positions of played games (every phase: selfplay_trace snapshots up to turn 400) and synthetic bear-offs of either
    colour with one to four checkers left (so that many turns end the game), plus one finished game."""
    tr = O.selfplay_trace(17, 0, 48, 400, cap=64, max_episode_steps=0, threads=4)
    lo = tr["lo"][::8].reshape(-1, 16)
    hi = tr["hi"][::8].reshape(-1, 16)
    live = (hi[:, 11] & S.FLAG_DONE) == 0
    lo, hi = lo[live][::3], hi[live][::3]
    rng = np.random.default_rng(3)
    boards, off_w, off_b, turn = [], [], [], []
    for j in range(160):
        b = np.zeros(24, int)
        left = int(rng.integers(1, 5))
        white = j % 2 == 0
        home = range(0, 6) if white else range(12, 18)       # the mover's home in the absolute frame
        for _ in range(left):
            b[rng.choice(list(home))] += 1 if white else -1
        other = int(rng.integers(0, 15))                     # the other side: 0 off (a mars) or some off
        b[11 if white else 23] = (-1 if white else 1) * (15 - other)
        boards.append(b)
        off_w.append(15 - left if white else other)
        off_b.append(other if white else 15 - left)
        turn.append(1 if white else -1)
    slo, shi = S.pack_states(np.array(boards), off_w=np.array(off_w), off_b=np.array(off_b), turn=np.array(turn),
                             steps=np.array([(j * 37) % 300 for j in range(160)]))
    flo, fhi = S.pack_states(np.array(boards[:1]), off_w=off_w[0], off_b=off_b[0], done=True)
    return np.concatenate([lo, slo, flo]), np.concatenate([hi, shi, fhi])


def test_afterstates_batch_equals_full_step():
    """o_afterstates_batch (the oracle's narde_afterstates_scan rows) against OracleEnv.set_state + full_step(dice, k) for
    every stored (position, k): doubles and plain dice, bear-offs, game-ending turns, a finished game (no actions), and
    lists longer than the capacity (only the first `cap` are written, the count is the whole list's)."""
    lo, hi = _afterstate_positions()
    n = lo.shape[0]
    dice = np.array([[1 + (i * 7) % 6, 1 + (i * 11 + i // 6) % 6] for i in range(n)], np.uint8)
    dice[::5, 1] = dice[::5, 0]                                  # every fifth position rolls doubles
    cap = 24
    counts, acts, as_lo, as_hi = O.afterstates_batch(lo, hi, dice, cap=cap, threads=4)
    want_counts, _ = O.enumerate_batch(lo, hi, dice, cap=cap)
    assert np.array_equal(counts, want_counts)
    assert counts[-1] == 0 and not as_lo[-1].any() and not as_hi[-1].any()
    u = S.unpack_states(lo, hi)
    pairs = ended = doubles = beyond = 0
    for i in range(n):
        stored = min(int(counts[i]), cap)
        beyond += int(counts[i]) > cap
        after = S.unpack_states(as_lo[i], as_hi[i])
        assert not as_lo[i, stored:].any() and not as_hi[i, stored:].any() and not acts[i, stored:].any()
        player = int(u["turn"][i])
        mover = u["board"][i] if player == 1 else S.rotate_board(u["board"][i])
        listed, _ = O.turn_enumerate(mover, u["off_w"][i] if player == 1 else u["off_b"][i], int(dice[i, 0]),
                                     int(dice[i, 1]), u["first_w"][i] if player == 1 else u["first_b"][i], cap=cap)
        for k in range(stored):
            e = O.OracleEnv()
            e.set_state(u["board"][i], u["off_w"][i], u["off_b"][i], u["first_w"][i], u["first_b"][i], player)
            _, _, done, cnt = e.full_step(dice[i], k, want_obs=False)
            assert cnt == counts[i]
            board, ow, ob, fw, fb, pl = e.state_tuple()
            got = (tuple(after["board"][k]), after["off_w"][k], after["off_b"][k], int(after["first_w"][k]),
                   int(after["first_b"][k]), after["turn"][k])
            assert got == (board, ow, ob, fw, fb, pl), (i, k)
            assert bool(after["done"][k]) == done and after["steps"][k] == (u["steps"][i] + 1) & 0xFFFF, (i, k)
            assert S.decode_action(int(acts[i, k]) & 0xFFFFFFFFFFFFFFFF) == [
                (f, 'off' if t == O.OFF else t) for f, t in listed[k]["moves"]], (i, k)
            pairs += 1
            ended += done
            doubles += int(dice[i, 0] == dice[i, 1])
    assert pairs > 3000 and ended > 50 and doubles > 500 and beyond > 20, (pairs, ended, doubles, beyond)
