"""ctypes wrapper over oracle/libnarde_oracle.so -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package (gym_narde_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libnarde_oracle.so")

OFF = -1
NONE = -2


class OGame(C.Structure):
    _fields_ = [
        ("board", C.c_int32 * 24),
        ("borne_off_white", C.c_int32),
        ("borne_off_black", C.c_int32),
        ("first_turn_white", C.c_int32),
        ("first_turn_black", C.c_int32),
    ]


class OEnv(C.Structure):
    _fields_ = [("game", OGame), ("current_player", C.c_int32)]


class OTurnAction(C.Structure):
    _fields_ = [
        ("n_moves", C.c_int32),
        ("moves", C.c_int32 * 8),
        ("key", C.c_int32),
        ("after", C.c_int32 * 24),
        ("after_off", C.c_int32),
    ]


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "narde_oracle.c")
    hdr = os.path.join(_HERE, "narde_oracle.h")
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(p) > os.path.getmtime(_LIB_PATH) for p in (src, hdr)
    )
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        i32p = C.POINTER(C.c_int32)
        L.o_game_init.argtypes = [C.POINTER(OGame)]
        L.o_rotate_board.argtypes = [i32p, i32p]
        L.o_violates_block_rule.argtypes = [i32p]
        L.o_violates_block_rule.restype = C.c_int
        L.o_get_valid_moves.argtypes = [C.POINTER(OGame), i32p, C.c_int, C.c_int, i32p]
        L.o_get_valid_moves.restype = C.c_int
        L.o_execute_rotated_move.argtypes = [C.POINTER(OGame), C.c_int, C.c_int, C.c_int]
        L.o_env_reset.argtypes = [C.POINTER(OEnv), i32p, C.c_int]
        L.o_env_reset.restype = C.c_int
        L.o_env_step.argtypes = [C.POINTER(OEnv), C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, i32p]
        L.o_turn_enumerate.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.POINTER(OTurnAction), C.POINTER(C.c_int64)]
        L.o_turn_enumerate.restype = C.c_int
        L.o_obs198.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.o_full_step.argtypes = [C.POINTER(OEnv), C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.POINTER(C.c_float), i32p, C.POINTER(C.c_float)]
        L.o_full_step.restype = C.c_int
        L.o_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.o_turn_dice.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, i32p, i32p, C.POINTER(C.c_uint32)]
        L.o_opening_player.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64]
        L.o_opening_player.restype = C.c_int
        L.o_selfplay.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_int64),
                                 C.POINTER(C.c_int64), C.POINTER(C.c_double)]
        L.o_selfplay.restype = C.c_int64
        u8p, vp = C.POINTER(C.c_uint8), C.c_void_p
        L.o_selfplay_trace.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_uint64, vp, vp, vp, C.c_int64,
                                       C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, vp, vp, vp, vp, vp,
                                       vp, vp, vp, vp, vp]
        L.o_selfplay_trace.restype = C.c_int64
        L.o_enumerate_batch.argtypes = [vp, vp, vp, C.c_int64, C.c_int, vp, vp]
        L.o_enumerate_batch.restype = None
        L.o_afterstates_batch.argtypes = [vp, vp, vp, C.c_int64, C.c_int, vp, vp, vp, vp]
        L.o_afterstates_batch.restype = None
        L.o_list_weight.argtypes = [C.c_int]
        L.o_list_weight.restype = C.c_uint64
        _lib = L
    return _lib


def _i32(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(C.POINTER(C.c_int32))


# ------------------------------------------------------------------------------------------
# Pythonic helpers mirroring the reference's object surface
# ------------------------------------------------------------------------------------------
class OracleNarde:
    """Mirror of gym_narde/envs/narde.py:Narde backed by the C oracle."""

    def __init__(self):
        self.g = OGame()
        lib().o_game_init(C.byref(self.g))

    @property
    def board(self):
        return np.ctypeslib.as_array(self.g.board)

    @board.setter
    def board(self, v):
        v = np.asarray(v, dtype=np.int32)
        for i in range(24):
            self.g.board[i] = int(v[i])

    def get_valid_moves(self, roll, current_player=1):
        r, rp = _i32(list(roll))
        out = np.zeros(96 * 2, dtype=np.int32)
        n = lib().o_get_valid_moves(C.byref(self.g), rp, len(r), int(current_player),
                                    out.ctypes.data_as(C.POINTER(C.c_int32)))
        return [(int(out[2 * i]), 'off' if out[2 * i + 1] == OFF else int(out[2 * i + 1])) for i in range(n)]

    def execute_rotated_move(self, move, current_player):
        to = OFF if move[1] == 'off' else int(move[1])
        lib().o_execute_rotated_move(C.byref(self.g), int(move[0]), to, int(current_player))

    def violates_block_rule(self, board):
        b, bp = _i32(board)
        return bool(lib().o_violates_block_rule(bp))


class OracleEnv:
    """Mirror of gym_narde/envs/narde_env.py:NardeEnv with the dice passed in explicitly."""

    def __init__(self):
        self.e = OEnv()
        lib().o_game_init(C.byref(self.e.game))
        self.e.current_player = 1

    def reset(self, rolls):
        r, rp = _i32(list(rolls))
        used = lib().o_env_reset(C.byref(self.e), rp, len(r))
        return self.obs(), used

    def obs(self):
        out = np.zeros(24, dtype=np.int32)
        g = self.e.game
        b = np.array(g.board[:], dtype=np.int32)
        if self.e.current_player == 1:
            return b
        return np.concatenate((-b[12:], -b[:12])).astype(np.int32)

    def step(self, dice, action):
        obs = np.zeros(24, dtype=np.int32)
        rew = C.c_int32(0)
        done = C.c_int32(0)
        lib().o_env_step(C.byref(self.e), int(dice[0]), int(dice[1]), int(action[0]), int(action[1]),
                         obs.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(rew), C.byref(done))
        return obs, int(rew.value), bool(done.value)

    def full_step(self, dice, action_idx, reward_mode=0, want_obs=True):
        obs = np.zeros(198, dtype=np.float32)
        rew = C.c_float(0)
        done = C.c_int32(0)
        n = lib().o_full_step(C.byref(self.e), int(dice[0]), int(dice[1]), int(action_idx), int(reward_mode),
                              C.byref(rew), C.byref(done),
                              obs.ctypes.data_as(C.POINTER(C.c_float)) if want_obs else None)
        return obs, float(rew.value), bool(done.value), n

    # convenience accessors
    @property
    def board(self):
        return np.array(self.e.game.board[:], dtype=np.int32)

    def state_tuple(self):
        g = self.e.game
        return (tuple(g.board[:]), g.borne_off_white, g.borne_off_black, g.first_turn_white,
                g.first_turn_black, self.e.current_player)

    def set_state(self, board, off_w=0, off_b=0, first_w=0, first_b=0, player=1):
        g = self.e.game
        for i in range(24):
            g.board[i] = int(board[i])
        g.borne_off_white, g.borne_off_black = int(off_w), int(off_b)
        g.first_turn_white, g.first_turn_black = int(first_w), int(first_b)
        self.e.current_player = int(player)


def turn_enumerate(board_mover, mover_off, d1, d2, first_turn, cap=8192, with_nodes=False):
    """Returns list of dicts (sorted canonical order) for the Tier-N full-turn enumeration."""
    b, bp = _i32(board_mover)
    arr = (OTurnAction * cap)()
    nodes = C.c_int64(0)
    n = lib().o_turn_enumerate(bp, int(mover_off), int(d1), int(d2), int(bool(first_turn)), cap, arr,
                               C.byref(nodes))
    out = []
    for i in range(min(n, cap)):
        a = arr[i]
        mv = [(a.moves[2 * k], a.moves[2 * k + 1]) for k in range(a.n_moves)]
        out.append({"moves": mv, "key": a.key, "after": tuple(a.after[:]), "after_off": a.after_off})
    if with_nodes:
        return out, n, nodes.value
    return out, n


def obs198(board_abs, off_w, off_b, player):
    b, bp = _i32(board_abs)
    out = np.zeros(198, dtype=np.float32)
    lib().o_obs198(bp, int(off_w), int(off_b), int(player), out.ctypes.data_as(C.POINTER(C.c_float)))
    return out


def philox4x32_10(ctr, key):
    c = (C.c_uint32 * 4)(*[int(x) & 0xFFFFFFFF for x in ctr])
    k = (C.c_uint32 * 2)(*[int(x) & 0xFFFFFFFF for x in key])
    o = (C.c_uint32 * 4)()
    lib().o_philox4x32_10(c, k, o)
    return [int(x) for x in o]


def turn_dice(seed, env, step):
    d1, d2, w = C.c_int32(0), C.c_int32(0), C.c_uint32(0)
    lib().o_turn_dice(int(seed), int(env), int(step), C.byref(d1), C.byref(d2), C.byref(w))
    return d1.value, d2.value, w.value


def opening_player(seed, env, step):
    return int(lib().o_opening_player(int(seed), int(env), int(step)))


def selfplay(seed, env_base, n_envs, n_steps, step0=0):
    """Full-rules random self-play in C (CPU baseline).  Returns (env_steps, sum_actions, episodes)."""
    a, e, c = C.c_int64(0), C.c_int64(0), C.c_double(0)
    n = lib().o_selfplay(int(seed), int(env_base), int(n_envs), int(n_steps), int(step0), C.byref(a), C.byref(e),
                         C.byref(c))
    return int(n), int(a.value), int(e.value)


def list_weights(cap):
    """The multipliers of o_selfplay_trace's action-list checksum, as int64 bit patterns [cap]."""
    return np.array([lib().o_list_weight(k) for k in range(cap)], dtype=np.uint64).view(np.int64)


def selfplay_trace(seed, env_base, n_envs, n_steps, step0=0, init=None, words=None, word_mode=1, cap=64,
                   reward_mode=0, autoreset=True, max_episode_steps=1000, threads=None, want_states=True,
                   with_obs=False):
    """o_selfplay_trace over envs [env_base, env_base + n_envs), split over `threads` host threads (ctypes
    releases the GIL; every thread plays a contiguous block of envs into the shared [n_steps, n_envs] arrays).
    init: (lo, hi) uint8 [n_envs, 16] start states or None (fresh games, roll-off at step0).
    words: uint32 [n_steps, n_envs] policy words or None (the turn's Philox word).
    Returns a dict of numpy arrays [n_steps, n_envs, ...] + "stats" int64[8] + "turns"."""
    from concurrent.futures import ThreadPoolExecutor
    L = lib()
    T, n = int(n_steps), int(n_envs)
    out = {"chosen": np.zeros((T, n), np.int64), "count": np.zeros((T, n), np.int32),
           "dice": np.zeros((T, n, 2), np.uint8), "done": np.zeros((T, n), np.uint8),
           "reward": np.zeros((T, n), np.float32), "hash": np.zeros((T, n), np.int64)}
    if want_states:
        out["lo"] = np.zeros((T, n, 16), np.uint8)
        out["hi"] = np.zeros((T, n, 16), np.uint8)
    if init is not None:
        ilo = np.ascontiguousarray(init[0], dtype=np.uint8).reshape(n, 16)
        ihi = np.ascontiguousarray(init[1], dtype=np.uint8).reshape(n, 16)
    if words is not None:
        words = np.ascontiguousarray(words).view(np.uint32).reshape(T, n)
    threads = int(threads or os.cpu_count() or 1)
    per = max(1, -(-n // threads))
    blocks = [(b, min(b + per, n)) for b in range(0, n, per)]
    stats = np.zeros((len(blocks), 8), np.int64)
    obs_chk = np.zeros(len(blocks), np.float64)

    def ptr(a, off):
        return None if a is None else a.ctypes.data + off * a.itemsize

    def run(k):
        b, e = blocks[k]
        return L.o_selfplay_trace(
            int(seed) & 0xFFFFFFFFFFFFFFFF, (int(env_base) + b) & 0xFFFFFFFF, e - b, T, int(step0),
            ptr(ilo, 16 * b) if init is not None else None, ptr(ihi, 16 * b) if init is not None else None,
            ptr(words, b) if words is not None else None, n, int(word_mode), int(cap), int(reward_mode),
            int(bool(autoreset)), int(max_episode_steps), n,
            ptr(out.get("lo"), 16 * b), ptr(out.get("hi"), 16 * b), ptr(out["chosen"], b), ptr(out["count"], b),
            ptr(out["dice"], 2 * b), ptr(out["done"], b), ptr(out["reward"], b), ptr(out["hash"], b),
            stats[k].ctypes.data, obs_chk[k:].ctypes.data if with_obs else None)

    if len(blocks) == 1:
        turns = run(0)
    else:
        with ThreadPoolExecutor(len(blocks)) as ex:
            turns = sum(ex.map(run, range(len(blocks))))
    st = stats.sum(0)
    st[6] = stats[:, 6].max()
    out["stats"] = st
    out["obs_checksum"] = float(obs_chk.sum())
    out["turns"] = int(turns)
    return out


def enumerate_batch(lo, hi, dice, cap=64, threads=None):
    """o_enumerate_batch on host threads: (counts int32 [n], list checksums int64 [n])."""
    from concurrent.futures import ThreadPoolExecutor
    L = lib()
    lo = np.ascontiguousarray(lo, np.uint8).reshape(-1, 16)
    hi = np.ascontiguousarray(hi, np.uint8).reshape(-1, 16)
    dice = np.ascontiguousarray(dice, np.uint8).reshape(-1, 2)
    n = lo.shape[0]
    counts, hashes = np.zeros(n, np.int32), np.zeros(n, np.int64)
    threads = int(threads or os.cpu_count() or 1)
    per = max(1, -(-n // (threads * 4)))

    def run(b):
        e = min(b + per, n)
        L.o_enumerate_batch(lo.ctypes.data + 16 * b, hi.ctypes.data + 16 * b, dice.ctypes.data + 2 * b, e - b, int(cap),
                            counts.ctypes.data + 4 * b, hashes.ctypes.data + 8 * b)

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(run, range(0, n, per)))
    return counts, hashes


def afterstates_batch(lo, hi, dice, cap=64, threads=None):
    """o_afterstates_batch on host threads: (counts int32 [n], actions int64 [n, cap], as_lo, as_hi uint8 [n, cap, 16]).
    Entry (i, k) for k < min(counts[i], cap) is canonical action k of env i and the packed state after it and the end of
    the turn, as narde_afterstates_scan writes row offsets[i] + k; the other entries are zero."""
    from concurrent.futures import ThreadPoolExecutor
    L = lib()
    lo = np.ascontiguousarray(lo, np.uint8).reshape(-1, 16)
    hi = np.ascontiguousarray(hi, np.uint8).reshape(-1, 16)
    dice = np.ascontiguousarray(dice, np.uint8).reshape(-1, 2)
    n, cap = lo.shape[0], int(cap)
    counts, actions = np.zeros(n, np.int32), np.zeros((n, cap), np.int64)
    as_lo, as_hi = np.zeros((n, cap, 16), np.uint8), np.zeros((n, cap, 16), np.uint8)
    threads = int(threads or os.cpu_count() or 1)
    per = max(1, -(-n // (threads * 4)))

    def run(b):
        e = min(b + per, n)
        L.o_afterstates_batch(lo.ctypes.data + 16 * b, hi.ctypes.data + 16 * b, dice.ctypes.data + 2 * b, e - b, cap,
                              counts.ctypes.data + 4 * b, actions.ctypes.data + 8 * cap * b,
                              as_lo.ctypes.data + 16 * cap * b, as_hi.ctypes.data + 16 * cap * b)

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(run, range(0, n, per)))
    return counts, actions, as_lo, as_hi
