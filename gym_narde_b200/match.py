"""Lock-step matches between two policies -- two afterstate nets, or a net and the random agent -- with the results tallied
on the device: the strength measurement of TD-Gammon-style training (checkpoint against checkpoint) and the reference's
evaluate_model.evaluate (a model against the random agent), for thousands of games at once.

Per lock-step turn, entirely on the device, every launch on one stream and without a host synchronisation:
    enumerate (narde_step_full, ENUMERATE_ONLY) -> split the counts by the seat that owns the side to move
    (narde_match_split_counts) -> per NET seat: afterstate rows of the envs it owns (narde_afterstates_scan) -> its net's
    scores (tcgen05 scorer) -> each env's choice by its owner's rule (narde_match_choose)
    -> side batch for lists longer than max_actions: gather -> enumerate -> split -> rows -> score -> choose -> scatter
    -> narde_step_chosen -> outcomes and tallies (narde_match_tally).
Every afterstate row is scored once, by the net whose seat is to move; a random seat produces no rows.  The rules are
stated in include/narde_b200.h (narde_match_split_counts / narde_match_choose / narde_match_tally).
"""
from __future__ import annotations

import math

from . import _cabi
from .actor import _SideBatch

_MODES = {"max": 0, "white_value": 1}
_CHECK_EVERY = 8      # play(): turns between two reads of the games tally


class _Pool:
    """One net seat's afterstate rows in one pass (main lists or side batch): the rows of the slots whose turn the seat
    owns, their scores, offsets and row count.  rows_cap > 0 bounds the rows (the side batch); then `eff` receives the
    length of each slot's scored prefix (0 when its rows did not fit), else every row fits and eff is the count itself."""

    def __init__(self, t, dev, n, rows, rows_cap=0):
        self.counts = t.zeros(n, dtype=t.int32, device=dev)      # the seat's share of the counts (split_counts)
        self.eff = t.zeros(n, dtype=t.int32, device=dev) if rows_cap else self.counts
        self.rows_cap = rows_cap
        self.as_lo = t.zeros((rows, 16), dtype=t.uint8, device=dev)
        self.as_hi = t.zeros((rows, 16), dtype=t.uint8, device=dev)
        self.scores = t.zeros(rows, dtype=t.float32, device=dev)
        self.offsets = t.zeros(n, dtype=t.int64, device=dev)
        self.rows_dev = t.zeros(1, dtype=t.int64, device=dev)
        self.scan_ws = t.zeros((n + 127) // 128 + 4, dtype=t.int64, device=dev)   # NARDE_AFTERSTATE_SCRATCH_WORDS(n), own

    def score(self, mlp, lo, hi, actions):
        _cabi.afterstates_scan(lo, hi, actions, self.counts, self.as_lo, self.as_hi, self.scan_ws, offsets=self.offsets,
                               rows_out=self.rows_dev, rows_cap=self.rows_cap,
                               counts_eff=self.eff if self.rows_cap else None)
        mlp.score_states(self.as_lo, self.as_hi, out=self.scores, rows_dev=self.rows_dev)

    def segments(self):
        return self.scores, self.offsets, self.eff


def _check_policies(policy_a, policy_b, mode_a, mode_b):
    """(is_net per seat, mode per seat) after validation; raises ValueError.  Needs no GPU."""
    from .mlp import AfterstateMLP
    nets, modes = [], []
    for name, pol, mode in (("a", policy_a, mode_a), ("b", policy_b, mode_b)):
        if isinstance(pol, str):
            if pol != "random":
                raise ValueError("policy_%s must be an AfterstateMLP or 'random', got %r" % (name, pol))
            if mode is not None:
                raise ValueError("mode_%s applies to a net only; policy_%s is 'random'" % (name, name))
            nets.append(False)
            modes.append(0)
        elif isinstance(pol, AfterstateMLP):
            mode = "white_value" if mode is None else mode
            if mode not in _MODES:
                raise ValueError("mode_%s must be 'max' or 'white_value', got %r" % (name, mode))
            nets.append(True)
            modes.append(_MODES[mode])
        else:
            raise ValueError("policy_%s must be an AfterstateMLP or 'random', got %r" % (name, type(pol).__name__))
    return nets, modes


class AfterstateMatch:
    def __init__(self, num_games, policy_a, policy_b, seed=0, mode_a=None, mode_b=None, max_actions=64,
                 max_episode_steps=1000, env_base=0, overflow_slots=None, overflow_cap=3072, overflow_rows=None):
        """num_games lock-step games of policy A against policy B.  A policy is an AfterstateMLP or "random"; mode_a /
        mode_b ("max" or "white_value", default "white_value") is AfterstateActor's mode of a net seat and must not be
        given for a random seat.

        Seats: game g = env_base + i.  A plays WHITE in even g and BLACK in odd g, so colours are balanced to within one
        game and the results depend only on (seed, g, turn): splitting the games over shards (env_base) changes nothing.

        A net's move is AfterstateActor(mode=...)'s greedy choice over every legal action (lists longer than max_actions
        go to a side batch: overflow_slots, overflow_cap and overflow_rows as AfterstateActor's); a random move is
        VecNardeEnv.step()'s uniform action.  The games run in a VecNardeEnv(num_games, seed, env_base=env_base,
        autoreset=False, max_actions, max_episode_steps) owned by the match (`env`).

        Rounds: play() plays one game in every env to its end.  Round 0 starts as env.reset() does; a later round resets
        every env at the current turn counter, so it plays new games.  A sequence of play() calls is reproducible from
        (seed, env_base, num_games).  A truncated game (max_episode_steps turns) counts as neither side's win.

        Device memory beyond the env's: per net seat num_games * max_actions afterstate rows (36 B each) -- on one turn up
        to every env can be owned by the same seat -- plus its side-batch rows."""
        nets, modes = _check_policies(policy_a, policy_b, mode_a, mode_b)
        n = int(num_games)
        if n < 1:
            raise ValueError("num_games must be >= 1, got %r" % (num_games,))
        if int(max_actions) < 1:
            raise ValueError("max_actions must be >= 1, got %r" % (max_actions,))
        if int(max_episode_steps) < 1:
            raise ValueError("max_episode_steps must be >= 1 (every game of a round must end), got %r" % (max_episode_steps,))
        from .vec_env import VecNardeEnv
        self.env = env = VecNardeEnv(n, seed=seed, env_base=env_base, autoreset=False, max_actions=max_actions,
                                     max_episode_steps=max_episode_steps)
        t, dev = env.torch, env.device
        self.torch, self.num_games, self.cap = t, n, env.max_actions
        self.nets = (policy_a if nets[0] else None, policy_b if nets[1] else None)
        self.kinds = (1 if nets[0] else 0) | (2 if nets[1] else 0)
        self.modes = tuple(modes)
        self.pools = tuple(_Pool(t, dev, n, n * self.cap) if net else None for net in nets)
        self.choice = t.zeros(n, dtype=t.int32, device=dev)
        self.value = t.zeros(n, dtype=t.float32, device=dev)
        self.dice = env.dice
        self.act_override = t.zeros(n, dtype=t.int64, device=dev)   # chosen actions beyond the stored lists (side batch)
        self.outcome = t.zeros(n, dtype=t.uint8, device=dev)        # 0 running, 1 A won, 2 B won, 3 truncated; +4 mars
        self.tallies = t.zeros(_cabi.MATCH_TALLIES, dtype=t.int64, device=dev)
        m = max(256, n // 16) if overflow_slots is None else int(overflow_slots)
        m = -(-m // 128) * 128            # whole tiles of the side batch's kernels
        self.side, self.side_pools = None, (None, None)
        if m > 0:
            self.side = _SideBatch(t, dev, m, int(overflow_cap))
            rows = int(overflow_rows) if overflow_rows is not None else 192 * m
            self.side_pools = tuple(_Pool(t, dev, m, rows, rows_cap=rows) if net else None for net in nets)
        self._enum_ws = t.zeros(_cabi.workspace_ints(n), dtype=t.int32, device=dev)
        self._graph = self._graph_args = None
        self.rounds = 0
        env.reset()

    # -- one turn -----------------------------------------------------------------------------------
    def _choose(self, lo, hi, actions, counts, cap, pools, choice, value, eff=None, env_idx=None):
        """Split the counts by owner, score each net seat's rows with its net, and choose per slot by the owner's rule."""
        env = self.env
        if self.kinds:
            _cabi.match_split_counts(hi, counts, env.env_base, self.kinds, *(p.counts if p else None for p in pools),
                                     env_idx=env_idx)
        for pool, mlp in zip(pools, self.nets):
            if pool is not None:
                pool.score(mlp, lo, hi, actions)
        _cabi.match_choose(hi, counts, cap, env.env_base, env.seed, self.kinds, self.modes,
                           [p.segments() if p else None for p in pools], choice, value, eff=eff, env_idx=env_idx,
                           step_dev=env._step_dev)

    def _enumerate_turn(self):
        env = self.env
        _cabi.step_full(env.lo, env.hi, env.env_base, env.seed, 0, actions=env.actions, counts=env.counts,
                        dice_out=self.dice, done=env.overflow, flags=_cabi.ENUMERATE_ONLY, workspace=self._enum_ws,
                        step_dev=env._step_dev)

    def _turn(self):
        """Every launch of a turn after the turn counter is set, on the current stream one after the other.  The side
        batch's enumeration runs without a workspace: no kernel of the turn waits on another one running beside it."""
        env, sb = self.env, self.side
        self._enumerate_turn()
        self._choose(env.lo, env.hi, env.actions, env.counts, self.cap, self.pools, self.choice, self.value)
        if sb is not None:
            _cabi.gather_overflow(env.lo, env.hi, self.dice, env.overflow, sb.lo, sb.hi, sb.dice, sb.idx, sb.ctrl,
                                  act_override=self.act_override)
            _cabi.enumerate_actions_fast(sb.lo, sb.hi, sb.dice, sb.actions, sb.counts, sb.ovf)
            # (eff into sb.counts_eff: a random owner's slot gets its whole count, so the scatter does not skip it)
            self._choose(sb.lo, sb.hi, sb.actions, sb.counts, sb.cap, self.side_pools, sb.choice, sb.value,
                         eff=sb.counts_eff, env_idx=sb.idx)
            _cabi.scatter_choice(sb.choice, sb.value, sb.idx, sb.counts_eff, sb.counts, sb.cap, self.choice, self.value,
                                 sb.ctrl, sb.actions, self.act_override)
        _cabi.step_chosen(env.lo, env.hi, env.env_base, env.seed, 0, self.dice, self.choice, env.actions, env.counts,
                          act_override=self.act_override, chosen=env.chosen, obs198=env.obs, reward=env.reward,
                          done=env.done, truncated=env.trunc, stats=env.stats, flags=env._step_flags(),
                          max_episode_steps=env.max_episode_steps, step_dev=env._step_dev)
        _cabi.match_tally(env.hi, env.done, env.trunc, env.env_base, self.outcome, self.tallies)

    def step(self):
        """One lock-step turn of every game (eager launches)."""
        env = self.env
        env.step_count += 1
        env._step_dev.fill_(env.step_count)
        self._turn()

    def step_graph(self):
        """step() as one CUDA-graph replay (captured on first use, and again when env._frozen_args() changed since)."""
        env, t = self.env, self.torch
        env.step_count += 1
        key = env._frozen_args()
        if self._graph is None or self._graph_args != key:
            self._warmup()
            env._step_dev.fill_(env.step_count - 1)
            t.cuda.synchronize(env.device)
            g = t.cuda.CUDAGraph()
            with t.cuda.graph(g):
                _cabi.advance_counter(env._step_dev)
                self._turn()
            self._graph, self._graph_args = g, key
        self._graph.replay()

    def _warmup(self):
        """First-use work that must not happen during capture (function attributes, lazy allocations): the read-only part
        of a turn once, outside the graph."""
        env = self.env
        saved = env._step_dev.clone()
        env._step_dev.fill_(env.step_count)
        self._enumerate_turn()
        self._choose(env.lo, env.hi, env.actions, env.counts, self.cap, self.pools, self.choice, self.value)
        env._step_dev.copy_(saved)

    # -- rounds and results ---------------------------------------------------------------------------
    def play(self):
        """One round: reset every env, then replay turns (step_graph) until every game has an outcome -- at most
        max_episode_steps turns.  Reads the games tally once every few turns (one small copy to the host each time).
        Returns this round's tallies as results() does."""
        env = self.env
        if self.rounds == 0:
            env.reset()                   # (turn counter 0, env stats cleared)
            self.tallies.zero_()
        else:
            _cabi.reset(env.lo, env.hi, env.env_base, env.seed, env.step_count)
        self.outcome.zero_()
        self.rounds += 1
        start = self.tallies.cpu()
        goal = int(start[0]) + self.num_games
        limit = env.max_episode_steps
        for turn in range(1, limit + 1):
            self.step_graph()
            if (turn % _CHECK_EVERY == 0 or turn == limit) and int(self.tallies[0].item()) >= goal:
                break
        end = self.tallies.cpu()
        if int(end[0]) < goal:
            raise RuntimeError("%d games still running after max_episode_steps turns" % (goal - int(end[0])))
        return _summary(end - start)

    def results(self):
        """Cumulative tallies over every round (one D2H copy): games, a_wins, b_wins, a_mars / b_mars (wins by mars),
        truncated, a_white_wins / b_white_wins (wins as WHITE), plies (summed lengths of the finished games, truncated ones
        included), and derived from them: a_win_share among decided games with its normal-approximation 95 % interval,
        and a_points / b_points with a mars counting 2 (the reference's mover12 reward)."""
        return _summary(self.tallies.cpu())

    def uncovered_envs(self):
        """Env turns so far whose choice was made among the first max_actions actions only (one D2H copy); -1 without a
        side batch."""
        return int(self.side.ctrl[2].item()) if self.side is not None else -1


def _summary(v):
    d = dict(zip(_cabi.MATCH_TALLY_NAMES, (int(x) for x in v.tolist())))
    decided = d["a_wins"] + d["b_wins"]
    if decided:
        p = d["a_wins"] / decided
        half = 1.96 * math.sqrt(p * (1.0 - p) / decided)
        d["a_win_share"], d["a_win_share_ci95"] = p, (p - half, p + half)
    else:
        d["a_win_share"], d["a_win_share_ci95"] = float("nan"), (float("nan"), float("nan"))
    d["a_points"] = d["a_wins"] + d["a_mars"]
    d["b_points"] = d["b_wins"] + d["b_mars"]
    return d
