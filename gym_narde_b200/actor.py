"""Batched afterstate actor (SURVEY.md section 8(f) rank 1): the device-resident replacement of
the per-move loop of DQNAgent.act (train_deepq_pytorch.py:411-600), greedy or exploring.

Per lock-step turn, entirely on the GPU and without a host synchronisation:
    roll (Philox) -> get_valid_actions (full legal-turn enumeration) -> afterstate of every legal
    action (narde_afterstates) -> Box(198) encoding + DecomposedDQN(198) forward + max_a Q on the
    tcgen05 tensor cores (narde_mlp_score_states) -> greedy choice per env (narde_segment_argmax), or
    epsilon-greedy / softmax once exploration is on (narde_segment_sample) -> VecNardeEnv.step(action_idx, dice).
"""
from __future__ import annotations

import math

from . import _cabi

_FLT_MAX = 3.4028234663852886e38


class _SideBatch:
    """Buffers of the second pass over the environments whose legal list exceeds env.max_actions."""

    def __init__(self, t, dev, m, cap):
        self.cap = cap
        self.lo = t.zeros((m, 16), dtype=t.uint8, device=dev)
        self.hi = t.zeros((m, 16), dtype=t.uint8, device=dev)
        self.dice = t.ones((m, 2), dtype=t.uint8, device=dev)
        self.idx = t.full((m,), -1, dtype=t.int32, device=dev)
        self.ctrl = t.zeros(4, dtype=t.int32, device=dev)
        self.actions = t.zeros((m, cap), dtype=t.int64, device=dev)
        self.counts = t.zeros(m, dtype=t.int32, device=dev)
        self.counts_eff = t.zeros(m, dtype=t.int32, device=dev)
        self.ovf = t.zeros(m, dtype=t.uint8, device=dev)
        self.ws = t.zeros(_cabi.workspace_ints(m), dtype=t.int32, device=dev)
        self.scan_ws = t.zeros((m + 127) // 128 + 4, dtype=t.int64, device=dev)
        self.offsets = t.zeros(m, dtype=t.int64, device=dev)
        self.rows_dev = t.zeros(1, dtype=t.int64, device=dev)
        self.choice = t.zeros(m, dtype=t.int32, device=dev)
        self.value = t.zeros(m, dtype=t.float32, device=dev)


def _score_side_batch(mlp, sb, lo, hi, dice, overflow, act_override=None, workspace=None):
    """A side batch up to its scores, on the current stream: gather the positions flagged in `overflow` -> enumerate them
    with the side capacity (workspace: narde_enumerate_fast's, None = order-dependent turns resolved inline) -> afterstate
    rows (bounded by sb.rows_cap) -> score."""
    _cabi.gather_overflow(lo, hi, dice, overflow, sb.lo, sb.hi, sb.dice, sb.idx, sb.ctrl, act_override=act_override)
    _cabi.enumerate_actions_fast(sb.lo, sb.hi, sb.dice, sb.actions, sb.counts, sb.ovf, workspace)
    _cabi.afterstates_scan(sb.lo, sb.hi, sb.actions, sb.counts, sb.as_lo, sb.as_hi, sb.scan_ws, offsets=sb.offsets,
                           rows_out=sb.rows_dev, rows_cap=sb.rows_cap, counts_eff=sb.counts_eff)
    # (the scorer keeps no state between launches, so this one may be queued beside the first pass's: its CTAs get their
    # SMs when those leave)
    mlp.score_states(sb.as_lo, sb.as_hi, out=sb.scores, rows_dev=sb.rows_dev)


class AfterstateActor:
    def __init__(self, env, mlp, mode="max", overflow_slots=None, overflow_cap=3072, overflow_rows=None, epsilon=0.0,
                 temperature=0.0):
        """env: VecNardeEnv(rules="full"); mlp: AfterstateMLP; mode: "max" (the mover maximises the score)
        or "white_value" (the net scores positions for WHITE: WHITE maximises, BLACK minimises).

        Exploration (DQNAgent.act's epsilon, decayed by the trainer; see set_exploration): each env turn explores with
        probability `epsilon` and then plays the env's own uniform random action (the one VecNardeEnv.step() plays
        without actions: epsilon=1 is exactly that policy); otherwise, with `temperature` > 0, it samples
        softmax(score / temperature) (the score negated for BLACK in "white_value" mode), else it plays the arg-max.
        The random words come from the env's Philox stream keyed by seed, global env id and turn number
        (include/narde_b200.h, narde_segment_sample): results do not depend on sharding and can be recomputed on the host.
        `value` holds the score of the action chosen.

        Every legal action is scored, as DQNAgent.act does (train_deepq_pytorch.py:430-507): environments whose list
        is longer than env.max_actions (doubles turns, up to ~1300 actions; 0.5-1 % of the envs in self-play) get a
        second pass with capacity `overflow_cap` (default 3072 >= C(18, 4) = 3060, the number of 4-multisets of 15 sources:
        every doubles turn fits; 2018 legal turns have been seen in self-play) in a side batch of `overflow_slots` environments (default N/16, at
        least 256) sharing `overflow_rows` afterstate rows (default 192 per slot).  Environments that do not fit --
        more overflowing envs than slots, a list longer than overflow_cap, or the row pool exhausted -- are counted in
        `uncovered_envs()` and keep the choice among their first max_actions actions; overflow_slots=0 switches the
        second pass off."""
        if env.rules != "full":
            raise ValueError("AfterstateActor needs rules='full'")
        if mode not in ("max", "white_value"):
            raise ValueError("mode must be 'max' or 'white_value'")
        t = env.torch
        self.env, self.mlp, self.mode = env, mlp, 0 if mode == "max" else 1
        n, cap, dev = env.num_envs, env.max_actions, env.device
        self.cap = cap
        self.as_lo = t.zeros((n * cap, 16), dtype=t.uint8, device=dev)   # afterstate planes, ragged rows packed
        self.as_hi = t.zeros((n * cap, 16), dtype=t.uint8, device=dev)
        self.scores = t.zeros(n * cap, dtype=t.float32, device=dev)
        self.offsets = t.zeros(n, dtype=t.int64, device=dev)
        self.rows_dev = t.zeros(1, dtype=t.int64, device=dev)
        self._scan_ws = t.zeros((n + 127) // 128 + 4, dtype=t.int64, device=dev)   # NARDE_AFTERSTATE_SCRATCH_WORDS(n)
        self.choice = t.zeros(n, dtype=t.int32, device=dev)
        self.value = t.zeros(n, dtype=t.float32, device=dev)
        self.dice = env.dice                                        # the turn's dice (written by the enumeration)
        self.act_override = t.zeros(n, dtype=t.int64, device=dev)   # chosen actions beyond the stored lists (side batch)
        m = max(256, n // 16) if overflow_slots is None else int(overflow_slots)
        m = -(-m // 128) * 128            # whole tiles of the side batch's kernels
        self.side = None
        if m > 0:
            self.side = sb = _SideBatch(t, dev, m, int(overflow_cap))
            rows = int(overflow_rows) if overflow_rows is not None else 192 * m
            sb.rows_cap = rows
            sb.as_lo = t.zeros((rows, 16), dtype=t.uint8, device=dev)
            sb.as_hi = t.zeros((rows, 16), dtype=t.uint8, device=dev)
            sb.scores = t.zeros(rows, dtype=t.float32, device=dev)
        self._graph = self._graph_args = None
        self._params = t.zeros(2, dtype=t.float32, device=dev)   # {epsilon, 1 / temperature}, read by the kernels
        self._sampling = False        # narde_segment_sample from the first time exploration is switched on
        self.epsilon = self.temperature = 0.0
        self.set_exploration(epsilon, temperature)
        self._s2 = t.cuda.Stream(device=dev) if self.side is not None else None
        self._enum_ws = t.zeros(_cabi.workspace_ints(n), dtype=t.int32, device=dev)

    def set_exploration(self, epsilon=None, temperature=None):
        """Set the exploration rate epsilon in [0, 1] and the softmax temperature (>= 0; 0 = arg-max) for the next
        turns; None keeps the current value.  The values live in device memory: changing them (e.g. decaying epsilon
        every episode) never recaptures step_graph()'s CUDA graph.  Only the first switch from greedy to exploring does,
        once."""
        eps = self.epsilon if epsilon is None else float(epsilon)
        tau = self.temperature if temperature is None else float(temperature)
        if not 0.0 <= eps <= 1.0:
            raise ValueError("epsilon must be in [0, 1], got %r" % (epsilon,))
        if not (math.isfinite(tau) and tau >= 0.0):
            raise ValueError("temperature must be finite and >= 0, got %r" % (temperature,))
        inv_tau = 1.0 / tau if tau > 0.0 else 0.0
        if inv_tau > _FLT_MAX:
            raise ValueError("temperature %r is too small: 1 / temperature overflows float32" % (temperature,))
        self.epsilon, self.temperature = eps, tau
        # (a stream-ordered copy: turns enqueued before it keep the old values, later ones see the new)
        self._params.copy_(self.env.torch.tensor([eps, inv_tau], dtype=self.env.torch.float32))
        if eps > 0.0 or tau > 0.0:
            self._sampling = True

    def afterstates(self, actions, counts):
        """Fill as_lo/as_hi with the afterstates of actions[i, :min(counts[i], cap)]; returns offsets [N]."""
        env = self.env
        # one launch: the device-wide exclusive scan of min(counts, cap) (decoupled look-back), the row count and the
        # rows themselves (narde_afterstates_scan) -- no host-side prefix sum, no torch ops
        _cabi.afterstates_scan(env.lo, env.hi, actions, counts, self.as_lo, self.as_hi, self._scan_ws, offsets=self.offsets,
                               rows_out=self.rows_dev)
        return self.offsets

    def _segment_choice(self, score, offsets, counts, hi, cap, choice, value, step, step_dev, env_idx=None):
        """The choice per env over its scores: narde_segment_argmax until exploration was first switched on, then
        narde_segment_sample (bit-equal to it with zero parameters)."""
        if not self._sampling:
            _cabi.segment_argmax(score, offsets, counts, hi, cap, self.mode, choice, value)
            return
        env = self.env
        _cabi.segment_sample(score, offsets, counts, hi, cap, self.mode, env.env_base, env.seed, step, self._params, choice,
                             value, env_idx=env_idx, step_dev=step_dev)

    def _side_prepare(self, step, step_dev):
        """Second pass (see __init__): gather -> enumerate with the large capacity -> afterstate rows -> score -> choice.  It only
        needs the first pass's enumeration (overflow flags), so it runs on a side stream BESIDE the first pass's rows / scorer /
        arg-max (small latency-bound kernels next to the one-CTA-per-SM scorer); fork / join with stream waits, which a
        CUDA-graph capture records as a branch."""
        sb, env, t = self.side, self.env, self.env.torch
        if sb is None:
            return
        self._s2.wait_stream(t.cuda.current_stream(env.device))
        with t.cuda.stream(self._s2):
            _score_side_batch(self.mlp, sb, env.lo, env.hi, self.dice, env.overflow, act_override=self.act_override,
                              workspace=sb.ws)
            # (the same rule over the whole list: the same coin and, per action index, the same noise as the first pass)
            self._segment_choice(sb.scores, sb.offsets, sb.counts_eff, sb.hi, sb.cap, sb.choice, sb.value, step, step_dev,
                                 env_idx=sb.idx)

    def _side_finish(self):
        """Second pass, after the join: scatter the side batch's choices into self.choice / self.value /
        self.act_override."""
        sb, env, t = self.side, self.env, self.env.torch
        if sb is None:
            return
        t.cuda.current_stream(env.device).wait_stream(self._s2)
        _cabi.scatter_choice(sb.choice, sb.value, sb.idx, sb.counts_eff, sb.counts, sb.cap, self.choice, self.value, sb.ctrl,
                             sb.actions, self.act_override)

    def uncovered_envs(self):
        """Env turns whose choice was made among the first max_actions actions only (one D2H copy)."""
        return int(self.side.ctrl[2].item()) if self.side is not None else -1

    def _choose_enumerated(self, step, step_dev=None):
        """The choice once this turn's lists are in env.actions / env.counts / env.overflow and its dice in self.dice:
        afterstate rows -> score -> arg-max (or sample), with the side batch beside them, then its scatter.  step / step_dev:
        the turn number the dice were rolled with, which keys the exploration's random words."""
        env = self.env
        self._side_prepare(step, step_dev)
        self.afterstates(env.actions, env.counts)
        self.mlp.score_states(self.as_lo, self.as_hi, out=self.scores, rows_dev=self.rows_dev)
        self._segment_choice(self.scores, self.offsets, env.counts, env.hi, self.cap, self.choice, self.value, step, step_dev)
        self._side_finish()

    def choose(self):
        """roll -> enumerate -> afterstates -> score -> greedy (or exploring) index.  Returns (choice [N] int32, dice [N,2]).
        The choice may be played by VecNardeEnv.step(choice, dice) as well as by step()."""
        self.env.roll()                   # (writes env.dice, which self.dice is)
        self.env.get_valid_actions(self.dice)
        self._choose_enumerated(self.env.step_count + 1)      # the turn number env.roll() used
        return self.choice, self.dice

    def _play_chosen(self):
        """narde_step_chosen: the lists of this turn are in env.actions / env.counts and the choice is made -- apply it and
        complete the turn (reward, termination, auto-reset, statistics, Box(198)) without enumerating the position again."""
        env = self.env
        _cabi.step_chosen(env.lo, env.hi, env.env_base, env.seed, 0, self.dice, self.choice, env.actions, env.counts,
                          act_override=self.act_override, chosen=env.chosen, obs198=env.obs, reward=env.reward, done=env.done,
                          truncated=env.trunc, stats=env.stats, flags=env._step_flags(),
                          max_episode_steps=env.max_episode_steps, step_dev=env._step_dev)

    def step(self):
        """One lock-step turn for all envs; returns VecNardeEnv.step's tuple."""
        env = self.env
        self.choose()
        env.step_count += 1
        env._step_dev.fill_(env.step_count)
        self._play_chosen()
        return env.obs, env.reward, env.terminated, env.truncated, env.info

    # -- the same turn as ONE CUDA-graph replay ---------------------------------------------------
    def _enumerate_turn(self):
        """This turn's legal lists and dice (Philox, step number read from the env's device counter)."""
        env = self.env
        _cabi.step_full(env.lo, env.hi, env.env_base, env.seed, 0, actions=env.actions, counts=env.counts,
                        dice_out=self.dice, done=env.overflow, flags=_cabi.ENUMERATE_ONLY, workspace=self._enum_ws,
                        step_dev=env._step_dev)

    def _enqueue_turn(self):
        """All launches of a greedy turn with the step number read from the env's device counter, so that the
        captured graph can be replayed: enumerate (Philox dice of the turn) -> afterstates -> score -> argmax ->
        fused step with the chosen indices (which re-derives the same dice from the same counter)."""
        _cabi.advance_counter(self.env._step_dev)
        self._enumerate_turn()
        self._choose_enumerated(0, step_dev=self.env._step_dev)
        self._play_chosen()

    def step_graph(self):
        """step() as one CUDA-graph replay (captured on first use, and again when env._frozen_args() or the greedy /
        exploring switch changed since; needs the env built with chunks=1)."""
        env, t = self.env, self.env.torch
        if len(env._chunks) != 1:
            raise ValueError("step_graph needs an unchunked env")
        env.step_count += 1
        key = (env._frozen_args(), self._sampling)
        if self._graph is None or self._graph_args != key:
            self._enqueue_turn_warmup()
            env._step_dev.fill_(env.step_count - 1)
            t.cuda.synchronize(env.device)
            g = t.cuda.CUDAGraph()
            with t.cuda.graph(g):
                self._enqueue_turn()
            self._graph, self._graph_args = g, key
        self._graph.replay()
        return env.obs, env.reward, env.terminated, env.truncated, env.info

    def _enqueue_turn_warmup(self):
        """First-use work that must not happen during capture (function attributes, lazy allocations): run the
        read-only part of a turn once, outside the graph."""
        env = self.env
        saved = env._step_dev.clone()
        self._enumerate_turn()
        self.afterstates(env.actions, env.counts)
        self.mlp.score_states(self.as_lo, self.as_hi, out=self.scores, rows_dev=self.rows_dev)
        env._step_dev.copy_(saved)
