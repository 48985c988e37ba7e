"""One-ply expectimax lookahead actor: the move choice of TD-Gammon and gnubg at 1-ply, batched on the GPU.

Per lock-step turn, entirely on the device and without a host synchronisation:
    first pass (AfterstateActor's enumerate -> afterstate rows -> tcgen05 scorer, side batch for long lists)
    -> top-K candidates per env (narde_segment_topk)
    -> P = N * K * 21 reply positions: every candidate afterstate with every roll of the opponent (narde_lookahead_expand)
    -> enumerate (narde_enumerate_fast) -> afterstate rows (narde_afterstates_scan, bounded pool) -> scorer
       -> the opponent's best reply (narde_segment_argmax mode 1), a side batch for reply lists longer than reply_cap
    -> expectimax value per candidate and the choice (narde_lookahead_reduce) -> narde_step_chosen.
The rule itself is stated in include/narde_b200.h (narde_segment_topk / narde_lookahead_reduce).
"""
from __future__ import annotations

from . import _cabi
from .actor import AfterstateActor, _SideBatch, _score_side_batch


class LookaheadActor:
    def __init__(self, env, mlp, candidates=8, reply_cap=64, reply_overflow_slots=None, reply_rows=None,
                 **first_pass_kwargs):
        """env: VecNardeEnv(rules="full"); mlp: AfterstateMLP scoring positions for WHITE (WHITE maximises, BLACK
        minimises: AfterstateActor's mode="white_value", the only mode in which expectimax is defined).

        Each turn, the `candidates` (K, 1..32) best actions by 0-ply score over the whole legal list (slot 0 = the greedy
        choice) are looked at one ply deeper: for each candidate afterstate and each of the opponent's 21 distinct rolls
        (weights 1 for doubles, 2 otherwise, out of 36), the opponent's best reply is scored, and the candidate's value v is
        the weighted mean of those replies (float32, roll order 1-1, 1-2, ..., 6-6).  A candidate that ends the game keeps
        its 0-ply score; a blocked roll counts as the candidate's 0-ply score.  The env plays the candidate with the best v
        (ties to the better 0-ply rank); `value` holds that v and `choice` the index of the action in the legal list.
        With candidates=1 the action is AfterstateActor(mode="white_value")'s, bit for bit.

        first_pass_kwargs (overflow_slots, overflow_cap, overflow_rows) configure the first pass exactly as
        AfterstateActor; lookahead is greedy, so mode must be "white_value" and epsilon / temperature 0.

        The reply stage runs the first pass's chain over P = N * K * 21 positions: lists stored up to `reply_cap` actions
        each; `reply_rows` afterstate rows (default P * min(reply_cap, 32)); lists longer than reply_cap go to a side
        batch of `reply_overflow_slots` positions (default max(256, P / 16)) with capacity 3072 (every doubles turn).  A
        candidate whose replies did not all fit is given v = NaN and never chosen over a defined one; its env is counted in
        uncovered_envs().

        Device memory of the reply stage, in bytes, with m = reply_overflow_slots and R = reply_rows:
            P * (8 * reply_cap + 64)   the stored reply lists (u64 action words) and the per-position buffers
          + R * 36                     afterstate rows (32 B) and their scores
          + m * (8 * 3072 + 192 * 36 + 80)   the reply side batch (192 rows per slot)
        e.g. N = 4096, K = 8: P = 688 128 positions, 352 MB of reply action words at reply_cap 64, 793 MB of rows at the
        default R = 32 * P, 1.36 GB of side batch at m = 43 008."""
        mode = first_pass_kwargs.pop("mode", "white_value")
        if mode != "white_value":
            raise ValueError("LookaheadActor needs mode='white_value' (a net that scores positions for WHITE); got %r" % (mode,))
        for name in ("epsilon", "temperature"):
            if float(first_pass_kwargs.pop(name, 0.0)) != 0.0:
                raise ValueError("LookaheadActor is greedy: %s must be 0" % name)
        k = int(candidates)
        if not 1 <= k <= _cabi.LOOKAHEAD_MAX_CANDIDATES:
            raise ValueError("candidates must be in [1, %d], got %r" % (_cabi.LOOKAHEAD_MAX_CANDIDATES, candidates))
        if int(reply_cap) < 1:
            raise ValueError("reply_cap must be >= 1")
        self.first = a = AfterstateActor(env, mlp, mode="white_value", **first_pass_kwargs)
        t = env.torch
        self.env, self.mlp, self.candidates = env, mlp, k
        n, dev = env.num_envs, env.device
        self.dice = a.dice
        self.choice, self.value = a.choice, a.value          # (narde_step_chosen plays them through the first pass's buffers)
        # candidates
        self.cand_idx = t.zeros((n, k), dtype=t.int32, device=dev)
        self.cand_score = t.zeros((n, k), dtype=t.float32, device=dev)
        self.cand_lo = t.zeros((n * k, 16), dtype=t.uint8, device=dev)
        self.cand_hi = t.zeros((n * k, 16), dtype=t.uint8, device=dev)
        self.cand_act = t.zeros((n, k), dtype=t.int64, device=dev)
        self.cand_count = t.zeros(n, dtype=t.int32, device=dev)
        self.cand_value = t.zeros((n, k), dtype=t.float32, device=dev)
        # reply positions
        p = self.positions = n * k * _cabi.LOOKAHEAD_ROLLS
        rcap = self.reply_cap = int(reply_cap)
        self.r_lo = t.zeros((p, 16), dtype=t.uint8, device=dev)
        self.r_hi = t.zeros((p, 16), dtype=t.uint8, device=dev)
        self.r_dice = t.ones((p, 2), dtype=t.uint8, device=dev)
        self.r_actions = t.zeros((p, rcap), dtype=t.int64, device=dev)
        self.r_counts = t.zeros(p, dtype=t.int32, device=dev)
        self.r_ovf = t.zeros(p, dtype=t.uint8, device=dev)
        rows = self.reply_rows = int(reply_rows) if reply_rows is not None else p * min(rcap, 32)
        self.r_as_lo = t.zeros((rows, 16), dtype=t.uint8, device=dev)
        self.r_as_hi = t.zeros((rows, 16), dtype=t.uint8, device=dev)
        self.r_scores = t.zeros(rows, dtype=t.float32, device=dev)
        self.r_offsets = t.zeros(p, dtype=t.int64, device=dev)
        self.r_rows_dev = t.zeros(1, dtype=t.int64, device=dev)
        self.r_scan_ws = t.zeros((p + 127) // 128 + 4, dtype=t.int64, device=dev)   # NARDE_AFTERSTATE_SCRATCH_WORDS(P)
        self.r_eff = t.zeros(p, dtype=t.int32, device=dev)
        self.r_choice = t.zeros(p, dtype=t.int32, device=dev)
        self.r_value = t.zeros(p, dtype=t.float32, device=dev)
        m = max(256, p // 16) if reply_overflow_slots is None else int(reply_overflow_slots)
        m = -(-m // 128) * 128
        self.reply_side = None
        if m > 0:
            self.reply_side = sb = _SideBatch(t, dev, m, 3072)
            sb.rows_cap = 192 * m
            sb.as_lo = t.zeros((sb.rows_cap, 16), dtype=t.uint8, device=dev)
            sb.as_hi = t.zeros((sb.rows_cap, 16), dtype=t.uint8, device=dev)
            sb.scores = t.zeros(sb.rows_cap, dtype=t.float32, device=dev)
        self._uncovered = t.zeros(1, dtype=t.int32, device=dev)
        self._graph = self._graph_args = None

    def uncovered_envs(self):
        """Env turns so far whose choice was not made over every legal action with every reply scored: the first pass's
        (AfterstateActor.uncovered_envs) plus those with a candidate of v = NaN because its replies did not fit (one D2H
        copy)."""
        return int(self._uncovered.item()) + max(0, self.first.uncovered_envs())

    # -- the launches of a turn ---------------------------------------------------------------------
    # Every launch of a turn goes to the current stream, one after the other, and the enumerations run without a workspace
    # (their order-dependent doubles turns resolved inline, no programmatic dependent kernel): no kernel of a lookahead turn
    # waits on another one that runs beside it.
    def _candidates(self):
        """First pass: the 0-ply scores of every legal action and the top-K of each env's whole list."""
        a, env = self.first, self.env
        out = (self.cand_idx, self.cand_score, self.cand_lo, self.cand_hi, self.cand_act, self.cand_count)
        a.afterstates(env.actions, env.counts)
        self.mlp.score_states(a.as_lo, a.as_hi, out=a.scores, rows_dev=a.rows_dev)
        _cabi.segment_topk(a.scores, a.offsets, env.counts, env.hi, 1, a.as_lo, a.as_hi, env.actions, *out)
        sb = a.side
        if sb is not None:
            # (act_override is cleared for every env here; narde_lookahead_reduce writes this turn's)
            _score_side_batch(self.mlp, sb, env.lo, env.hi, self.dice, env.overflow, act_override=a.act_override)
            _cabi.segment_topk(sb.scores, sb.offsets, sb.counts, sb.hi, 1, sb.as_lo, sb.as_hi, sb.actions, *out,
                               env_idx=sb.idx, counts_eff=sb.counts_eff, ctrl=sb.ctrl)

    def _replies(self):
        """The opponent's best reply for every (candidate, roll): r_value, with r_counts the legal counts and r_eff the
        length of the list prefix each reply was chosen from."""
        _cabi.lookahead_expand(self.cand_lo, self.cand_hi, self.cand_count, self.r_lo, self.r_hi, self.r_dice)
        _cabi.enumerate_actions_fast(self.r_lo, self.r_hi, self.r_dice, self.r_actions, self.r_counts, self.r_ovf)
        _cabi.afterstates_scan(self.r_lo, self.r_hi, self.r_actions, self.r_counts, self.r_as_lo, self.r_as_hi, self.r_scan_ws,
                               offsets=self.r_offsets, rows_out=self.r_rows_dev, rows_cap=self.reply_rows,
                               counts_eff=self.r_eff)
        self.mlp.score_states(self.r_as_lo, self.r_as_hi, out=self.r_scores, rows_dev=self.r_rows_dev)
        # (counts_eff, not the counts: a position whose rows did not fit has none to read)
        _cabi.segment_argmax(self.r_scores, self.r_offsets, self.r_eff, self.r_hi, self.reply_cap, 1, self.r_choice,
                             self.r_value)
        sb = self.reply_side
        if sb is not None:
            _score_side_batch(self.mlp, sb, self.r_lo, self.r_hi, self.r_dice, self.r_ovf)
            _cabi.segment_argmax(sb.scores, sb.offsets, sb.counts_eff, sb.hi, sb.cap, 1, sb.choice, sb.value)
            # the side batch's replies over the whole list replace the prefix's: value, and as "choice" the length of the list
            # they were chosen from (r_eff stays shorter than the count where the side batch did not cover the position)
            _cabi.scatter_choice(sb.counts_eff, sb.value, sb.idx, sb.counts_eff, sb.counts, sb.cap, self.r_eff, self.r_value,
                                 sb.ctrl)

    def _choose_enumerated(self):
        """The choice once this turn's lists are in env.actions / env.counts / env.overflow and its dice in self.dice."""
        env, a = self.env, self.first
        self._candidates()
        self._replies()
        _cabi.lookahead_reduce(env.hi, self.cand_idx, self.cand_score, self.cand_hi, self.cand_act, self.cand_count, a.cap,
                               self.r_value, self.r_counts, self.r_eff, self.choice, self.value, act_override=a.act_override,
                               cand_value=self.cand_value, uncovered=self._uncovered)

    def choose(self):
        """roll -> enumerate -> candidates -> replies -> expectimax choice.  Returns (choice [N] int32, dice [N,2]).  An index
        beyond env.max_actions is played through act_override by step(); VecNardeEnv.step(choice, dice) cannot play it."""
        self.env.roll()
        self.env.get_valid_actions(self.dice)
        self._choose_enumerated()
        return self.choice, self.dice

    def step(self):
        """One lock-step turn for all envs; returns VecNardeEnv.step's tuple."""
        env = self.env
        self.choose()
        env.step_count += 1
        env._step_dev.fill_(env.step_count)
        self.first._play_chosen()
        return env.obs, env.reward, env.terminated, env.truncated, env.info

    def _enqueue_turn(self):
        _cabi.advance_counter(self.env._step_dev)
        self.first._enumerate_turn()
        self._choose_enumerated()
        self.first._play_chosen()

    def step_graph(self):
        """step() as one CUDA-graph replay without a host synchronisation (captured on first use, and again when
        env._frozen_args() changed since; needs the env built with chunks=1)."""
        env, t = self.env, self.env.torch
        if len(env._chunks) != 1:
            raise ValueError("step_graph needs an unchunked env")
        env.step_count += 1
        key = env._frozen_args()
        if self._graph is None or self._graph_args != key:
            self.first._enqueue_turn_warmup()
            env._step_dev.fill_(env.step_count - 1)
            t.cuda.synchronize(env.device)
            g = t.cuda.CUDAGraph()
            with t.cuda.graph(g):
                self._enqueue_turn()
            self._graph, self._graph_args = g, key
        self._graph.replay()
        return env.obs, env.reward, env.terminated, env.truncated, env.info
