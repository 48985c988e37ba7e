"""VecNardeEnv -- N lock-step Narde games on one B200, same calls as the reference NardeEnv.

Mirrors gym_narde/envs/narde_env.py (reset/step/observation/reward) over a batch:
  rules="full"      README contract (Tier N): full legal-turn enumeration (max-dice, higher-die,
                    per-turn head rule, doubles up to 4 half-moves), Box(198) observation,
                    reward +1 iff WHITE wins (or the reference's mover 1/2 with reward="mover12").
  rules="reference" the reference code's exact behaviour (Tier R): NardeEnv.step quirks included,
                    int32[24] mover-perspective observation, reward 1/2 to the mover.
All state lives in HBM as two [N,16] uint8 planes; every method enqueues hand-written sm_100a
kernels through the C ABI (gym_narde_b200/_cabi.py).  There is no CPU path.
"""
from __future__ import annotations

from . import _cabi


class VecNardeEnv:
    def __init__(self, num_envs, seed=0, rules="full", reward=None, max_actions=64, device="cuda",
                 env_base=0, autoreset=None, max_episode_steps=1000, write_actions=True, chunks=None,
                 graph=True):
        torch = _cabi.require_cuda()
        _cabi.load()
        if rules not in ("full", "reference"):
            raise ValueError("rules must be 'full' or 'reference'")
        self.torch = torch
        self.num_envs = int(num_envs)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.rules = rules
        self.reward_mode = reward or ("white01" if rules == "full" else "mover12")
        if self.reward_mode not in ("white01", "mover12"):
            raise ValueError("reward must be 'white01' or 'mover12'")
        self.max_actions = int(max_actions)
        self.device = torch.device(device)
        self.env_base = int(env_base)
        # autoreset: rules="full" resets finished games inside the fused step (default on).  The reference-exact step
        # has no reset inside (NardeEnv.step, narde_env.py:27-103: the caller resets), so asking for it is an error
        # rather than a silently ignored flag; use reset_done() between steps.
        if rules == "reference" and autoreset:
            raise ValueError("autoreset=True is not available with rules='reference' (call reset_done() instead)")
        self.autoreset = bool(rules == "full") if autoreset is None else bool(autoreset)
        self.max_episode_steps = int(max_episode_steps)
        self.write_actions = bool(write_actions)
        self.step_count = 0  # Philox step counter (global, shared by all envs)
        self.use_graph = bool(graph)
        self._graphs = {}    # action-input key -> (captured CUDA graph of one step, the input buffer, _frozen_args())
        n, dev = self.num_envs, self.device
        self.lo = torch.zeros((n, 16), dtype=torch.uint8, device=dev)
        self.hi = torch.zeros((n, 16), dtype=torch.uint8, device=dev)
        self.dice = torch.zeros((n, 2), dtype=torch.uint8, device=dev)
        self.counts = torch.zeros(n, dtype=torch.int32, device=dev)
        self.chosen = torch.zeros(n, dtype=torch.int64, device=dev)
        self.actions = torch.zeros((n, self.max_actions), dtype=torch.int64, device=dev)
        self.overflow = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)        # terminated (0/1)
        self.trunc = torch.zeros(n, dtype=torch.uint8, device=dev)       # truncated (0/1)
        # zero-copy bool views: step() launches exactly one kernel and no torch ops
        self.terminated = self.done.view(torch.bool)
        self.truncated = self.trunc.view(torch.bool)
        self.stats = torch.zeros(_cabi.NUM_STATS, dtype=torch.int64, device=dev)
        # The fused step is launched as `chunks` independent sub-batches (multiples of the 128-env CTA
        # tile) on separate CUDA streams: the small CTA-per-env kernel for order-dependent doubles turns
        # of one chunk overlaps the main kernel of the next, and the tail of one wave is filled by
        # another chunk's CTAs.  Results do not depend on the chunking (global env ids).
        if chunks is None:
            chunks = 1
        per = -(-n // (128 * chunks)) * 128
        self._chunks = [(b, min(b + per, n)) for b in range(0, n, per)]
        self._streams = [torch.cuda.Stream(device=dev) for _ in self._chunks[1:]]
        # deferred-turn lists (see narde_b200.h: NARDE_WORKSPACE_INTS(n) int32 per call)
        self._workspaces = [torch.zeros(_cabi.workspace_ints(e - b), dtype=torch.int32, device=dev) for b, e in self._chunks]
        self._enum_ws = torch.zeros(_cabi.workspace_ints(n), dtype=torch.int32, device=dev)   # get_valid_actions' deferred-turn list
        # graph-replayed steps of an unchunked env let the kernels advance the step counter and clear the list
        # themselves (DEVICE_ADVANCE: two graph nodes fewer per step); that workspace is never shared with other calls
        self._ws_adv = torch.zeros(_cabi.workspace_ints(n), dtype=torch.int32, device=dev) if len(self._chunks) == 1 else None
        # device-resident copy of step_count: kernel arguments stay frozen, so a step is one graph replay
        self._step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.action_in = torch.zeros(n, dtype=torch.int32, device=dev)   # persistent policy input (graph-replayable)
        self.info = {"dice": self.dice, "counts": self.counts, "chosen": self.chosen}
        if rules == "full":
            self.obs = torch.zeros((n, 198), dtype=torch.float32, device=dev)
            self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
        else:
            self.obs = torch.zeros((n, 24), dtype=torch.int32, device=dev)
            self.reward = torch.zeros(n, dtype=torch.int32, device=dev)

    # -- gym-style API -----------------------------------------------------------------------
    def reset(self, *, seed=None, options=None):
        """NardeEnv.reset (narde_env.py:105-120) for every env; returns (obs, {})."""
        if seed is not None:
            self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.step_count = 0
        self._step_dev.zero_()
        _cabi.reset(self.lo, self.hi, self.env_base, self.seed, 0)
        self.stats.zero_()
        return self.observe(), {}

    def reset_done(self):
        """Reset the envs whose last step ended the game (terminated or truncated), like a caller of the reference env
        does after `done`; returns the refreshed observation.  (rules="full" with autoreset does this inside the step.)"""
        t = self.torch
        mask = t.bitwise_or(self.done, self.trunc)
        _cabi.reset(self.lo, self.hi, self.env_base, self.seed, self.step_count, mask=mask)
        return self.observe()

    def observe(self):
        if self.rules == "full":
            _cabi.obs198(self.lo, self.hi, self.obs)
        else:
            _cabi.obs24(self.lo, self.hi, self.obs)
        return self.obs

    def roll(self):
        """The dice the NEXT step will use (Philox stream); [N,2] uint8."""
        _cabi.roll_dice(self.dice, self.env_base, self.seed, self.step_count + 1)
        return self.dice

    def get_valid_moves(self, dice4):
        """Narde.get_valid_moves for every env (narde.py:58-92).  dice4: [N,4] uint8, 0-padded.
        Returns (moves [N,96,2] uint8 with 255 = 'off', counts [N] int32)."""
        t = self.torch
        moves = t.zeros((self.num_envs, _cabi.MAX_HALF_MOVES, 2), dtype=t.uint8, device=self.device)
        counts = t.zeros(self.num_envs, dtype=t.int32, device=self.device)
        _cabi.half_moves(self.lo, self.hi, dice4, moves, counts)
        return moves, counts

    def get_valid_actions(self, dice=None):
        """README get_valid_actions(roll): all legal full-turn actions per env.
        Returns (actions [N,max_actions] int64 bit patterns, counts [N], overflow [N])."""
        if dice is None:
            dice = self.roll()
        _cabi.enumerate_actions_fast(self.lo, self.hi, dice, self.actions, self.counts, self.overflow, self._enum_ws)
        return self.actions, self.counts, self.overflow

    def step(self, actions=None, dice=None, fraction=False):
        """One lock-step turn for all envs.

        rules="full":      actions = int32 [N] indices into get_valid_actions (None = uniform random
                           from the Philox stream); dice = optional [N,2] uint8 override.  With
                           fraction=True the int32 values are read as u32 fractions f and env i plays
                           action floor(f * count_i / 2^32) (a policy that cannot know the counts of a
                           roll made inside the step, e.g. a host-side sampler).
        rules="reference": actions = int32 [N,2] codes (from*24+to) exactly as NardeEnv.step takes
                           them; dice default to the Philox stream.
        Returns (obs, reward, terminated, truncated, info)."""
        t = self.torch
        self.step_count += 1
        if self.rules == "full":
            flags = self._step_flags(fraction=fraction and actions is not None)
            # A captured graph freezes the kernel arguments, so graphs are cached per action-input buffer
            # (identified by its device pointer; the tensor is kept alive by the cache) and replayed when the
            # same persistent buffer is passed again.  Up to 8 buffers are cached; anything else (fresh
            # tensors, explicit dice) is launched directly.
            key = None
            if self.use_graph and dice is None:
                if actions is None:
                    key = "random"
                elif actions.is_contiguous() and actions.dtype == t.int32 and actions.numel() == self.num_envs:
                    key = (actions.data_ptr(), bool(fraction))
                    if key not in self._graphs and len(self._graphs) >= 8:
                        key = None
            if key is not None:
                ent = self._graphs.get(key)
                if ent is None or ent[2] != self._frozen_args():
                    ent = self._graphs[key] = (self._capture(actions, dice, flags), actions, self._frozen_args())
                ent[0].replay()
            else:
                self._step_dev.fill_(self.step_count)
                self._launch_full(actions, dice, flags)
        else:
            if actions is None:
                raise ValueError("rules='reference' needs action codes [N,2]")
            if dice is None:
                _cabi.roll_dice(self.dice, self.env_base, self.seed, self.step_count)
                dice = self.dice
            _cabi.step_ref(self.lo, self.hi, dice, actions, self.obs, self.reward, self.done,
                           max_episode_steps=self.max_episode_steps, truncated=self.trunc)
        return self.obs, self.reward, self.terminated, self.truncated, self.info

    def _step_flags(self, fraction=False, packed=False):
        """The flags word of this env's full-rules step launches."""
        return ((_cabi.REWARD_MOVER12 if self.reward_mode == "mover12" else 0) | (_cabi.AUTORESET if self.autoreset else 0)
                | (_cabi.ACTION_FRACTION if fraction else 0) | (_cabi.PACK_RESULT if packed else 0))

    def _frozen_args(self):
        """The kernel arguments a captured CUDA graph freezes that reset(seed=...) and load_state_dict() can change.  Every
        holder of a captured graph (this env's step caches, HostPipeline, AfterstateActor) records this value at capture
        and captures again when it differs before a replay."""
        return self.seed, self.env_base

    def _launch_full(self, actions, dice, flags, dev_advance=False):
        """Enqueue one fused step: every chunk on its own stream (fork/join around the current stream).
        dev_advance (unchunked envs, graph capture): the step index is the device counter + 1 and the kernels store
        it back themselves."""
        t = self.torch
        main = t.cuda.current_stream(self.device)
        if dev_advance:
            flags |= _cabi.DEVICE_ADVANCE
        for k, (b, e) in enumerate(self._chunks):
            stream = main if k == 0 else self._streams[k - 1]
            if k:
                stream.wait_stream(main)
            with t.cuda.stream(stream):
                _cabi.step_full(self.lo[b:e], self.hi[b:e], self.env_base + b, self.seed, 0,
                                dice_in=None if dice is None else dice[b:e],
                                action_idx=None if actions is None else actions[b:e],
                                actions=self.actions[b:e] if self.write_actions else None,
                                counts=self.counts[b:e], dice_out=self.dice[b:e], chosen=self.chosen[b:e],
                                obs198=self.obs[b:e], reward=self.reward[b:e], done=self.done[b:e],
                                stats=self.stats, flags=flags, max_episode_steps=self.max_episode_steps,
                                truncated=self.trunc[b:e], workspace=self._ws_adv if dev_advance else self._workspaces[k],
                                step_dev=self._step_dev)
        for s_ in self._streams:
            main.wait_stream(s_)

    def _capture(self, actions, dice, flags):
        """Capture one step (counter advance + all chunk launches) into a CUDA graph.  The first replay
        performs the step, so nothing is executed here."""
        t = self.torch
        self._step_dev.fill_(self.step_count - 1)
        t.cuda.synchronize(self.device)
        g = t.cuda.CUDAGraph()
        with t.cuda.graph(g):
            if self._ws_adv is not None:
                self._launch_full(actions, dice, flags, dev_advance=True)
            else:
                _cabi.advance_counter(self._step_dev)
                self._launch_full(actions, dice, flags)
        return g

    # -- host-facing step: host buffers in, host buffers out, one graph replay ---------------------------
    def host_io(self):
        """Pinned host buffers of step_host(): write `actions` (int32 [N]; indices, or u32 fractions with
        fraction=True), read `reward` (float32 [N]), `done` and `truncated` (uint8 [N])."""
        t = self.torch
        if getattr(self, "_hio", None) is None:
            n = self.num_envs
            self._hio = {"actions": t.zeros(n, dtype=t.int32).pin_memory(),
                         "reward": t.zeros(n, dtype=t.float32).pin_memory(),
                         "done": t.zeros(n, dtype=t.uint8).pin_memory(),
                         "truncated": t.zeros(n, dtype=t.uint8).pin_memory(),
                         "result": t.zeros(n, dtype=t.uint8).pin_memory(),
                         # obs="packed": the state planes after the turn, the 32-byte encoding of Box(198)
                         "lo": t.zeros((n, 16), dtype=t.uint8).pin_memory(),
                         "hi": t.zeros((n, 16), dtype=t.uint8).pin_memory(),
                         # obs="compact": one 20-byte record per env (state + result bits, include/narde_b200.h)
                         "rec": t.zeros((n, 20), dtype=t.uint8).pin_memory()}
            self._hio_graphs = {}
        return self._hio

    def step_host(self, fraction=False, packed=False, actions=None, dma_in=False, obs=None):
        """One lock-step turn driven from the host (rules="full") with ZERO-COPY I/O: every CTA of the fused step
        fetches its envs' action words from the pinned host buffer with one bulk asynchronous copy (512 B over
        PCIe into shared memory, overlapped with the state load and the dice), and reward / done / truncated are
        written STRAIGHT into the pinned host buffers (page-locked memory is mapped into the device address space;
        posted PCIe writes from inside the kernel).  No copy operations, no stream round trips: 0.120 ms/step at
        131 072 envs against 0.110 for the device-resident step and 0.141 with a DMA in front (dma_in=True).
        One CUDA-graph replay per turn.  Asynchronous:
        synchronise the stream (or an event) before reading the host buffers; write the next actions only after
        that.  Box(198) stays in `self.obs` on the device; self.reward / self.done are NOT updated by this call.
        packed=True: one byte per env in host_io()["result"] instead (bit 0 terminated, bit 1 truncated, bits 2-3
        the reward 0/1/2) -- a sixth of the PCIe write traffic.
        actions: another pinned int32 [N] host tensor to read this turn's choices from (e.g. a row of a ring the
        policy fills ahead); one graph is cached per buffer (up to 32).
        obs="packed": the OBSERVATION crosses to the host as well, in its packed form -- the kernel also writes every
        env's 32-byte state record (after the turn, after an auto-reset) into host_io()["lo"] / ["hi"]; Box(198) is a
        function of exactly those bytes (gym_narde_b200.expand_obs198(lo, hi) gives the float32 [N,198] rows, bit-equal
        to the device's), so 32 B per env cross PCIe instead of 792.
        obs="compact": observation AND result in ONE 20-byte record per env in host_io()["rec"] (24 points of 5 bits, off
        counts, side to move, flags, terminated / truncated / reward bits, episode steps;
        gym_narde_b200.state.unpack_compact(rec) -> the same lo / hi planes and the result byte); reward / done /
        truncated / result are not written separately.  2.6 MB instead of 4.3 MB per 131 072 envs: the posted PCIe
        writes end before the kernel does."""
        t = self.torch
        if self.rules != "full":
            raise ValueError("step_host needs rules='full'")
        io = self.host_io()
        self.step_count += 1
        flags = self._step_flags(fraction, packed)
        src = io["actions"] if actions is None else actions
        if not (src.is_pinned() and src.dtype == t.int32 and src.is_contiguous() and src.numel() == self.num_envs):
            raise _cabi.NardeCudaError("step_host actions must be a pinned contiguous int32 [N] host tensor")
        if obs not in (None, "packed", "compact"):
            raise ValueError("obs must be None (Box(198) stays on the device), 'packed' or 'compact'")
        compact = obs == "compact"
        if len(self._chunks) != 1:
            raise _cabi.NardeCudaError("step_host needs an unchunked env (chunks=1)")
        key = (src.data_ptr(), bool(fraction), bool(packed), bool(dma_in), obs)
        ent = self._hio_graphs.get(key)
        if ent is None and len(self._hio_graphs) >= 32:
            raise _cabi.NardeCudaError("step_host: more than 32 distinct host action buffers")
        if ent is None or ent[2] != self._frozen_args():
            self._step_dev.fill_(self.step_count - 1)
            t.cuda.synchronize(self.device)
            g = t.cuda.CUDAGraph()
            with t.cuda.graph(g):
                if dma_in:
                    self.action_in.copy_(src, non_blocking=True)
                adv = self._ws_adv is not None
                if adv:
                    flags |= _cabi.DEVICE_ADVANCE
                else:
                    _cabi.advance_counter(self._step_dev)
                # dma_in=False: the kernel fetches its CTA's action words from the host buffer itself (one bulk
                # asynchronous copy of 512 B per CTA into shared memory)
                _cabi.step_full(self.lo, self.hi, self.env_base, self.seed, 0, action_idx=self.action_in if dma_in else src,
                                actions=self.actions if self.write_actions else None, counts=self.counts,
                                dice_out=self.dice, chosen=self.chosen, obs198=self.obs,
                                reward=None if (packed or compact) else io["reward"],
                                done=None if compact else (io["result"] if packed else io["done"]),
                                stats=self.stats, flags=flags, max_episode_steps=self.max_episode_steps,
                                truncated=None if (packed or compact) else io["truncated"],
                                workspace=self._ws_adv if adv else self._workspaces[0], step_dev=self._step_dev,
                                mirror_lo=io["lo"] if obs == "packed" else (io["rec"] if compact else None),
                                mirror_hi=io["hi"] if obs == "packed" else None)
            ent = self._hio_graphs[key] = (g, src, self._frozen_args())
        ent[0].replay()
        return io

    def host_pipeline(self, depth=8, fraction=False):
        """A window of `depth` lock-step turns driven from pinned host buffers as ONE CUDA graph with the copies
        on their own streams: the H2D copy of turn t+1's actions and the D2H copy of turn t-1's results overlap
        the kernels of turn t (see HostPipeline)."""
        return HostPipeline(self, depth, fraction)

    def episode_stats(self):
        """Device-side counters as a dict (one D2H copy)."""
        v = self.stats.cpu().tolist()
        return dict(zip(_cabi.STAT_NAMES, v))

    # -- checkpoint: the SoA planes + the Philox (seed, step) are the complete state -----------
    def state_dict(self):
        return {"lo": self.lo.clone(), "hi": self.hi.clone(), "seed": self.seed, "step_count": self.step_count,
                "env_base": self.env_base, "rules": self.rules}

    def load_state_dict(self, sd):
        self.lo.copy_(sd["lo"])
        self.hi.copy_(sd["hi"])
        self.seed, self.step_count, self.env_base = sd["seed"], sd["step_count"], sd["env_base"]
        self._step_dev.fill_(self.step_count)

    def close(self):
        pass


class HostPipeline:
    """`depth` consecutive turns of a VecNardeEnv(rules="full") with host-side inputs and outputs.

    actions [depth, N] int32 (pinned): the policy's choices for the next `depth` turns (indices, or u32 fractions
    of the legal list with fraction=True); reward [depth, N] float32, done and truncated [depth, N] uint8 (pinned)
    receive every turn's results.  run() replays one captured graph: per turn a DMA of that turn's actions on a
    copy-in stream (double-buffered on the device, so it overlaps the previous turn's kernels) and the fused step,
    which writes its results straight into the pinned host rows (zero-copy, no device-to-host copies).
    Asynchronous: synchronise before reading the host buffers.  Box(198) of the last turn stays in env.obs."""

    def __init__(self, env, depth=8, fraction=False):
        t = env.torch
        if env.rules != "full" or len(env._chunks) != 1:
            raise ValueError("HostPipeline needs an unchunked rules='full' env")
        self.env, self.depth, self.fraction = env, int(depth), bool(fraction)
        n, dev = env.num_envs, env.device
        self.actions = t.zeros((depth, n), dtype=t.int32).pin_memory()
        self.reward = t.zeros((depth, n), dtype=t.float32).pin_memory()
        self.done = t.zeros((depth, n), dtype=t.uint8).pin_memory()
        self.truncated = t.zeros((depth, n), dtype=t.uint8).pin_memory()
        self._d_act = [t.zeros(n, dtype=t.int32, device=dev) for _ in range(2)]
        self._s_in = t.cuda.Stream(device=dev)
        self._graph = self._graph_args = None

    def _capture(self):
        env, t, D = self.env, self.env.torch, self.depth
        flags = env._step_flags(self.fraction)
        env._step_dev.fill_(env.step_count)
        t.cuda.synchronize(env.device)
        g = t.cuda.CUDAGraph()
        with t.cuda.graph(g):
            main = t.cuda.current_stream(env.device)
            ev_in = [t.cuda.Event() for _ in range(D)]
            ev_c = [t.cuda.Event() for _ in range(D)]
            self._s_in.wait_stream(main)
            for k in range(D):
                b = k & 1
                with t.cuda.stream(self._s_in):
                    if k >= 2:
                        self._s_in.wait_event(ev_c[k - 2])          # turn k-2 has consumed this device buffer
                    self._d_act[b].copy_(self.actions[k], non_blocking=True)
                    ev_in[k].record(self._s_in)
                main.wait_event(ev_in[k])
                adv = env._ws_adv is not None
                if not adv:
                    _cabi.advance_counter(env._step_dev)
                _cabi.step_full(env.lo, env.hi, env.env_base, env.seed, 0, action_idx=self._d_act[b],
                                actions=env.actions if env.write_actions else None, counts=env.counts,
                                dice_out=env.dice, chosen=env.chosen, obs198=env.obs, reward=self.reward[k],
                                done=self.done[k], stats=env.stats, flags=flags | (_cabi.DEVICE_ADVANCE if adv else 0),
                                max_episode_steps=env.max_episode_steps, truncated=self.truncated[k],
                                workspace=env._ws_adv if adv else env._workspaces[0], step_dev=env._step_dev)
                ev_c[k].record(main)
            main.wait_stream(self._s_in)
        return g

    def run(self):
        """Play the next `depth` turns (one graph replay)."""
        if self._graph is None or self._graph_args != self.env._frozen_args():
            self._graph, self._graph_args = self._capture(), self.env._frozen_args()
        self._graph.replay()
        self.env.step_count += self.depth
