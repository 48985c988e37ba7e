#!/usr/bin/env python
"""bench.py -- legal-move-enumerated Narde env steps/s on N B200s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port on host cores)
    python bench.py ... --dump-outputs DIR                    # + the last timed turn's outputs as DIR/<name>.npy

Workload (config.workload): BASELINE config 4's per-GPU shard -- 131072 lock-step environments per
GPU (1M environments at 8 GPUs), full-rules random self-play: per env turn = Philox dice ->
full legal-turn enumeration (written to HBM) -> uniform action -> apply -> termination/reward ->
auto-reset -> Box(198) observation.  One "step" = --turns-per-step (default 128) lock-step turns of all envs of the
GPU, each turn ONE graph replay (main kernel + its programmatic dependent) timed on its own with CUDA events and
the L2 flushed (untimed) in front of it -- so that the timed region lasts hundreds of milliseconds (clock samples)
while every launch is still timed cold.  Prints ONE JSON line on rank 0.

After the timing the SAME env object plays 64 more turns that are recorded and compared, env turn by env turn, with
the C oracle (oracle/narde_oracle.c o_selfplay_trace) replaying them from the same positions on all host cores: that
run is both the `cpu_baseline` (same positions, dice, policy: same_config true) and the parity check
(`parity_checked_env_turns`).  The unmodified Python reference (baseline/_ref, vendored by baseline/fetch_ref.py) is
timed on the same cores beside it.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "legal-move-enumerated env steps/sec"
UNIT = "env_steps/s"
SEED = 0x5EED


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


_POLLER = r"""
import sys, time
import pynvml as n
n.nvmlInit()
pci = sys.argv[1]
h = n.nvmlDeviceGetHandleByPciBusId(pci.encode()) if pci != "-" else n.nvmlDeviceGetHandleByIndex(int(sys.argv[2]))
print("max", n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM), flush=True)
while True:
    try:
        print(time.time(), n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), int(n.nvmlDeviceGetCurrentClocksEventReasons(h)),
              n.nvmlDeviceGetPowerUsage(h) / 1000.0, flush=True)
    except Exception as e:
        print("err", e, flush=True)
    time.sleep(0.001)
"""


class ClockSampler:
    """SM clock + clock-event (throttle) reasons sampled DURING the timed region.

    A helper PROCESS polls NVML every ~1 ms for the whole run (a thread would be starved by the launch
    loop holding the GIL; `nvidia-smi -lms` is too coarse for a timed region of tens of milliseconds);
    mark()/stop() keep the samples whose timestamps fall inside the timed region."""
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
            ("sw_power_cap", 0x4), ("hw_power_brake_slowdown", 0x80))

    def __init__(self, gpu_index, pci_bus_id=None):
        self.rows = []
        self.sm_max = None
        self.t0 = self.t1 = None
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _POLLER, pci_bus_id or "-", str(gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = line.split()
            try:
                if f[0] == "max":
                    self.sm_max = float(f[1])
                elif f[0] != "err":
                    self.rows.append((float(f[0]), float(f[1]), int(f[2]), float(f[3])))
            except (ValueError, IndexError):
                pass

    def wait_ready(self, timeout=20.0):
        t = time.time()
        while self.proc is not None and not self.rows and time.time() - t < timeout and self.proc.poll() is None:
            time.sleep(0.01)

    def start(self):
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        time.sleep(0.01)
        self.proc.terminate()
        rows = [r for r in self.rows if self.t0 <= r[0] <= self.t1]
        bits = 0
        for r in rows:
            bits |= r[2]
        return {"sm_mhz": statistics.median(r[1] for r in rows) if rows else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(k for k, b in self.BITS if bits & b), "samples": len(rows),
                "power_w_max": max(r[3] for r in rows) if rows else None,
                "source": "NVML polled every ~1 ms by a helper process; samples inside the timed region only"}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port (C restatement of the reference's algorithm) and the Python reference on the host cores
# ------------------------------------------------------------------------------------------
def steady_state_positions(n_envs, burn_in, seed=SEED, env_base=0):
    """The CUDA arm's workload for the CPU arm when no GPU produced the positions: `burn_in` turns of the same
    self-play from fresh games, played by the oracle itself (untimed).  Returns (lo, hi) uint8 [n,16]."""
    from oracle import oracle as O
    tr = O.selfplay_trace(seed, env_base, n_envs, burn_in, step0=0, cap=64)
    return tr["lo"][-1].copy(), tr["hi"][-1].copy()


def cpu_trace(init, n_envs, n_steps, step0, seed=SEED, env_base=0, cap=64, want_states=False):
    """Timed oracle run: n_envs envs x n_steps turns from `init` on all host cores (threads; ctypes releases the
    GIL), doing everything a CUDA step does per env turn (dice, enumeration, list, choice, apply, reward, reset,
    Box(198) row).  Returns (trace dict, seconds)."""
    from oracle import oracle as O
    t0 = time.perf_counter()
    tr = O.selfplay_trace(seed, env_base, n_envs, n_steps, step0=step0, init=init, cap=cap, want_states=want_states,
                          with_obs=True)
    return tr, time.perf_counter() - t0


def _pyref_setup():
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref, "gym_narde", "envs", "narde_env.py")):
        return None
    for p in (os.path.join(ROOT, "tests"), ref):
        if p not in sys.path:
            sys.path.insert(0, p)
    import gymnasium_stub
    gymnasium_stub.install()
    from gym_narde.envs.narde_env import NardeEnv
    return NardeEnv


def _pyref_worker(args):
    """One process of the Python-reference timing (SURVEY 8d CPU rows i / ii): independent reference NardeEnv episodes
    for `seconds` of wall time.  mode "step": NardeEnv.step with valid-random codes drawn from get_valid_moves on the
    env's own dice (the global numpy RNG is rewound so that step() re-rolls the same two dice); mode "enum": the same
    plus the (move1, move2) pair enumeration the reference's agent does before every step (one get_valid_moves call
    per first move on the remaining die, train_deepq_pytorch.py:430-507)."""
    mode, seconds, seed = args
    import numpy as np
    NardeEnv = _pyref_setup()
    np.random.seed(seed)
    env = NardeEnv()
    env.reset()
    code = lambda m: m[0] * 24 + (0 if m[1] == "off" else m[1])
    n = eps = ep_steps = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        st = np.random.get_state()
        dice = [int(np.random.randint(1, 7)), int(np.random.randint(1, 7))]
        np.random.set_state(st)                      # env.step() rolls these same dice again (narde_env.py:29)
        moves = env.game.get_valid_moves(dice, env.current_player)
        if mode == "enum" and moves:
            pairs = []
            for m1 in moves:
                rest = list(dice)
                if m1[1] == "off":                    # the first die large enough pays for a bear-off, else the largest
                    need = m1[0] + 1
                    rest.remove(next((d for d in rest if d >= need), max(rest)))
                else:
                    dist = m1[0] - m1[1]
                    rest.remove(dist if dist in rest else rest[0])
                seconds_moves = env.game.get_valid_moves(rest, env.current_player)
                pairs += [(code(m1), code(m2)) for m2 in seconds_moves] or [(code(m1), 0)]
            action = pairs[(n * 2654435761) % len(pairs)]
        elif moves:
            action = (code(moves[(n * 2654435761) % len(moves)]), code(moves[(n * 40503) % len(moves)]))
        else:
            action = (0, 0)
        _, _, done, _, _ = env.step(action)
        n += 1
        ep_steps += 1
        if done or ep_steps >= 1000:                  # gym_narde/__init__.py:6 max_episode_steps
            env.reset()
            eps += 1
            ep_steps = 0
    return n, eps, time.perf_counter() - t0


def python_reference_rates(cores, seconds=5.0):
    """The unmodified Python reference on `cores` processes (spawn); None when baseline/_ref is absent."""
    if _pyref_setup() is None:
        return None
    import multiprocessing as mp
    out = {"cores": cores, "seconds_per_row": seconds, "source": "baseline/_ref (unmodified files of the original gym-narde, gymnasium stubbed)"}
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        for mode, key in (("step", "NardeEnv_step_valid_random"), ("enum", "pair_enumeration_plus_step")):
            res = pool.map(_pyref_worker, [(mode, seconds, 1000 + c) for c in range(cores)])
            rate = sum(r[0] / r[2] for r in res)
            out[key] = {"env_steps_per_s": rate, "per_core": rate / cores, "episodes": sum(r[1] for r in res)}
    return out


def run_reference_arm(args):
    """--impl reference: the reference algorithm's CPU implementation on all host cores -- the oracle port
    (oracle/narde_oracle.c o_selfplay_trace), on the CUDA arm's workload: the same seed and env ids, steady-state
    positions after the same burn-in (played untimed by the oracle itself on a bounded sample of the envs), the same
    dice / policy stream, one Box(198) row per env turn.  One "step" = SAMPLE_ENVS envs x SAMPLE_TURNS turns."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    n_envs, turns = 4096, 64
    init = steady_state_positions(n_envs, args.burn_in)
    step0 = args.burn_in
    for _ in range(max(args.warmup, 1)):
        cpu_trace(init, n_envs, 8, step0)
    tot = acts = 0
    t_all = 0.0
    for k in range(args.steps):
        tr, dt = cpu_trace(init, n_envs, turns, step0, want_states=True)
        init, step0 = (tr["lo"][-1].copy(), tr["hi"][-1].copy()), step0 + turns
        tot += tr["turns"]
        acts += int(tr["stats"][5])
        t_all += dt
    value = tot / t_all
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": "config4 shard positions: full-rules random self-play after %d burn-in turns (same seed, env ids, dice "
                               "and policy stream as the CUDA arm), bounded sample of %d envs x %d turns per step" % (args.burn_in, n_envs, turns),
                   "sample_envs": n_envs, "turns_per_step": turns, "mean_legal_actions": acts / max(tot, 1), "action_capacity": 64},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d envs x %d turns per step x %d steps on %d host threads (oracle/narde_oracle.c o_selfplay_trace)" % (n_envs, turns, args.steps, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_python_reference:
        line["python_reference"] = python_reference_rates(cores, 4.0)
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------
def run_cuda_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0 and world > 1:
        print("warning: --gpus %d but WORLD_SIZE %d" % (args.gpus, world), file=sys.stderr)

    from gym_narde_b200 import VecNardeEnv, _cabi

    E, K, W, R = args.envs_per_gpu, args.steps, args.warmup, args.turns_per_step
    nvtx = torch.cuda.nvtx
    env = VecNardeEnv(E, seed=SEED, max_actions=args.cap, env_base=rank * E, device=dev, chunks=args.chunks,
                      graph=not args.no_graph)
    env.reset()
    # ---- config 4's cross-rank clause: the first 50 turns of rank 1's shard, re-played on rank 0's GPU from the same
    # global env ids, must leave bit-identical states / outputs (results depend on (seed, global env id, step) only)
    cross = None
    CR = 50
    nvtx.range_push("burn_in")
    for t in range(args.burn_in):           # de-correlate game phases: steady-state self-play mix
        env.step()
        if world > 1 and t + 1 == CR:
            mine = torch.cat([env.lo.view(-1), env.hi.view(-1), env.counts.view(torch.uint8), env.chosen.view(torch.uint8)])
            other = torch.empty_like(mine)
            if rank == 1:
                other.copy_(mine)
            dist.broadcast(other, src=1)
            if rank == 0:
                twin = VecNardeEnv(E, seed=SEED, max_actions=args.cap, env_base=1 * E, device=dev, graph=not args.no_graph)
                twin.reset()
                for _ in range(CR):
                    twin.step()
                replay = torch.cat([twin.lo.view(-1), twin.hi.view(-1), twin.counts.view(torch.uint8), twin.chosen.view(torch.uint8)])
                cross = {"replayed_rank": 1, "on_rank": 0, "turns": CR, "envs": E,
                         "bit_identical": bool(torch.equal(replay, other))}
                del twin
    nvtx.range_pop()
    torch.cuda.synchronize()

    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(step_fn, n_steps):
        """Per-launch CUDA events on the launching stream; L2 flushed (untimed) in front of every launch."""
        evs = []
        for _ in range(n_steps):
            if flush is not None:
                flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    def pct(v, q):
        v = sorted(v)
        return v[min(len(v) - 1, int(q * len(v)))]

    # ---- device-resident arm: `value` ----
    for _ in range(W * min(R, 8)):
        env.step()
    stats0 = env.stats.clone()
    props = torch.cuda.get_device_properties(dev)
    try:
        pci = "%08X:%02X:%02X.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
    except Exception:
        pci = None
    sampler = ClockSampler(local_rank, pci)
    sampler.wait_ready()
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    nvtx.range_push("timed_value")
    ms = timed_loop(lambda: env.step(), K * R)            # K steps of R turns; every turn = one graph replay
    nvtx.range_pop()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t_wall0)
    clocks = sampler.stop()
    dstats = (env.stats - stats0).cpu().tolist()
    dumped = None
    if args.dump_outputs and rank == 0:      # before any further turn overwrites the last timed one
        dumped = dump_step_outputs(env, args.dump_outputs)
    total_ms = sum(ms)
    A = dstats[5] / float(E * K * R)
    # stored list entries per env turn = min(count, cap): what the kernel really writes (roofline bytes)
    stored = 0
    for _ in range(32):
        env.step()
        stored += int(env.counts.clamp(max=args.cap).sum().item())
    A_stored = stored / (32.0 * E)
    # side figure: the same turns back to back in ONE device interval, no L2 flush (what a pipeline of steps sees: the
    # launch latency and the exact kernel's last microseconds hide behind the next turn; a turn writes ~126 MB of
    # outputs per GPU on top of the previous turn's, as much as the L2 holds)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_b2b = 256
    t0.record()
    for _ in range(n_b2b):
        env.step()
    t1.record()
    torch.cuda.synchronize()
    ms_b2b = t0.elapsed_time(t1) / n_b2b

    # ---- end-to-end arm: host action choices in (pinned) -> step -> reward/done out (pinned) ----
    # uniformly random u32 fractions (fraction=True), FRESH every turn from a pinned pool the "host policy" filled
    # ahead: the same i.i.d. uniform self-play policy as the device arm (a constant fraction per env is a different,
    # more expensive game: 0.147 instead of 0.110 ms/step with device-resident inputs)
    POOL = 16
    h_pool = torch.randint(-(1 << 31), (1 << 31) - 1, (POOL, E), dtype=torch.int64).to(torch.int32).pin_memory()
    e2e_t = [0]
    d_idx = env.action_in                                    # persistent device input of VecNardeEnv.step
    h_rew = torch.zeros(E, dtype=torch.float32).pin_memory()
    h_done = torch.zeros(E, dtype=torch.uint8).pin_memory()

    def e2e_step_copies():
        e2e_t[0] += 1
        d_idx.copy_(h_pool[e2e_t[0] % POOL], non_blocking=True)        # H2D: this step's inputs (action choices)
        obs, rew, term, trunc, info = env.step(d_idx, fraction=True)   # public API call (graph replay)
        h_rew.copy_(rew, non_blocking=True)                  # D2H: this step's results
        h_done.copy_(env.done, non_blocking=True)

    io = env.host_io()                                       # pinned host result buffers of the host-facing step

    def e2e_step():
        # public API call with HOST buffers, zero-copy: the fused step fetches this turn's action choices from pinned
        # host memory (one bulk copy per CTA) and writes reward / done / truncated into pinned host memory
        e2e_t[0] += 1
        env.step_host(fraction=True, actions=h_pool[e2e_t[0] % POOL])

    def e2e_step_obs():
        # the same, and the OBSERVATION crosses PCIe too, in its packed form (32-byte state records written by the
        # kernel into pinned host memory; gym_narde_b200.expand_obs198 decodes them to Box(198) rows on the host)
        e2e_t[0] += 1
        # (obs="compact": observation and result in ONE 20-byte record per env -- 24 points of 5 bits, off counts, side to
        # move, flags, terminated / truncated / reward bits, steps -- 2.6 MB per turn instead of 4.2 MB of planes plus
        # three result arrays: the posted PCIe writes end before the kernel does)
        env.step_host(fraction=True, actions=h_pool[e2e_t[0] % POOL], obs="compact")

    for _ in range(max(W, POOL + 1)):          # one graph per pool buffer is captured on first use: all of them now
        e2e_step()
    barrier()
    nvtx.range_push("timed_e2e")
    ms_e2e = timed_loop(e2e_step, K * R)
    nvtx.range_pop()
    barrier()
    total_e2e = sum(ms_e2e)
    for _ in range(max(W, POOL + 1)):
        e2e_step_obs()
    barrier()
    ms_e2e_pobs = timed_loop(e2e_step_obs, K * R)
    barrier()
    total_e2e_pobs = sum(ms_e2e_pobs)
    k_side = min(K * R, 200)
    for _ in range(W):
        e2e_step_copies()
    ms_e2e_copies = timed_loop(e2e_step_copies, k_side)
    barrier()

    # ---- end-to-end, pipelined: VecNardeEnv.host_pipeline -- windows of 8 turns as ONE CUDA graph whose per-turn
    # H2D (action choices) / D2H (reward, done bits) copies run on copy streams, double-buffered on the device, so
    # the copies of neighbouring turns overlap the kernels.  Every turn still copies its own inputs in and its own
    # results out; timed as one device interval over K turns; no L2 flush is possible inside it, but a turn writes
    # ~120 MB of outputs (Box(198) 104 MB + action lists + ...) on top of the previous turn's, more than the L2. ----
    depth = 8
    pipe = env.host_pipeline(depth=depth, fraction=True)
    pipe.actions.copy_(h_pool[:depth])
    n_rep = max(1, (k_side + depth - 1) // depth)

    def e2e_pipelined(reps):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            pipe.run()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1)

    e2e_pipelined(2)
    barrier()
    ms_pipe_turn = e2e_pipelined(n_rep) / (n_rep * depth)     # per turn
    barrier()

    # ---- end-to-end with the whole Box(198) batch copied to the host as well (a host-side policy) ----
    h_obs = torch.empty((E, 198), dtype=torch.float32).pin_memory()

    def e2e_obs_step():
        e2e_step_copies()
        h_obs.copy_(env.obs, non_blocking=True)

    k_obs = max(3, min(K * R, 20))
    for _ in range(2):
        e2e_obs_step()
    barrier()
    ms_e2e_obs = timed_loop(e2e_obs_step, k_obs)
    barrier()

    # ---- config 2 side measurement (4096 lock-step envs, same kernel) ----
    small = VecNardeEnv(4096, seed=SEED, max_actions=args.cap, env_base=0, device=dev)
    small.reset()
    for _ in range(args.burn_in):
        small.step()
    torch.cuda.synchronize()
    ms_small = timed_loop(lambda: small.step(), min(K * R, 50))

    # ---- Tier R side measurement: the reference CODE's exact NardeEnv.step (narde_env.py:27-103) batched ----
    ref_env = VecNardeEnv(E, seed=SEED, rules="reference", device=dev)
    ref_env.reset()
    codes = torch.randint(0, 576, (E, 2), dtype=torch.int32, device=dev)
    for _ in range(30):
        ref_env.step(codes)
    torch.cuda.synchronize()
    ms_ref = timed_loop(lambda: ref_env.step(codes), min(K * R, 50))
    tier_r = {"value": E * len(ms_ref) / (sum(ms_ref) * 1e-3), "unit": "reference-exact env steps/s (rank 0)", "envs": E,
              "ms_per_step": sum(ms_ref) / len(ms_ref),
              "note": "k_roll_dice + k_step_ref: NardeEnv.step semantics of the reference code (2 dice, <= 2 half-moves, its "
                      "quirks), int32[24] observation, uniformly random action codes as examples/play_random_agent.py samples them"}

    # ---- config 5 side measurement: afterstate scoring with the tcgen05 MLP, 64K envs (rank 0's GPU) ----
    cfg5 = cfg3 = None
    if not args.no_config5 and rank == 0:
        cfg5 = config5_afterstate_scoring(torch, dev, args, timed_loop)
    if not args.no_config3 and rank == 0:
        cfg3 = config3_enumeration_microbench(torch, dev, args, timed_loop, measured_peaks()[0])

    # ---- policy-weight broadcast (config 4: NCCL broadcast of the packed DecomposedDQN(198) weights) ----
    bcast_ms = None
    if world > 1:
        from gym_narde_b200 import dist as ndist
        wp = torch.zeros(557056 // 2 + 16, dtype=torch.int16, device=dev)   # packed operand stages (~0.56 MB bf16)
        bs = torch.zeros(1088, dtype=torch.float32, device=dev)
        if rank == 0:
            wp.fill_(7)
            bs.fill_(0.5)
        ndist.broadcast_policy([wp, bs], src=0)                               # warm-up / communicator setup
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ndist.broadcast_policy([wp, bs], src=0)
        b.record()
        torch.cuda.synchronize()
        assert int(wp[0].item()) == 7 and float(bs[0].item()) == 0.5
        bcast_ms = a.elapsed_time(b)

    # ---- parity at the benchmarked configuration + the CPU baseline on the SAME work (rank 0, N = 1) ----
    parity = cpu = pyref = None
    if not args.no_cpu_baseline and world == 1:
        parity, cpu, pyref = parity_and_cpu_baseline(torch, env, args, cfg3)

    # ---- reduce over ranks (MAX time), gather episode stats with NCCL ----
    tmax = torch.tensor([total_ms, total_e2e, ms_pipe_turn, total_e2e_pobs], dtype=torch.float64, device=dev)
    st = env.stats.clone()
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        gathered = [torch.zeros_like(st) for _ in range(world)]
        dist.all_gather(gathered, st)                        # config 4: allgather of episode stats
        st_all = torch.stack(gathered)
    else:
        st_all = st[None]
    total_ms_max, total_e2e_max, ms_pipe_max, total_e2e_pobs_max = tmax.cpu().tolist()

    if rank == 0:
        peak, peak_src = measured_peaks()
        units = world * E * K * R
        value = units / (total_ms_max * 1e-3)
        e2e_value = units / (total_e2e_max * 1e-3)
        bytes_per_unit = 871 + 8 * A_stored                  # SURVEY 8(d): B_step(A), A = list entries actually stored
        kernel_ms = total_ms / (K * R)                       # rank-0 kernels of one turn (main + programmatic dependent)
        achieved = E * bytes_per_unit / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_src, ncu_counters = None, None, None
        cands = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.startswith("r02") and f.endswith("_step_full_v2.json"))
        if cands:                                            # ncu --set full of this round's kernel on this workload
            try:
                prof = json.load(open(os.path.join(ROOT, "profiles", cands[-1])))["launches"][0]
                traffic = prof.get("dram_bytes_per_launch")
                traffic_src = "ncu --set full, profiles/%s (per launch)" % cands[-1]
                pm = prof.get("metrics", {})
                num = lambda k: float(str(pm.get(k, "nan")).split()[0])
                ncu_counters = {"issue_slots_busy_pct": num("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                                "active_threads_per_warp_instruction": num("smsp__thread_inst_executed_per_inst_executed.ratio"),
                                "warp_instructions_per_launch": num("smsp__inst_executed.sum"),
                                "warps_active_pct": num("sm__warps_active.avg.pct_of_peak_sustained_active"),
                                "stall_cycles_per_issue": prof.get("warp_stalls_per_issue"),
                                "source": "profiles/%s (the committed capture of this kernel; not re-measured in this run)" % cands[-1]}
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8/u32 bit arithmetic (obs f32)", "data": "synthetic",
            "config": {"workload": "config4 shard: %d lock-step envs/GPU full-rules random self-play (1M envs at 8 GPUs)" % E,
                       "envs_per_gpu": E, "action_capacity": args.cap, "burn_in_steps": args.burn_in,
                       "turns_per_step": R, "ms_per_turn": total_ms_max / (K * R),
                       "ms_per_turn_p50": pct(ms, 0.5), "ms_per_turn_p95": pct(ms, 0.95),
                       "mean_legal_actions": A, "mean_stored_actions": A_stored, "max_legal_actions": int(st_all[:, 6].max().item()),
                       "l2": "flushed in front of every timed launch (256 MiB fill, untimed)" if flush is not None else "not flushed",
                       "parallelism": "env-sharded x%d, no data-path collective" % world},
            "roofline": {"bound": "hbm", "kernel": "k_step_full_v2<128,true> + its programmatic dependent k_step_deferred (order-dependent doubles turns, overlaps the tail), timed together as one turn", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_env_step": bytes_per_unit, "kernel_ms": kernel_ms, "launches_timed": K * R,
                         "ncu_counters": ncu_counters},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * E * R, "d2h_bytes_per_step": 6 * E * R,
                    "ms_per_step": total_e2e_max / K, "ms_per_turn": total_e2e_max / (K * R), "observation": "Box(198) stays in HBM (device-resident policy); see e2e_with_obs",
                    "note": "VecNardeEnv.step_host(fraction=True, actions=pool row), zero-copy, one CUDA-graph replay per turn: every CTA of the fused step bulk-copies its envs' int32 action choices (fresh u32 fractions of the legal list, pinned pool) from host memory into shared memory, and reward f32 / done u8 / truncated u8 are written by the kernel straight into pinned host memory"},
            "e2e_with_obs": {"value": units / (total_e2e_pobs_max * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 4 * E * R,
                             "d2h_bytes_per_step": 20 * E * R, "ms_per_turn": total_e2e_pobs_max / (K * R),
                             "frac_of_value": (units / (total_e2e_pobs_max * 1e-3)) / value,
                             "observation": "compact: one 20-byte record per env (the state -- a lossless encoding of Box(198) -- and the turn's result bits; gym_narde_b200.state.unpack_compact + expand_obs198 decode it) is written by the kernel into pinned host memory",
                             "note": "step_host(fraction=True, obs='compact'): actions in, observation + terminated / truncated / reward out in one record per env, all through pinned host memory, no copy operations (the 32-byte planes + one result byte, obs='packed', packed=True: 0.122 ms per turn)"},
            "e2e_explicit_copies": {"value": world * E * k_side / (sum(ms_e2e_copies) * 1e-3), "unit": UNIT, "ms_per_turn": sum(ms_e2e_copies) / k_side,
                                    "note": "the same turn with cudaMemcpyAsync H2D / D2H around VecNardeEnv.step (rank 0's time)"},
            "e2e_pipelined": {"value": world * E / (ms_pipe_max * 1e-3), "unit": UNIT, "ms_per_turn": ms_pipe_max,
                              "note": "VecNardeEnv.host_pipeline(depth=8, fraction=True): 8 turns per CUDA-graph replay, every turn with its "
                                      "own DMA of pinned action choices on a copy-in stream (double-buffered on the device) and its results "
                                      "written by the kernel straight into pinned host rows; one device interval, no L2 flush (a turn's "
                                      "outputs exceed the L2)"},
            "e2e_obs_to_host": {"value": world * E * k_obs / (sum(ms_e2e_obs) * 1e-3), "unit": UNIT, "turns": k_obs,
                                "d2h_bytes_per_turn": 5 * E + 792 * E, "ms_per_turn": sum(ms_e2e_obs) / k_obs,
                                "note": "explicit copies plus the full float32 Box(198) batch copied D2H every turn (PCIe-bound; rank 0's time)"},
            # per turn: k_step_full_v2 + k_step_deferred (+ k_advance_counter when a chunked env replays a graph)
            "gpu_launches": K * R * ((3 if (env.use_graph and env._ws_adv is None) else 2) * len(env._chunks)),
            "wall_ms": wall_ms, "clocks": clocks,
            "config2_4096_envs": {"value": 4096 * len(ms_small) / (sum(ms_small) * 1e-3), "unit": UNIT,
                                  "ms_per_turn": sum(ms_small) / len(ms_small)},
            "episode_stats": {k: int(v) for k, v in zip(_cabi.STAT_NAMES, st_all.sum(0).tolist())},
        }
        line["tier_r_reference_rules_step"] = tier_r
        if bcast_ms is not None:
            line["policy_broadcast_ms"] = bcast_ms
        if cross is not None:
            line["cross_rank_shard_check"] = cross
        if dumped is not None:
            line["dumped_outputs"] = dumped
        if cfg5 is not None:
            line["config5_afterstate_scoring"] = cfg5
        line["back_to_back"] = {"ms_per_turn": ms_b2b, "value_rank0": E / (ms_b2b * 1e-3), "turns": n_b2b,
                                "note": "rank 0: 256 graph-replayed turns in one CUDA-event interval, L2 NOT flushed (side figure; "
                                        "`value` is the flushed, individually timed one)"}
        if cfg3 is not None:
            cfg3.pop("_sample", None)
            line["config3_enumeration_microbench"] = cfg3
        if parity is not None:
            line["parity"] = parity
            line["parity_checked_env_turns"] = parity["checked_env_turns"]
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if pyref is not None:
            line["python_reference"] = pyref
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_ENVS = 65536    # 832 bytes of float32 outputs per env: a sample of this many envs stays under 64 MB


def dump_step_outputs(env, out_dir):
    """--dump-outputs: what the last VecNardeEnv.step() returned, as float32 DIR/<name>.npy.  step() returns the env's
    persistent output buffers, so right after the timed loop they hold the last timed turn.  Every array keeps the same
    rows: all envs, or a fixed seeded sample of DUMP_ENVS of them.  The arguments fix the inputs (seed, env ids, number
    of turns), so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    torch = env.torch
    n = env.num_envs
    rows = np.arange(n) if n <= DUMP_ENVS else np.sort(np.random.default_rng(SEED).choice(n, DUMP_ENVS, replace=False))
    idx = torch.from_numpy(rows).to(env.device)
    info = env.info
    arrays = {"obs": env.obs, "reward": env.reward, "terminated": env.terminated, "truncated": env.truncated,
              "dice": info["dice"], "counts": info["counts"]}
    arrays = {k: v[idx].to(torch.float32).cpu().numpy() for k, v in arrays.items()}
    # a turn action is four u16 half-moves (include/narde_b200.h): column k holds bits 16k..16k+15, exact in float32
    arrays["chosen"] = info["chosen"][idx].cpu().numpy().view(np.uint16).reshape(-1, 4).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    return {"dir": out_dir, "turn": env.step_count, "envs": int(len(rows)), "arrays": sorted(arrays)}


def parity_and_cpu_baseline(torch, env, args, cfg3):
    """The one place of the CUDA arm that executes oracle/: as the CPU baseline and as the checker.

    The env object that was just timed plays P more turns through the same call (graph replay), every turn's outputs
    are kept on the device; the C oracle then replays the SAME turns from the SAME start positions on all host cores
    (timed: the cpu_baseline, same_config true) for as many of the envs as fit ~12 s of CPU work, and every env turn
    of that sample is compared: packed state, legal-action count, checksum of the stored list, chosen action, dice,
    reward, terminated / truncated.  Then config 3's 10 k-position subsample against the oracle's enumeration."""
    import numpy as np
    from oracle import oracle as O
    O.build()
    E, P, cap = env.num_envs, 96, env.max_actions      # 96 turns = one period of the (synchronised) game phases
    cores = os.cpu_count() or 1
    step0 = env.step_count
    init_lo, init_hi = env.lo.cpu().numpy(), env.hi.cpu().numpy()
    w = torch.from_numpy(O.list_weights(cap)).to(env.device)
    keep = torch.arange(cap, device=env.device)[None, :]
    rec = {k: [] for k in ("lo", "hi", "count", "chosen", "dice", "reward", "done", "hash")}
    for _ in range(P):
        env.step()
        rec["lo"].append(env.lo.clone())
        rec["hi"].append(env.hi.clone())
        rec["count"].append(env.counts.clone())
        rec["chosen"].append(env.chosen.clone())
        rec["dice"].append(env.dice.clone())
        rec["reward"].append(env.reward.clone())
        rec["done"].append(env.done | (env.trunc << 1))
        m = keep < env.counts.clamp(max=cap)[:, None]
        rec["hash"].append((torch.where(m, env.actions, torch.zeros_like(env.actions)) * w[None, :]).sum(1))
    torch.cuda.synchronize()
    # rate probe, then a sample sized to ~12 s of CPU work
    _, dt = cpu_trace((init_lo[:2048], init_hi[:2048]), 2048, 8, step0, env.seed, env.env_base, cap)
    rate = 2048 * 8 / dt
    M = int(min(E, max(4096, (12.0 * rate / P) // 1024 * 1024)))
    tr, dt = cpu_trace((init_lo[:M], init_hi[:M]), M, P, step0, env.seed, env.env_base, cap, want_states=True)
    equal, first_bad = True, None
    for key in ("count", "dice", "hash", "chosen", "reward", "done", "lo", "hi"):
        got = torch.stack(rec[key])[:, :M].cpu().numpy()
        if not (got == tr[key]).all():
            equal = False
            bad = np.argwhere((got != tr[key]).reshape(P, M, -1).any(2))[0]
            first_bad = {"field": key, "turn": int(step0 + bad[0] + 1), "env": int(bad[1])}
            break
    parity = {"checked_env_turns": int(tr["turns"]) if equal else 0, "equal": equal, "envs": M, "turns": P,
              "path": "VecNardeEnv.step() of the timed env object (graph replay, DEVICE_ADVANCE, cap %d), every env turn vs oracle/narde_oracle.c o_selfplay_trace" % cap,
              "fields": "state planes, legal-action count, stored-list checksum, chosen action, dice, reward, terminated/truncated"}
    if first_bad:
        parity["first_mismatch"] = first_bad
    if cfg3 is not None and "_sample" in cfg3:      # config 3: 10 k-position subsample against the oracle (SURVEY 8d)
        lo3, hi3, d3, c3, a3 = cfg3["_sample"]
        wn = O.list_weights(a3.shape[1]).view(np.uint64)
        m3 = np.arange(a3.shape[1])[None, :] < np.minimum(c3, a3.shape[1])[:, None]
        with np.errstate(over="ignore"):
            h3 = (np.where(m3, a3.view(np.uint64), 0) * wn[None, :]).sum(1, dtype=np.uint64).view(np.int64)
        oc, oh = O.enumerate_batch(lo3, hi3, d3, a3.shape[1])
        cfg3["subsample_equals_oracle"] = bool((oc == c3).all() and (oh == h3).all())
        cfg3["subsample_positions"] = int(len(oc))
        parity["config3_subsample_equal"] = cfg3["subsample_equals_oracle"]
    A_cpu = float(tr["stats"][5]) / max(tr["turns"], 1)
    cpu = {"value": tr["turns"] / dt, "unit": UNIT, "cores": cores, "kind": "port", "same_config": True,
           "mean_legal_actions": A_cpu,
           "sample": "%d of the GPU arm's %d envs x %d turns from the GPU arm's own steady-state positions (same seed, env ids, dice, policy, "
                     "cap; one Box(198) row per env turn), %d env turns in %.1f s on %d host threads (oracle/narde_oracle.c o_selfplay_trace)" % (M, E, P, tr["turns"], dt, cores)}
    pyref = None if args.no_python_reference else python_reference_rates(cores, 5.0)
    if pyref is not None:
        cpu["python_reference_NardeEnv_step_per_s"] = pyref["NardeEnv_step_valid_random"]["env_steps_per_s"]
        cpu["python_reference_pair_enumeration_step_per_s"] = pyref["pair_enumeration_plus_step"]["env_steps_per_s"]
    if not equal:
        print("PARITY FAILURE: %s" % json.dumps(first_bad), file=sys.stderr)
    return parity, cpu, pyref


def config3_enumeration_microbench(torch, dev, args, timed_loop, peak):
    """BASELINE config 3 (SURVEY 8d): get_valid_actions over 1M synthetic positions, seed 1234, three strata
    (gym_narde_b200/workloads.py:config3_positions).  The 10 k-position subsample is checked against the ORACLE in
    parity_and_cpu_baseline (the only place of this arm that touches oracle/)."""
    from gym_narde_b200 import _cabi
    from gym_narde_b200.workloads import config3_positions
    n = 1 << 20
    lo, hi, dice, strata_rng = config3_positions(dev, n=n, seed=1234)
    cap = args.cap
    actions = torch.zeros((n, cap), dtype=torch.int64, device=dev)
    counts = torch.zeros(n, dtype=torch.int32, device=dev)
    ovf = torch.zeros(n, dtype=torch.uint8, device=dev)
    ws = torch.zeros(_cabi.workspace_ints(n), dtype=torch.int32, device=dev)
    run = lambda: _cabi.enumerate_actions_fast(lo, hi, dice, actions, counts, ovf, ws)
    for _ in range(3):
        run()
    k = max(5, min(args.steps * args.turns_per_step, 20))
    ms = timed_loop(run, k)
    mean_ms = sum(ms) / k
    g = torch.Generator(device=dev).manual_seed(99)
    sub = torch.randperm(n, device=dev, generator=g)[:10000]
    sample = (lo[sub].cpu().numpy(), hi[sub].cpu().numpy(), dice[sub].cpu().numpy(), counts[sub].cpu().numpy(),
              actions[sub].cpu().numpy())
    A = float(counts.float().mean().item())
    bytes_per = 38 + 8 * float(counts.clamp(max=cap).float().mean().item())
    strata = {}
    for name, (a, b) in strata_rng.items():
        strata[name] = {"positions": b - a, "mean_legal": float(counts[a:b].float().mean().item()),
                        "max_legal": int(counts[a:b].max().item())}
    return {"positions": n, "positions_per_s": n / (mean_ms * 1e-3), "ms": mean_ms, "cap": cap, "mean_legal_actions": A,
            "max_legal_actions": int(counts.max().item()), "overflow_positions": int(ovf.sum().item()),
            "deferred_exact_positions": int(ws[0].item()), "strata": strata, "_sample": sample,
            "achieved_GBps": n * bytes_per / (mean_ms * 1e-3) / 1e9, "hbm_frac": n * bytes_per / (mean_ms * 1e-3) / 1e9 / peak,
            "algorithmic_bytes_per_position": bytes_per}


def config5_afterstate_scoring(torch, dev, args, timed_loop):
    """BASELINE config 5: DecomposedDQN(198) (train_deepq_pytorch.py:184-236, torch.manual_seed(0) random init) over
    all legal afterstates of 65536 envs: enumerate -> afterstates -> Box(198) encode + 3-layer MLP + max_a Q
    on the tcgen05 tensor cores -> greedy choice -> env step, all on the device (AfterstateActor)."""
    import torch.nn as nn
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    torch.manual_seed(0)
    fn = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU()).to(dev)
    head = nn.Linear(256, 576).to(dev)
    mlp = AfterstateMLP.from_module(fn, head)
    E5 = 65536
    env = VecNardeEnv(E5, seed=SEED, max_actions=args.cap, device=dev)
    actor = AfterstateActor(env, mlp)
    env.reset()
    for _ in range(60):                      # random self-play burn-in, then greedy turns
        env.step()
    for _ in range(5):
        actor.step_graph()
    torch.cuda.synchronize()
    k = max(5, min(args.steps, 30))
    rows = []

    side_rows = []

    def greedy_step():
        actor.step_graph()                   # one CUDA-graph replay per greedy turn
        rows.append(actor.rows_dev.clone())
        side_rows.append(actor.side.rows_dev.clone())

    ms_actor = timed_loop(greedy_step, k)
    mean_rows = float(torch.stack(rows).float().mean().item())
    # the scorer alone on the last step's afterstates (same rows, L2 flushed between launches)
    ms_mlp = timed_loop(lambda: mlp.score_states(actor.as_lo, actor.as_hi, out=actor.scores, rows_dev=actor.rows_dev), k)
    last_rows = int(actor.rows_dev.item())
    flop_row = 2 * (198 * 256 + 256 * 256 + 256 * 576)
    mlp_ms = sum(ms_mlp) / len(ms_mlp)
    tfl = last_rows * flop_row / (mlp_ms * 1e-3) / 1e12
    peak_tf, peak_burst = 1361.0, 1596.6
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        try:
            d = json.load(open(pk))
            peak_tf = float(d["bf16_tflops_sustained"])
            peak_burst = float(d.get("bf16_tflops", peak_burst))
        except Exception:
            pass
    mean_side = float(torch.stack(side_rows).float().mean().item())
    return {"envs": E5, "greedy_env_steps_per_s": E5 * k / (sum(ms_actor) * 1e-3), "ms_per_greedy_step": sum(ms_actor) / k,
            "ms_per_greedy_step_outside_the_scorer": sum(ms_actor) / k - mlp_ms,
            "afterstate_rows_per_step": mean_rows, "side_batch_rows_per_step": mean_side,
            "env_turns_not_fully_scored": actor.uncovered_envs(),
            "scorer_rows": last_rows, "scorer_ms": mlp_ms,
            "scorer_rows_per_s": last_rows / (mlp_ms * 1e-3), "scorer_tflops": tfl,
            "scorer_frac_of_bf16_peak": tfl / peak_tf, "bf16_peak_tflops": peak_tf,
            "scorer_frac_of_bf16_burst_peak": tfl / peak_burst, "bf16_burst_peak_tflops": peak_burst,
            "flops_per_row": flop_row, "dtype": "bf16 operands, fp32 accumulate (tcgen05)",
            "note": "greedy turn = one CUDA-graph replay: enumerate -> afterstate rows + their offsets (one launch) -> k_mlp<states in, "
                    "row-max out> (Box(198) encoded in-kernel from 32-byte afterstates; weights random init) -> arg-max -> second pass over "
                    "the envs whose list exceeds the stored capacity (side batch: every legal action is scored) -> fused step.  The scorer "
                    "alone is timed in isolation on the last turn's rows (burst peak is its comparator; the sustained one the turn's)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=131072)
    ap.add_argument("--cap", type=int, default=64)
    ap.add_argument("--burn-in", type=int, default=300)
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--chunks", type=int, default=None)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--no-config3", action="store_true")
    ap.add_argument("--no-python-reference", action="store_true")
    ap.add_argument("--turns-per-step", type=int, default=128,
                    help="lock-step turns (graph replays, each timed on its own with a flushed L2) that make one 'step'")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what VecNardeEnv.step() returned on the last timed turn as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the CUDA path's outputs; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_cuda_arm(args)


if __name__ == "__main__":
    main()
