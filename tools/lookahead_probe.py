"""GPU: what a one-ply lookahead turn costs (gym_narde_b200.LookaheadActor).  For N envs x K candidates: random-init
DecomposedDQN(198), cap 64, reply_cap 64, 60 random burn-in turns, step_graph() warmed, then `--turns` replays timed with
CUDA events (one pair around the whole window, and per turn).  Per setting it reports ms per turn; reply positions
(N * K * 21) and the rows the scorer scored per turn (first pass, its side batch, replies, the reply side batch: the
device row counters, read after five untimed turns and after the last timed one); the scorer's share of the last timed
turn -- score_states alone on that turn's row buffers and counts, timed with events -- and its achieved FLOP/s at
527 360 FLOP per row (2 * (198*256 + 256*256 + 256*576)); device memory allocated by the actor.  Prints the card and its power limit, then one JSON line per setting."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn as nn
from gym_narde_b200 import AfterstateMLP, LookaheadActor, VecNardeEnv

FLOP_PER_ROW = 2 * (198 * 256 + 256 * 256 + 256 * 576)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (a query only; the measurement does not depend on it)
        q = "unknown (%s)" % e
    return name, q


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _scorer_ms(actor, reps):
    """score_states alone over the four row buffers of the last turn, with their device row counts."""
    a, mlp = actor.first, actor.mlp
    bufs = [(a.as_lo, a.as_hi, a.scores, a.rows_dev), (actor.r_as_lo, actor.r_as_hi, actor.r_scores, actor.r_rows_dev)]
    for sb in (a.side, actor.reply_side):
        if sb is not None:
            bufs.append((sb.as_lo, sb.as_hi, sb.scores, sb.rows_dev))
    for lo, hi, out, rows in bufs:
        mlp.score_states(lo, hi, out=out, rows_dev=rows)
    s, e = _events()
    s.record()
    for _ in range(reps):
        for lo, hi, out, rows in bufs:
            mlp.score_states(lo, hi, out=out, rows_dev=rows)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def _rows(actor):
    a = actor.first
    r = {"first_pass": int(a.rows_dev.item()), "replies": int(actor.r_rows_dev.item())}
    r["first_side"] = int(a.side.rows_dev.item()) if a.side is not None else 0
    r["reply_side"] = int(actor.reply_side.rows_dev.item()) if actor.reply_side is not None else 0
    return r


def run(n, k, mlp, turns):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    env = VecNardeEnv(n, seed=0x5EED, max_actions=64)
    actor = LookaheadActor(env, mlp, candidates=k, reply_cap=64)
    mem = torch.cuda.memory_allocated() - base
    env.reset()
    for _ in range(60):
        env.step()
    rows = []
    for _ in range(5):                   # untimed: the row counts of a few turns
        actor.step()
        rows.append(_rows(actor))
    for _ in range(3):
        actor.step_graph()
    torch.cuda.synchronize()
    s, e = _events()
    per = []
    s.record()
    for _ in range(turns):
        a, b = _events()
        a.record()
        actor.step_graph()
        b.record()
        per.append((a, b))
    e.record()
    torch.cuda.synchronize()
    ms_window = s.elapsed_time(e) / turns
    ms_turn = [a.elapsed_time(b) for a, b in per]
    # the scorer alone on the row buffers and row counts the last timed turn left, against that turn's own time
    scorer = _scorer_ms(actor, 10)
    last = _rows(actor)
    scored = sum(last.values())
    mean_rows = {key: statistics.mean(r[key] for r in rows) for key in rows[0]}
    return {"envs": n, "candidates": k, "reply_cap": 64, "turns": turns, "ms_per_turn": ms_window,
            "ms_per_turn_median": statistics.median(ms_turn), "reply_positions": actor.positions,
            "rows_per_turn_mean_of_5": mean_rows, "rows_last_turn": last,
            "last_turn_ms": ms_turn[-1], "scorer_ms_last_turn_rows": scorer, "scorer_share_of_last_turn": scorer / ms_turn[-1],
            "scorer_tflops": scored * FLOP_PER_ROW / (scorer * 1e-3) / 1e12,
            "actor_device_mb": mem / 2 ** 20, "max_allocated_mb": torch.cuda.max_memory_allocated() / 2 ** 20,
            "uncovered_envs": actor.uncovered_envs()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[1024, 4096, 16384])
    ap.add_argument("--candidates", type=int, nargs="+", default=[1, 4, 8])
    ap.add_argument("--turns", type=int, default=50)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    name, limits = card()
    head_line = "card: %s | power.limit, clocks.max.sm: %s" % (name, limits)
    print(head_line, flush=True)
    torch.manual_seed(0)
    fn = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU()).cuda()
    mlp = AfterstateMLP.from_module(fn, nn.Linear(256, 576).cuda())
    lines = [head_line]
    for n in args.envs:
        for k in args.candidates:
            torch.cuda.reset_peak_memory_stats()
            r = run(n, k, mlp, args.turns)
            r.update(card=name, power_limit_and_max_sm_clock=limits)
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
