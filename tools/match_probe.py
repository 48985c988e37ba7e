"""GPU: what a lock-step match turn costs (gym_narde_b200.AfterstateMatch).  65 536 games, cap 64, random-init
DecomposedDQN(198) nets (torch seeds 0 and 1), 60 random burn-in turns, step_graph() warmed, then `--turns` replays timed
with CUDA events, for net vs net, net vs random and random vs random, beside AfterstateActor.step_graph() (greedy
self-play of the seed-0 net) on the same settings.  Per setting: ms per turn; the rows the scorer scored on the last timed
turn (the pools' device row counters) against the rows of the net-owned envs (min(count, cap) summed over the envs whose
side to move a net seat owns, plus the side batch's): every row scored once; and score_states alone on the main pools' rows
of that turn (timed with events: the scorer's share of the turn); and the wall time and games/s of one full
play() (every game to its end, max_episode_steps 1000).  Prints the card and its power limit, then one JSON line per
setting."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.nn as nn
from gym_narde_b200 import AfterstateActor, AfterstateMatch, AfterstateMLP, VecNardeEnv
from lookahead_probe import card


def _net(seed):
    torch.manual_seed(seed)
    fn = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU()).cuda()
    return AfterstateMLP.from_module(fn, nn.Linear(256, 576).cuda())


def _time(step, turns):
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(turns):
        step()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / turns


def _scorer_ms(bufs, reps=10):
    """score_states alone over (net, lo, hi, out, rows_dev) buffers as the last turn left them, timed with events."""
    for mlp, lo, hi, out, rows in bufs:
        mlp.score_states(lo, hi, out=out, rows_dev=rows)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        for mlp, lo, hi, out, rows in bufs:
            mlp.score_states(lo, hi, out=out, rows_dev=rows)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def _rows(pools):
    return sum(int(p.rows_dev.item()) for p in pools if p is not None)


def run_match(n, a, b, turns, seed):
    m = AfterstateMatch(n, a, b, seed=seed)
    for _ in range(60):
        m.env.step()
    ms = _time(m.step_graph, turns)
    hi = m.env.hi.cpu().numpy()
    m.step_graph()
    counts = np.minimum(m.env.counts.cpu().numpy(), m.cap)
    g = m.env.env_base + np.arange(n)
    a_owns = hi[:, 10].view(np.int8) == np.where(g % 2 == 0, 1, -1)
    net_owned = (a_owns & (m.kinds & 1 != 0)) | (~a_owns & (m.kinds & 2 != 0))
    side = m.side_pools
    r = {"ms_per_turn": ms, "rows_scored_last_turn": _rows(m.pools), "rows_of_net_owned_envs": int(counts[net_owned].sum()),
         "side_rows_scored_last_turn": _rows(side),
         "scorer_ms_main_pools_last_turn": _scorer_ms([(net, p.as_lo, p.as_hi, p.scores, p.rows_dev)
                                                       for net, p in zip(m.nets, m.pools) if p is not None])}
    t0 = time.perf_counter()
    res = m.play()
    wall = time.perf_counter() - t0
    r.update(play_wall_s=wall, play_games_per_s=n / wall, play_results=res, play_turns=m.env.step_count,
             uncovered_envs=m.uncovered_envs())
    return r


def run_actor(n, net, turns, seed):
    env = VecNardeEnv(n, seed=seed, autoreset=False, max_actions=64)
    actor = AfterstateActor(env, net, mode="white_value")
    env.reset()
    for _ in range(60):
        env.step()
    ms = _time(actor.step_graph, turns)
    actor.step_graph()
    return {"ms_per_turn": ms, "rows_scored_last_turn": int(actor.rows_dev.item()),
            "scorer_ms_main_pools_last_turn": _scorer_ms([(net, actor.as_lo, actor.as_hi, actor.scores, actor.rows_dev)]),
            "side_rows_scored_last_turn": int(actor.side.rows_dev.item()), "uncovered_envs": actor.uncovered_envs()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=65536)
    ap.add_argument("--turns", type=int, default=30)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    name, limits = card()
    lines = ["card: %s | power.limit, clocks.max.sm: %s" % (name, limits)]
    print(lines[-1], flush=True)
    na, nb = _net(0), _net(1)
    n, seed = args.games, 0x5EED
    settings = [("greedy_actor_selfplay", lambda: run_actor(n, na, args.turns, seed)),
                ("net_vs_net", lambda: run_match(n, na, nb, args.turns, seed)),
                ("net_vs_random", lambda: run_match(n, na, "random", args.turns, seed)),
                ("random_vs_random", lambda: run_match(n, "random", "random", args.turns, seed))]
    greedy = None
    for label, fn in settings:
        r = fn()
        if label == "greedy_actor_selfplay":
            greedy = r["ms_per_turn"]
        r = dict(setting=label, games=n, cap=64, turns=args.turns, vs_greedy_turn=r["ms_per_turn"] / greedy, **r)
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
