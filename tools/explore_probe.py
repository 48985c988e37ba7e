"""GPU: what exploration costs the afterstate actor's turn.  Config 5's setup (65 536 envs, cap 64, random-init
DecomposedDQN(198), 60 random burn-in turns, step_graph() replays timed one by one with CUDA events, L2 flushed in front
of each): the greedy turn against epsilon 0.1, temperature 1, both, and epsilon 1, timed in alternating rounds.
Prints the card and its power limit, then one JSON line (ms per turn: mean and median per setting, ratio to greedy,
uncovered_envs())."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn as nn
from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor

SETTINGS = (("greedy", None), ("eps0.1", (0.1, 0.0)), ("tau1", (0.0, 1.0)), ("eps0.1+tau1", (0.1, 1.0)), ("eps1", (1.0, 0.0)))


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (a query only; the measurement does not depend on it)
        q = "unknown (%s)" % e
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--cap", type=int, default=64)
    ap.add_argument("--turns", type=int, default=20, help="timed turns per setting and round")
    ap.add_argument("--rounds", type=int, default=4)
    args = ap.parse_args()
    name, limits = card()
    print("card: %s | power.limit, clocks.max.sm: %s" % (name, limits), flush=True)
    torch.manual_seed(0)
    fn = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU()).cuda()
    head = nn.Linear(256, 576).cuda()
    mlp = AfterstateMLP.from_module(fn, head)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    actors = {}
    for label, params in SETTINGS:
        env = VecNardeEnv(args.envs, seed=0x5EED, max_actions=args.cap)
        actor = AfterstateActor(env, mlp)
        if params is not None:
            actor.set_exploration(*params)
        env.reset()
        for _ in range(60):
            env.step()
        for _ in range(5):
            actor.step_graph()
        actors[label] = actor
    torch.cuda.synchronize()
    ms = {label: [] for label, _ in SETTINGS}
    for _ in range(args.rounds):
        for label, _ in SETTINGS:
            actor, evs = actors[label], []
            for _ in range(args.turns):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                actor.step_graph()
                b.record()
                evs.append((a, b))
            torch.cuda.synchronize()
            ms[label] += [a.elapsed_time(b) for a, b in evs]
    g = statistics.mean(ms["greedy"])
    out = {"card": name, "power_limit_and_max_sm_clock": limits, "envs": args.envs, "cap": args.cap,
           "turns_per_setting": args.turns * args.rounds, "l2": "flushed in front of every timed turn"}
    for label, _ in SETTINGS:
        out[label] = {"ms_mean": statistics.mean(ms[label]), "ms_median": statistics.median(ms[label]),
                      "ratio_to_greedy": statistics.mean(ms[label]) / g,
                      "uncovered_envs": actors[label].uncovered_envs()}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
