"""GPU (-m gpu): the greedy and lookahead actors against the oracle at the sizes bench.py and tools/lookahead_probe.py
run, with the actors' default pools.

The reference tests of test_gpu_actor_reference.py and test_gpu_lookahead.py run a few thousand envs with a side batch
slot for every env.  Some paths only run, or only run hard, at the benchmarked sizes: narde_afterstates_scan's look-back
over thousands of tiles (5 376 reply tiles at N = 4096, K = 8; 21 504 at N = 16 384), the scorer over hundreds of
persistent rounds, the side batches' default sizes (N / 16 slots) with thousands of gathered envs, and the greedy
side batch on its own stream beside a first pass that fills the GPU.  Here:

- config 5 as bench.py times it (65 536 envs, cap 64, mode "max", the seed-0 nn.Linear net, step_graph()): every
  choice within bound() of the float64 net over the oracle's full lists; the same shape with exact scorers, bit for bit;
- score_states over 29 M packed rows (a lookahead turn at N = 16 384) with a device row count below the buffer;
- LookaheadActor at the probe's settings (K = 8, cap and reply_cap 64): bit for bit with an exact scorer at N = 4096
  and 16 384, within the bound with the probe's net at N = 4096;
- both actors give the same states and choices whether one env holds every game or two half-size envs split them by
  env_base, each with its own default pools.

Each test prints the env turns it checked, the choices beyond the stored list, the side-batch rows and its wall time
(-s).
"""
import time

import numpy as np
import pytest
import torch

from test_gpu_actor_reference import _Turn, _actor, _design, _play, check_exact_turn, check_within_bound
from test_gpu_lookahead import _LookTurn, _lookahead, check_look_bound, check_look_turn
from test_gpu_mlp_reference import SENTINEL, _cuda, _mlp, _nan_buffer
from test_mlp_reference_cpu import EXACT_DESIGNS, check_premise, default_net, ref_q, synthetic_states

pytestmark = pytest.mark.gpu

SEED = 0x5EED          # bench.py's and the probe's seed
E5 = 65536             # bench.py config 5's envs
CAP = 64               # bench.py's --cap default, the probe's cap and reply_cap
K = 8                  # the probe's candidates


def _net():
    """bench.py config 5's and the probe's scorer: nn.Linear's default init under torch.manual_seed(0)."""
    W, b = default_net(0, 1.0)
    return tuple(w.cuda() for w in W), tuple(v.cuda() for v in b)


def _greedy(design, mode, n=E5, env_base=0):
    """config5_afterstate_scoring's env and actor: no pool arguments, 60 random turns."""
    return _actor(design, CAP, mode, n=n, max_episode_steps=1000, seed=SEED, env_base=env_base)


def _look(design, n, env_base=0):
    """tools/lookahead_probe.py's env and actor: no pool arguments, 60 random turns."""
    return _lookahead(design, K, CAP, CAP, n=n, seed=SEED, env_base=env_base, slot_per_env=False)


# ---------------------------------------------------------------------------------------------------------------
# the greedy actor at config 5's shape
# ---------------------------------------------------------------------------------------------------------------
def test_config5_as_benchmarked_is_within_the_bound():
    """bench.py config 5 (65 536 envs, cap 64, mode "max", the seed-0 net, default pools, step_graph()), 20 turns after
    60 random ones: the rule of check_within_bound against the oracle's full lists scored by the float64 net, the action
    played is the oracle's action at the choice, and every env was covered.  Some choices come from the side batch."""
    t0 = time.time()
    W, b = _net()
    env, actor = _greedy((W, b), "max")
    seen = dict(turns=0, decided=0, near=0, beyond=0, side_rows=0)
    for t in range(20):
        lo, hi, dice = _play(env, actor, True)
        ref = _Turn(lo, hi, dice, env.counts, W, b, 0, emulate=False, with_bound=True)
        choice, chosen = actor.choice.cpu().numpy(), env.chosen.cpu().numpy()
        d, e = check_within_bound(ref, choice, actor.value.cpu().numpy(), t)
        live = np.flatnonzero(ref.counts > 0)
        assert np.array_equal(chosen[live], ref.acts[live, choice[live]]), ("action", t)
        seen["turns"] += len(live)
        seen["decided"] += d
        seen["near"] += e
        seen["beyond"] += int((choice[live] >= CAP).sum())
        seen["side_rows"] += int(actor.side.rows_dev.item())
    uncovered = actor.uncovered_envs()
    print("config 5, seed-0 net: %s, uncovered %d, %.1f s" % (seen, uncovered, time.time() - t0))
    assert uncovered == 0
    assert seen["beyond"] > 0 and seen["side_rows"] > 0, seen
    assert seen["decided"] > 100000, seen


@pytest.mark.parametrize("design,mode", [("perm", "max"), ("sparse", "white_value")])
def test_config5_shape_with_an_exact_scorer_is_bit_exact(design, mode):
    """config 5's env and default pools with an exact scorer, 30 turns alternating step() and step_graph(): choice,
    value and the action played equal the reference bit for bit (check_exact_turn) for every env."""
    t0 = time.time()
    W, b = _design(design)
    env, actor = _greedy((W, b), mode)
    seen = dict(turns=0, beyond=0, side_rows=0)
    for t in range(30):
        lo, hi, dice = _play(env, actor, t % 2 == 1)
        ref = _Turn(lo, hi, dice, env.counts, W, b, 1 if mode == "white_value" else 0, emulate=True, premise=(t == 0))
        choice = actor.choice.cpu().numpy()
        rows, want_k = check_exact_turn(ref, choice, actor.value.cpu().numpy(), env.chosen.cpu().numpy(),
                                        (design, mode, t))
        seen["turns"] += len(rows)
        seen["beyond"] += int((want_k[rows] >= CAP).sum())
        seen["side_rows"] += int(actor.side.rows_dev.item())
    uncovered = actor.uncovered_envs()
    print("config 5 shape, exact %s %s: %s, uncovered %d, %.1f s" % (design, mode, seen, uncovered, time.time() - t0))
    assert uncovered == 0
    assert seen["beyond"] > 0, seen


# ---------------------------------------------------------------------------------------------------------------
# the scorer at lookahead row counts
# ---------------------------------------------------------------------------------------------------------------
def test_score_states_at_lookahead_row_counts():
    """score_states (k_mlp<states, max>) over 29 M packed rows, about one N = 16 384 lookahead turn (765 persistent
    rounds), with device row counts below the buffer's: every row below the count equals the exact reference, every row
    at or past it keeps a sentinel.  The input repeats a 99 991-row period (not a multiple of the 128-row tile), so one
    period's float64 reference checks them all."""
    from gym_narde_b200.state import expand_obs198
    t0 = time.time()
    d = _cuda(EXACT_DESIGNS["sparse"]())
    mlp = _mlp(d)
    period = 99_991
    lo_p, hi_p = synthetic_states(period, 31)
    x = torch.from_numpy(expand_obs198(lo_p, hi_p)).cuda()
    q = check_premise(x, d["W"], d["b"])
    assert torch.equal(q, ref_q(x, d["W"], d["b"]))
    want = q.max(1).values.float()
    n = 29_000_000
    reps = -(-n // period)
    lo = torch.from_numpy(lo_p).cuda().repeat(reps, 1)[:n].contiguous()
    hi = torch.from_numpy(hi_p).cuda().repeat(reps, 1)[:n].contiguous()
    try:
        for rows in (n - 777, 8_388_608 + 129):
            out = _nan_buffer(n)
            mlp.score_states(lo, hi, out=out, rows_dev=torch.tensor([rows], dtype=torch.int64, device="cuda"))
            torch.cuda.synchronize()
            for r0 in range(0, rows, period):
                got = out[r0:min(r0 + period, rows)]
                bad = (got.view(torch.int32) != want[:got.shape[0]].view(torch.int32)).nonzero()
                assert len(bad) == 0, (rows, r0, len(bad), int(bad[0]))
            assert (out[rows:].view(torch.int32) == SENTINEL).all(), rows
            del out
    finally:
        del lo, hi
        torch.cuda.empty_cache()
    print("score_states: %d rows, %d periods, %.1f s" % (n, reps, time.time() - t0))


# ---------------------------------------------------------------------------------------------------------------
# the lookahead actor at the probe's settings
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,turns", [(4096, 4), (16384, 2)])
def test_lookahead_at_the_probe_settings_is_bit_exact(n, turns):
    """LookaheadActor(env, mlp, candidates=8) with cap and reply_cap 64 and default pools, an exact scorer, after 60
    random turns: choice, value and the action played equal _LookTurn bit for bit for every env (N = 4096: step() and
    step_graph() alternating; N = 16 384: step_graph()).  Every env was covered, the reply side batch scored rows, and
    lookahead played another action than greedy somewhere."""
    t0 = time.time()
    W, b = _design("sparse")
    env, actor = _look((W, b), n)
    seen = dict(turns=0, blocked=0, terminal=0, reply_side=0, beyond=0, differ=0)
    side_rows = reply_rows = 0
    for t in range(turns):
        lo, hi, dice = _play(env, actor, n > 4096 or t % 2 == 1)
        ref = _LookTurn(lo, hi, dice, K, W, b, premise=(t == 0))
        check_look_turn(ref, env, actor, CAP, CAP, seen, (n, t))
        side_rows += int(actor.reply_side.rows_dev.item())
        reply_rows += ref.reply_rows
    uncovered = actor.uncovered_envs()
    print("lookahead N=%d K=%d exact sparse: %s, reply rows %d, reply side-batch rows %d, positions %d, uncovered %d, "
          "%.1f s" % (n, K, seen, reply_rows, side_rows, actor.positions, uncovered, time.time() - t0))
    assert uncovered == 0
    assert side_rows > 0 and seen["reply_side"] > 0 and seen["differ"] > 0, (seen, side_rows)


def test_lookahead_at_the_probe_settings_with_the_probe_net():
    """The probe's seed-0 net at N = 4096, K = 8, default pools, two turns: check_look_bound over the actor's own
    candidates."""
    t0 = time.time()
    W, b = _net()
    env, actor = _look((W, b), 4096)
    decided = near = 0
    for t in range(2):
        lo, hi, dice = _play(env, actor, t == 1)
        cands = (actor.cand_idx.cpu().numpy(), actor.cand_count.cpu().numpy())
        ref = _LookTurn(lo, hi, dice, K, W, b, emulate=False, with_bound=True, cands=cands)
        d, e = check_look_bound(ref, actor, K, t)
        decided += d
        near += e
    uncovered = actor.uncovered_envs()
    print("lookahead N=4096 K=%d seed-0 net: %d env turns decided by more than 2B, %d near-ties, uncovered %d, %.1f s"
          % (K, decided, near, uncovered, time.time() - t0))
    assert uncovered == 0
    assert decided > 40


# ---------------------------------------------------------------------------------------------------------------
# sharding
# ---------------------------------------------------------------------------------------------------------------
def _same_shards(whole, halves, what):
    """whole: (env, actor) over every env; halves: two (env, actor) over the first and second half.  Every actor, each
    with its own default pools, has covered every env so far (when slots run out, which envs get one follows the order of
    atomics, so an uncovered env would make the comparison below depend on timing); states, the action played and the
    choice agree."""
    uncovered = [a.uncovered_envs() for _, a in [whole] + list(halves)]
    assert uncovered == [0, 0, 0], ("uncovered envs (whole, first half, second half)", what, uncovered)
    (env, actor), parts = whole, halves
    for name, get in (("lo", lambda e, a: e.lo), ("hi", lambda e, a: e.hi), ("chosen", lambda e, a: e.chosen),
                      ("choice", lambda e, a: a.choice)):
        a, b = get(env, actor), torch.cat([get(e, x) for e, x in parts])
        bad = (a != b).reshape(a.shape[0], -1).any(1).nonzero().flatten()
        assert len(bad) == 0, (name, what, len(bad), bad[:5].tolist())


def test_greedy_actor_does_not_depend_on_sharding():
    """config 5: one env of 65 536 games against two of 32 768 (env_base 0 and 32 768), each actor with its own default
    pools, 10 turns (step() and step_graph() alternating): every env covered, the same states, actions and choices."""
    t0 = time.time()
    W, b = _net()
    whole = _greedy((W, b), "max")
    halves = [_greedy((W, b), "max", n=E5 // 2, env_base=base) for base in (0, E5 // 2)]
    beyond = 0
    for t in range(10):
        for env, actor in [whole] + halves:
            _play(env, actor, t % 2 == 1)
        _same_shards(whole, halves, t)
        beyond += int((whole[1].choice >= CAP).sum().item())
    print("greedy sharding: %d env turns, %d choices beyond cap, uncovered 0 in every actor, %.1f s"
          % (10 * E5, beyond, time.time() - t0))
    assert beyond > 0


def test_lookahead_does_not_depend_on_sharding():
    """The probe's settings at N = 4096 (5 376 reply tiles) against two envs of 2048 (2 688 each), default pools, the
    seed-0 net, 3 turns: every env covered, the same states, actions and choices."""
    t0 = time.time()
    W, b = _net()
    whole = _look((W, b), 4096)
    halves = [_look((W, b), 2048, env_base=base) for base in (0, 2048)]
    differ = 0
    for t in range(3):
        for env, actor in [whole] + halves:
            _play(env, actor, t % 2 == 1)
        _same_shards(whole, halves, t)
        differ += int((whole[1].choice != whole[1].cand_idx[:, 0]).sum().item())
    print("lookahead sharding: %d env turns, %d where lookahead is not greedy, uncovered 0 in every actor, %.1f s"
          % (3 * 4096, differ, time.time() - t0))
    assert differ > 0
