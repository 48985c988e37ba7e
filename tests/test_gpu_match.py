"""AfterstateMatch (gym_narde_b200/match.py; narde_match_split_counts / narde_match_choose / narde_match_tally): lock-step
games between two policies with the results tallied on the device.

- The seat rule, the outcome and the tallies in numpy, against the host build of the kernels' helpers
  (tests/hostsim/match_hostsim.cpp); argument validation and the wrappers without a GPU.
- (-m gpu) the same net on both seats plays AfterstateActor's self-play; random against random plays VecNardeEnv.step().
- (-m gpu) two different exact nets, and a net against the random agent, to the end of every game against the oracle:
  every choice is ref_choice of the owner's float64 net over the oracle's full list (uniform_index for a random owner),
  the oracle replays the match from its choices, and the outcomes and tallies equal a host recount and the env's stats.
- (-m gpu) sharding over env_base and successive rounds.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from test_gpu_actor_reference import _Turn, _design, same_floats
from test_gpu_explore import uniform_index
from test_mlp_reference_cpu import default_net

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("games", "a_wins", "b_wins", "a_mars", "b_mars", "truncated", "a_white_wins", "b_white_wins", "plies")


# ---------------------------------------------------------------------------------------------------------------
# the rules in numpy
# ---------------------------------------------------------------------------------------------------------------
def a_colour(g):
    """A plays WHITE (+1) in even games, BLACK (-1) in odd ones."""
    return np.where(np.asarray(g) % 2 == 0, 1, -1)


def owner(g, turn):
    """0 when A owns the side to move, 1 when B does."""
    return np.where(np.asarray(turn) == a_colour(g), 0, 1)


def outcome_of(g, off_w, off_b, terminated, truncated):
    """The outcome code: 1 A won, 2 B won, 3 truncated, + 4 mars (the loser has none off); 0 running."""
    winner = np.where(np.asarray(off_w) == 15, 1, -1)
    code = np.where(winner == a_colour(g), 1, 2)
    mars = np.where(winner == 1, off_b, off_w) == 0
    code = code + 4 * mars
    return np.where(terminated, code, np.where(truncated, 3, 0)).astype(np.uint8)


def tallies_of(g, code, plies):
    code, g = np.asarray(code), np.asarray(g)
    r, done = code & 3, code != 0
    aw = a_colour(g) == 1
    return np.array([done.sum(), (r == 1).sum(), (r == 2).sum(), (code == 5).sum(), (code == 6).sum(), (r == 3).sum(),
                     ((r == 1) & aw).sum(), ((r == 2) & ~aw).sum(), np.where(done, plies, 0).sum()], np.int64)


def meta_of(off_w, off_b, turn, flags=0):
    return (np.asarray(off_w, np.uint32) | (np.asarray(off_b, np.uint32) << 8)
            | ((np.asarray(turn) & 0xFF).astype(np.uint32) << 16) | (np.uint32(flags) << 24)).astype(np.uint32)


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "hostsim", "match_hostsim.cpp")
    lib = str(tmp_path_factory.mktemp("match_hostsim") / "libmatch_hostsim.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", lib, src])
    L = C.CDLL(lib)
    L.hs_rule_sign.restype = C.c_float
    L.hs_rule_sign.argtypes = [C.c_int, C.c_uint32]
    L.hs_uniform_pick.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_int]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_hostsim_seat_rule_and_split(hostsim):
    rng = np.random.default_rng(1)
    n = 5000
    g = rng.integers(0, 1 << 40, n).astype(np.uint64)
    turn = rng.choice([-1, 1], n)
    meta = meta_of(rng.integers(0, 15, n), rng.integers(0, 15, n), turn)
    counts = rng.integers(0, 3000, n).astype(np.int32)
    want = owner(g.astype(np.int64), turn)
    assert abs(int((want == 0).sum()) - n // 2) < n // 10
    for kinds in range(4):
        own, ca, cb = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
        hostsim.hs_match_split(_p(g), _p(meta), _p(counts), C.c_int64(n), C.c_int(kinds), _p(own), _p(ca), _p(cb))
        assert np.array_equal(own, want)
        assert np.array_equal(ca, np.where((want == 0) & bool(kinds & 1), counts, 0)), kinds
        assert np.array_equal(cb, np.where((want == 1) & bool(kinds & 2), counts, 0)), kinds


def test_hostsim_outcome_and_tallies(hostsim):
    rng = np.random.default_rng(2)
    n = 6000
    g = rng.integers(0, 1 << 20, n).astype(np.uint64)
    winner_white = rng.random(n) < 0.5
    loser_off = np.where(rng.random(n) < 0.3, 0, rng.integers(1, 15, n))
    off_w = np.where(winner_white, 15, loser_off)
    off_b = np.where(winner_white, loser_off, 15)
    kind = rng.integers(0, 3, n)                       # 0 running, 1 terminated, 2 truncated
    off_w = np.where(kind == 1, off_w, rng.integers(0, 15, n))
    off_b = np.where(kind == 1, off_b, rng.integers(0, 15, n))
    term, trunc = (kind == 1).astype(np.uint8), (kind == 2).astype(np.uint8)
    meta = meta_of(off_w, off_b, rng.choice([-1, 1], n))
    plies = rng.integers(1, 1000, n).astype(np.int32)
    out, tal = np.zeros(n, np.uint8), np.zeros(9, np.int64)
    hostsim.hs_match_tally(_p(g), _p(meta), _p(term), _p(trunc), _p(plies), C.c_int64(n), _p(out), _p(tal))
    gi = g.astype(np.int64)
    want = outcome_of(gi, off_w, off_b, term != 0, trunc != 0)
    assert np.array_equal(out, want)
    assert set(np.unique(want)) == {0, 1, 2, 3, 5, 6}
    assert np.array_equal(tal, tallies_of(gi, want, plies))


def test_hostsim_sign_and_uniform_pick(hostsim):
    for mode in (0, 1):
        for turn in (1, -1):
            assert hostsim.hs_rule_sign(mode, int(meta_of(3, 4, turn))) == (-1.0 if mode == 1 and turn == -1 else 1.0)
    rng = np.random.default_rng(3)
    for _ in range(200):
        seed, g, step, c = int(rng.integers(0, 1 << 63)), int(rng.integers(0, 1 << 31)), int(rng.integers(0, 1 << 40)), \
            int(rng.integers(1, 4000))
        assert hostsim.hs_uniform_pick(seed, g, step, c) == int(uniform_index(seed, g, step, c))


def test_argument_validation_without_a_gpu():
    from gym_narde_b200 import AfterstateMatch, AfterstateMLP
    net = AfterstateMLP.__new__(AfterstateMLP)          # (validation only looks at the type)
    bad = [dict(policy_a="random", policy_b="random", mode_a="max"),
           dict(policy_a=net, policy_b="random", mode_b="white_value"),
           dict(policy_a=net, policy_b=net, mode_a="min"),
           dict(policy_a="greedy", policy_b="random"),
           dict(policy_a=object(), policy_b="random"),
           dict(policy_a="random", policy_b="random", num_games=0),
           dict(policy_a="random", policy_b="random", max_episode_steps=0)]
    for kw in bad:
        kw.setdefault("num_games", 4)
        with pytest.raises(ValueError):
            AfterstateMatch(**kw)


def test_match_wrappers_have_no_cpu_fallback():
    from gym_narde_b200 import _cabi
    u8, i32, i64, f32 = torch.uint8, torch.int32, torch.int64, torch.float32
    z = lambda dt, *shape: torch.zeros(shape, dtype=dt)
    n = 4
    hi, counts = z(u8, n, 16), z(i32, n)
    pool = (z(f32, 32), z(i64, n), z(i32, n))
    calls = [("match_split_counts", (hi, counts, 0, 3, z(i32, n), z(i32, n))),
             ("match_choose", (hi, counts, 8, 0, 0, 3, (0, 1), (pool, pool), z(i32, n), z(f32, n))),
             ("match_choose", (hi, counts, 8, 0, 0, 0, (0, 0), (None, None), z(i32, n), z(f32, n))),
             ("match_tally", (hi, z(u8, n), z(u8, n), 0, z(u8, n), z(i64, 9)))]
    for name, args in calls:
        with pytest.raises(_cabi.NardeCudaError):
            getattr(_cabi, name)(*args)
    with pytest.raises(_cabi.NardeCudaError):   # a net seat without its pool
        _cabi.match_choose(hi, counts, 8, 0, 0, 1, (0, 0), (None, None), z(i32, n), z(f32, n))
    lib = _cabi.load()
    assert lib.narde_match_split_counts(None, None, 0, 0, None, 0, None, None, None) == 0
    assert lib.narde_match_split_counts(None, None, 4, 0, None, 0, None, None, None) == -1
    assert lib.narde_match_choose(None, None, 4, 8, 0, None, 0, 0, None, 0, 0, 0, *([None] * 6), None, None, None,
                                  None) == -1
    assert lib.narde_match_tally(None, None, None, 4, 0, None, None, None) == -1


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _mlp(design):
    from gym_narde_b200 import AfterstateMLP
    W, b = design
    return AfterstateMLP(W[0], b[0], W[1], b[1], W[2], b[2])


def _cuda_net(seed):
    W, b = default_net(seed, 1.0)
    return tuple(w.cuda() for w in W), tuple(v.cuda() for v in b)


SELFPLAY_RUNS = [(8, "max", False), (8, "white_value", True), (64, "max", True), (64, "white_value", False)]


@pytest.mark.gpu
@pytest.mark.parametrize("cap,mode,graph", SELFPLAY_RUNS)
def test_same_net_on_both_seats_is_selfplay(cap, mode, graph):
    """AfterstateMatch(net, net) plays AfterstateActor(net, mode)'s self-play: after 60 identical random turns, 40 turns
    with the same states, choices, values and played actions, bit for bit (the same tcgen05 scorer on the same rows)."""
    from gym_narde_b200 import AfterstateActor, AfterstateMatch, VecNardeEnv
    n, seed = 2000, 77 + cap
    net = _mlp(_cuda_net(0))
    match = AfterstateMatch(n, net, net, seed=seed, mode_a=mode, mode_b=mode, max_actions=cap, overflow_slots=n)
    env = VecNardeEnv(n, seed=seed, autoreset=False, max_actions=cap)
    actor = AfterstateActor(env, net, mode=mode, overflow_slots=n)
    env.reset()
    for _ in range(60):
        env.step()
        match.env.step()
    beyond = 0
    for t in range(40):
        actor.step_graph() if graph else actor.step()
        match.step_graph() if graph else match.step()
        assert torch.equal(env.lo, match.env.lo) and torch.equal(env.hi, match.env.hi), t
        live = env.counts > 0
        assert torch.equal(env.counts, match.env.counts), t
        assert torch.equal(actor.choice[live], match.choice[live]), t
        assert same_floats(actor.value[live].cpu().numpy(), match.value[live].cpu().numpy()), t
        assert torch.equal(env.chosen, match.env.chosen), t
        beyond += int((match.choice[live] >= cap).sum())
    assert actor.uncovered_envs() == 0 and match.uncovered_envs() == 0
    if cap == 8:
        assert beyond > 100, beyond


def _flags_masked(hi, trunc):
    """hi planes with FLAG_DONE cleared where a game was truncated (the match freezes those, the env does not)."""
    hi = hi.copy()
    hi[trunc, 11] &= ~np.uint8(4)
    return hi


@pytest.mark.gpu
def test_random_against_random_is_the_env_step():
    """Random against random is VecNardeEnv.step()'s uniform policy: bit-equal states and played actions of every running
    game until every game has ended (terminated, or truncated at 80 turns)."""
    from gym_narde_b200 import AfterstateMatch, VecNardeEnv
    n, seed, T = 3000, 11, 80
    match = AfterstateMatch(n, "random", "random", seed=seed, max_actions=8, max_episode_steps=T, overflow_slots=n)
    env = VecNardeEnv(n, seed=seed, autoreset=False, max_actions=8, max_episode_steps=T)
    env.reset()
    for t in range(T):
        running = match.outcome.cpu().numpy() == 0
        if not running.any():
            break
        env.step()
        match.step() if t % 2 else match.step_graph()
        trunc = env.trunc.cpu().numpy() != 0
        r = np.flatnonzero(running)
        assert np.array_equal(env.lo.cpu().numpy()[r], match.env.lo.cpu().numpy()[r]), t
        assert np.array_equal(env.hi.cpu().numpy()[r], _flags_masked(match.env.hi.cpu().numpy(), trunc)[r]), t
        assert np.array_equal(env.chosen.cpu().numpy()[r], match.env.chosen.cpu().numpy()[r]), t
    out = match.outcome.cpu().numpy()
    assert (out != 0).all() and (out == 3).any() and ((out & 3) != 3).any(), np.bincount(out)
    assert match.uncovered_envs() == 0


def _oracle_match(net_a, net_b, n, T, seed):
    """Play a match to the end of every game, checking each turn's choices against the oracle's full lists and the
    owner's float64 net (ref_choice; uniform_index for a random owner).  Returns the per-turn choices, the match, the
    per-turn record of the running games and its counts."""
    from oracle import oracle as O
    from gym_narde_b200 import AfterstateMatch
    seats = []
    for spec in (net_a, net_b):
        if spec == "random":
            seats.append(("random", None, None))
        else:
            design, mode = spec
            W, b = _design(design)
            seats.append((_mlp((W, b)), (W, b), mode))
    match = AfterstateMatch(n, seats[0][0], seats[1][0], seed=seed, mode_a=seats[0][2], mode_b=seats[1][2],
                            max_episode_steps=T, overflow_slots=n)
    env = match.env
    g = np.arange(n)
    words, rec, live_turns, random_turns, beyond = [], [], 0, 0, 0
    for t in range(1, T + 1):
        running = match.outcome.cpu().numpy() == 0
        if not running.any():
            break
        lo, hi = env.lo.cpu().numpy(), env.hi.cpu().numpy()
        match.step_graph() if t % 2 else match.step()
        dice, counts = match.dice.cpu().numpy(), env.counts.cpu().numpy()
        choice, value, chosen = match.choice.cpu().numpy(), match.value.cpu().numpy(), env.chosen.cpu().numpy()
        words.append(choice.copy())
        rec.append((running, env.lo.cpu().numpy(), env.hi.cpu().numpy(), env.done.cpu().numpy(), env.trunc.cpu().numpy(),
                    env.reward.cpu().numpy()))
        turn = hi[:, 10].view(np.int8)
        own = owner(g, turn)
        live = running & (counts > 0)
        for p, (pol, Wb, mode) in enumerate(seats):
            sel = np.flatnonzero(live & (own == p))
            if len(sel) == 0:
                continue
            if pol == "random":
                width = int(counts[sel].max())
                ocounts, acts, _, _ = O.afterstates_batch(lo[sel], hi[sel], dice[sel], cap=width)
                assert np.array_equal(ocounts, counts[sel]), t
                want = uniform_index(seed, sel, t, counts[sel])
                assert np.array_equal(choice[sel], want), (t, "random")
                assert (value[sel] == 0).all()
                random_turns += len(sel)
            else:
                ref = _Turn(lo[sel], hi[sel], dice[sel], torch.from_numpy(counts[sel]), Wb[0], Wb[1],
                            1 if mode == "white_value" else 0, emulate=True)
                want, want_v = ref.choice()
                bad = np.flatnonzero(choice[sel] != want)
                assert len(bad) == 0, (t, p, [(int(sel[i]), int(choice[sel[i]]), int(want[i])) for i in bad[:5]])
                assert same_floats(value[sel], want_v), (t, p)
                acts = ref.acts
            assert np.array_equal(chosen[sel], acts[np.arange(len(sel)), want]), (t, p, "action")
            beyond += int((want >= match.cap).sum())
            live_turns += len(sel)
    assert (match.outcome.cpu().numpy() != 0).all()
    assert match.uncovered_envs() == 0
    return np.array(words, np.int32), match, rec, (live_turns, random_turns, beyond)


def _check_against_trace(words, match, rec, seed, T):
    """The oracle replays the match from its choices (autoreset off): the same states, done bits and rewards of every
    running game on every turn; the outcomes and tallies equal a host recount and agree with the env's own statistics."""
    from oracle import oracle as O
    env, n = match.env, match.num_games
    tr = O.selfplay_trace(seed, 0, n, len(words), words=words, word_mode=0, autoreset=False, max_episode_steps=T)
    g = np.arange(n)
    for t, (running, lo, hi, done, trunc, reward) in enumerate(rec):
        r = np.flatnonzero(running)
        d = tr["done"][t][r]
        assert np.array_equal(tr["lo"][t][r], lo[r]), t
        assert np.array_equal(tr["hi"][t][r], _flags_masked(hi, trunc != 0)[r]), t
        assert np.array_equal(d & 1, done[r]) and np.array_equal((d >> 1) & 1, trunc[r]), t
        assert np.array_equal(tr["reward"][t][r], reward[r]), t
    # replay the match turn by turn on the host from the trace: the outcome of each game is fixed by its first done turn
    out = np.zeros(n, np.uint8)
    plies = np.zeros(n, np.int64)
    for t in range(len(words)):
        d = tr["done"][t]
        new = (out == 0) & (d != 0)
        hi = tr["hi"][t]
        code = outcome_of(g, hi[:, 8], hi[:, 9], (d & 1) != 0, (d & 2) != 0)
        out = np.where(new, code, out)
        plies = np.where(new, t + 1, plies)
    assert (out != 0).all()
    assert np.array_equal(out, match.outcome.cpu().numpy())
    tallies = tallies_of(g, out, plies)
    got = match.tallies.cpu().numpy()
    assert np.array_equal(got, tallies), (got, tallies)
    res = match.results()
    assert [res[k] for k in NAMES] == tallies.tolist()
    st = env.episode_stats()
    assert st["episodes"] == tallies[0] and st["white_wins"] + st["black_wins"] == tallies[1] + tallies[2]
    assert st["mars"] == tallies[3] + tallies[4] and st["episode_steps"] == tallies[8]
    # the final states: every game stopped at its end (a truncated one frozen), as the trace's state at its end turn
    end = plies - 1
    lo_end, hi_end = tr["lo"][end, g], tr["hi"][end, g]
    trunc = out == 3
    assert np.array_equal(env.lo.cpu().numpy(), lo_end)
    assert np.array_equal(_flags_masked(env.hi.cpu().numpy(), trunc), hi_end)
    return tr, out


@pytest.mark.gpu
@pytest.mark.parametrize("a,b", [(("perm", "max"), ("sparse", "white_value")), (("sparse", "white_value"), "random")],
                         ids=["net_vs_net", "net_vs_random"])
def test_match_against_the_oracle(a, b):
    """Two exact nets in different modes, and an exact net against the random agent, 3000 games to the end of every game
    (90 turns at most: truncations occur): every live env turn's choice, value and played action is the reference's;
    the oracle's replay from the match's choices, the outcomes, the tallies and the env's statistics agree."""
    n, T, seed = 3000, 90, 4242
    words, match, rec, (live, rnd, beyond) = _oracle_match(a, b, n, T, seed)
    tr, out = _check_against_trace(words, match, rec, seed, T)
    assert (out == 3).any() and ((out & 3) != 3).any(), np.bincount(out)
    if b == "random":
        assert rnd > 0
    assert beyond > 0
    print("%s vs %s: %d env turns checked (%d random), %d choices beyond the stored list, outcomes %s, %s"
          % (a, b, live, rnd, beyond, np.bincount(out, minlength=8).tolist(), match.results()))


@pytest.mark.gpu
def test_sharded_matches_give_the_same_outcomes():
    """Two half-size matches (env_base 0 and N/2) play the same games as one full match: the same outcomes and, summed,
    the same tallies."""
    from gym_narde_b200 import AfterstateMatch
    n, T = 4096, 120
    na, nb = _mlp(_cuda_net(0)), _mlp(_cuda_net(1))
    full = AfterstateMatch(n, na, nb, seed=5, mode_a="max", max_episode_steps=T)
    rf = full.play()
    halves = [AfterstateMatch(n // 2, na, nb, seed=5, mode_a="max", max_episode_steps=T, env_base=b) for b in (0, n // 2)]
    rh = [h.play() for h in halves]
    assert full.uncovered_envs() == 0 and all(h.uncovered_envs() == 0 for h in halves)
    assert torch.equal(full.outcome, torch.cat([h.outcome for h in halves]))
    for k in NAMES:
        assert rf[k] == rh[0][k] + rh[1][k], k
    assert rf["games"] == n


@pytest.mark.gpu
def test_rounds_play_new_games_reproducibly():
    """Two rounds of play() give different games; a second match with the same seed reproduces both; results() is their
    sum."""
    from gym_narde_b200 import AfterstateMatch
    net = _mlp(_cuda_net(0))
    runs = []
    for _ in range(2):
        m = AfterstateMatch(1024, net, "random", seed=9, max_episode_steps=80)
        rounds = []
        for _ in range(2):
            r = m.play()
            rounds.append((r, m.outcome.clone()))
        runs.append((rounds, m.results()))
    (r0, o0), (r1, o1) = runs[0][0]
    assert r0["games"] == r1["games"] == 1024
    assert not torch.equal(o0, o1) or r0["plies"] != r1["plies"]
    for (ra, oa), (rb, ob) in zip(runs[0][0], runs[1][0]):
        assert ra == rb and torch.equal(oa, ob)
    total = runs[0][1]
    for k in NAMES:
        assert total[k] == r0[k] + r1[k], k
    assert total["a_points"] == total["a_wins"] + total["a_mars"]
    lo, hi = total["a_win_share_ci95"]
    assert lo <= total["a_win_share"] <= hi
