"""Exploration of the afterstate actor (epsilon-greedy and softmax, narde_segment_sample).

The random words are recomputed on the host by a numpy Philox4x32-10 (checked against the oracle's, which the
Random123 known answers pin) with the stream layout of include/narde_b200.h: key = seed, counter = (global env id,
step_lo, step_hi, stream), stream 2 = the epsilon coin, 3 + (k << 8) = the Gumbel noise of action k, word z of
stream 0 = the env's own uniform action.  CPU tests run without a device; the rest are marked gpu."""
import math

import numpy as np
import pytest

M32 = np.uint64(0xFFFFFFFF)


def philox(c0, c1, c2, c3, seed):
    """Philox4x32-10 on uint32 arrays (broadcast); key = the 64-bit seed.  Returns the four words as uint64 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def words(seed, g, step, stream):
    return philox(g, step & 0xFFFFFFFF, step >> 32, stream, seed)


def explores(seed, g, step, eps):
    """The epsilon coin: (x >> 8) < floor(eps * 2^24), eps as the float32 the device reads."""
    return (words(seed, g, step, 2)[0] >> np.uint64(8)) < np.uint64(math.floor(float(np.float32(eps)) * 2.0 ** 24))


def uniform_index(seed, g, step, c):
    return ((words(seed, g, step, 0)[2] * np.asarray(c, dtype=np.uint64)) >> np.uint64(32)).astype(np.int64)


def gumbel64(seed, g, step, k):
    u = ((words(seed, g, step, 3 + (np.asarray(k, dtype=np.uint64) << np.uint64(8)))[0] >> np.uint64(9)).astype(np.float64)
         + 0.5) * 2.0 ** -23
    return -np.log(-np.log(u))


# -- CPU -------------------------------------------------------------------------------------
def test_numpy_philox_equals_the_oracle():
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    ctr = rng.integers(0, 2 ** 32, (64, 4), dtype=np.uint64)
    seeds = rng.integers(0, 2 ** 63, 64)
    for j in range(64):
        got = philox(*ctr[j], int(seeds[j]))
        want = O.philox4x32_10([int(x) for x in ctr[j]], [int(seeds[j]) & 0xFFFFFFFF, int(seeds[j]) >> 32])
        assert [int(w) for w in got] == want


def test_gumbel_uniform_stays_inside_the_open_interval_in_float32():
    for x in (0, (1 << 32) - 1):
        u = (np.float32(x >> 9) + np.float32(0.5)) * np.float32(2.0 ** -23)
        assert np.float32(0) < u < np.float32(1)
        assert np.isfinite(-np.log(-np.log(u)))


def test_segment_sample_wrapper_has_no_cpu_fallback():
    import torch
    from gym_narde_b200 import _cabi
    z = lambda dt, *shape: torch.zeros(shape, dtype=dt)
    n, cap, m = 4, 8, 32
    with pytest.raises(_cabi.NardeCudaError):
        _cabi.segment_sample(z(torch.float32, n * cap), z(torch.int64, n), z(torch.int32, n), z(torch.uint8, n, 16), cap, 0,
                             0, 1, 1, z(torch.float32, 2), z(torch.int32, n))
    with pytest.raises(_cabi.NardeCudaError):
        _cabi.gather_overflow(z(torch.uint8, n, 16), z(torch.uint8, n, 16), z(torch.uint8, n, 2), z(torch.uint8, n),
                              z(torch.uint8, m, 16), z(torch.uint8, m, 16), z(torch.uint8, m, 2), z(torch.int32, m),
                              z(torch.int32, 4), act_override=z(torch.int64, n))


def test_set_exploration_rejects_out_of_range_values():
    from gym_narde_b200 import AfterstateActor
    a = AfterstateActor.__new__(AfterstateActor)     # (the checks come before any device work)
    a.epsilon = a.temperature = 0.0
    for eps in (-0.1, 1.01, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            a.set_exploration(epsilon=eps)
    for tau in (-1.0, float("inf"), float("nan"), 1e-45):
        with pytest.raises(ValueError):
            a.set_exploration(temperature=tau)
    assert a.epsilon == 0.0 and a.temperature == 0.0


# -- GPU -------------------------------------------------------------------------------------
def _mlp():
    import torch
    import torch.nn as nn
    from gym_narde_b200 import AfterstateMLP
    torch.manual_seed(0)
    fn = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU()).cuda()
    head = nn.Linear(256, 576).cuda()
    return AfterstateMLP.from_module(fn, head)


def _same(a, b, t):
    import torch
    for name in ("lo", "hi", "obs", "reward", "done", "trunc", "chosen"):
        assert torch.equal(getattr(a, name), getattr(b, name)), (name, t)


@pytest.mark.gpu
def test_epsilon_one_plays_the_envs_own_random_policy():
    """epsilon=1: actor.step() and step_graph() play bit for bit what VecNardeEnv.step() plays without actions (at
    cap 8 most lists overflow: the side batch samples over the whole list)."""
    from gym_narde_b200 import VecNardeEnv, AfterstateActor
    mlp = _mlp()
    n, cap, base = 2048, 8, 3 * 2048
    a = VecNardeEnv(n, seed=17, max_actions=cap, env_base=base, max_episode_steps=60)
    b = VecNardeEnv(n, seed=17, max_actions=cap, env_base=base, max_episode_steps=60)
    actor = AfterstateActor(a, mlp, overflow_slots=n, overflow_rows=400 * n, epsilon=1.0)
    a.reset()
    b.reset()
    for t in range(100):
        if t % 3 == 0:
            actor.step()
        else:
            actor.step_graph()
        b.step()
        _same(a, b, t)
    assert a.episode_stats() == b.episode_stats() and a.episode_stats()["episodes"] > 0
    assert a.episode_stats()["overflows"] > 1000
    assert actor.uncovered_envs() == 0


@pytest.mark.gpu
def test_epsilon_coin_is_exact():
    """epsilon=0.3: the envs that explored are exactly the host's coin, they played the uniform index, and the others
    played narde_segment_argmax of the same scores; value = the chosen action's score."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateActor, _cabi
    mlp = _mlp()
    n, cap, base, seed = 4096, 64, 12345, 23
    for mode in ("max", "white_value"):
        env = VecNardeEnv(n, seed=seed, max_actions=cap, env_base=base)
        actor = AfterstateActor(env, mlp, mode=mode, overflow_slots=0, epsilon=0.3)
        env.reset()
        g = np.arange(n, dtype=np.uint64) + np.uint64(base)
        greedy = torch.zeros(n, dtype=torch.int32, device="cuda")
        explored_total = 0
        for t in range(40):
            step = env.step_count + 1
            choice, dice = actor.choose()
            _cabi.segment_argmax(actor.scores, actor.offsets, env.counts, env.hi, cap, actor.mode, greedy)
            c = env.counts.clamp(max=cap).cpu().numpy().astype(np.int64)
            got = choice.cpu().numpy().astype(np.int64)
            ex = explores(seed, g, step, 0.3) & (c > 0)
            assert np.array_equal(got[ex], uniform_index(seed, g, step, c)[ex]), (mode, t)
            assert np.array_equal(got[~ex], greedy.cpu().numpy()[~ex]), (mode, t)
            live = c > 0
            off = actor.offsets.cpu().numpy()
            sc = actor.scores.cpu().numpy()
            assert np.array_equal(actor.value.cpu().numpy()[live], sc[(off + got)[live]]), (mode, t)
            explored_total += int(ex.sum())
            env.step(choice, dice=dice)
        assert 0.27 < explored_total / (40 * n) < 0.33


def _host_sample(seed, g, step, scores, offsets, c, sign, inv_tau):
    """float64 Gumbel-max over ragged segments: (argmax, gap between the two best perturbed values, top value)."""
    m = len(c)
    K = int(c.sum())
    seg = np.repeat(np.arange(m), c)
    k = np.arange(K) - np.repeat(np.cumsum(c) - c, c)
    v = sign[seg] * scores[np.repeat(offsets, c) + k].astype(np.float64) * inv_tau + gumbel64(seed, g[seg], step, k)
    order = np.lexsort((k, -v, seg))          # per segment: best first, ties to the lowest index
    first = np.cumsum(c) - c
    best = order[first[c > 0]]
    idx = np.zeros(m, np.int64)
    top = np.zeros(m)
    gap = np.full(m, np.inf)
    idx[c > 0] = k[best]
    top[c > 0] = v[best]
    two = c > 1
    gap[two] = v[best[two[c > 0]]] - v[order[first[two] + 1]]
    return idx, gap, top


@pytest.mark.gpu
def test_softmax_agrees_with_a_float64_host_recomputation():
    """temperature 1 (epsilon 0): every choice, of the main pass and of the side batch (indices >= cap included), is
    the float64 Gumbel-max of the same scores and words, except near-ties (<= 0.1 % of the envs)."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateActor
    mlp = _mlp()
    n, cap, base, seed = 3072, 8, 777, 41
    for mode in ("max", "white_value"):
        env = VecNardeEnv(n, seed=seed, max_actions=cap, env_base=base)
        actor = AfterstateActor(env, mlp, mode=mode, overflow_slots=n, overflow_rows=400 * n, temperature=1.0)
        inv_tau = float(actor._params[1].item())
        env.reset()
        g = np.arange(n, dtype=np.uint64) + np.uint64(base)
        envs = near = beyond = 0
        for t in range(25):
            step = env.step_count + 1
            turn = env.hi[:, 10].view(torch.int8).cpu().numpy().astype(np.float64)
            sign = np.where(turn == 1, 1.0, -1.0) if mode == "white_value" else np.ones(n)
            choice, dice = actor.choose()
            got = choice.cpu().numpy().astype(np.int64)
            c = env.counts.clamp(max=cap).cpu().numpy().astype(np.int64)
            want, gap, top = _host_sample(seed, g, step, actor.scores.cpu().numpy(), actor.offsets.cpu().numpy(), c, sign,
                                          inv_tau)
            sb = actor.side
            slot_env = sb.idx.cpu().numpy().astype(np.int64)
            ce = sb.counts_eff.cpu().numpy().astype(np.int64)
            used = (slot_env >= 0) & (ce > 0)
            e = slot_env[used]
            sw, sgap, stop = _host_sample(seed, g[e], step, sb.scores.cpu().numpy(), sb.offsets.cpu().numpy()[used],
                                          ce[used], sign[e], inv_tau)
            want[e], gap[e], top[e] = sw, sgap, stop
            live = env.counts.cpu().numpy() > 0
            tie = gap <= 1e-4 * np.maximum(np.abs(top), 1.0)
            assert np.array_equal(got[live & ~tie], want[live & ~tie]), (mode, t)
            envs += int(live.sum())
            near += int((live & tie).sum())
            beyond += int((got[e] >= cap).sum())
            env.step(choice, dice=dice)
        assert near <= 0.001 * envs, (near, envs)
        assert beyond > 500, beyond
        assert actor.uncovered_envs() == 0


def _tv_bound(p, samples, envs):
    """E[TV] <= 1/2 sum_k sqrt(p_k (1 - p_k) / N), plus McDiarmid's deviation at 1e-6 / envs (one sample moves TV by
    at most 1/N)."""
    return 0.5 * np.sqrt(p * (1 - p) / samples).sum() + math.sqrt(math.log(envs / 1e-6) / (2 * samples))


@pytest.mark.gpu
def test_softmax_frequencies_match_the_distribution():
    """One turn's scores sampled at 4000 turn numbers: per env, the empirical frequencies are within a total-variation
    bound of softmax(sign * score / tau) (mixed with epsilon-uniform), for the thread kernel (cap 128) and the warp
    kernel (cap 256)."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateActor, _cabi
    mlp = _mlp()
    n, samples = 256, 4000
    env = VecNardeEnv(n, seed=8, max_actions=256)
    actor = AfterstateActor(env, mlp, mode="white_value")
    env.reset()
    for _ in range(6):
        env.step()
    actor.choose()
    counts, off = env.counts.cpu().numpy().astype(np.int64), actor.offsets.cpu().numpy()
    sc = actor.scores.cpu().numpy().astype(np.float64)
    turn = env.hi[:, 10].view(torch.int8).cpu().numpy()
    sign = np.where(turn == 1, 1.0, -1.0)
    spread = np.median([np.ptp(sc[off[i]:off[i] + min(counts[i], 256)]) for i in range(n) if counts[i] > 1])
    tau = float(spread) / 3.0                 # a few units of log-probability between the best and the worst action
    params = torch.zeros(2, dtype=torch.float32, device="cuda")
    out = torch.zeros((samples, n), dtype=torch.int32, device="cuda")
    checked = 0
    for cap in (128, 256):
        c = np.minimum(counts, cap)
        for eps in (0.0, 0.3):
            params.copy_(torch.tensor([eps, 1.0 / tau]))
            ptau = float(params[1].item())
            for s in range(samples):
                _cabi.segment_sample(actor.scores, actor.offsets, env.counts, env.hi, cap, 1, 0, 99, 1000 + s, params,
                                     out[s])
            got = out.cpu().numpy()
            for i in range(n):
                if c[i] < 2:
                    continue
                z = sign[i] * sc[off[i]:off[i] + c[i]] * ptau
                p = np.exp(z - z.max())
                p = (1 - eps) * p / p.sum() + eps / c[i]
                freq = np.bincount(got[:, i], minlength=c[i]) / samples
                assert len(freq) == c[i]
                tv = 0.5 * np.abs(freq - p).sum()
                assert tv < _tv_bound(p, samples, n), (cap, eps, i, tv)
                checked += 1
    assert checked > 4 * 200


@pytest.mark.gpu
def test_zero_parameters_are_the_greedy_choice():
    """narde_segment_sample with {0, 0}: index and value bit-equal to narde_segment_argmax, thread and warp kernels."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateActor, _cabi
    mlp = _mlp()
    n = 4096
    env = VecNardeEnv(n, seed=4, max_actions=256)
    actor = AfterstateActor(env, mlp)
    env.reset()
    for _ in range(10):
        env.step()
    actor.choose()
    params = torch.zeros(2, dtype=torch.float32, device="cuda")
    for cap in (64, 128, 256):
        for mode in (0, 1):
            i1, v1 = torch.full((n,), -3, dtype=torch.int32, device="cuda"), torch.full((n,), 7.0, device="cuda")
            i2, v2 = torch.full((n,), -4, dtype=torch.int32, device="cuda"), torch.full((n,), 8.0, device="cuda")
            _cabi.segment_argmax(actor.scores, actor.offsets, env.counts, env.hi, cap, mode, i1, v1)
            _cabi.segment_sample(actor.scores, actor.offsets, env.counts, env.hi, cap, mode, 0, 4, 11, params, i2, v2)
            assert torch.equal(i1, i2) and torch.equal(v1.view(torch.int32), v2.view(torch.int32)), (cap, mode)


@pytest.mark.gpu
def test_graph_replay_follows_the_exploration_schedule_without_recapture():
    """step_graph() with exploration equals eager step() turns given the same epsilon / temperature schedule; the
    switch greedy -> exploring recaptures once, later changes replay the same graph."""
    from gym_narde_b200 import VecNardeEnv, AfterstateActor
    mlp = _mlp()
    n, cap = 2048, 8
    envs = [VecNardeEnv(n, seed=13, max_actions=cap, env_base=n) for _ in range(2)]
    actors = [AfterstateActor(e, mlp, mode="white_value", overflow_slots=n, overflow_rows=400 * n) for e in envs]
    for e in envs:
        e.reset()
    schedule = [(0.0, 0.0)] * 3 + [(0.1, 0.0)] * 4 + [(0.1, 1.0)] * 4 + [(0.0, 0.05)] * 4 + [(0.5, 0.3)] * 4 + \
        [(1.0, 0.0)] * 3 + [(0.0, 0.0)] * 3 + [(0.05, 2.0)] * 5
    graphs = []
    for t, (eps, tau) in enumerate(schedule):
        for a in actors:
            a.set_exploration(epsilon=eps, temperature=tau)
        actors[0].step()
        actors[1].step_graph()
        graphs.append(actors[1]._graph)
        _same(envs[0], envs[1], t)
        assert np.array_equal(actors[0].value.cpu().numpy().view(np.int32), actors[1].value.cpu().numpy().view(np.int32))
    assert envs[0].episode_stats() == envs[1].episode_stats()
    assert graphs[0] is graphs[2] and graphs[3] is not graphs[0]
    assert all(gr is graphs[3] for gr in graphs[3:])
    assert actors[1].uncovered_envs() == 0


@pytest.mark.gpu
def test_exploration_does_not_depend_on_sharding():
    """Two half-size envs (env_base 0 and n/2) with exploration play the turns of one full env."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateActor
    mlp = _mlp()
    n, cap = 2048, 8
    full = VecNardeEnv(n, seed=29, max_actions=cap)
    halves = [VecNardeEnv(n // 2, seed=29, max_actions=cap, env_base=b) for b in (0, n // 2)]
    kw = dict(overflow_slots=n, overflow_rows=400 * n, epsilon=0.2, temperature=0.5)
    actors = [AfterstateActor(e, mlp, **kw) for e in [full] + halves]
    for e in [full] + halves:
        e.reset()
    for t in range(40):
        for a in actors:
            a.step()
        for name in ("lo", "hi", "chosen", "reward"):
            assert torch.equal(getattr(full, name), torch.cat([getattr(h, name) for h in halves])), (name, t)


@pytest.mark.gpu
def test_choose_then_env_step_leaves_no_stale_override():
    """choose() + VecNardeEnv.step(choice, dice) leaves the side batch's overrides unconsumed; a later actor.step() must
    not play them (the gather of the next turn clears them).  Against a twin that only uses choose() + env.step()."""
    from gym_narde_b200 import VecNardeEnv, AfterstateActor
    mlp = _mlp()
    n, cap = 2048, 6
    a = VecNardeEnv(n, seed=37, max_actions=cap)
    b = VecNardeEnv(n, seed=37, max_actions=cap)
    actor_a = AfterstateActor(a, mlp, overflow_slots=n, overflow_rows=400 * n)
    actor_b = AfterstateActor(b, mlp, overflow_slots=n, overflow_rows=400 * n)
    a.reset()
    b.reset()
    for t in range(40):
        if t % 2 == 0:
            choice, dice = actor_a.choose()
            a.step(choice, dice=dice)
        else:
            actor_a.step()
        choice, dice = actor_b.choose()
        b.step(choice, dice=dice)
        _same(a, b, t)
    assert actor_a.uncovered_envs() == 0
