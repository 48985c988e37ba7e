"""The afterstate actor's choice against the oracle and a float64 reference, and its segment, scan and side-batch kernels
at their edges.

- ref_choice() is the documented choice rule in numpy (include/narde_b200.h, narde_segment_argmax): the arg-max of
  sign * score over the first min(count, cap) entries, ties to the lowest index, an empty segment gives (0, 0), a NaN
  never beats a number and an all-NaN segment gives index 0 with its value.  The CPU tests pin it.
- (-m gpu) narde_segment_argmax / narde_segment_sample on hand-made scores at caps around the thread-per-env / warp-per-env
  switch; narde_afterstates_scan with a bounded row pool; narde_gather_overflow_clear + narde_scatter_choice directly.
- (-m gpu) AfterstateActor end to end: oracle afterstates (o_afterstates_batch) -> Box(198) on the host -> float64 net
  (ref_q of test_mlp_reference_cpu) -> ref_choice, with exact scorers (every choice, action and value bit for bit),
  a realistic scorer (within bound()), and a side batch too small for the turn.
"""
import numpy as np
import pytest
import torch

from test_mlp_reference_cpu import EXACT_DESIGNS, argmax_design, bound, check_premise, default_net, ref_q

NAN, INF = float("nan"), float("inf")


# ---------------------------------------------------------------------------------------------------------------
# host reference of the choice
# ---------------------------------------------------------------------------------------------------------------
def ref_choice(scores, counts, sign, cap):
    """(index int32 [n], value float32 [n]) of the choice per env.  scores: float32 [n, W], row i holding env i's
    segment from column 0 (W >= min(counts, cap)); sign: +1 / -1 per env.  Over the first c = min(count, cap) entries:
    the arg-max of sign * score with ties to the lowest index; a NaN never beats a number; all NaN -> index 0; c == 0
    -> (0, 0).  The value is the unsigned score of the chosen entry."""
    scores = np.asarray(scores, np.float32).reshape(len(counts), -1)
    c = np.clip(np.asarray(counts, np.int64), 0, cap)
    v = scores * np.asarray(sign, np.float32)[:, None]
    valid = np.arange(scores.shape[1])[None, :] < c[:, None]
    num = valid & ~np.isnan(v)
    with np.errstate(invalid="ignore"):
        top = np.where(num, v, -np.inf).max(1, initial=-np.inf)
        hit = num & (v == top[:, None])
    idx = np.where(hit.any(1), hit.argmax(1), 0).astype(np.int32)
    val = np.where(c > 0, scores[np.arange(len(c)), idx] if scores.shape[1] else 0.0, 0.0).astype(np.float32)
    return idx, val


def _loop_choice(scores, counts, sign, cap):
    """ref_choice written as the plain loop of the rule (checks the vectorised form)."""
    idx, val = np.zeros(len(counts), np.int32), np.zeros(len(counts), np.float32)
    for i, row in enumerate(scores):
        c = max(0, min(int(counts[i]), cap))
        best = None
        for k in range(c):
            x = np.float32(sign[i]) * np.float32(row[k])
            if np.isnan(x):
                continue
            if best is None or x > best[0]:
                best = (x, k)
        if c:
            idx[i] = 0 if best is None else best[1]
            val[i] = row[idx[i]]
    return idx, val


def same_floats(a, b):
    """Bit-equal float32 arrays, where a NaN matches any NaN (the payload of a NaN is not part of the contract)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(np.all((a.view(np.int32) == b.view(np.int32)) | (np.isnan(a) & np.isnan(b))))


def test_ref_choice_rule():
    s = np.float32
    cases = [  # (scores, count, sign, cap, index, value)
        ([1, 3, 3, 2], 4, 1, 64, 1, 3),                 # ties: lowest index
        ([1, 3, 3, 2], 4, -1, 64, 0, 1),                # BLACK to move in mode 1 takes the minimum
        ([1, 3, 5, 2], 2, 1, 64, 1, 3),                 # only the first `count`
        ([1, 3, 5, 2], 4, 1, 2, 1, 3),                  # only the first `cap`
        ([7, 8], 0, 1, 64, 0, 0),                       # empty
        ([NAN, 1, 2], 3, 1, 64, 2, 2),                  # NaN first loses
        ([0, NAN, 2], 3, 1, 64, 2, 2),
        ([NAN, NAN], 2, -1, 64, 0, NAN),                # all NaN: index 0 and its value
        ([NAN, -INF], 2, 1, 64, 1, -INF),               # -inf is a number
        ([-INF, -INF], 2, 1, 64, 0, -INF),
        ([1, INF, INF], 3, 1, 64, 1, INF),
        ([INF, 1, -INF], 3, -1, 64, 2, -INF),
        ([-1, -0.0, 0.0], 3, 1, 64, 1, -0.0),           # -0 == +0: the lower index, its own sign
        ([-1, 0.0, -0.0], 3, -1, 64, 0, -1),
        ([1, 0.0, -0.0], 3, -1, 64, 1, 0.0),
    ]
    for scores, count, sign, cap, k, v in cases:
        idx, val = ref_choice(np.array([scores], s), [count], [sign], cap)
        assert idx[0] == k and same_floats(val, [v]), (scores, count, sign, cap, idx[0], val[0])


def test_ref_choice_equals_the_plain_loop():
    rng = np.random.default_rng(1)
    n, w = 4000, 40
    sc = rng.integers(-3, 4, (n, w)).astype(np.float32)          # small integers: many ties
    sc[rng.random((n, w)) < 0.15] = NAN
    sc[rng.random((n, w)) < 0.05] = INF
    sc[rng.random((n, w)) < 0.05] = -INF
    sc[rng.random((n, w)) < 0.1] = -0.0
    sc[rng.random(n) < 0.05] = NAN                               # some all-NaN rows
    counts = rng.integers(0, w + 1, n)
    sign = rng.choice([-1, 1], n)
    for cap in (1, 7, 33, 64):
        a, b = ref_choice(sc, counts, sign, cap), _loop_choice(sc, counts, sign, cap)
        assert np.array_equal(a[0], b[0]) and same_floats(a[1], b[1]), cap


# ---------------------------------------------------------------------------------------------------------------
# (a) the segment kernels on hand-made scores
# ---------------------------------------------------------------------------------------------------------------
CAPS = (1, 31, 32, 33, 127, 128, 129, 256, 3072)
PATTERNS = ("equal", "lanes", "last", "inf", "all_neg_inf", "zeros_neg_first", "zeros_pos_first", "nan_first",
            "nan_lane", "all_nan", "nan_some", "random")


def _pattern(name, n, rng):
    """sign * score of a segment of n entries."""
    v = rng.standard_normal(n).astype(np.float32)
    if name == "equal":
        v[:] = 1.5
    elif name == "lanes":                       # equal maxima in different lanes: k, k + 32, k + 33
        v = -np.abs(v) - 1
        k = (n // 3) % 32 if n > 66 else 0
        for j in (k, k + 32, k + 33):
            if j < n:
                v[j] = 2.0
    elif name == "last":                        # the last lane of the last trip
        v = -np.abs(v) - 1
        v[n - 1] = 3.0
    elif name == "inf":
        v[::5] = -INF
        v[n // 2] = INF
        if n // 2 + 32 < n:
            v[n // 2 + 32] = INF
    elif name == "all_neg_inf":
        v[:] = -INF
    elif name.startswith("zeros"):
        v = -np.abs(v) - 1
        a, b = n // 4, (n // 2 if n > 2 else n - 1)
        v[b] = 0.0 if name == "zeros_neg_first" else -0.0
        v[a] = -0.0 if name == "zeros_neg_first" else 0.0
    elif name == "nan_first":
        v[0] = NAN
    elif name == "nan_lane":                    # a NaN first in its lane, the maximum later in the same lane
        v[:] = 0.0
        v[1 % n] = NAN
        v[33 if n > 33 else n - 1] = 5.0
    elif name == "all_nan":
        v[:] = NAN
    elif name == "nan_some":
        v[rng.random(n) < 0.2] = NAN
    return v


def _segments(cap, seed):
    """Envs of every (count, pattern, side to move): flat scores with a gap after each segment, and the dense rows of
    ref_choice.  The gap holds +inf in the mover's sign, so a read past the segment would win."""
    rng = np.random.default_rng(seed)
    counts = sorted({0, 1, cap - 1, cap, cap + 1, 3 * cap + 5})
    envs = [(c, p, t) for c in counts for p in PATTERNS for t in (1, -1)]
    n = len(envs)
    width = max(1, min(max(counts), cap))
    dense = np.zeros((n, width), np.float32)
    flat, offsets, cnt, turn, pats = [], np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int8), []
    at = 0
    for i, (c, p, t) in enumerate(envs):
        stored = min(c, cap)
        v = _pattern(p, max(stored, 1), rng)[:stored]
        offsets[i], cnt[i], turn[i] = at, c, t
        pats.append(p)
        flat.append(v)              # (the sign is applied per mode below)
        flat.append(np.full(1 + i % 3, INF, np.float32))
        at += stored + 1 + i % 3
        dense[i, :stored] = v
    return flat, dense, offsets, cnt, turn, pats


def _gpu_segments(flat, dense, offsets, counts, turn, mode):
    sign = np.where((turn == 1) | (mode == 0), 1.0, -1.0).astype(np.float32)
    sc = np.concatenate([part * sign[i // 2] for i, part in enumerate(flat)]).astype(np.float32)
    hi = np.zeros((len(counts), 16), np.uint8)
    hi[:, 10] = turn.view(np.uint8)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return sign, dense * sign[:, None], cu(sc), cu(offsets), cu(counts), cu(hi)   # (dense * sign: the stored rows)


def _run_argmax(score, off, cnt, hi, cap, mode):
    from gym_narde_b200 import _cabi
    n = cnt.shape[0]
    idx = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    val = torch.full((n,), 0x7FC0DEAD, dtype=torch.int32, device="cuda").view(torch.float32)
    _cabi.segment_argmax(score, off, cnt, hi, cap, mode, idx, val)
    return idx.cpu().numpy(), val.cpu().numpy()


def _run_sample(score, off, cnt, hi, cap, mode, params, env_idx=None, env_base=0, seed=0, step=0):
    from gym_narde_b200 import _cabi
    n = cnt.shape[0]
    idx = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    val = torch.full((n,), 0x7FC0DEAD, dtype=torch.int32, device="cuda").view(torch.float32)
    p = torch.tensor(params, dtype=torch.float32, device="cuda")
    _cabi.segment_sample(score, off, cnt, hi, cap, mode, env_base, seed, step, p, idx, val, env_idx=env_idx)
    return idx.cpu().numpy(), val.cpu().numpy()


def _mismatches(got, want, pats, counts, what):
    bad = [(pats[i], int(counts[i]), int(got[0][i]), float(got[1][i]), int(want[0][i]), float(want[1][i]))
           for i in range(len(pats)) if got[0][i] != want[0][i] or not same_floats(got[1][i:i + 1], want[1][i:i + 1])]
    return "%s: %d mismatches (pattern, count, kernel index, value, reference index, value): %s" % (what, len(bad), bad[:6])


@pytest.mark.gpu
@pytest.mark.parametrize("cap", CAPS)
def test_segment_kernels_on_hand_made_scores(cap):
    """narde_segment_argmax and narde_segment_sample ({0, 0}: greedy) equal ref_choice bit for bit on every pattern, count
    and side to move, in both modes; for cap <= 128 the warp-per-env kernel (the same segments launched with cap 129)
    equals the thread-per-env one.  narde_segment_sample {1, 0} (every env explores) plays the env's uniform action
    of the Philox stream and leaves the outputs of env_idx = -1 slots untouched."""
    from oracle import oracle as O
    flat, dense, offsets, counts, turn, pats = _segments(cap, cap)
    for mode in (0, 1):
        sign, raw, score, off, cnt, hi = _gpu_segments(flat, dense, offsets, counts, turn, mode)
        want = ref_choice(raw, counts, sign, cap)
        got = _run_argmax(score, off, cnt, hi, cap, mode)
        assert np.array_equal(got[0], want[0]) and same_floats(got[1], want[1]), _mismatches(
            got, want, pats, counts, "segment_argmax cap %d mode %d" % (cap, mode))
        got0 = _run_sample(score, off, cnt, hi, cap, mode, (0.0, 0.0), seed=5, step=9)
        assert np.array_equal(got0[0], got[0]) and same_floats(got0[1], got[1]), _mismatches(
            got0, want, pats, counts, "segment_sample {0, 0} cap %d mode %d" % (cap, mode))
        if cap <= 128:
            clamped = torch.clamp(cnt, max=cap)
            warp = _run_argmax(score, off, clamped, hi, 129, mode)
            assert np.array_equal(warp[0], got[0]) and same_floats(warp[1], got[1]), _mismatches(
                warp, got, pats, counts, "warp kernel vs thread kernel cap %d mode %d" % (cap, mode))
        # epsilon 1: every env with actions explores; slots of -1 are skipped
        n = len(counts)
        eidx = np.array([-1 if i % 5 == 3 else 1000 + 3 * i for i in range(n)], np.int32)
        env_base, seed, step = 7, 0xC0FFEE, 11
        got1 = _run_sample(score, off, cnt, hi, cap, mode, (1.0, 0.0), env_idx=torch.from_numpy(eidx).cuda(),
                           env_base=env_base, seed=seed, step=step)
        for i in range(n):
            c = min(int(counts[i]), cap)
            if eidx[i] < 0:
                assert got1[0][i] == -7 and got1[1][i:i + 1].view(np.int32)[0] == 0x7FC0DEAD, i
                continue
            z = O.turn_dice(seed, env_base + int(eidx[i]), step)[2]
            k = (z * c) >> 32 if c else 0
            v = raw[i, k] if c else np.float32(0)
            assert got1[0][i] == k and same_floats(got1[1][i:i + 1], [v]), (cap, mode, i, pats[i], got1[0][i], k)


@pytest.mark.gpu
@pytest.mark.parametrize("cap", (32, 128, 129, 3072))
def test_gumbel_sampler_never_picks_a_nan(cap):
    """narde_segment_sample with temperature 1: an index inside the segment whose score is a number whenever the segment
    has one (index 0 for an all-NaN segment), and the value of that index."""
    flat, dense, offsets, counts, turn, pats = _segments(cap, 100 + cap)
    for mode in (0, 1):
        sign, raw, score, off, cnt, hi = _gpu_segments(flat, dense, offsets, counts, turn, mode)
        for step in range(4):
            idx, val = _run_sample(score, off, cnt, hi, cap, mode, (0.0, 1.0), seed=3, step=step)
            for i in range(len(counts)):
                c = min(int(counts[i]), cap)
                if c == 0:
                    assert idx[i] == 0 and val[i] == 0, (cap, mode, i)
                    continue
                assert 0 <= idx[i] < c and same_floats(val[i:i + 1], raw[i, idx[i]:idx[i] + 1]), (cap, mode, i)
                if np.isnan(raw[i, :c]).all():
                    assert idx[i] == 0, (cap, mode, i, pats[i])
                else:
                    assert not np.isnan(raw[i, idx[i]]), (cap, mode, step, i, pats[i], int(idx[i]))


# ---------------------------------------------------------------------------------------------------------------
# (b) narde_afterstates_scan with a bounded row pool
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,cap", [(1, 12), (127, 64), (129, 12), (3000, 64), (131072, 12)])
def test_afterstates_scan_row_pool(n, cap):
    """offsets = exclusive prefix sums of min(counts, cap) (numpy), *rows_out clipped to rows_cap, counts_eff = 0 for every
    env whose rows do not all fit; rows below rows_cap equal the unbounded call's, rows at and beyond it keep a
    sentinel.  rows_cap: unbounded, 1, an env boundary, one row into an env, one past the total."""
    from gym_narde_b200 import VecNardeEnv, _cabi
    env = VecNardeEnv(n, seed=40 + n, max_actions=cap)
    env.reset()
    for _ in range(25):
        env.step()
    acts, counts, _ = env.get_valid_actions()
    c = np.minimum(counts.cpu().numpy(), cap).astype(np.int64)
    off = np.cumsum(c) - c
    total = int(c.sum())
    R = max(n * cap, total + 2)
    scratch = torch.zeros(n // 128 + 5, dtype=torch.int64, device="cuda")

    def run(rows_cap):
        lo2 = torch.full((R, 16), 0xAB, dtype=torch.uint8, device="cuda")
        hi2 = torch.full_like(lo2, 0xCD)
        offs = torch.full((n,), -7, dtype=torch.int64, device="cuda")
        rows = torch.full((1,), -5, dtype=torch.int64, device="cuda")
        ce = torch.full((n,), -9, dtype=torch.int32, device="cuda")
        _cabi.afterstates_scan(env.lo, env.hi, acts, counts, lo2, hi2, scratch, offsets=offs, rows_out=rows,
                               rows_cap=rows_cap, counts_eff=ce)
        return lo2.cpu().numpy(), hi2.cpu().numpy(), offs.cpu().numpy(), int(rows.item()), ce.cpu().numpy()

    lo0, hi0, off0, rows0, ce0 = run(0)
    assert np.array_equal(off0, off) and rows0 == total and np.array_equal(ce0, c)
    assert (lo0[total:] == 0xAB).all() and (hi0[total:] == 0xCD).all()
    mid = np.flatnonzero((off >= total // 2) & (c > 0))
    boundary = int(off[mid[0]]) if len(mid) and off[mid[0]] > 0 else total
    into = np.flatnonzero(c >= 2)
    one_in = int(off[into[len(into) // 2]]) + 1 if len(into) else 1
    for rc in sorted({1, boundary, one_in, total + 1}):
        lo2, hi2, off2, rows2, ce2 = run(rc)
        k = min(rc, total)
        assert np.array_equal(off2, off), rc
        assert rows2 == k, (rc, rows2, total)
        assert np.array_equal(ce2, np.where(off + c <= rc, c, 0)), rc
        assert np.array_equal(lo2[:k], lo0[:k]) and np.array_equal(hi2[:k], hi0[:k]), rc
        assert (lo2[k:] == 0xAB).all() and (hi2[k:] == 0xCD).all(), rc


# ---------------------------------------------------------------------------------------------------------------
# (c) the side batch's gather and scatter
# ---------------------------------------------------------------------------------------------------------------
FINISHED_HI = np.array([0] * 8 + [15, 0, 1, 4] + [0] * 4, np.uint8)   # off_w 15, WHITE, terminated (k_gather_overflow)


@pytest.mark.gpu
@pytest.mark.parametrize("m", (32, 64, 128))
def test_gather_and_scatter(m):
    """narde_gather_overflow_clear: every overflowing env at most once, all of them when they fit, exactly m otherwise,
    entry k in slot (k mod T) * 32 + k / T (T = m / 32; compared as sets: the order of entries follows atomics); unused
    slots are finished games with dice 0x0101 and index -1; act_override is zeroed; ctrl[2] grows by seen - m.
    narde_scatter_choice: only gathered envs change, slots with counts_eff == 0 are skipped and counted, slots with
    counts > cap are counted and still scattered, act_out is the chosen word, ctrl[0] is 0 again.  Calls repeat on the
    same ctrl buffer."""
    from gym_narde_b200 import _cabi
    rng = np.random.default_rng(m)
    n, cap = 1500, 48
    T = m // 32
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    ctrl = torch.zeros(4, dtype=torch.int32, device="cuda")
    missed = 0
    for rep, seen in enumerate((m - 5, m, m + 17, m - 1, 3 * m)):
        lo = rng.integers(0, 256, (n, 16), dtype=np.uint8)
        hi = rng.integers(0, 256, (n, 16), dtype=np.uint8)
        dice = rng.integers(1, 7, (n, 2), dtype=np.uint8)
        ovf = np.zeros(n, np.uint8)
        ovf[rng.choice(n, seen, replace=False)] = 1 + rng.integers(0, 3, seen)
        sub_lo = torch.full((m, 16), 0x5A, dtype=torch.uint8, device="cuda")
        sub_hi = torch.full_like(sub_lo, 0x5A)
        sub_dice = torch.full((m, 2), 9, dtype=torch.uint8, device="cuda")
        sub_idx = torch.full((m,), -3, dtype=torch.int32, device="cuda")
        act_override = torch.full((n,), 77, dtype=torch.int64, device="cuda")
        _cabi.gather_overflow(cu(lo), cu(hi), cu(dice), cu(ovf), sub_lo, sub_hi, sub_dice, sub_idx, ctrl,
                              act_override=act_override)
        g_idx, g_lo, g_hi, g_dice = (t.cpu().numpy() for t in (sub_idx, sub_lo, sub_hi, sub_dice))
        ctrl_g = ctrl.cpu().numpy()
        got = min(seen, m)
        missed += max(0, seen - m)
        assert ctrl_g[0] == seen and ctrl_g[1] == 0 and ctrl_g[2] == missed, (rep, ctrl_g)
        used = np.flatnonzero(g_idx >= 0)
        assert set(used.tolist()) == {(k % T) * 32 + k // T for k in range(got)}, rep
        envs = g_idx[used]
        assert len(set(envs.tolist())) == got and ovf[envs].all(), rep
        assert np.array_equal(g_lo[used], lo[envs]) and np.array_equal(g_hi[used], hi[envs]), rep
        assert np.array_equal(g_dice[used], dice[envs]), rep
        free = np.flatnonzero(g_idx < 0)
        assert (g_idx[free] == -1).all() and (g_lo[free] == 0).all() and (g_hi[free] == FINISHED_HI).all(), rep
        assert (g_dice[free] == 1).all(), rep
        assert int(act_override.abs().sum().item()) == 0, rep
        # scatter
        sub_choice = rng.integers(0, cap, m).astype(np.int32)
        sub_value = rng.standard_normal(m).astype(np.float32)
        eff = rng.integers(1, cap + 1, m).astype(np.int32)
        eff[rng.random(m) < 0.25] = 0
        sub_counts = rng.integers(1, 2 * cap, m).astype(np.int32)
        sub_actions = rng.integers(1, 2 ** 62, (m, cap), dtype=np.int64)
        choice = torch.full((n,), -4, dtype=torch.int32, device="cuda")
        value = torch.full((n,), -8.5, dtype=torch.float32, device="cuda")
        act_out = torch.full((n,), 5, dtype=torch.int64, device="cuda")
        _cabi.scatter_choice(cu(sub_choice), cu(sub_value), sub_idx, cu(eff), cu(sub_counts), cap, choice, value, ctrl,
                             cu(sub_actions), act_out)
        ch, va, ao, ctrl_s = (t.cpu().numpy() for t in (choice, value, act_out, ctrl))
        want_ch, want_va, want_ao = np.full(n, -4, np.int32), np.full(n, -8.5, np.float32), np.full(n, 5, np.int64)
        for s in used:
            if eff[s] == 0:
                missed += 1
                continue
            missed += int(sub_counts[s] > cap)
            i = g_idx[s]
            want_ch[i], want_va[i], want_ao[i] = sub_choice[s], sub_value[s], sub_actions[s, sub_choice[s]]
        assert np.array_equal(ch, want_ch) and same_floats(va, want_va) and np.array_equal(ao, want_ao), rep
        assert ctrl_s[0] == 0 and ctrl_s[1] == 0 and ctrl_s[2] == missed, (rep, ctrl_s, missed)


# ---------------------------------------------------------------------------------------------------------------
# (d, e, f) the actor end to end against the oracle and the float64 net
# ---------------------------------------------------------------------------------------------------------------
def _design(name):
    d = argmax_design() if name == "argmax" else EXACT_DESIGNS[name]()
    return tuple(w.cuda() for w in d["W"]), tuple(v.cuda() for v in d["b"])


class _Turn:
    """The oracle's view of one actor turn: the full legal lists of the positions before it and the float64 scores of
    every afterstate, row per (env, k)."""

    def __init__(self, lo, hi, dice, counts_dev, W, b, mode, emulate, premise=False, with_bound=False):
        from oracle import oracle as O
        from gym_narde_b200.state import expand_obs198
        self.counts = counts_dev.cpu().numpy()
        width = max(1, int(self.counts.max()))
        counts, self.acts, as_lo, as_hi = O.afterstates_batch(lo, hi, dice, cap=width)
        assert np.array_equal(counts, self.counts), "the enumeration's counts differ from the oracle's"
        mask = np.arange(width)[None, :] < counts[:, None]
        x = torch.from_numpy(expand_obs198(as_lo[mask], as_hi[mask])).cuda()
        if premise:
            check_premise(x, W, b)
        q = ref_q(x, W, b, emulate=emulate).max(1).values
        self.sign = np.where((mode == 1) & (hi[:, 10].view(np.int8) != 1), -1.0, 1.0).astype(np.float32)
        self.mask = mask
        self.q = np.zeros(mask.shape, np.float64)
        self.q[mask] = q.cpu().numpy()
        if with_bound:
            self.bnd = np.zeros(mask.shape, np.float64)
            self.bnd[mask] = bound(x, W, b).max(1).values.cpu().numpy()
        self.rows = int(mask.sum())

    def choice(self, cap=1 << 30, prefix=None):
        """ref_choice over each env's first min(count, cap) actions (prefix: per-env cap)."""
        sc = self.q.astype(np.float32)
        if prefix is None:
            return ref_choice(sc, self.counts, self.sign, cap)
        return ref_choice(sc, np.minimum(self.counts, prefix), self.sign, cap)


def _actor(design, cap, mode, n=3001, max_episode_steps=90, **kw):
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    W, b = design
    env = VecNardeEnv(n, seed=1234 + cap, max_actions=cap, max_episode_steps=max_episode_steps)
    mlp = AfterstateMLP(W[0], b[0], W[1], b[1], W[2], b[2])
    actor = AfterstateActor(env, mlp, mode=mode, **kw)
    env.reset()
    for _ in range(60):                       # random self-play: positions of every phase when the greedy turns start
        env.step()
    return env, actor


def _play(env, actor, graph):
    lo, hi = env.lo.cpu().numpy(), env.hi.cpu().numpy()
    actor.step_graph() if graph else actor.step()
    return lo, hi, actor.dice.cpu().numpy()


EXACT_RUNS = [("perm", 64, "max", False), ("sparse", 64, "white_value", True), ("argmax", 8, "white_value", False),
              ("perm", 8, "max", True)]


@pytest.mark.gpu
@pytest.mark.parametrize("design,cap,mode,graph", EXACT_RUNS)
def test_actor_plays_the_reference_choice_with_an_exact_scorer(design, cap, mode, graph):
    """An exact scorer (every afterstate score is a float32 value that any summation order reproduces): for every live env
    of every turn, the actor's choice is ref_choice over the oracle's full legal list scored by the float64 net, the action
    played is the oracle's action at that index, and value is the reference score bit for bit.  Cap 8 sends most lists
    through the side batch; 100 turns cross bear-offs, auto-resets and max_episode_steps truncations."""
    W, b = _design(design)
    m = 1 if mode == "white_value" else 0
    env, actor = _actor((W, b), cap, mode, overflow_slots=3072)
    checked = beyond = ends = truncs = bearoffs = 0
    for t in range(100):
        lo, hi, dice = _play(env, actor, graph)
        ref = _Turn(lo, hi, dice, env.counts, W, b, m, emulate=True, premise=(t % 25 == 0))
        choice, value, chosen = actor.choice.cpu().numpy(), actor.value.cpu().numpy(), env.chosen.cpu().numpy()
        want_k, want_v = ref.choice()
        live = ref.counts > 0
        bad = np.flatnonzero(live & (choice != want_k))
        assert len(bad) == 0, ("choice", design, cap, mode, t, len(bad), [(int(i), int(ref.counts[i]), int(choice[i]),
                                                                           int(want_k[i])) for i in bad[:5]])
        assert same_floats(value[live], want_v[live]), ("value", design, cap, mode, t)
        assert (choice[~live] == 0).all() and (value[~live] == 0).all(), t
        rows = np.flatnonzero(live)
        assert np.array_equal(chosen[rows], ref.acts[rows, want_k[rows]]), ("action", t)
        checked += len(rows)
        beyond += int((want_k[live] >= cap).sum())
        ends += int((env.done.cpu().numpy() != 0).sum())
        truncs += int((env.trunc.cpu().numpy() != 0).sum())
        half = (chosen[rows].astype(np.uint64)[:, None] >> np.arange(0, 64, 16, dtype=np.uint64)) & np.uint64(0xFFFF)
        bearoffs += int(((half != 0xFFFF) & ((half >> np.uint64(8)) == 255)).any(1).sum())
    assert actor.uncovered_envs() == 0
    assert ends > 0 and truncs > 0 and bearoffs > 0, (ends, truncs, bearoffs)
    if cap == 8:
        assert beyond > 100, beyond           # the side batch decided turns
    print("exact %s cap %d %s %s: %d env turns checked (%d choices beyond the stored list, %d games ended, %d truncated)"
          % (design, cap, mode, "step_graph" if graph else "step", checked, beyond, ends, truncs))


@pytest.mark.gpu
@pytest.mark.parametrize("scale", (1.0, 4.0))
def test_actor_with_a_realistic_scorer_is_within_the_bound(scale):
    """nn.Linear's default init (x1, x4): where the best plain-float64 score beats the second by more than twice bound(),
    the actor plays the reference's action; elsewhere the chosen action's score is within 2 * bound of the best; value
    is within bound() of the plain score of the chosen row."""
    W, b = default_net(0, scale)
    W, b = tuple(w.cuda() for w in W), tuple(v.cuda() for v in b)
    decided = near = 0
    for mode in ("max", "white_value"):
        env, actor = _actor((W, b), 64, mode, overflow_slots=3072)
        for t in range(25):
            lo, hi, dice = _play(env, actor, False)
            ref = _Turn(lo, hi, dice, env.counts, W, b, 1 if mode == "white_value" else 0, emulate=False, with_bound=True)
            choice, value = actor.choice.cpu().numpy(), actor.value.cpu().numpy().astype(np.float64)
            live = np.flatnonzero(ref.counts > 0)
            signed = np.where(ref.mask, ref.q * ref.sign[:, None], -np.inf)
            order = np.argsort(-signed, axis=1, kind="stable")
            best = signed[np.arange(len(signed)), order[:, 0]]
            second = np.where(ref.counts > 1, signed[np.arange(len(signed)), order[:, min(1, signed.shape[1] - 1)]],
                              -np.inf)
            lim = np.where(ref.mask, ref.bnd, 0).max(1)
            clear = best - second > 2 * lim
            for i in live:
                k = choice[i]
                assert 0 <= k < ref.counts[i], (mode, t, i)
                if clear[i]:
                    assert k == order[i, 0], (mode, t, i, k, order[i, 0], best[i] - second[i], lim[i])
                else:
                    assert signed[i, k] >= best[i] - 2 * lim[i], (mode, t, i)
                assert abs(value[i] - ref.q[i, k]) <= ref.bnd[i, k], (mode, t, i, value[i], ref.q[i, k], ref.bnd[i, k])
            decided += int(clear[live].sum())
            near += int((~clear[live]).sum())
        assert actor.uncovered_envs() == 0
    share = near / max(1, decided + near)
    print("realistic x%g: %d env turns decided by more than 2 bound, %d near-ties (%.4f)" % (scale, decided, near, share))
    assert decided > 10000


@pytest.mark.gpu
def test_actor_with_a_bounded_side_batch_scores_a_prefix_and_counts_it():
    """A side batch too small for the turn (128 slots for ~2500 overflowing envs, overflow_cap 40, a row pool that runs
    out mid-turn): every env plays either the full-list reference choice or the reference choice over the prefix it was
    scored on (its first max_actions or its first overflow_cap actions); envs of the second kind are no more than the
    growth of uncovered_envs(); the action played is always one of the oracle's legal actions."""
    W, b = _design("sparse")
    cap, ocap = 8, 40
    env, actor = _actor((W, b), cap, "white_value", overflow_slots=32, overflow_cap=ocap, overflow_rows=2000)
    assert actor.side.idx.shape[0] == 128
    checked = prefixed = 0
    before = actor.uncovered_envs()
    for t in range(40):
        lo, hi, dice = _play(env, actor, t % 2 == 1)
        ref = _Turn(lo, hi, dice, env.counts, W, b, 1, emulate=True)
        choice, value, chosen = actor.choice.cpu().numpy(), actor.value.cpu().numpy(), env.chosen.cpu().numpy()
        full, short, side = ref.choice(), ref.choice(prefix=cap), ref.choice(prefix=ocap)
        live = np.flatnonzero(ref.counts > 0)
        other = 0
        for i in live:
            k = choice[i]
            assert chosen[i] == ref.acts[i, k], (t, i)            # a legal action, the one at the chosen index
            assert same_floats(value[i:i + 1], ref.q[i, k:k + 1].astype(np.float32)), (t, i)
            if k == full[0][i]:
                continue
            assert k == short[0][i] or k == side[0][i], (t, i, k, full[0][i], short[0][i], side[0][i])
            other += 1
        after = actor.uncovered_envs()
        assert other <= after - before, (t, other, after - before)
        before = after
        checked += len(live)
        prefixed += other
    print("bounded side batch: %d env turns checked, %d decided on a prefix, %d uncovered" % (checked, prefixed, before))
    assert prefixed > 100
