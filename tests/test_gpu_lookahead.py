"""The one-ply expectimax lookahead (include/narde_b200.h: narde_segment_topk, narde_lookahead_expand,
narde_lookahead_reduce; gym_narde_b200.LookaheadActor) against a numpy statement of its rule and the oracle.

- ref_topk / ref_values / ref_choice (test_gpu_actor_reference) are the rule in numpy, checked against plain loops and
  against the host build of the kernels' helpers (tests/hostsim/lookahead_hostsim.cpp).
- (-m gpu) the three kernels on hand-made inputs.
- (-m gpu) LookaheadActor end to end: the oracle's full legal lists (o_afterstates_batch) of every position and of every
  (candidate, roll) reply position, scored by the float64 net (ref_q of test_mlp_reference_cpu), through the numpy rule:
  with exact scorers bit for bit, with a realistic scorer within bound(), and with pools too small for the turn.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from test_gpu_actor_reference import _gpu_segments, _segments, ref_choice, same_floats
from test_mlp_reference_cpu import EXACT_DESIGNS, argmax_design, bound, check_premise, default_net, ref_q

NAN, INF = float("nan"), float("inf")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLLS = [(a, b) for a in range(1, 7) for b in range(a, 7)]
WEIGHTS = np.array([1.0 if a == b else 2.0 for a, b in ROLLS], np.float32)
FINISHED_HI = np.array([0] * 8 + [15, 0, 1, 4] + [0] * 4, np.uint8)   # off_w 15, WHITE, terminated


# ---------------------------------------------------------------------------------------------------------------
# the rule in numpy
# ---------------------------------------------------------------------------------------------------------------
def ref_topk(scores, counts, sign, K):
    """Step 1: (idx int32 [n, K], -1 beyond got; got int32 [n]) -- the first min(K, count) entries of each row of
    sign * scores in the order of the choice rule: numbers before NaN, larger first, ties (-0 == +0, NaN and NaN) to the
    lower index."""
    scores = np.asarray(scores, np.float32)
    n, w = scores.shape
    c = np.asarray(counts, np.int64)
    v = scores * np.asarray(sign, np.float32)[:, None]
    k = np.broadcast_to(np.arange(w), (n, w))
    valid = k < c[:, None]
    cat = np.where(~valid, 2, np.where(np.isnan(v), 1, 0))
    key = np.where(cat == 0, -v, 0.0).astype(np.float64)
    key[key == 0] = 0.0                                              # -0 and +0 sort as equals
    order = np.lexsort((k, key, cat), axis=1)[:, :K]
    got = np.minimum(c, K).astype(np.int32)
    idx = np.where(np.arange(order.shape[1])[None, :] < got[:, None], order, -1).astype(np.int32)
    if idx.shape[1] < K:
        idx = np.concatenate([idx, np.full((n, K - idx.shape[1]), -1, np.int32)], 1)
    return idx, got


def _loop_topk(scores, counts, sign, K):
    """ref_topk as repeated plain-loop arg-max rounds, each over the entries after the previous pick."""
    def before(v, k, w, j):
        if np.isnan(v) != np.isnan(w):
            return not np.isnan(v)
        if np.isnan(v) or v == w:
            return k < j
        return v > w
    n = len(counts)
    idx, got = np.full((n, K), -1, np.int32), np.zeros(n, np.int32)
    for i in range(n):
        prev = None
        for r in range(K):
            best = None
            for k in range(int(counts[i])):
                v = np.float32(sign[i]) * np.float32(scores[i][k])
                if prev is not None and not before(prev[0], prev[1], v, k):
                    continue
                if best is None or before(v, k, best[0], best[1]):
                    best = (v, k)
            if best is None:
                break
            idx[i, r], prev = best[1], best
            got[i] = r + 1
    return idx, got


def ref_values(s0, terminal, r, count, eff):
    """Step 3 per candidate: (v float32 [c], unfit bool [c]) from s0 [c], terminal [c] and r / count / eff [c, 21]."""
    s0 = np.asarray(s0, np.float32)
    acc = np.zeros(len(s0), np.float32)
    unfit = np.zeros(len(s0), bool)
    for d in range(21):
        x = np.where(count[:, d] == 0, s0, np.asarray(r[:, d], np.float32)).astype(np.float32)
        unfit |= (count[:, d] > 0) & (eff[:, d] < count[:, d])
        acc = (acc + WEIGHTS[d] * x).astype(np.float32)
    unfit &= ~np.asarray(terminal, bool)
    with np.errstate(invalid="ignore"):
        v = np.where(terminal, s0, np.where(unfit, np.float32(NAN), acc / np.float32(36.0))).astype(np.float32)
    return v, unfit


def _loop_values(s0, terminal, r, count, eff):
    v, unfit = np.zeros(len(s0), np.float32), np.zeros(len(s0), bool)
    for c in range(len(s0)):
        if terminal[c]:
            v[c] = s0[c]
            continue
        acc = np.float32(0)
        for d, (a, b) in enumerate(ROLLS):
            if count[c, d] == 0:
                x = np.float32(s0[c])
            elif eff[c, d] < count[c, d]:
                unfit[c] = True
                continue
            else:
                x = np.float32(r[c, d])
            acc = np.float32(acc + np.float32(1 if a == b else 2) * x)
        v[c] = np.float32(NAN) if unfit[c] else np.float32(acc / np.float32(36))
    return v, unfit


def ref_pick(v, got, sign):
    """Step 4: the slot per env -- ref_choice over the candidates' v (a NaN never wins, all NaN -> slot 0)."""
    return ref_choice(v, got, sign, v.shape[1])[0]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the rule, the roll table and the host build of the kernels' helpers
# ---------------------------------------------------------------------------------------------------------------
def test_roll_table():
    assert len(ROLLS) == 21 and len(set(ROLLS)) == 21 and WEIGHTS.sum() == 36
    assert ROLLS[0] == (1, 1) and ROLLS[1] == (1, 2) and ROLLS[6] == (2, 2) and ROLLS[-1] == (6, 6)
    outcomes = {}
    for a in range(1, 7):
        for b in range(1, 7):
            outcomes[tuple(sorted((a, b)))] = outcomes.get(tuple(sorted((a, b))), 0) + 1
    assert [outcomes[r] for r in ROLLS] == WEIGHTS.astype(int).tolist()


def _random_scores(rng, n, w):
    sc = rng.integers(-3, 4, (n, w)).astype(np.float32)          # small integers: many ties
    sc[rng.random((n, w)) < 0.15] = NAN
    sc[rng.random((n, w)) < 0.05] = INF
    sc[rng.random((n, w)) < 0.05] = -INF
    sc[rng.random((n, w)) < 0.1] = -0.0
    sc[rng.random(n) < 0.05] = NAN                               # some all-NaN rows
    return sc


def test_ref_topk_equals_the_plain_loop_and_starts_with_the_choice():
    rng = np.random.default_rng(3)
    n, w = 1500, 40
    sc = _random_scores(rng, n, w)
    counts = rng.integers(0, w + 1, n)
    sign = rng.choice([-1, 1], n)
    for K in (1, 2, 7, 32, 45):
        a, b = ref_topk(sc, counts, sign, K), _loop_topk(sc, counts, sign, K)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), K
        live = counts > 0
        assert np.array_equal(a[0][live, 0], ref_choice(sc, counts, sign, w)[0][live]), K


def _random_replies(rng, n):
    s0 = rng.integers(-4, 5, n).astype(np.float32) * np.float32(0.25)
    s0[rng.random(n) < 0.05] = NAN
    terminal = rng.random(n) < 0.1
    r = (rng.integers(-8, 9, (n, 21)) * 0.125).astype(np.float32)
    r[rng.random((n, 21)) < 0.01] = NAN
    count = rng.integers(1, 40, (n, 21)).astype(np.int32)
    count[rng.random((n, 21)) < 0.08] = 0                         # blocked rolls
    eff = count.copy()
    eff[rng.random((n, 21)) < 0.01] = 0                           # rows did not fit
    short = rng.random((n, 21)) < 0.01
    eff[short] = np.minimum(eff[short], 8)                        # a prefix only (reply side batch missed it)
    count[rng.random(n) < 0.05] = 0                               # every roll blocked
    return s0, terminal, r, count, eff


def test_ref_values_equal_the_plain_loop():
    rng = np.random.default_rng(4)
    s0, terminal, r, count, eff = _random_replies(rng, 3000)
    a, b = ref_values(s0, terminal, r, count, eff), _loop_values(s0, terminal, r, count, eff)
    assert same_floats(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert a[1].any() and (terminal & ~a[1]).any() and ((count == 0).all(1) & ~terminal).any()
    # the hand cases of step 3
    one = lambda s, t, rr, cc, ee: ref_values(np.array([s], np.float32), np.array([t]), np.array([rr], np.float32),
                                               np.array([cc], np.int32), np.array([ee], np.int32))[0][0]
    flat = [1.0] * 21
    assert one(0.5, False, flat, [3] * 21, [3] * 21) == np.float32(1.0)
    assert one(0.5, False, flat, [0] * 21, [0] * 21) == np.float32(0.5)            # every roll blocked: s0
    assert one(0.25, True, flat, [3] * 21, [0] * 21) == np.float32(0.25)           # terminal: s0 exactly, no NaN
    assert np.isnan(one(0.5, False, flat, [3] * 21, [3] * 20 + [0]))              # one roll did not fit
    assert np.isnan(one(0.5, False, flat, [30] * 21, [30] * 20 + [8]))            # one roll scored on a prefix
    two = [2.0] + [0.0] * 20                                                       # 1-1 weighs 1, 1-2 weighs 2
    assert one(0.0, False, two, [1] * 21, [1] * 21) == np.float32(2.0 / 36)
    assert one(0.0, False, [0.0, 2.0] + [0.0] * 19, [1] * 21, [1] * 21) == np.float32(4.0 / 36)


def test_ref_pick():
    s = np.float32
    cases = [  # (v, got, sign, slot)
        ([1, 3, 3], 3, 1, 1), ([1, 3, 3], 3, -1, 0), ([NAN, 1, 2], 3, 1, 2), ([NAN, NAN, NAN], 3, 1, 0),
        ([2, NAN, 2], 3, 1, 0), ([1, 5, 9], 2, 1, 1), ([7], 0, 1, 0), ([-0.0, 0.0], 2, 1, 0), ([NAN, -INF], 2, -1, 1),
    ]
    for v, got, sign, slot in cases:
        assert ref_pick(np.array([v], s), [got], [sign])[0] == slot, (v, got, sign)


@pytest.fixture(scope="module")
def la_hostsim(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "hostsim", "lookahead_hostsim.cpp")
    lib = str(tmp_path_factory.mktemp("la_hostsim") / "liblookahead_hostsim.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", lib, src])
    return C.CDLL(lib)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_hostsim_roll_table(la_hostsim):
    for d, (a, b) in enumerate(ROLLS):
        ab, w = np.zeros(2, np.int32), np.zeros(1, np.float32)
        la_hostsim.hs_la_roll(C.c_int(d), _p(ab), _p(w))
        assert tuple(ab) == (a, b) and w[0] == WEIGHTS[d], d


def test_hostsim_helpers_follow_the_numpy_rule(la_hostsim):
    """The kernels' la_topk, la_candidate_value and la_pick, compiled for the host, equal ref_topk, ref_values and
    ref_pick bit for bit."""
    rng = np.random.default_rng(5)
    n, w = 3000, 70
    sc = _random_scores(rng, n, w)
    counts = rng.integers(0, w + 1, n).astype(np.int32)
    sign = rng.choice([-1, 1], n).astype(np.float32)
    for K in (1, 7, 32):
        idx, got = np.full((n, K), -1, np.int32), np.zeros(n, np.int32)
        la_hostsim.hs_la_topk(_p(sc), C.c_int64(n), C.c_int(w), _p(counts), _p(sign), C.c_int(K), _p(idx), _p(got))
        want = ref_topk(sc, counts, sign, K)
        assert np.array_equal(idx, want[0]) and np.array_equal(got, want[1]), K
    s0, terminal, r, count, eff = _random_replies(rng, 4000)
    v, unfit = np.zeros(4000, np.float32), np.zeros(4000, np.uint8)
    t8 = terminal.astype(np.uint8)
    la_hostsim.hs_la_value(_p(s0), _p(t8), _p(r), _p(count), _p(eff), C.c_int64(4000), _p(v), _p(unfit))
    want = ref_values(s0, terminal, r, count, eff)
    assert same_floats(v, want[0]) and np.array_equal(unfit.astype(bool), want[1])
    K = 8
    vv = v.reshape(500, K)
    cnt = rng.integers(0, K + 1, 500).astype(np.int32)
    sg = rng.choice([-1, 1], 500).astype(np.float32)
    slot = np.zeros(500, np.int32)
    la_hostsim.hs_la_pick(_p(vv), C.c_int64(500), C.c_int(K), _p(cnt), _p(sg), _p(slot))
    assert np.array_equal(slot, ref_pick(vv, cnt, sg))


def test_new_entries_reject_bad_arguments_without_a_gpu():
    from gym_narde_b200 import _cabi
    lib = _cabi.load()
    nul = [None] * 13
    assert lib.narde_segment_topk(None, None, None, None, 0, 8, 1, 4, *nul) == 0
    assert lib.narde_segment_topk(None, None, None, None, 4, 8, 1, 4, *nul) == -1
    assert lib.narde_lookahead_expand(None, None, None, 0, 4, None, None, None, None) == 0
    assert lib.narde_lookahead_expand(None, None, None, 4, 4, None, None, None, None) == -1
    assert lib.narde_lookahead_reduce(None, None, None, None, None, None, 0, 4, 8, *[None] * 9) == 0
    assert lib.narde_lookahead_reduce(None, None, None, None, None, None, 4, 4, 8, *[None] * 9) == -1
    u8, i32, i64, f32 = torch.uint8, torch.int32, torch.int64, torch.float32
    z = lambda dt, *shape: torch.zeros(shape, dtype=dt)
    n, k, cap = 4, 3, 8
    p = n * k * 21
    cands = (z(i32, n, k), z(f32, n, k), z(u8, n * k, 16), z(u8, n * k, 16), z(i64, n, k), z(i32, n))
    calls = [
        ("segment_topk", (z(f32, n * cap), z(i64, n), z(i32, n), z(u8, n, 16), 1, z(u8, n * cap, 16), z(u8, n * cap, 16),
                          z(i64, n, cap)) + cands),
        ("segment_topk", (z(f32, n * cap), z(i64, n), z(i32, n), z(u8, n, 16), 1, z(u8, n * cap, 16), z(u8, n * cap, 16),
                          z(i64, n, cap), z(i32, n, 33)) + cands[1:]),
        ("lookahead_expand", (cands[2], cands[3], cands[5], z(u8, p, 16), z(u8, p, 16), z(u8, p, 2))),
        ("lookahead_reduce", (z(u8, n, 16),) + cands[:2] + (cands[3], cands[4], cands[5], cap, z(f32, p), z(i32, p),
                                                            z(i32, p), z(i32, n), z(f32, n))),
    ]
    for name, args in calls:
        with pytest.raises(_cabi.NardeCudaError):
            getattr(_cabi, name)(*args)


def test_constructor_rejects_max_mode_and_exploration():
    from gym_narde_b200.lookahead import LookaheadActor

    class _Env:
        rules = "full"
    for kw in ({"mode": "max"}, {"epsilon": 0.1}, {"temperature": 1.0}, {"candidates": 0}, {"candidates": 33}):
        with pytest.raises(ValueError):
            LookaheadActor(_Env(), None, **kw)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the kernels on hand-made inputs
# ---------------------------------------------------------------------------------------------------------------
def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cand_buffers(m, K):
    return (torch.full((m, K), -7, dtype=torch.int32, device="cuda"),
            torch.full((m, K), 0x7FC0DEAD, dtype=torch.int32, device="cuda").view(torch.float32),
            torch.full((m * K, 16), 0x5A, dtype=torch.uint8, device="cuda"),
            torch.full((m * K, 16), 0x5B, dtype=torch.uint8, device="cuda"),
            torch.full((m, K), 9, dtype=torch.int64, device="cuda"),
            torch.full((m,), -3, dtype=torch.int32, device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("cap", (31, 128, 129, 3072))
@pytest.mark.parametrize("K", (1, 7, 32))
def test_segment_topk_on_hand_made_scores(cap, K):
    """narde_segment_topk on every pattern, count and side to move of the segment tests, in both modes, at caps around
    the thread / warp switch: the candidates of ref_topk, their scores, rows and action words; slots beyond the count
    untouched.  Then the same segments as a side batch (env_idx, counts_eff, ctrl) overwriting a larger batch."""
    from gym_narde_b200 import _cabi
    flat, dense, offsets, counts, turn, pats = _segments(cap, 7 * cap + K)
    n = len(counts)
    rng = np.random.default_rng(cap + K)
    rows = int(offsets[-1]) + len(flat[-2]) + len(flat[-1]) + 4
    as_lo = rng.integers(0, 256, (rows, 16), dtype=np.uint8)
    as_hi = rng.integers(0, 256, (rows, 16), dtype=np.uint8)
    acts = rng.integers(1, 2 ** 62, (n, cap), dtype=np.int64)
    c = np.minimum(counts, cap)
    for mode in (0, 1):
        sign, raw, score, off, cnt, hi = _gpu_segments(flat, dense, offsets, counts, turn, mode)
        wid, got = ref_topk(raw, c, sign, K)
        out = _cand_buffers(n, K)
        _cabi.segment_topk(score, off, cnt, hi, mode, cu(as_lo), cu(as_hi), cu(acts), *out)
        g_idx, g_sc, g_lo, g_hi, g_act, g_cnt = (t.cpu().numpy() for t in out)
        assert np.array_equal(g_cnt, got), (cap, K, mode)
        for i in range(n):
            j = np.arange(got[i])
            k = wid[i, j]
            assert np.array_equal(g_idx[i, j], k), (cap, K, mode, i, pats[i], int(counts[i]), g_idx[i, :got[i]], k)
            assert same_floats(g_sc[i, j], raw[i, k]), (cap, K, mode, i)
            assert np.array_equal(g_lo[i * K + j], as_lo[offsets[i] + k]) and np.array_equal(g_hi[i * K + j], as_hi[offsets[i] + k])
            assert np.array_equal(g_act[i, j], acts[i, k])
            assert (g_idx[i, got[i]:] == -7).all() and (g_lo[i * K + got[i]:(i + 1) * K] == 0x5A).all(), (cap, K, i)
        # as a side batch: slot s -> env eidx[s] of a batch of n + 9 envs; counts_eff 0 skips (and counts) a slot
        big = n + 9
        eidx = rng.permutation(big)[:n].astype(np.int32)
        eidx[rng.random(n) < 0.2] = -1
        eff = c.astype(np.int32).copy()
        eff[rng.random(n) < 0.2] = 0
        ctrl = torch.tensor([5, 0, 3, 0], dtype=torch.int32, device="cuda")
        out = _cand_buffers(big, K)
        _cabi.segment_topk(score, off, cnt, hi, mode, cu(as_lo), cu(as_hi), cu(acts), *out, env_idx=cu(eidx),
                           counts_eff=cu(eff), ctrl=ctrl)
        g_idx, g_sc, g_lo, g_hi, g_act, g_cnt = (t.cpu().numpy() for t in out)
        want_cnt = np.full(big, -3, np.int32)
        missed = 0
        for s in range(n):
            if eidx[s] < 0:
                continue
            if eff[s] == 0:
                missed += 1
                continue
            missed += int(counts[s] > cap)
            e = eidx[s]
            want_cnt[e] = got[s]
            assert np.array_equal(g_idx[e, :got[s]], wid[s, :got[s]]), (cap, K, mode, s)
            assert np.array_equal(g_act[e, :got[s]], acts[s, wid[s, :got[s]]]), (cap, K, mode, s)
        assert np.array_equal(g_cnt, want_cnt), (cap, K, mode)
        untouched = np.setdiff1d(np.arange(big), eidx[(eidx >= 0) & (eff > 0)])
        assert (g_idx[untouched] == -7).all() and (g_act[untouched] == 9).all()
        assert ctrl.cpu().tolist() == [0, 0, 3 + missed, 0], (ctrl.cpu().tolist(), missed)


@pytest.mark.gpu
@pytest.mark.parametrize("K", (1, 5, 32))
def test_lookahead_expand_on_hand_made_candidates(K):
    from gym_narde_b200 import _cabi
    rng = np.random.default_rng(K)
    n = 301
    c_lo = rng.integers(0, 256, (n * K, 16), dtype=np.uint8)
    c_hi = rng.integers(0, 256, (n * K, 16), dtype=np.uint8)
    cnt = rng.integers(0, K + 1, n).astype(np.int32)
    p = n * K * 21
    lo = torch.full((p, 16), 0xEE, dtype=torch.uint8, device="cuda")
    hi = torch.full_like(lo, 0xEE)
    dice = torch.zeros((p, 2), dtype=torch.uint8, device="cuda")
    _cabi.lookahead_expand(cu(c_lo), cu(c_hi), cu(cnt), lo, hi, dice)
    lo, hi, dice = lo.cpu().numpy(), hi.cpu().numpy(), dice.cpu().numpy()
    slot = np.arange(p) // 21
    live = (slot % K) < cnt[slot // K]
    want_lo = np.where(live[:, None], c_lo[slot], 0)
    want_hi = np.where(live[:, None], c_hi[slot], FINISHED_HI[None, :])
    assert np.array_equal(lo, want_lo) and np.array_equal(hi, want_hi)
    assert np.array_equal(dice, np.array(ROLLS, np.uint8)[np.arange(p) % 21])


@pytest.mark.gpu
@pytest.mark.parametrize("K", (1, 4, 32))
def test_lookahead_reduce_on_hand_made_replies(K):
    """Every case of step 3 (blocked rolls, rolls that did not fit or were scored on a prefix, terminal candidates,
    NaN replies) and of step 4 (ties, NaN, all NaN, no candidate), for both sides to move: choice, value, act_override
    (the word only for an index >= cap), cand_value and the uncovered count."""
    from gym_narde_b200 import _cabi
    rng = np.random.default_rng(40 + K)
    n, cap = 2000, 16
    s0, terminal, r, count, eff = _random_replies(rng, n * K)
    s0[rng.random(n * K) < 0.3] = 0.5                                  # ties of v
    r[rng.random(n * K) < 0.3] = np.float32(0.5)
    got = rng.integers(0, K + 1, n).astype(np.int32)
    cand_idx = rng.integers(0, 2 * cap, (n, K)).astype(np.int32)
    cand_act = rng.integers(1, 2 ** 62, (n, K), dtype=np.int64)
    cand_hi = rng.integers(0, 256, (n * K, 16), dtype=np.uint8)
    cand_hi[:, 11] = np.where(terminal, cand_hi[:, 11] | 4, cand_hi[:, 11] & ~np.uint8(4))
    hi = np.zeros((n, 16), np.uint8)
    turn = rng.choice([-1, 1], n).astype(np.int8)
    hi[:, 10] = turn.view(np.uint8)
    choice = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    value = torch.full((n,), -1.0, dtype=torch.float32, device="cuda")
    act = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    cval = torch.full((n, K), 0x7FC0DEAD, dtype=torch.int32, device="cuda").view(torch.float32)
    unc = torch.tensor([11], dtype=torch.int32, device="cuda")
    _cabi.lookahead_reduce(cu(hi), cu(cand_idx), cu(s0.reshape(n, K)), cu(cand_hi), cu(cand_act), cu(got), cap,
                           cu(r.reshape(-1)), cu(count.reshape(-1)), cu(eff.reshape(-1)), choice, value, act_override=act,
                           cand_value=cval, uncovered=unc)
    v, unfit = ref_values(s0, terminal, r, count, eff)
    v, unfit = v.reshape(n, K), unfit.reshape(n, K)
    live = np.arange(K)[None, :] < got[:, None]
    sign = np.where(turn == 1, 1, -1).astype(np.float32)
    slot = ref_pick(v, got, sign)
    rows = np.arange(n)
    want_choice = np.where(got > 0, cand_idx[rows, slot], 0)
    want_value = np.where(got > 0, v[rows, slot], 0).astype(np.float32)
    want_act = np.where((got > 0) & (want_choice >= cap), cand_act[rows, slot], 0)
    g_cval = cval.cpu().numpy()
    assert np.array_equal(choice.cpu().numpy(), want_choice)
    assert same_floats(value.cpu().numpy(), want_value)
    assert np.array_equal(act.cpu().numpy(), want_act)
    assert same_floats(g_cval[live], v[live]) and (g_cval[~live].view(np.int32) == 0x7FC0DEAD).all()
    assert int(unc.item()) == 11 + int((unfit & live).any(1).sum())
    assert ((np.isnan(v) | ~live).all(1) & (got > 0)).any()                       # an env whose candidates are all NaN
    if K > 1:
        assert (live & (v == 0.5)).sum(1).max() > 1                                # ties of v


# ---------------------------------------------------------------------------------------------------------------
# GPU: LookaheadActor end to end against the oracle
# ---------------------------------------------------------------------------------------------------------------
def _design(name):
    d = argmax_design() if name == "argmax" else EXACT_DESIGNS[name]()
    return tuple(w.cuda() for w in d["W"]), tuple(v.cuda() for v in d["b"])


def _score_rows(lo, hi, W, b, emulate, with_bound, premise=False, chunk=1 << 18):
    """max_a Q of packed rows (numpy [r, 16] x2) by the float64 net: (q float64 [r], bound float64 [r] or None).
    premise: assert that the design is exact on the first chunk (check_premise)."""
    from gym_narde_b200.state import expand_obs198
    q, bd = np.zeros(len(lo)), np.zeros(len(lo)) if with_bound else None
    for s in range(0, len(lo), chunk):
        x = expand_obs198(cu(lo[s:s + chunk]), cu(hi[s:s + chunk]))
        if premise and s == 0:
            check_premise(x, W, b)
        q[s:s + chunk] = ref_q(x, W, b, emulate=emulate).max(1).values.cpu().numpy()
        if with_bound:
            bd[s:s + chunk] = bound(x, W, b).max(1).values.cpu().numpy()
    return q, bd


def _full_lists(lo, hi, dice):
    """o_afterstates_batch over the whole legal lists: (counts [n], acts [n, w], as_lo, as_hi [n, w, 16])."""
    from oracle import oracle as O
    counts, acts, a_lo, a_hi = O.afterstates_batch(lo, hi, dice, cap=32)
    long = np.flatnonzero(counts > 32)
    if len(long) == 0:
        return counts, acts, a_lo, a_hi
    w = int(counts.max())
    c2, a2, l2, h2 = O.afterstates_batch(lo[long], hi[long], dice[long], cap=w)
    acts = np.concatenate([acts, np.zeros((len(lo), w - 32), np.int64)], 1)
    a_lo = np.concatenate([a_lo, np.zeros((len(lo), w - 32, 16), np.uint8)], 1)
    a_hi = np.concatenate([a_hi, np.zeros((len(lo), w - 32, 16), np.uint8)], 1)
    acts[long], a_lo[long], a_hi[long] = a2, l2, h2
    return counts, acts, a_lo, a_hi


def _scored(lo, hi, dice, W, b, emulate, with_bound, premise=False):
    counts, acts, a_lo, a_hi = _full_lists(lo, hi, dice)
    mask = np.arange(acts.shape[1])[None, :] < counts[:, None]
    q, bd = _score_rows(a_lo[mask], a_hi[mask], W, b, emulate, with_bound, premise)
    s = np.zeros(mask.shape, np.float64)
    s[mask] = q
    bnd = None
    if with_bound:
        bnd = np.zeros(mask.shape, np.float64)
        bnd[mask] = bd
    return counts, acts, a_lo, a_hi, s, bnd


def _sign(hi):
    return np.where(hi[:, 10].view(np.int8) == 1, 1.0, -1.0).astype(np.float32)


def _best_replies(lo, hi, dice, W, b, emulate, with_bound, chunk=1 << 16):
    """The opponent's side of every reply position, `chunk` positions at a time (so _scored's [positions, longest list]
    arrays stay small at millions of positions): (legal counts [p], the score of the choice over the whole list
    float32 [p], the largest bound() of its rows [p] or None)."""
    p = len(lo)
    rc, best = np.zeros(p, np.int32), np.zeros(p, np.float32)
    rb = np.zeros(p) if with_bound else None
    for s in range(0, p, chunk):
        e = min(s + chunk, p)
        c, _, _, _, q, bd = _scored(lo[s:e], hi[s:e], dice[s:e], W, b, emulate, with_bound)
        rc[s:e] = c
        best[s:e] = ref_choice(q.astype(np.float32), c, _sign(hi[s:e]), q.shape[1])[1]
        if with_bound:
            rb[s:e] = np.where(np.arange(bd.shape[1])[None, :] < c[:, None], bd, 0).max(1)
    return rc, best, rb


class _LookTurn:
    """The reference of one lookahead turn from the positions before it: the first pass over the oracle's full lists, the
    top-K, the oracle's full reply lists of every (candidate, roll), each scored by the float64 net, and the numpy rule.
    cands: the candidate indices to evaluate (default: the reference's own top-K)."""

    def __init__(self, lo, hi, dice, K, W, b, emulate=True, with_bound=False, cands=None, premise=False):
        n = len(lo)
        self.counts, self.acts, a_lo, a_hi, self.q, self.bnd = _scored(lo, hi, dice, W, b, emulate, with_bound, premise)
        self.sign = _sign(hi)
        self.s0 = self.q.astype(np.float32)
        self.idx, self.got = ref_topk(self.s0, self.counts, self.sign, K)
        if cands is not None:
            self.idx, self.got = cands
        live = np.arange(K)[None, :] < self.got[:, None]
        ii, jj = np.nonzero(live)
        kk = self.idx[ii, jj]
        c_lo, c_hi = a_lo[ii, kk], a_hi[ii, kk]
        p_lo, p_hi = np.repeat(c_lo, 21, 0), np.repeat(c_hi, 21, 0)
        p_dice = np.tile(np.array(ROLLS, np.uint8), (len(ii), 1))
        rc, r_best, rb = _best_replies(p_lo, p_hi, p_dice, W, b, emulate, with_bound)
        self.reply_rows = int(rc.sum())
        self.terminal = np.zeros((n, K), bool)
        self.terminal[ii, jj] = (c_hi[:, 11] & 4) != 0
        self.r_counts = np.zeros((n, K, 21), np.int32)
        self.r_counts[ii, jj] = rc.reshape(-1, 21)
        s0c = np.zeros((n, K), np.float32)
        s0c[ii, jj] = self.s0[ii, kk]
        self.s0c = s0c
        v, _ = ref_values(s0c[ii, jj], self.terminal[ii, jj], r_best.reshape(-1, 21), rc.reshape(-1, 21),
                          rc.reshape(-1, 21))
        self.v = np.zeros((n, K), np.float32)
        self.v[ii, jj] = v
        self.slot = ref_pick(self.v, self.got, self.sign)
        rows = np.arange(n)
        self.choice = np.where(self.got > 0, self.idx[rows, self.slot], 0)
        self.value = np.where(self.got > 0, self.v[rows, self.slot], 0).astype(np.float32)
        self.live_slots = live
        if with_bound:
            b_env = np.where(self.counts[:, None] > np.arange(self.bnd.shape[1])[None, :], self.bnd, 0).max(1)
            per = np.zeros(n)
            np.maximum.at(per, np.repeat(ii, 21), rb)
            self.B = np.maximum(b_env, per)


def _lookahead(design, K, cap, reply_cap, n=512, seed=None, env_base=0, slot_per_env=True, **kw):
    """env and actor after 60 random turns; seed None: 77 + cap + K.  slot_per_env: a first-pass side batch slot for
    every env unless kw sets overflow_slots (False: the actor's default pools, as far as kw leaves them)."""
    from gym_narde_b200 import AfterstateMLP, LookaheadActor, VecNardeEnv
    W, b = design
    env = VecNardeEnv(n, seed=77 + cap + K if seed is None else seed, max_actions=cap, env_base=env_base)
    mlp = AfterstateMLP(W[0], b[0], W[1], b[1], W[2], b[2])
    if slot_per_env:
        kw.setdefault("overflow_slots", n)
    actor = LookaheadActor(env, mlp, candidates=K, reply_cap=reply_cap, **kw)
    env.reset()
    for _ in range(60):                       # random self-play: positions of every phase
        env.step()
    return env, actor


def _play(env, actor, graph):
    lo, hi = env.lo.cpu().numpy(), env.hi.cpu().numpy()
    actor.step_graph() if graph else actor.step()
    return lo, hi, actor.dice.cpu().numpy()


def check_look_turn(ref, env, actor, cap, reply_cap, seen, what):
    """The exact-scorer rule of one lookahead turn: choice, value and the action played equal the reference bit for bit
    for every env.  Adds to `seen` what the turn crossed: live env turns, blocked replies, terminal candidates, reply
    lists longer than reply_cap, candidates beyond the stored list, envs where lookahead played another action than
    greedy."""
    choice, value, chosen = actor.choice.cpu().numpy(), actor.value.cpu().numpy(), env.chosen.cpu().numpy()
    live = ref.counts > 0
    bad = np.flatnonzero(choice != ref.choice)
    assert len(bad) == 0, ("choice", what, len(bad),
                           [(int(i), int(ref.counts[i]), int(choice[i]), int(ref.choice[i])) for i in bad[:5]])
    assert same_floats(value, ref.value), ("value", what,
                                           np.flatnonzero(value.view(np.int32) != ref.value.view(np.int32))[:5])
    rows = np.flatnonzero(live)
    assert np.array_equal(chosen[rows], ref.acts[rows, ref.choice[rows]]), ("action", what)
    ls = ref.live_slots
    seen["turns"] += int(live.sum())
    seen["blocked"] += int(((ref.r_counts == 0) & (ls & ~ref.terminal)[:, :, None]).sum())
    seen["terminal"] += int((ref.terminal & ls).sum())
    seen["reply_side"] += int(((ref.r_counts > reply_cap) & ls[:, :, None]).sum())
    seen["beyond"] += int(((ref.idx >= cap) & ls).sum())
    seen["differ"] += int((live & (ref.choice != ref.idx[:, 0])).sum())


def check_look_bound(ref, actor, K, what):
    """The realistic-scorer rule of one lookahead turn (ref: a _LookTurn with_bound over the actor's own candidates),
    B = the largest bound() over an env's first-pass and reply rows: the candidates are within 2B of the reference's K-th
    best 0-ply score; where the reference's best and second-best v differ by more than 2B the actor plays the reference's
    best, elsewhere an action whose reference v is within 2B of the best.  Returns (decided, near-ties)."""
    c_idx, c_cnt = actor.cand_idx.cpu().numpy(), actor.cand_count.cpu().numpy()
    choice = actor.choice.cpu().numpy()
    decided = near = 0
    for i in np.flatnonzero(ref.counts > 0):
        B = ref.B[i]
        g = int(c_cnt[i])
        assert g == min(K, ref.counts[i]), (what, i)
        signed0 = ref.sign[i] * ref.q[i, :ref.counts[i]]
        kth_best = np.sort(signed0)[::-1][g - 1]
        assert (ref.sign[i] * ref.q[i, c_idx[i, :g]] >= kth_best - 2 * B).all(), (what, i)
        sv = ref.sign[i] * ref.v[i, :g].astype(np.float64)
        order = np.argsort(-sv, kind="stable")
        slot = int(np.flatnonzero(c_idx[i, :g] == choice[i])[0])
        if g > 1 and sv[order[0]] - sv[order[1]] > 2 * B:
            assert slot == order[0], (what, i, slot, order[0], sv, B)
            decided += 1
        else:
            assert sv[slot] >= sv[order[0]] - 2 * B, (what, i)
            near += 1
    return decided, near


EXACT_RUNS = [("perm", 32, 8, 64, True), ("sparse", 4, 64, 8, False), ("argmax", 1, 8, 8, True),
              ("argmax", 4, 8, 64, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("design,K,cap,reply_cap,graph", EXACT_RUNS)
def test_lookahead_plays_the_reference_with_an_exact_scorer(design, K, cap, reply_cap, graph):
    """With an exact scorer, for every env of every turn: choice, the action played and value equal the numpy rule over the
    oracle's full lists bit for bit, and nothing is uncovered.  The run crosses blocked replies, terminal candidates,
    reply lists longer than reply_cap (the reply side batch), candidates beyond the first pass's stored list, and (K > 1)
    turns where lookahead plays another action than greedy."""
    W, b = _design(design)
    n = 512
    env, actor = _lookahead((W, b), K, cap, reply_cap, n=n, reply_overflow_slots=n * K * 21 // (1 if reply_cap == 8 else 4))
    seen = dict(turns=0, blocked=0, terminal=0, reply_side=0, beyond=0, differ=0)
    for t in range(30):
        lo, hi, dice = _play(env, actor, graph)
        ref = _LookTurn(lo, hi, dice, K, W, b, premise=(t % 10 == 0))
        check_look_turn(ref, env, actor, cap, reply_cap, seen, (design, K, cap, reply_cap, t))
    assert actor.uncovered_envs() == 0
    print("lookahead exact %s K=%d cap %d reply_cap %d %s: %s" % (design, K, cap, reply_cap,
                                                                  "step_graph" if graph else "step", seen))
    assert seen["blocked"] > 0 and seen["terminal"] > 0 and seen["reply_side"] > 0, seen
    if cap == 8:
        assert seen["beyond"] > 0, seen
    if K > 1:
        assert seen["differ"] >= 0.01 * seen["turns"], seen


@pytest.mark.gpu
def test_one_candidate_plays_the_greedy_actor():
    """candidates=1 and AfterstateActor(mode="white_value") on two envs of the same seed: the same choices, actions and
    states for 100 turns (the second through step_graph)."""
    from gym_narde_b200 import AfterstateActor, AfterstateMLP, LookaheadActor, VecNardeEnv
    W, b = default_net(3, 1.0)
    W, b = tuple(w.cuda() for w in W), tuple(v.cuda() for v in b)
    mlp = AfterstateMLP(W[0], b[0], W[1], b[1], W[2], b[2])
    envs = [VecNardeEnv(1024, seed=99, max_actions=16) for _ in range(2)]
    # (side batches with a slot for every env: when more lists overflow than there are slots, which envs get one follows
    # the order of atomics, and the uncovered ones choose over their stored prefix)
    greedy = AfterstateActor(envs[0], mlp, mode="white_value", overflow_slots=1024)
    look = LookaheadActor(envs[1], mlp, candidates=1, overflow_slots=1024)
    for e in envs:
        e.reset()
    for t in range(100):
        greedy.step()
        look.step() if t < 50 else look.step_graph()
        assert torch.equal(greedy.choice, look.choice), t
        assert torch.equal(envs[0].chosen, envs[1].chosen), t
        assert torch.equal(envs[0].lo, envs[1].lo) and torch.equal(envs[0].hi, envs[1].hi), t
    assert greedy.uncovered_envs() == 0 and look.first.uncovered_envs() == 0    # (replies do not change the choice at K = 1)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", (1.0, 4.0))
def test_lookahead_with_a_realistic_scorer_is_within_the_bound(scale):
    """nn.Linear's init (x1, x4), B = the largest bound() over an env's first-pass and reply rows.  The candidates are
    within 2B of the reference's K-th best 0-ply score; over the actor's own candidates, where the reference's best and
    second-best v differ by more than 2B the actor plays the reference's best, elsewhere an action whose reference v is
    within 2B of the best."""
    W, b = default_net(1, scale)
    W, b = tuple(w.cuda() for w in W), tuple(v.cuda() for v in b)
    K = 4
    env, actor = _lookahead((W, b), K, 64, 64, n=256)
    decided = near = 0
    for t in range(8):
        lo, hi, dice = _play(env, actor, False)
        cands = (actor.cand_idx.cpu().numpy(), actor.cand_count.cpu().numpy())
        ref = _LookTurn(lo, hi, dice, K, W, b, emulate=False, with_bound=True, cands=cands)
        d, e = check_look_bound(ref, actor, K, (scale, t))
        decided += d
        near += e
    print("lookahead realistic x%g: %d env turns decided by more than 2B, %d near-ties" % (scale, decided, near))
    assert decided > 20


@pytest.mark.gpu
def test_lookahead_with_bounded_pools_counts_what_it_could_not_score():
    """reply_rows and reply_overflow_slots too small for the turn: uncovered_envs() grows by the number of envs with a
    NaN candidate value; every other env is exact; in a counted env every candidate's value is the reference's or NaN and
    the choice follows step 4 over those values."""
    W, b = _design("sparse")
    K, cap, rcap, n = 4, 64, 8, 512
    env, actor = _lookahead((W, b), K, cap, rcap, n=n, reply_rows=n * K * 21 * 3, reply_overflow_slots=256)
    before, counted, exact = actor.uncovered_envs(), 0, 0
    for t in range(12):
        lo, hi, dice = _play(env, actor, t % 2 == 1)
        ref = _LookTurn(lo, hi, dice, K, W, b)
        choice, value, cval = actor.choice.cpu().numpy(), actor.value.cpu().numpy(), actor.cand_value.cpu().numpy()
        ls = ref.live_slots
        nan_env = (np.isnan(cval) & ls).any(1)
        after = actor.uncovered_envs()
        assert after - before == int(nan_env.sum()), (t, after - before, int(nan_env.sum()))
        before = after
        ok = ~nan_env
        assert np.array_equal(choice[ok], ref.choice[ok]) and same_floats(value[ok], ref.value[ok]), t
        for i in np.flatnonzero(nan_env):
            g = ref.got[i]
            got_v = cval[i, :g]
            assert np.all(np.isnan(got_v) | (got_v.view(np.int32) == ref.v[i, :g].view(np.int32))), (t, i)
            slot = ref_pick(got_v[None, :], [g], [ref.sign[i]])[0]
            assert choice[i] == ref.idx[i, slot] and same_floats(value[i:i + 1], got_v[slot:slot + 1]), (t, i)
        counted += int(nan_env.sum())
        exact += int(ok.sum())
    print("bounded pools: %d env turns counted, %d exact" % (counted, exact))
    assert counted > 0 and exact > 0
