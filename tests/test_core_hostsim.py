"""CPU: the CUDA path's per-environment core (narde_core.cuh / narde_env.cuh compiled by g++ into the
test-only host harness) against the oracle and the golden fixtures.  Same checks as the -m gpu
parity tests, so the rules arithmetic is proven before it ever reaches the GPU."""
import numpy as np

import parity as P


def test_golden_valid_moves(hostsim):
    assert P.check_golden_valid_moves(hostsim) > 1000


def test_golden_step_traces(hostsim):
    assert P.check_golden_step_traces(hostsim) > 2000


def test_tier_n_kat(hostsim):
    assert P.check_tier_n_kat(hostsim) > 300


def test_half_moves_selfplay_and_synthetic(hostsim):
    lo, hi = P.pack_corpus(P.selfplay_corpus(25, 1))
    n = lo.shape[0]
    rng = np.random.RandomState(0)
    dice4 = np.zeros((n, 4), np.uint8)
    k = rng.randint(0, 3, size=n)
    d = rng.randint(1, 7, size=(n, 4))
    dice4[:, 0] = d[:, 0]
    dice4[k >= 1, 1] = d[k >= 1, 1]
    four = k == 2
    dice4[four] = d[four, :1]
    P.check_half_moves_vs_oracle(hostsim, lo, hi, dice4)
    b, off, ft = P.synthetic_boards(3000, 2)
    lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 3)
    dice4 = np.zeros((3000, 4), np.uint8)
    dice4[:, :2] = P.random_dice(3000, 4)
    P.check_half_moves_vs_oracle(hostsim, lo, hi, dice4)


def test_enumerate_selfplay(hostsim):
    lo, hi = P.pack_corpus(P.selfplay_corpus(25, 5))
    assert P.check_enumerate_vs_oracle(hostsim, lo, hi, P.random_dice(lo.shape[0], 6, 0.3)) > 0


def test_enumerate_synthetic_block_rule_heavy(hostsim):
    b, off, ft = P.synthetic_boards(5000, 7)
    lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 8)
    assert P.check_enumerate_vs_oracle(hostsim, lo, hi, P.random_dice(5000, 9, 0.5)) > 0


def test_enumerate_overflow_reports_true_count(hostsim):
    b, off, ft = P.synthetic_boards(500, 17)
    lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 18)
    P.check_enumerate_vs_oracle(hostsim, lo, hi, P.random_dice(500, 19, 0.7), cap=8)


def test_enumerate_fast_path(hostsim):
    """narde_enumerate_fast (fused-step phases in enumerate-only mode, exact phases for deferred turns)
    against the oracle on the same corpora; the states must come back untouched."""
    hostsim.enumerate_fast = True
    try:
        lo, hi = P.pack_corpus(P.selfplay_corpus(25, 5))
        assert P.check_enumerate_vs_oracle(hostsim, lo, hi, P.random_dice(lo.shape[0], 6, 0.3)) > 0
        b, off, ft = P.synthetic_boards(3000, 7)
        lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 8)
        assert P.check_enumerate_vs_oracle(hostsim, lo, hi, P.random_dice(3000, 9, 0.5)) > 0
        P.check_enumerate_vs_oracle(hostsim, lo[:500].copy(), hi[:500].copy(), P.random_dice(500, 19, 0.7), cap=8)
    finally:
        hostsim.enumerate_fast = False


def test_step_ref_lockstep(hostsim):
    assert P.check_step_ref_lockstep(hostsim, 64, 500, 42) > 0


def test_step_full_lockstep_autoreset(hostsim):
    assert P.check_step_full_lockstep(hostsim, 96, 260, 0x5EED) > 50


def test_step_full_lockstep_mover_reward_no_autoreset(hostsim):
    P.check_step_full_lockstep(hostsim, 48, 220, 99, cap=4, flags=1)


def test_step_full_caller_actions_index_and_fraction(hostsim):
    # caller-chosen actions: clamped int32 indices, and u32 fractions of the legal list (flag 32)
    P.check_step_full_lockstep(hostsim, 64, 150, 31, action_mode="index")
    P.check_step_full_lockstep(hostsim, 64, 150, 32, action_mode="fraction")


def test_obs198(hostsim):
    lo, hi = P.pack_corpus(P.selfplay_corpus(10, 21))
    P.check_obs198(hostsim, lo, hi)


def _v1_v2_equal(hostsim, lo, hi, **kw):
    import numpy as np
    outs = []
    for per_thread in (True, False):
        hostsim.per_thread = per_thread
        l, h = lo.copy(), hi.copy()
        o = hostsim.step_full(l, h, **kw)
        outs.append((l, h, o))
    hostsim.per_thread = False
    (l1, h1, o1), (l2, h2, o2) = outs
    assert (l1 == l2).all() and (h1 == h2).all()
    for k in o1:
        if k == "deferred":
            continue
        if o1[k] is None:
            assert o2[k] is None
            continue
        if k == "actions":
            cap = o1[k].shape[1]
            m = np.arange(cap)[None, :] < np.minimum(o1["counts"], cap)[:, None]
            assert (o1[k][m] == o2[k][m]).all()
        else:
            assert (o1[k] == o2[k]).all(), k
    o1["deferred"] = o2["deferred"]
    return o1


def test_block_kernel_tile_128_equals_per_thread_body(hostsim):
    """The library uses 32-env one-warp CTAs for batches <= 16384 and 128-env CTAs above (NARDE_TILE=64 selects the
    64-env / 128-thread tile: two threads per env in the item phases); force both large tiles on
    small inputs so that all three are checked here (the other tests run the 32-env tile)."""
    import ctypes as C
    hostsim.lib.hs_set_small_batch(C.c_int64(0))
    try:
        for tile in (64, 128):
            hostsim.lib.hs_set_tile(C.c_int(tile))
            test_block_kernel_equals_per_thread_body(hostsim)
            P.check_step_full_lockstep(hostsim, 200, 120, 0xBEEF)
            P.check_step_full_lockstep(hostsim, 67, 60, 0xF00D + tile, cap=4)
    finally:
        hostsim.lib.hs_set_small_batch(C.c_int64(16384))
        hostsim.lib.hs_set_tile(C.c_int(128))


def test_block_kernel_equals_per_thread_body(hostsim):
    """The CTA-cooperative phases (narde_block.cuh) and the per-thread body (narde_env.cuh) must agree
    bit for bit: synthetic block-rule-heavy boards, ragged batch sizes, given dice / given indices."""
    import numpy as np
    b, off, ft = P.synthetic_boards(3001, 31)
    lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 32)
    dice = P.random_dice(3001, 33, 0.4)
    o = _v1_v2_equal(hostsim, lo, hi, seed=5, step=9, dice_in=dice, cap=48, flags=0)
    assert o["counts"].max() > 48
    assert o["deferred"] > 20      # block-rule doubles turns went through the CTA-per-env exact phases
    idx = np.random.RandomState(1).randint(-2, 80, size=3001).astype(np.int32)
    _v1_v2_equal(hostsim, lo, hi, seed=5, step=9, dice_in=dice, action_idx=idx, cap=16, flags=1)
    _v1_v2_equal(hostsim, lo, hi, seed=5, step=9, cap=0, flags=2, want_actions=False)
    for n in (1, 127, 128, 129, 300):
        _v1_v2_equal(hostsim, lo[:n].copy(), hi[:n].copy(), seed=n, step=3, cap=64, flags=2)
    lo, hi = P.pack_corpus(P.selfplay_corpus(30, 41))
    for step in range(1, 6):
        _v1_v2_equal(hostsim, lo, hi, seed=77, step=step, cap=32, flags=2)
    # without a workspace the block-rule doubles turns are resolved inline: same results
    hostsim.defer = False
    try:
        b, off, ft = P.synthetic_boards(2000, 51)
        lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 52)
        o = _v1_v2_equal(hostsim, lo, hi, seed=5, step=9, dice_in=P.random_dice(2000, 53, 0.6), cap=48, flags=0)
        assert o["deferred"] == 0
    finally:
        hostsim.defer = True


def test_block_kernel_fallback_paths(hostsim):
    """The rare CTA whose level-2 doubles items do not fit the item table (searching iterator) or the per-item
    offset table (contiguous chunks, every item counted again in the emit phase): forced here through the
    test-only hook of the host build, on both tiles, against the per-thread body and the oracle."""
    import ctypes as C
    for force in (1, 2):
        hostsim.lib.hs_set_force_slow(C.c_int(force))
        try:
            test_block_kernel_equals_per_thread_body(hostsim)
            P.check_step_full_lockstep(hostsim, 96, 100, 0xFA11 + force)
            hostsim.lib.hs_set_small_batch(C.c_int64(0))
            test_block_kernel_equals_per_thread_body(hostsim)
        finally:
            hostsim.lib.hs_set_small_batch(C.c_int64(16384))
            hostsim.lib.hs_set_force_slow(C.c_int(0))


def test_exact_kernel_multi_window_levels(hostsim):
    """The exact (block-rule) doubles phases test a level's candidates in windows of 1024, with a team of one warp
    (long lists) or of the whole 128-thread CTA (short lists).  Test-only hooks of the host build shrink the window
    to 8 so that ordinary positions take the multi-window route (actions stored window by window, the chosen action
    read back from the stored list or found by the second pass: cap 0 / 4) and select the 128-thread team."""
    import ctypes as C
    for force in (4, 8, 12):
        hostsim.lib.hs_set_force_slow(C.c_int(force))
        try:
            test_block_kernel_equals_per_thread_body(hostsim)
            b, off, ft = P.synthetic_boards(4000, 61)
            lo, hi, _, _ = P.pack_mover_boards(b, off, ft, 62)
            dice = P.random_dice(4000, 63, 0.8)
            o = _v1_v2_equal(hostsim, lo, hi, seed=7, step=2, dice_in=dice, cap=4, flags=0)
            assert o["deferred"] > 50
            _v1_v2_equal(hostsim, lo, hi, seed=8, step=3, dice_in=dice, cap=0, flags=0, want_actions=False)
            hostsim.enumerate_fast = True
            try:
                assert P.check_enumerate_vs_oracle(hostsim, lo[:1500].copy(), hi[:1500].copy(), dice[:1500], cap=8) > 0
            finally:
                hostsim.enumerate_fast = False
        finally:
            hostsim.lib.hs_set_force_slow(C.c_int(0))


def test_oracle_bulk_trace_equals_stepwise_hostsim(hostsim):
    """o_selfplay_trace (the C bulk trace the full-size GPU parity test and bench.py compare against) agrees field by
    field with step-by-step calls: Philox policy, caller indices / fractions, TimeLimit truncation, no auto-reset."""
    turns, eps = P.check_trace_vs_backend(hostsim, 300, 260, 0xBEEF, cap=16)
    assert turns == 300 * 260 and eps > 300
    P.check_trace_vs_backend(hostsim, 200, 120, 11, action_mode="index", cap=8)
    P.check_trace_vs_backend(hostsim, 200, 120, 12, action_mode="fraction", cap=64)
    _, eps = P.check_trace_vs_backend(hostsim, 150, 130, 13, max_episode_steps=40, cap=4)
    assert eps >= 150 * 3                                   # every env truncated three times
    turns, _ = P.check_trace_vs_backend(hostsim, 150, 260, 14, flags=1, cap=4)   # mover reward, finished envs idle
    assert turns < 150 * 260


def test_hostsim_rebuilds_when_any_included_file_changes(monkeypatch, tmp_path):
    """The host harness is rebuilt when a file that hostsim.cpp includes, directly or through another header, is newer
    than the library: a stale library would test old code."""
    import os
    import re
    import subprocess

    import support

    def includes(path, seen):
        with open(path) as f:
            names = re.findall(r'^\s*#\s*include\s+"([^"]+)"', f.read(), re.M)
        for name in names:
            dep = os.path.realpath(os.path.join(os.path.dirname(path), name))
            if dep not in seen:
                seen.add(dep)
                includes(dep, seen)
        return seen

    deps = includes(os.path.join(support.ROOT, "tests", "hostsim", "hostsim.cpp"), set())
    assert any(d.endswith("narde_deferred.cuh") for d in deps)
    lib = str(tmp_path / "libnarde_hostsim.so")
    open(lib, "wb").close()
    monkeypatch.setattr(support, "_HS_LIB", lib)
    builds = []
    monkeypatch.setattr(subprocess, "check_call", lambda cmd, **kw: builds.append(cmd))
    for dep in sorted(deps):
        # the library is newer than every file but `dep`
        monkeypatch.setattr(os.path, "getmtime",
                            lambda p, dep=dep: 1.0 if p == lib else 2.0 if os.path.realpath(p) == dep else 0.0)
        builds.clear()
        support.build_hostsim()
        assert builds, f"a change to {dep} leaves the host harness stale"
