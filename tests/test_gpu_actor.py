"""GPU (-m gpu): the batched afterstate-greedy actor (enumerate -> afterstates -> tcgen05 score -> argmax -> step).

Integer pieces are bit-exact: every afterstate row equals the state the (oracle-validated) fused step
produces when that action is played; the greedy index equals torch's segment arg-max of the same scores."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _net():
    import torch
    import torch.nn as nn
    torch.manual_seed(0)
    fn = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU()).cuda()
    head = nn.Linear(256, 576).cuda()
    return fn, head


def test_afterstates_equal_fused_step_results():
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n, cap = 3000, 96
    env = VecNardeEnv(n, seed=21, max_actions=cap, autoreset=False, max_episode_steps=0)
    actor = AfterstateActor(env, mlp)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    checked = 0
    for t in range(130):
        dice = env.roll().clone()
        acts, counts, ovf = env.get_valid_actions(dice)
        acts, counts = acts.clone(), counts.clone()
        off = actor.afterstates(acts, counts).clone()
        c = counts.clamp(max=cap).long()
        assert int(actor.rows_dev.item()) == int(c.sum().item())
        idx = (torch.rand(n, device="cuda", generator=g) * c.clamp(min=1)).long().clamp(max=cap - 1)
        done_before = env.done.bool().clone()
        env.step(idx.to(torch.int32), dice=dice)
        live = (c > 0) & ~done_before
        rows = (off + idx)[live]
        assert torch.equal(actor.as_lo[rows], env.lo[live]) and torch.equal(actor.as_hi[rows], env.hi[live]), t
        checked += int(live.sum().item())
    assert checked > 200000


def test_actor_choice_is_segment_argmax_and_step_plays_it():
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n, cap = 2048, 64
    for mode in ("max", "white_value"):
        env = VecNardeEnv(n, seed=9, max_actions=cap)
        actor = AfterstateActor(env, mlp, mode=mode, overflow_slots=0)   # the first pass alone (stored lists only)
        env.reset()
        for t in range(60):
            turn = env.hi[:, 10].view(torch.int8).clone()          # +1 WHITE / -1 BLACK to move
            choice, dice = actor.choose()
            counts = env.counts.clone()
            c = counts.clamp(max=cap).long()
            K = int(actor.rows_dev.item())
            # scores of the packed afterstate rows == row max of forward_states on the same rows
            q = mlp.forward_states(actor.as_lo[:K].contiguous(), actor.as_hi[:K].contiguous())
            assert torch.equal(actor.scores[:K], q.max(1).values)
            # dense [n, cap] view of the ragged scores, -inf padded
            dense = torch.full((n, cap), float("-inf"), device="cuda")
            col = torch.arange(cap, device="cuda")[None, :].expand(n, cap)
            mask = col < c[:, None]
            dense[mask] = actor.scores[:K]
            if mode == "white_value":
                dense = torch.where(mask, dense * turn.float()[:, None], dense)
            want = dense.argmax(1)
            live = c > 0
            assert torch.equal(choice.long()[live], want[live]), (mode, t)
            chosen_act = env.actions[torch.arange(n, device="cuda"), choice.long()].clone()
            env.step(choice, dice=dice)
            assert torch.equal(env.chosen[live], chosen_act[live])


def test_actor_graph_replay_equals_eager_turns():
    """AfterstateActor.step_graph (one CUDA-graph replay per greedy turn, step number read from the device
    counter) plays exactly the turns of the eager step()."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n, cap = 4096, 64
    envs = [VecNardeEnv(n, seed=13, max_actions=cap) for _ in range(2)]
    actors = [AfterstateActor(e, mlp) for e in envs]
    for e in envs:
        e.reset()
        for _ in range(30):
            e.step()
    for t in range(50):
        actors[0].step()
        actors[1].step_graph()
        assert torch.equal(envs[0].lo, envs[1].lo) and torch.equal(envs[0].hi, envs[1].hi), t
        assert torch.equal(envs[0].obs, envs[1].obs) and torch.equal(envs[0].reward, envs[1].reward)
        assert torch.equal(envs[0].chosen, envs[1].chosen)
    assert envs[0].episode_stats() == envs[1].episode_stats()


def test_afterstates_scan_equals_host_prefix_sum_version():
    """narde_afterstates_scan (offsets by an in-kernel decoupled look-back scan, rows dealt to threads) against
    narde_afterstates fed with torch's exclusive prefix sum: offsets, row count, rows and row->env map, at ragged
    sizes around the 128-env tile, with one scratch buffer reused across calls of different sizes."""
    import ctypes as C
    import torch
    from gym_narde_b200 import VecNardeEnv, _cabi
    lib = _cabi.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t: C.c_void_p(t.data_ptr())
    scratch = torch.zeros(131072 // 128 + 5, dtype=torch.int64, device="cuda")
    # (131 072 envs: 1024 tiles, more than are resident at once -- the look-back really waits on other CTAs)
    for n, cap, steps in ((1, 8, 3), (127, 16, 10), (129, 64, 25), (3000, 24, 40), (4096, 64, 60), (131072, 12, 45)):
        env = VecNardeEnv(n, seed=77 + n, max_actions=cap)
        env.reset()
        for _ in range(steps):
            env.step()
        acts, counts, _ = env.get_valid_actions()
        c = counts.clamp(max=cap).long()
        off_ref = torch.cumsum(c, 0) - c
        K = int(c.sum().item())
        ref_lo = torch.zeros((K + 1, 16), dtype=torch.uint8, device="cuda")
        ref_hi = torch.zeros_like(ref_lo)
        ref_env = torch.full((K + 1,), -1, dtype=torch.int32, device="cuda")
        _cabi.afterstates(env.lo, env.hi, acts, counts, off_ref, ref_lo, ref_hi, ref_env)
        for rep in range(2):           # the scratch words are left ready for the next call
            lo2, hi2 = torch.zeros_like(ref_lo), torch.zeros_like(ref_hi)
            env2 = torch.full_like(ref_env, -1)
            off = torch.full((n,), -7, dtype=torch.int64, device="cuda")
            rows = torch.zeros(1, dtype=torch.int64, device="cuda")
            assert lib.narde_afterstates_scan(P(env.lo), P(env.hi), P(acts), P(counts), n, cap, P(off), P(rows), P(lo2),
                                              P(hi2), P(env2), P(scratch), 0, None, st) == 0
            assert int(rows.item()) == K
            assert torch.equal(off, off_ref)
            assert torch.equal(lo2, ref_lo) and torch.equal(hi2, ref_hi) and torch.equal(env2, ref_env)


def test_actor_scores_every_legal_action_beyond_the_stored_capacity():
    """ADVICE r1: the greedy choice must look at EVERY legal action (DQNAgent.act, train_deepq_pytorch.py:430-507), not
    at the first env.max_actions.  With a tiny stored capacity most envs overflow; the actor's choice (main pass +
    side-batch pass) must equal the arg-max over the complete list enumerated with a capacity that holds everything."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor, _cabi
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n, cap, big = 1536, 8, 2048
    for mode in ("max", "white_value"):
        env = VecNardeEnv(n, seed=31, max_actions=cap)
        actor = AfterstateActor(env, mlp, mode=mode, overflow_slots=n, overflow_cap=big, overflow_rows=400 * n)
        env.reset()
        acts_b = torch.zeros((n, big), dtype=torch.int64, device="cuda")
        cnt_b = torch.zeros(n, dtype=torch.int32, device="cuda")
        ws = torch.zeros(_cabi.workspace_ints(n), dtype=torch.int32, device="cuda")
        overflowed = beyond = 0
        for t in range(70):
            turn = env.hi[:, 10].view(torch.int8).clone().float()
            choice, dice = actor.choose()
            _cabi.enumerate_actions_fast(env.lo, env.hi, dice, acts_b, cnt_b, None, ws)
            c = cnt_b.long()
            assert int(c.max().item()) <= big
            off = torch.cumsum(c, 0) - c
            K = int(c.sum().item())
            lo2 = torch.zeros((K + 1, 16), dtype=torch.uint8, device="cuda")
            hi2 = torch.zeros_like(lo2)
            _cabi.afterstates(env.lo, env.hi, acts_b, cnt_b, off, lo2, hi2)
            sc = mlp.score_states(lo2[:K].contiguous(), hi2[:K].contiguous())
            dense = torch.full((n, int(c.max().item()) + 1), float("-inf"), device="cuda")
            col = torch.arange(dense.shape[1], device="cuda")[None, :]
            mask = col < c[:, None]
            dense[mask] = sc
            if mode == "white_value":
                dense = torch.where(mask, dense * turn[:, None], dense)
            want = dense.argmax(1)
            live = c > 0
            assert torch.equal(choice.long()[live], want[live]), (mode, t)
            overflowed += int((c > cap).sum().item())
            beyond += int((want[live] >= cap).sum().item())
            chosen_act = acts_b[torch.arange(n, device="cuda"), choice.long()].clone()
            env.step(choice, dice=dice)
            assert torch.equal(env.chosen[live], chosen_act[live])     # the step plays it although it was never stored
        assert overflowed > 10000 and beyond > 3000, (overflowed, beyond)
        assert actor.uncovered_envs() == 0
    # a side batch that is too small: nothing breaks, the misses are counted
    env = VecNardeEnv(n, seed=31, max_actions=cap)
    actor = AfterstateActor(env, mlp, overflow_slots=16, overflow_cap=32, overflow_rows=256)
    env.reset()
    for t in range(30):
        actor.step()
    assert actor.uncovered_envs() > 0


def test_step_chosen_equals_fused_step_with_the_same_choice():
    """narde_step_chosen (what AfterstateActor.step plays: apply the chosen action, complete the turn, no second
    enumeration) against narde_step_full(action_idx=choice, dice) on a twin env: states, Box(198), reward, terminated /
    truncated, chosen action and episode statistics, through auto-resets, truncation and choices beyond the stored lists."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n = 3000
    for cap, mode, max_steps in ((64, "max", 1000), (6, "white_value", 40)):
        a = VecNardeEnv(n, seed=5, max_actions=cap, max_episode_steps=max_steps)
        b = VecNardeEnv(n, seed=5, max_actions=cap, max_episode_steps=max_steps, graph=False)
        actor = AfterstateActor(a, mlp, mode=mode, overflow_slots=n, overflow_cap=2048, overflow_rows=300 * n)
        a.reset()
        b.reset()
        beyond = 0
        for t in range(150):
            actor.step()
            beyond += int((actor.choice >= cap).sum().item())
            b.step(actor.choice.clone(), dice=a.dice.clone())
            assert torch.equal(a.lo, b.lo) and torch.equal(a.hi, b.hi), (cap, t)
            assert torch.equal(a.obs, b.obs) and torch.equal(a.reward, b.reward), (cap, t)
            assert torch.equal(a.done, b.done) and torch.equal(a.trunc, b.trunc), (cap, t)
            assert torch.equal(a.chosen, b.chosen) and torch.equal(a.counts, b.counts), (cap, t)
        assert a.episode_stats() == b.episode_stats()
        assert a.episode_stats()["episodes"] > 0
        if cap == 6:
            assert beyond > 1000          # actions that were never stored in the main batch's lists were played
        assert int(actor.act_override.abs().sum().item()) == 0   # every override was consumed


def test_short_or_mistyped_buffers_are_refused_before_any_launch():
    """A short `out`, an int32 rows_dev and a short afterstate buffer raise NardeCudaError, and nothing is launched: the
    outputs keep their sentinel values."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, _cabi
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n, cap = 512, 16
    env = VecNardeEnv(n, seed=3, max_actions=cap)
    env.reset()
    acts, counts, _ = env.get_valid_actions()
    torch.cuda.synchronize()
    score = torch.full((n - 1,), 7.0, device="cuda")
    q = torch.full((n, 575), 7.0, device="cuda")
    score_full = torch.full((n,), 7.0, device="cuda")
    rows = torch.full((1,), -5, dtype=torch.int64, device="cuda")
    with pytest.raises(_cabi.NardeCudaError, match="out must have shape"):
        mlp.score_states(env.lo, env.hi, out=score)
    with pytest.raises(_cabi.NardeCudaError, match="out must have shape"):
        mlp.forward_states(env.lo, env.hi, out=q)
    with pytest.raises(_cabi.NardeCudaError, match="out must have shape"):
        mlp.forward(env.obs, out=score_full)                      # q rows are [K,576], not [K]
    with pytest.raises(_cabi.NardeCudaError, match="rows_dev must have dtype"):
        mlp.score_states(env.lo, env.hi, out=score_full, rows_dev=torch.full((1,), n, dtype=torch.int32, device="cuda"))
    scratch = torch.zeros(n // 128 + 4, dtype=torch.int64, device="cuda")
    short = [torch.zeros((n * cap - 1, 16), dtype=torch.uint8, device="cuda") for _ in range(2)]
    with pytest.raises(_cabi.NardeCudaError, match="as_lo must have at least"):
        _cabi.afterstates_scan(env.lo, env.hi, acts, counts, *short, scratch, rows_out=rows)     # rows_cap 0: n * cap rows
    with pytest.raises(_cabi.NardeCudaError, match="as_lo must have at least"):
        _cabi.afterstates_scan(env.lo, env.hi, acts, counts, *short, scratch, rows_out=rows, rows_cap=n * cap)
    torch.cuda.synchronize()
    assert (score == 7).all() and (q == 7).all() and (score_full == 7).all()
    assert int(rows.item()) == -5 and int(scratch.abs().sum().item()) == 0


def test_captured_graphs_follow_a_loaded_env_base():
    """env_base is a frozen kernel argument of every captured graph, like the seed: after load_state_dict() of a state
    with another env_base (same seed), the replays of AfterstateActor.step_graph(), HostPipeline.run() and the env's own
    step graph play the turns of a freshly built env given the same state."""
    import torch
    from gym_narde_b200 import VecNardeEnv, AfterstateMLP, AfterstateActor
    fn, head = _net()
    mlp = AfterstateMLP.from_module(fn, head)
    n, cap, depth = 2048, 64, 4
    src = VecNardeEnv(n, seed=11, max_actions=cap, env_base=5 * n)
    src.reset()
    for _ in range(20):
        src.step()
    sd = src.state_dict()

    def fresh():
        e = VecNardeEnv(n, seed=99, max_actions=cap)
        e.load_state_dict(sd)
        return e

    a = VecNardeEnv(n, seed=11, max_actions=cap)
    actor = AfterstateActor(a, mlp)
    a.reset()
    for _ in range(3):
        actor.step_graph()                  # captured with env_base 0
    a.load_state_dict(sd)
    b = fresh()
    actor_b = AfterstateActor(b, mlp)
    for t in range(3):
        actor.step_graph()
        actor_b.step()
        assert torch.equal(a.lo, b.lo) and torch.equal(a.hi, b.hi) and torch.equal(a.chosen, b.chosen), t

    a = VecNardeEnv(n, seed=11, max_actions=cap)
    a.reset()
    pipe = a.host_pipeline(depth=depth)
    pipe.run()
    a.step()                                # the env's own graph of a Philox-random step
    a.load_state_dict(sd)
    b = fresh()
    acts = torch.randint(0, 12, (depth, n), generator=torch.Generator().manual_seed(2), dtype=torch.int32)
    pipe.actions.copy_(acts)
    pipe.run()
    want_r = []
    for k in range(depth):
        b.step(acts[k].cuda())
        want_r.append(b.reward.cpu())
    torch.cuda.synchronize()
    assert torch.equal(a.lo, b.lo) and torch.equal(a.hi, b.hi) and torch.equal(pipe.reward, torch.stack(want_r))
    a.step()
    b.step()
    assert torch.equal(a.lo, b.lo) and torch.equal(a.hi, b.hi) and torch.equal(a.dice, b.dice)
