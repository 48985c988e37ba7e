"""GPU (-m gpu): the tcgen05 afterstate MLP (k_mlp, k_mlp2sm in gym_narde_b200/csrc/narde_mlp.cu) against the float64
reference of test_mlp_reference_cpu.py.

- Exact designs (dyadic weights and inputs, every partial sum an fp32 value): every entry, with and without the
  cluster-pair kernel, at row counts that cross tile, slot-pair and persistent-round boundaries, must equal the
  emulating reference bit for bit.
- The score epilogue: a planted maximum in every column block and half, all-negative rows, row-dependent arg-max.
- Realistic weights: |kernel - plain float64 net| <= bound() element by element, at three weight scales and with
  every Q-value negative.
- Stores stop at the row count, rows_dev clamps to [0, K] (also between replays of one CUDA graph), and row offsets
  past 2^31 elements of Q are addressed correctly.
"""
import contextlib

import numpy as np
import pytest
import torch

from test_mlp_reference_cpu import (EXACT_DESIGNS, OUT, argmax_design, bound, check_premise, default_net,
                                    move1_codes, planted_design, ref_q, synthetic_states)

pytestmark = pytest.mark.gpu

ROUND = 148 * 2 * 128          # rows of one persistent round: 148 CTAs x 2 slots x 128 rows
ROWS = (1, 127, 128, 129, 255, 256, 257, ROUND, ROUND + 1, 2 * ROUND + 129, 3 * ROUND + 77)
SENTINEL = 0x7FC0DEAD          # a NaN bit pattern no kernel writes


@contextlib.contextmanager
def cluster_pair(on):
    from gym_narde_b200 import _cabi
    lib = _cabi.load()
    lib.narde_mlp_use_cluster_pair(1 if on else 0)
    try:
        yield
    finally:
        lib.narde_mlp_use_cluster_pair(0)


def _mlp(d):
    from gym_narde_b200.mlp import AfterstateMLP
    w_move2 = torch.cat([d["W3m"], d["w2b_t"].T], dim=1)
    return AfterstateMLP(d["W"][0], d["b"][0], d["W"][1], d["b"][1], d["W"][2], d["b"][2], w_move2, d["b3m"])


def _cuda(d):
    return {k: (tuple(t.cuda() for t in v) if isinstance(v, tuple) else v.cuda()) for k, v in d.items()}


@pytest.fixture(scope="module")
def inputs():
    """3 * ROUND + 77 rows: real positions of played games (both colours to move, some bearing off) interleaved with
    synthetic ones (every point count, every off count); Box(198) rows from the host decoder; move1 codes."""
    from gym_narde_b200 import VecNardeEnv
    from gym_narde_b200.state import expand_obs198
    n = ROWS[-1]
    env = VecNardeEnv(n // 2, seed=21)
    env.reset()
    for _ in range(60):
        env.step()
    lo_r, hi_r = env.lo.cpu().numpy(), env.hi.cpu().numpy()
    lo_s, hi_s = synthetic_states(n - n // 2, 22)
    perm = np.random.default_rng(23).permutation(n)
    lo, hi = np.concatenate([lo_r, lo_s])[perm], np.concatenate([hi_r, hi_s])[perm]
    x = expand_obs198(lo, hi)
    del env
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return dict(lo=t(lo), hi=t(hi), x=t(x), m1=move1_codes(n, 24).cuda())


def _exact_ref(d, data, move2):
    W = (d["W"][0], d["W"][1], d["W3m"] if move2 else d["W"][2])
    b = (d["b"][0], d["b"][1], d["b3m"] if move2 else d["b"][2])
    m1 = data["m1"] if move2 else None
    q = check_premise(data["x"], W, b, move1=m1, w2b_t=d["w2b_t"])
    assert torch.equal(q, ref_q(data["x"], W, b, move1=m1, w2b_t=d["w2b_t"]))
    q32 = q.float()
    assert torch.equal(q32.double(), q)
    return q32


def _first_mismatch(got, want):
    bad = (got != want).nonzero()
    i = tuple(bad[0].tolist())
    return "%d mismatches, first at %s: kernel %r, reference %r" % (len(bad), i, got[i].item(), want[i].item())


def _entries(mlp, data):
    """name -> (call(K), reference key): the seven entries of the kernel."""
    lo, hi, x, m1 = data["lo"], data["hi"], data["x"], data["m1"]
    return {
        "forward": (lambda k: mlp.forward(x[:k]), "q"),
        "score": (lambda k: mlp.score(x[:k]), "s"),
        "forward_states": (lambda k: mlp.forward_states(lo[:k], hi[:k]), "q"),
        "score_states": (lambda k: mlp.score_states(lo[:k], hi[:k]), "s"),
        "score_states_2sm": (lambda k: mlp.score_states_2sm(lo[:k], hi[:k]), "s"),
        "forward_move2": (lambda k: mlp.forward(x[:k], m1[:k]), "q2"),
        "forward_states_move2": (lambda k: mlp.forward_states(lo[:k], hi[:k], m1[:k]), "q2"),
    }


@pytest.mark.parametrize("design", sorted(EXACT_DESIGNS))
def test_exact_design_is_bit_exact_on_every_entry(design, inputs):
    d = _cuda(EXACT_DESIGNS[design]())
    ref = {"q": _exact_ref(d, inputs, False), "q2": _exact_ref(d, inputs, True)}
    ref["s"] = ref["q"].max(1).values
    mlp = _mlp(d)
    for name, (call, key) in _entries(mlp, inputs).items():
        for pair in ((False,) if name == "score_states_2sm" else (False, True)):
            with cluster_pair(pair):
                for k in ROWS:
                    got = call(k)
                    want = ref[key][:k]
                    assert torch.equal(got, want), (design, name, "pair" if pair else "default", k,
                                                    _first_mismatch(got, want))


@pytest.mark.parametrize("top", [3.0, -1.0])
def test_score_finds_a_planted_maximum_in_every_block_and_half(top, inputs):
    """Layer 3 = 0, every bias -5 but one: the score is that bias, wherever its column is (both halves of every
    job, both sides of each 32-column chunk) and also when the whole row is negative."""
    lo, hi, x = inputs["lo"], inputs["hi"], inputs["x"]
    for col in (0, 31, 32, 127, 128, 255, 256, 383, 384, 511, 512, 543, 544, 575):
        mlp = _mlp(_cuda(planted_design(col, top)))
        for k in (257, ROUND + 1):
            want = torch.full((k,), top, device="cuda")
            runs = {"score_states_2sm": mlp.score_states_2sm(lo[:k], hi[:k])}
            for pair in (False, True):
                with cluster_pair(pair):
                    runs["score/%d" % pair] = mlp.score(x[:k])
                    runs["score_states/%d" % pair] = mlp.score_states(lo[:k], hi[:k])
            for name, got in runs.items():
                assert torch.equal(got, want), (col, top, k, name, _first_mismatch(got, want))


def test_score_follows_a_row_dependent_argmax(inputs):
    d = _cuda(argmax_design())
    q = check_premise(inputs["x"], d["W"], d["b"])
    a = q.argmax(1)
    for c0, n in ((0, 128), (128, 128), (256, 128), (384, 128), (512, 32), (544, 32)):
        assert ((a >= c0) & (a < c0 + n)).any(), c0           # the design peaks in every block and half
    want = q.float().max(1).values
    mlp = _mlp(d)
    lo, hi, x = inputs["lo"], inputs["hi"], inputs["x"]
    k = len(want)
    runs = {"score_states_2sm": mlp.score_states_2sm(lo, hi)}
    for pair in (False, True):
        with cluster_pair(pair):
            runs["score/%d" % pair] = mlp.score(x)
            runs["score_states/%d" % pair] = mlp.score_states(lo, hi)
    for name, got in runs.items():
        assert torch.equal(got, want[:k]), (name, _first_mismatch(got, want))


def _realistic(kind):
    if kind == "he":
        g = torch.Generator().manual_seed(9)
        W = tuple(torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5 for o, i in ((256, 198), (256, 256), (576, 256)))
        b = (torch.zeros(256), torch.zeros(256), torch.zeros(576))
        return W, b
    return default_net(0, float(kind))


@pytest.mark.parametrize("kind", ["1", "4", "16", "he"])
def test_realistic_weights_stay_within_the_float64_bound(kind):
    """Default nn.Linear init times 1, 4 and 16, and a He init whose layer-3 bias makes every Q-value negative:
    |q - plain float64 net| <= bound() element by element, on 4096 observations of played games (fp32 rows) and
    40 000 packed states (multi-round)."""
    from gym_narde_b200 import VecNardeEnv
    from gym_narde_b200.mlp import AfterstateMLP
    from gym_narde_b200.state import expand_obs198
    W, b = _realistic(kind)
    W, b = tuple(w.cuda() for w in W), tuple(v.cuda() for v in b)
    env = VecNardeEnv(40000, seed=31)
    env.reset()
    for _ in range(50):
        env.step()
    lo, hi = env.lo.clone(), env.hi.clone()
    x_states = torch.from_numpy(expand_obs198(lo.cpu().numpy(), hi.cpu().numpy())).cuda()
    x_obs = env.observe()[:4096].contiguous()
    del env
    if kind == "he":
        top = ref_q(torch.cat([x_obs, x_states]), W, b, emulate=False).max().item()
        b = (b[0], b[1], b[2] - (top + 1.0))
    mlp = AfterstateMLP(W[0], b[0], W[1], b[1], W[2], b[2])
    worst = 0.0
    for x, runs in ((x_obs, {"forward": lambda: mlp.forward(x_obs), "score": lambda: mlp.score(x_obs)}),
                    (x_states, {"forward_states": lambda: mlp.forward_states(lo, hi),
                                "score_states": lambda: mlp.score_states(lo, hi),
                                "score_states_2sm": lambda: mlp.score_states_2sm(lo, hi)})):
        plain, bnd = ref_q(x, W, b, emulate=False), bound(x, W, b)
        if kind == "he":
            assert (plain < 0).all()
        for name, run in runs.items():
            got = run().double()
            if got.dim() == 1:
                err, lim = (got - plain.max(1).values).abs(), bnd.max(1).values
            else:
                err, lim = (got - plain).abs(), bnd
            ratio = (err / lim).max().item()
            worst = max(worst, ratio)
            assert ratio <= 1.0, (kind, name, ratio, err.max().item())
    print("realistic weights %s: largest err/bound %.3f" % (kind, worst))


def _nan_buffer(*shape):
    return torch.full(shape, SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


def _bits(t):
    return t.view(torch.int32)


def test_stores_stop_at_the_row_count(inputs):
    """out = big[:K] of a NaN-filled buffer: every entry fills rows < K and leaves big[K:] bitwise untouched."""
    d = _cuda(EXACT_DESIGNS["perm"]())
    mlp = _mlp(d)
    lo, hi, x, m1 = inputs["lo"], inputs["hi"], inputs["x"], inputs["m1"]
    for k in (1, 129, ROUND + 1):
        calls = {
            "forward": (OUT, lambda o: mlp.forward(x[:k], out=o)),
            "forward_states": (OUT, lambda o: mlp.forward_states(lo[:k], hi[:k], out=o)),
            "forward_move2": (OUT, lambda o: mlp.forward(x[:k], m1[:k], out=o)),
            "forward_states_move2": (OUT, lambda o: mlp.forward_states(lo[:k], hi[:k], m1[:k], out=o)),
            "score": (None, lambda o: mlp.score(x[:k], out=o)),
            "score_states": (None, lambda o: mlp.score_states(lo[:k], hi[:k], out=o)),
            "score_states_2sm": (None, lambda o: mlp.score_states_2sm(lo[:k], hi[:k], out=o)),
        }
        for name, (cols, call) in calls.items():
            for pair in ((False,) if name == "score_states_2sm" else (False, True)):
                big = _nan_buffer(k + 300, *(() if cols is None else (cols,)))
                with cluster_pair(pair):
                    call(big[:k])
                    want = call(None)
                assert torch.equal(big[:k], want), (name, pair, k)
                assert (_bits(big[k:]) == SENTINEL).all(), (name, pair, k)


def _rows_dev_cases(k):
    return (0, -5, 1, k - 1, k, k + 1000)


def test_rows_dev_is_clamped_to_zero_and_the_row_count(inputs):
    """score_states / score_states_2sm with a device row count: rows below min(max(rows_dev, 0), K) equal the
    result without it, every other row keeps the sentinel.  lo / hi / out are prefixes of larger buffers, so even a
    kernel that ignored the clamp would stay inside its allocations, and show."""
    d = _cuda(EXACT_DESIGNS["sparse"]())
    mlp = _mlp(d)
    k = ROUND + 1
    lo, hi = inputs["lo"][:k], inputs["hi"][:k]      # rows k.. of the same buffers exist
    full = mlp.score_states(lo, hi)
    calls = {"score_states": lambda o, rd: mlp.score_states(lo, hi, out=o, rows_dev=rd),
             "score_states_2sm": lambda o, rd: mlp.score_states_2sm(lo, hi, out=o, rows_dev=rd)}
    for name, call in calls.items():
        for pair in ((False,) if name == "score_states_2sm" else (False, True)):
            for rd in _rows_dev_cases(k):
                big = _nan_buffer(k + 1100)
                with cluster_pair(pair):
                    call(big[:k], torch.tensor([rd], dtype=torch.int64, device="cuda"))
                n = min(max(rd, 0), k)
                assert torch.equal(big[:n], full[:n]), (name, pair, rd)
                assert (_bits(big[n:]) == SENTINEL).all(), (name, pair, rd)


@pytest.mark.parametrize("name", ["score_states", "score_states_2sm"])
def test_rows_dev_changes_between_graph_replays(name, inputs):
    d = _cuda(EXACT_DESIGNS["sparse"]())
    mlp = _mlp(d)
    k = 2 * ROUND + 129
    lo, hi = inputs["lo"][:k], inputs["hi"][:k]
    full = mlp.score_states(lo, hi)
    big = _nan_buffer(k + 1100)
    rd = torch.tensor([k], dtype=torch.int64, device="cuda")
    run = getattr(mlp, name)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run(lo, hi, out=big[:k], rows_dev=rd)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run(lo, hi, out=big[:k], rows_dev=rd)
    for v in _rows_dev_cases(k) + (ROUND, 129):
        _bits(big).fill_(SENTINEL)
        rd.fill_(v)
        g.replay()
        torch.cuda.synchronize()
        n = min(max(v, 0), k)
        assert torch.equal(big[:n], full[:n]), (name, v)
        assert (_bits(big[n:]) == SENTINEL).all(), (name, v)
    del g


def test_q_rows_past_2_to_the_31_elements(inputs):
    """forward_states at 3 800 000 rows: element offsets of Q pass 2^31 (row 3 728 271).  The input repeats the
    113 741-row set (a period that is not a multiple of the 128-row tile), so every period must equal the same exact
    reference."""
    d = _cuda(EXACT_DESIGNS["perm"]())
    mlp = _mlp(d)
    want = _exact_ref(d, inputs, False)
    period = want.shape[0]
    n = 3_800_000
    assert (n - 1) * OUT > 2 ** 31
    reps = -(-n // period)
    lo = inputs["lo"].repeat(reps, 1)[:n].contiguous()
    hi = inputs["hi"].repeat(reps, 1)[:n].contiguous()
    q = mlp.forward_states(lo, hi)
    torch.cuda.synchronize()
    try:
        for r0 in range(0, n, period):
            got = q[r0:r0 + period]
            assert torch.equal(got, want[:got.shape[0]]), (r0, _first_mismatch(got, want[:got.shape[0]]))
    finally:
        del q, lo, hi
        torch.cuda.empty_cache()
