"""GPU (-m gpu): the tcgen05 afterstate-scoring MLP against the fp32 torch reference of the same net.

Architecture = DecomposedDQN.forward(x) with state_size 198 (train_deepq_pytorch.py:184-236),
torch.manual_seed(0) default nn.Linear init (BASELINE config 5: random-init weights).  This is the
one floating-point kernel of the path: tolerance (bf16 operands, fp32 accumulate) is stated below."""
import numpy as np
import pytest

from test_mlp_reference_cpu import bound, ref_q

pytestmark = pytest.mark.gpu

ABS_TOL = 5e-3          # |q_kernel - q_fp32| on Q-values of magnitude ~0.1-0.5 (measured 7e-4; SURVEY 7.10 asks <= 1e-2)
ARGMAX_AGREEMENT = 0.95  # floor only: bf16 rounding flips near-ties among 576 random-init Q-values; the measured figure is
                         # printed by __graft_entry__.smoke(), and every flip must be a near-tie (checked below)


def _reference_net():
    import torch
    import torch.nn as nn
    torch.manual_seed(0)
    feature_network = nn.Sequential(nn.Linear(198, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU())
    move1_head = nn.Linear(256, 576)
    return feature_network.cuda(), move1_head.cuda()


def test_mlp_matches_fp32_reference_on_real_observations():
    import torch
    from gym_narde_b200 import VecNardeEnv
    from gym_narde_b200.mlp import AfterstateMLP
    fn, head = _reference_net()
    mlp = AfterstateMLP.from_module(fn, head)
    env = VecNardeEnv(4096, seed=3)
    env.reset()
    for _ in range(40):
        obs, *_ = env.step()
    for rows in (4096, 1, 127, 129, 1000):
        x = obs[:rows].contiguous()
        q = mlp(x)
        with torch.no_grad():
            ref = head(fn(x))
        err = (q - ref).abs().max().item()
        assert err < ABS_TOL, (rows, err)
        if rows == 4096:
            am, rm = q.argmax(1), ref.argmax(1)
            agree = (am == rm).float().mean().item()
            assert agree > ARGMAX_AGREEMENT, agree
            # where the arg-max differs, the float64 net itself has the two candidates within the kernel's error
            # bound of each (a near-tie): gap <= bound[a_kernel] + bound[a_ref]
            W = tuple(lin.weight.data for lin in (fn[0], fn[2], head))
            b = tuple(lin.bias.data for lin in (fn[0], fn[2], head))
            ref64, bnd = ref_q(x, W, b, emulate=False), bound(x, W, b)
            am, rm = q.argmax(1), ref64.argmax(1)
            diff = am != rm
            gap = ref64.gather(1, rm[:, None]) - ref64.gather(1, am[:, None])
            lim = bnd.gather(1, rm[:, None]) + bnd.gather(1, am[:, None])
            assert (gap[diff] <= lim[diff]).all(), (gap[diff] - lim[diff]).max().item()
    # exactness of the data path: with bf16-representable weights/inputs the only error is accumulation order
    torch.manual_seed(1)
    xb = torch.randint(0, 2, (512, 198), device="cuda").float()
    for lin in (fn[0], fn[2], head):
        lin.weight.data = lin.weight.data.to(torch.bfloat16).float()
    mlp2 = AfterstateMLP.from_module(fn, head)
    with torch.no_grad():
        h1 = torch.relu(fn[0](xb)).to(torch.bfloat16).float()
        h2 = torch.relu(fn[2](h1)).to(torch.bfloat16).float()
        ref2 = head(h2)
    assert (mlp2(xb) - ref2).abs().max().item() < 2e-3


def test_mlp_state_input_and_score_modes_agree_with_forward():
    """The in-kernel Box(198) encoding (packed states in) feeds the MMAs the same bf16 operands as the
    fp32 observation rows, so Q-values are bit-identical; score = row max of those Q-values."""
    import torch
    from gym_narde_b200 import VecNardeEnv
    from gym_narde_b200.mlp import AfterstateMLP
    fn, head = _reference_net()
    mlp = AfterstateMLP.from_module(fn, head)
    env = VecNardeEnv(3000, seed=11)
    env.reset()
    for _ in range(70):                      # mid-game and bear-off positions, both colours to move
        env.step()
    obs = env.observe().clone()
    for rows in (3000, 1, 128, 129, 257, 1000):
        lo, hi, x = env.lo[:rows].contiguous(), env.hi[:rows].contiguous(), obs[:rows].contiguous()
        q = mlp.forward(x)
        qs = mlp.forward_states(lo, hi)
        assert torch.equal(q, qs), rows
        assert torch.equal(mlp.score(x), q.max(dim=1).values), rows
        assert torch.equal(mlp.score_states(lo, hi), q.max(dim=1).values), rows


def test_mlp_cluster_pair_variant_is_bit_identical():
    """The opt-in cluster-pair kernel (two CTAs share each weight stage through TMA multicast, stages released by
    tcgen05.commit multicast to both CTAs) computes the same bits as the default kernel, for ragged row counts
    (odd tile counts leave one CTA of a pair with empty rounds)."""
    import torch
    from gym_narde_b200 import VecNardeEnv, _cabi
    from gym_narde_b200.mlp import AfterstateMLP
    fn, head = _reference_net()
    mlp = AfterstateMLP.from_module(fn, head)
    env = VecNardeEnv(40000, seed=2)
    env.reset()
    for _ in range(50):
        env.step()
    lib = _cabi.load()
    for rows in (40000, 129, 1, 38017):
        lo, hi = env.lo[:rows].contiguous(), env.hi[:rows].contiguous()
        a_q, a_s = mlp.forward_states(lo, hi), mlp.score_states(lo, hi)
        lib.narde_mlp_use_cluster_pair(1)
        try:
            b_q, b_s = mlp.forward_states(lo, hi), mlp.score_states(lo, hi)
            torch.cuda.synchronize()
        finally:
            lib.narde_mlp_use_cluster_pair(0)
        assert torch.equal(a_q, b_q) and torch.equal(a_s, b_s), rows


def test_mlp_cta_group2_scorer_is_bit_identical():
    """k_mlp2sm: clusters of two CTAs, tcgen05.mma cta_group::2 (M = 256 over both CTAs' tiles, each CTA holds half
    of the B operand), peer hand-offs through remote mbarrier arrives and commit multicast.  Same bits as the
    default scorer, including ragged row counts that leave a CTA of the pair without rows."""
    import torch
    from gym_narde_b200 import VecNardeEnv
    from gym_narde_b200.mlp import AfterstateMLP
    fn, head = _reference_net()
    mlp = AfterstateMLP.from_module(fn, head)
    env = VecNardeEnv(50000, seed=8)
    env.reset()
    for _ in range(60):
        env.step()
    for rows in (50000, 1, 128, 129, 257, 40001):
        lo, hi = env.lo[:rows].contiguous(), env.hi[:rows].contiguous()
        a = mlp.score_states(lo, hi)
        b = mlp.score_states_2sm(lo, hi)
        torch.cuda.synchronize()
        assert torch.equal(a, b), rows


def test_mlp_move2_head_matches_fp32_reference():
    """DecomposedDQN.forward(x, selected_move1) (train_deepq_pytorch.py:203-233): the move2 Q-values, with the one-hot
    half of move2_head applied as a gathered weight column in the kernel's epilogue.  Same tolerance as forward(x);
    the fp32 observation rows and the packed states give bit-identical results."""
    import torch
    import torch.nn as nn
    from gym_narde_b200 import VecNardeEnv
    from gym_narde_b200.mlp import AfterstateMLP
    fn, head = _reference_net()
    move2_head = nn.Linear(256 + 576, 576).cuda()      # drawn after move1_head from the same generator, as in the reference
    mlp = AfterstateMLP.from_module(fn, head, move2_head)
    env = VecNardeEnv(3000, seed=5)
    env.reset()
    for _ in range(50):
        env.step()
    obs = env.observe().clone()
    g = torch.Generator(device="cuda").manual_seed(7)
    for rows in (3000, 1, 127, 129, 1000):
        x = obs[:rows].contiguous()
        m1 = torch.randint(0, 576, (rows,), device="cuda", generator=g)
        q2 = mlp.forward(x, m1)
        with torch.no_grad():
            feats = fn(x)
            onehot = torch.zeros(rows, 576, device="cuda").scatter_(1, m1.unsqueeze(1), 1)
            ref = move2_head(torch.cat((feats, onehot), dim=1))
        err = (q2 - ref).abs().max().item()
        assert err < ABS_TOL, (rows, err)
        assert torch.equal(q2, mlp.forward_states(env.lo[:rows].contiguous(), env.hi[:rows].contiguous(), m1)), rows
        # the move1 path is untouched by the extra mode
        with torch.no_grad():
            assert (mlp.forward(x) - head(feats)).abs().max().item() < ABS_TOL
    # edge codes 0 and 575, int32 and int64 index tensors
    x = obs[:256].contiguous()
    for code in (0, 575):
        m1 = torch.full((256,), code, device="cuda", dtype=torch.int32)
        with torch.no_grad():
            ref = fn(x) @ move2_head.weight[:, :256].t() + move2_head.weight[:, 256 + code] + move2_head.bias
        assert (mlp.forward(x, m1) - ref).abs().max().item() < ABS_TOL
    mlp_no = AfterstateMLP.from_module(fn, head)
    with pytest.raises(Exception):
        mlp_no.forward(x, m1)
