"""A float64 reference of the tcgen05 afterstate MLP (gym_narde_b200/csrc/narde_mlp.cu), its error bound, the exact
test designs, and the CPU checks of all three plus the packed weight layout.

test_gpu_mlp_reference.py runs the kernel against what this module computes:
- ref_q(emulate=True) follows the kernel's data path (bf16 operands, fp32 bias, ReLU, bf16 hidden activations);
  ref_q(emulate=False) is the plain float64 net.
- bound() is a first-order bound on |kernel - plain float64|, element by element, that scales with the weights.
- The exact designs have dyadic weights, biases and inputs whose partial sums all fit in fp32 (check_premise), so
  the kernel's output does not depend on the order it accumulates in and must equal ref_q(emulate=True) bit for bit.
"""
import math
import os
import re

import numpy as np
import pytest
import torch

from gym_narde_b200.mlp import pack_weights
from gym_narde_b200.state import expand_obs198, pack_states

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MLP_CU = os.path.join(ROOT, "gym_narde_b200", "csrc", "narde_mlp.cu")

IN, HID, OUT, K1 = 198, 256, 576, 208
FRAC = (97, 195)          # the off/15 features of Box(198): the only inputs that are not multiples of 1/2
U_BF16 = 2.0 ** -8        # unit roundoff of bf16 (8 significant bits, round to nearest even)
U_FP32 = 2.0 ** -24
PREMISE_BITS = 16         # every partial sum within 2^16 quanta: 8 bits of margin below fp32's 24


# ---------------------------------------------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------------------------------------------
def bf16(t):
    """The kernel's rounding of an fp32 value to bf16 (round to nearest even), back in float64."""
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def clamp_move1(move1):
    return move1.to(torch.int64).clamp(0, OUT - 1)


def ref_q(x, W, b, move1=None, w2b_t=None, emulate=True):
    """Q-values [K, 576] in float64.  W = (w1, w2, w3) as torch Linear weights ([out, in]), b = (b1, b2, b3).
    move1 (with w2b_t [576, 576]): the move2 mode, layer 3 plus the fp32 row w2b_t[clamp(move1, 0, 575)].
    emulate=True mirrors the kernel: x and W rounded to bf16, products summed in float64 plus the fp32 bias, ReLU,
    hidden activations rounded to bf16 before the next layer.  emulate=False is the plain float64 net."""
    r = bf16 if emulate else (lambda t: t.to(torch.float64))
    h = r(x)
    for w, bb in zip(W[:2], b[:2]):
        h = torch.relu(h @ r(w).T + bb.to(torch.float64))
        if emulate:
            h = bf16(h)
    q = h @ r(W[2]).T + b[2].to(torch.float64)
    if move1 is not None:
        q = q + w2b_t.to(torch.float64)[clamp_move1(move1)]
    return q


def bound(x, W, b, move1=None, w2b_t=None):
    """Bound on |kernel - ref_q(emulate=False)| per element of Q, in float64.

    The kernel rounds x and W to bf16 exactly as ref_q(emulate=True) does; what it may do differently is the order of
    its fp32 sums, whose error is at most n * U_FP32 times the sum of |terms| for n terms (products, bias, and the
    move2 gather; bf16 products are exact in fp32).  Those errors are carried through the layers as intervals around
    the kernel's possible activations: |W| widens them, and ReLU and the bf16 rounding of the hidden activations are
    monotone, so the interval's end points map to end points (a rounding that may go either way widens the interval
    by that one bf16 step).  The output's interval, plus its centre's distance from the plain float64 net, bounds the
    kernel's error.  It scales with the weights, unlike a fixed tolerance, and is tight enough to be useful: the worst
    case of the first-order propagation through |W| alone is about 1000 times the observed error.  Most of the error
    is the bf16 rounding, which the bound knows exactly, so a kernel's err / bound is close to (but at most) 1."""
    lo = hi = bf16(x)
    plain = x.to(torch.float64)
    for layer in range(3):
        w, bb = bf16(W[layer]), b[layer].to(torch.float64)
        wa = w.abs()
        c, r = (lo + hi) / 2, (hi - lo) / 2
        zc = c @ w.T + bb
        mag = torch.maximum(lo.abs(), hi.abs()) @ wa.T + bb.abs()
        plain = plain @ W[layer].to(torch.float64).T + bb
        n_terms = w.shape[1] + 1
        if layer == 2 and move1 is not None:
            gather = w2b_t.to(torch.float64)[clamp_move1(move1)]
            zc, plain, mag = zc + gather, plain + gather, mag + gather.abs()
            n_terms += 1
        # + float64 slack: zc is itself a float64 sum of n_terms terms
        zr = r @ wa.T + n_terms * (U_FP32 + 2.0 ** -50) * mag
        if layer == 2:
            return (zc - plain).abs() + zr
        lo, hi = bf16(torch.relu(zc - zr)), bf16(torch.relu(zc + zr))
        plain = torch.relu(plain)


def _quantum(t):
    """Largest power of two dividing each float64 element (inf for 0)."""
    m, ex = torch.frexp(t)
    mant = (m.abs() * 2.0 ** 53).to(torch.int64)
    low = mant & -mant
    q = torch.ldexp(low.to(torch.float64), ex.to(torch.float64) - 53)
    return torch.where(t == 0, torch.full_like(t, math.inf), q)


def check_premise(x, W, b, move1=None, w2b_t=None, chunk=8192):
    """Asserts that the design is exact: weights are bf16 values and, for every output of every layer, the sum of
    |terms| (products, bias, and the move2 gather) is at most 2^16 times the largest power of two dividing all of
    them -- so every partial sum, in any order, is an exact fp32 value.  W must be sparse (a few nonzeros per row).
    Returns the emulated Q-values in float64, summed term by term: a second computation of ref_q(emulate=True)."""
    Wd = [w.to(torch.float64) for w in W]
    for layer, w in enumerate(Wd):
        assert torch.equal(bf16(w), w), "layer %d weights are not bf16 values" % layer
    sparse = []
    for w in Wd:
        nz = w != 0
        nnz = int(nz.sum(1).max())
        idx = torch.argsort(nz.to(torch.int8), dim=1, descending=True, stable=True)[:, :nnz]
        sparse.append((idx, w.gather(1, idx)))
    out = []
    for r0 in range(0, x.shape[0], chunk):
        h = bf16(x[r0:r0 + chunk])
        for layer, (idx, vals) in enumerate(sparse):
            terms = [h[:, idx] * vals, b[layer].to(torch.float64)[None, :, None].expand(h.shape[0], -1, 1)]
            if layer == 2 and move1 is not None:
                terms.append(w2b_t.to(torch.float64)[clamp_move1(move1[r0:r0 + chunk])][:, :, None])
            terms = torch.cat(terms, dim=2)
            s_abs, q = terms.abs().sum(2), _quantum(terms).amin(2)
            bad = s_abs > 2.0 ** PREMISE_BITS * q
            assert not bad.any(), "premise fails at layer %d, output (row, col) %s: sum|terms| %s, quantum %s" % (
                layer, tuple((bad.nonzero()[0] + torch.tensor([r0, 0], device=bad.device)).tolist()),
                s_abs[bad][0].item(), q[bad][0].item())
            h = terms.sum(2)
            if layer < 2:
                h = bf16(torch.relu(h))
        out.append(h)
    return torch.cat(out)


# ---------------------------------------------------------------------------------------------------------------
# designs: dict(W=(w1, w2, w3), b=(b1, b2, b3), W3m, b3m, w2b_t) of float32 CPU tensors.  W3m / b3m: the first 256
# input columns and bias of move2_head (different from the move1 head, so a mix-up of the two packs shows);
# w2b_t[m] = move2_head.weight[:, 256 + m]
# ---------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _randint(g, lo, hi, shape):
    return torch.randint(lo, hi, shape if isinstance(shape, tuple) else (shape,), generator=g)


def _sign(g, n):
    return (_randint(g, 0, 2, n) * 2 - 1).to(torch.float64)


def _head(g, src, n_in):
    """Layer 3 of the chain designs: column c reads hidden unit src[c] with weight +-2^{-1,0,1}; bias in 2^-4 steps."""
    w = torch.zeros(OUT, n_in, dtype=torch.float64)
    w[torch.arange(OUT), src] = _sign(g, OUT) * 2.0 ** _randint(g, -1, 2, OUT).to(torch.float64)
    return w, _randint(g, -128, 129, OUT).to(torch.float64) / 16


def _every_unit_read(g):
    """576 hidden-unit indices, every one of the 256 units read at least twice, in random column order."""
    src = torch.cat([torch.randperm(HID, generator=g), torch.randperm(HID, generator=g),
                     torch.randperm(HID, generator=g)[:OUT - 2 * HID]])
    return src[torch.randperm(OUT, generator=g)]


def _finish(W, b, W3m, b3m, g):
    w2b_t = _randint(g, -64, 65, (OUT, OUT)).to(torch.float64) / 16
    f = lambda t: t.to(torch.float32)
    return dict(W=tuple(map(f, W)), b=tuple(map(f, b)), W3m=f(W3m), b3m=f(b3m), w2b_t=f(w2b_t))


def perm_design(seed=0):
    """Signed permutation chain.  Hidden unit n of layer 1 reads input src1[n] (all 198 inputs are read, 58 of them
    twice) with weight +-2^{-1,0,1}; layer 2 is a signed scaled permutation; each of the 576 outputs reads one hidden
    unit.  Biases keep every routed value positive through ReLU and every hidden value a bf16 value: on integer-ish
    paths h = 2^e (x + m) or 2^e (7 + m - x) (x a multiple of 1/2 in [0, 6], m in 0..3), then 2^e' (h' + m) or
    2^e' (11 + m - h'); the off/15 paths keep weight +1 and bias 0.  A transposed, shifted or dropped (n, k) anywhere
    gives a wrong value in a known column."""
    g = _gen(1000 + seed)
    src1 = torch.cat([torch.randperm(IN, generator=g), _randint(g, 0, IN, HID - IN)])[torch.randperm(HID, generator=g)]
    frac1 = (src1 == FRAC[0]) | (src1 == FRAC[1])
    e1 = torch.where(frac1, 0, _randint(g, -1, 2, HID)).to(torch.float64)
    s1 = torch.where(frac1, 1.0, _sign(g, HID))
    m1 = _randint(g, 0, 4, HID).to(torch.float64)
    w1 = torch.zeros(HID, IN, dtype=torch.float64)
    w1[torch.arange(HID), src1] = s1 * 2.0 ** e1
    b1 = torch.where(frac1, 0.0, torch.where(s1 > 0, m1, 7 + m1) * 2.0 ** e1)
    src2 = torch.randperm(HID, generator=g)
    frac2 = frac1[src2]
    e2 = torch.where(frac2, 0, _randint(g, -1, 2, HID)).to(torch.float64)
    s2 = torch.where(frac2, 1.0, _sign(g, HID))
    m2 = _randint(g, 0, 4, HID).to(torch.float64)
    w2 = torch.zeros(HID, HID, dtype=torch.float64)
    w2[torch.arange(HID), src2] = s2 * 2.0 ** e2
    b2 = torch.where(frac2, 0.0, torch.where(s2 > 0, m2, 11 + m2) * 2.0 ** (e1[src2] + e2))
    w3, b3 = _head(g, _every_unit_read(g), HID)
    w3m, b3m = _head(g, _every_unit_read(g), HID)
    return _finish((w1, w2, w3), (b1, b2, b3), w3m, b3m, g)


def _sparse(g, n_out, n_in, nnz, e, cols):
    """n_out x n_in with nnz nonzeros per row, at distinct columns drawn from `cols`, values +-{1, 2} * 2^-e."""
    w = torch.zeros(n_out, n_in, dtype=torch.float64)
    cols = torch.as_tensor(cols)
    for n in range(n_out):
        k = cols[torch.randperm(len(cols), generator=g)[:nnz]]
        w[n, k] = _sign(g, nnz) * _randint(g, 1, 3, nnz).to(torch.float64) * 2.0 ** -e
    return w


def sparse_design(seed=0):
    """Sparse small-integer blocks: six nonzeros per row in layers 1 and 2, four per output in layer 3, values
    +-{1, 2} * 2^-e, scattered over every K stage (real accumulation, not routing); the off/15 inputs are left to
    off15_design."""
    g = _gen(2000 + seed)
    cols1 = [k for k in range(IN) if k not in FRAC]
    w1 = _sparse(g, HID, IN, 6, 2, cols1)
    b1 = _randint(g, 0, 17, HID).to(torch.float64) / 8
    w2 = _sparse(g, HID, HID, 6, 2, range(HID))
    b2 = _randint(g, 0, 17, HID).to(torch.float64) / 8
    w3 = _sparse(g, OUT, HID, 4, 3, range(HID))
    w3m = _sparse(g, OUT, HID, 4, 3, range(HID))
    b3, b3m = (_randint(g, -128, 129, OUT).to(torch.float64) / 16 for _ in range(2))
    return _finish((w1, w2, w3), (b1, b2, b3), w3m, b3m, g)


def off15_design(seed=0):
    """Layer 1 reads only the two off/15 inputs (97: White's, 195: Black's; K stages 3 and 6, the second in the 16-K
    tail stage): h = relu(a x97 + c x195 + b), a, c in {0, +-1, +-2}; bf16(n/15) has a 2^-11 quantum.  Layer 2 is a
    permutation, each output reads one hidden unit with weight +-1."""
    g = _gen(3000 + seed)
    w1 = torch.zeros(HID, IN, dtype=torch.float64)
    ac = _randint(g, -2, 3, (HID, 2)).to(torch.float64)
    ac[(ac == 0).all(1), 0] = 1.0
    w1[:, FRAC[0]], w1[:, FRAC[1]] = ac[:, 0], ac[:, 1]
    b1 = _randint(g, 2, 5, HID).to(torch.float64)
    w2 = torch.zeros(HID, HID, dtype=torch.float64)
    w2[torch.arange(HID), torch.randperm(HID, generator=g)] = 1.0
    b2 = torch.zeros(HID, dtype=torch.float64)
    heads = []
    for _ in range(2):
        src = _every_unit_read(g)
        w = torch.zeros(OUT, HID, dtype=torch.float64)
        w[torch.arange(OUT), src] = _sign(g, OUT)
        heads += [w, _randint(g, -128, 129, OUT).to(torch.float64) / 16]
    return _finish((w1, w2, heads[0]), (b1, b2, heads[1]), heads[2], heads[3], g)


def argmax_design(seed=0):
    """Row-dependent arg-max: hidden unit u < 48 carries the (n-3)/2 excess feature of one colour on one point
    (inputs 4p+3 and 98+4p+3, values 0..6 in halves); output c reads unit c mod 48 with weight 1, and distinct biases
    pi(c) * 2^-10 break ties.  The arg-max of a row is the column, among those reading its largest excess, with the
    largest pi: it lands in every column block and half across positions."""
    g = _gen(4000 + seed)
    feats = [4 * p + 3 for p in range(24)] + [98 + 4 * p + 3 for p in range(24)]
    w1 = torch.zeros(HID, IN, dtype=torch.float64)
    w1[torch.arange(48), torch.tensor(feats)] = 1.0
    w2 = torch.zeros(HID, HID, dtype=torch.float64)
    w2[torch.arange(48), torch.arange(48)] = 1.0
    z = torch.zeros(HID, dtype=torch.float64)
    w3 = torch.zeros(OUT, HID, dtype=torch.float64)
    w3[torch.arange(OUT), torch.arange(OUT) % 48] = 1.0
    b3 = torch.randperm(OUT, generator=g).to(torch.float64) * 2.0 ** -10
    return _finish((w1, w2, w3), (z, z, b3), w3, b3, g)


def planted_design(col, top, seed=0):
    """Layer 3 weights 0, every bias -5 except column `col` (bias `top`): every row's score is exactly `top`.
    Layers 1 and 2: the default nn.Linear init (they only feed zeros)."""
    g = _gen(5000 + seed)
    w1 = (torch.rand(HID, IN, generator=g, dtype=torch.float64) * 2 - 1) / math.sqrt(IN)
    w2 = (torch.rand(HID, HID, generator=g, dtype=torch.float64) * 2 - 1) / math.sqrt(HID)
    b1 = (torch.rand(HID, generator=g, dtype=torch.float64) * 2 - 1) / math.sqrt(IN)
    b2 = (torch.rand(HID, generator=g, dtype=torch.float64) * 2 - 1) / math.sqrt(HID)
    w3 = torch.zeros(OUT, HID, dtype=torch.float64)
    b3 = torch.full((OUT,), -5.0, dtype=torch.float64)
    b3[col] = top
    return _finish((w1, w2, w3), (b1, b2, b3), w3, b3, g)


EXACT_DESIGNS = {"perm": perm_design, "sparse": sparse_design, "off15": off15_design}


def synthetic_states(n, seed):
    """n packed states through the package's own encoder: every point empty with probability 1/2, else +-1..15;
    off counts 0..15 for both colours; either side to move.  The kernel only decodes bytes, so the positions need
    not be reachable."""
    rng = np.random.default_rng(seed)
    boards = rng.integers(1, 16, (n, 24)) * rng.choice([-1, 1], (n, 24)) * (rng.random((n, 24)) < 0.5)
    return pack_states(boards, off_w=rng.integers(0, 16, n), off_b=rng.integers(0, 16, n),
                       turn=rng.choice([-1, 1], n))


def move1_codes(n, seed):
    """Per-row first-move codes: random in [0, 576), with 0, 575 and the out-of-range -1, 576 and 2^31 - 1 (which
    must act as 0, 575, 575) in the first rows and every 11th row."""
    rng = np.random.default_rng(seed)
    m = rng.integers(0, OUT, n).astype(np.int64)
    special = np.array([2 ** 31 - 1, 0, 575, -1, 576], np.int64)
    m[0::11] = special[np.arange(len(m[0::11])) % len(special)]
    m[:len(special)] = special[:n]
    return torch.from_numpy(m.astype(np.int32))


def default_net(seed=0, scale=1.0):
    """nn.Linear's default init of the three layers (torch.manual_seed(seed)), every weight and bias times `scale`."""
    import torch.nn as nn
    torch.manual_seed(seed)
    layers = [nn.Linear(IN, HID), nn.Linear(HID, HID), nn.Linear(HID, OUT)]
    return (tuple(l.weight.data * scale for l in layers), tuple(l.bias.data * scale for l in layers))


# ---------------------------------------------------------------------------------------------------------------
# packed weight layout (mlp.pack_weights) against the kernel's job table
# ---------------------------------------------------------------------------------------------------------------
def kernel_jobs():
    """The five GEMM jobs (w_off, nb, k, b_off, col0) of c_jobs in narde_mlp.cu, evaluated from the source."""
    src = open(MLP_CU).read()
    consts = dict(re.findall(r"constexpr int (k\w+) = (\d+);", src))
    body = re.search(r"Job c_jobs\[5\] = \{(.*?)\};", src, re.S).group(1)
    jobs = []
    for row in re.findall(r"\{([^{}]*)\}", body):
        fields = []
        for f in row.split(","):
            expr = re.sub(r"\bk\w+\b", lambda m: consts[m.group(0)], f)
            assert re.fullmatch(r"[\d\s*+\-()]+", expr), expr
            fields.append(eval(expr))
        jobs.append(tuple(fields))
    assert len(jobs) == 5
    return jobs


def decode_pack(wpack, jobs, two_sm=False):
    """Inverse of the documented layout, written from the description alone: per job block, stages of 32 K (the
    last one shorter), each nb x klen at offset(n, k) = (k/8)*(nb*16) + (n/8)*128 + (n%8)*16 + (k%8)*2 bytes;
    two_sm: each stage is [rows 0..nb/2 | rows nb/2..nb], every half in that layout with nb/2 rows.
    Returns the [nb, k] bf16 bit patterns (uint16) of each block."""
    flat = wpack.cpu().numpy().view(np.uint16)
    blocks = []
    for w_off, nb, k, _, _ in jobs:
        blk = np.zeros((nb, k), np.uint16)
        at = w_off
        for k0 in range(0, k, 32):
            klen = min(32, k - k0)
            for n0, n1 in (((0, nb // 2), (nb // 2, nb)) if two_sm else ((0, nb),)):
                m = n1 - n0
                n, kk = np.arange(m)[:, None], np.arange(klen)[None, :]
                off = at + (kk // 8) * (m * 16) + (n // 8) * 128 + (n % 8) * 16 + (kk % 8) * 2
                blk[n0:n1, k0:k0 + klen] = flat[off // 2]
                at += m * klen * 2
        blocks.append(blk)
    return blocks


def _bits(w):
    return w.to(torch.float32).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def _coded(shape, axis):
    """Weights whose bf16 bit pattern is 0x3C00 + (row or column index): distinct along `axis`."""
    idx = torch.arange(shape[axis]).reshape([-1 if a == axis else 1 for a in range(2)]).expand(shape)
    return (0x3C00 + idx).to(torch.int16).contiguous().view(torch.bfloat16).to(torch.float32)


def test_kernel_job_table_matches_the_packer():
    jobs = kernel_jobs()
    assert [(nb, k) for _, nb, k, _, _ in jobs] == [(256, K1), (256, HID), (256, HID), (256, HID), (64, HID)]
    at = 0
    for w_off, nb, k, _, _ in jobs:
        assert w_off == at
        at += nb * k * 2
    # bias layout: b1 | b2 | b3, and layer 3's jobs cover columns 0..575 in order
    assert [b for _, _, _, b, _ in jobs] == [0, 256, 512, 768, 1024]
    assert [c for _, _, _, _, c in jobs[2:]] == [0, 256, 512]
    assert all(b == 512 + c for _, _, _, b, c in jobs[2:])
    W, b = default_net()
    for two_sm in (False, True):
        wpack, bias = pack_weights(W[0], b[0], W[1], b[1], W[2], b[2], two_sm=two_sm)
        assert wpack.dtype == torch.int16 and wpack.numel() * 2 == at, (two_sm, wpack.numel() * 2, at)
        assert torch.equal(bias, torch.cat(b))


@pytest.mark.parametrize("two_sm", [False, True])
def test_packed_layout_round_trips_through_the_documented_decoder(two_sm):
    jobs = kernel_jobs()
    g = _gen(7)
    shapes = ((HID, IN), (HID, HID), (OUT, HID))
    weight_sets = [[_coded(s, 0) for s in shapes], [_coded(s, 1) for s in shapes],
                   [torch.randn(s, generator=g) for s in shapes]]
    zeros = [torch.zeros(n) for n in (HID, HID, OUT)]
    for W in weight_sets:
        wpack, _ = pack_weights(W[0], zeros[0], W[1], zeros[1], W[2], zeros[2], two_sm=two_sm)
        blocks = decode_pack(wpack, jobs, two_sm)
        w1p = np.zeros((HID, K1), np.uint16)
        w1p[:, :IN] = _bits(W[0])
        want = [w1p, _bits(W[1])] + [_bits(W[2][n0:n0 + 256]) for n0 in (0, 256, 512)]
        for j, (got, exp) in enumerate(zip(blocks, want)):
            assert got.shape == exp.shape and np.array_equal(got, exp), (two_sm, j, np.argwhere(got != exp)[:5])


def _cpu_inputs(n=600, seed=11):
    lo, hi = synthetic_states(n, seed)
    return torch.from_numpy(expand_obs198(lo, hi)), move1_codes(n, seed)


@pytest.mark.parametrize("name", sorted(EXACT_DESIGNS) + ["argmax"])
def test_exact_designs_satisfy_their_premise(name):
    """Every exact design is exact on every input (check_premise), and its term-by-term sum is ref_q(emulate=True)."""
    d = argmax_design() if name == "argmax" else EXACT_DESIGNS[name]()
    x, m1 = _cpu_inputs()
    for w3, b3, mv in ((d["W"][2], d["b"][2], None), (d["W3m"], d["b3m"], m1)):
        W, b = (d["W"][0], d["W"][1], w3), (d["b"][0], d["b"][1], b3)
        exact = check_premise(x, W, b, move1=mv, w2b_t=d["w2b_t"])
        assert torch.equal(exact, ref_q(x, W, b, move1=mv, w2b_t=d["w2b_t"]))
        assert torch.equal(exact.float().double(), exact)          # Q-values are fp32 values


def test_perm_design_is_bf16_exact_and_routes_every_input():
    """With bf16 inputs the permutation chain loses nothing to rounding: emulate == plain.  Every input reaches the
    output and ReLU never clips, so a dropped or misplaced input changes some Q-value."""
    d = perm_design()
    x, _ = _cpu_inputs()
    x = bf16(x).float()
    assert torch.equal(ref_q(x, d["W"], d["b"], emulate=True), ref_q(x, d["W"], d["b"], emulate=False))
    assert (d["W"][0] != 0).any(0).all() and (d["W"][1] != 0).any(0).all() and (d["W"][2] != 0).any(0).all()
    h = x.double()
    for w, bb in zip(d["W"][:2], d["b"][:2]):
        h = h @ w.double().T + bb.double()
        assert (h >= 0).all()


def test_argmax_design_peaks_in_every_block_and_half():
    d = argmax_design()
    x, _ = _cpu_inputs(4000, 12)
    a = ref_q(x, d["W"], d["b"]).argmax(1)
    regions = set()
    for lo_, n in ((0, 256), (256, 256), (512, 64)):
        for h in (0, 1):
            c0 = lo_ + h * n // 2
            regions.add(bool(((a >= c0) & (a < c0 + n // 2)).any()))
    assert regions == {True}


def test_move1_codes_are_clamped_in_the_reference():
    d = perm_design()
    x, _ = _cpu_inputs(5)
    W, b = (d["W"][0], d["W"][1], d["W3m"]), (d["b"][0], d["b"][1], d["b3m"])
    q = ref_q(x, W, b, move1=torch.tensor([2 ** 31 - 1, 0, 575, -1, 576], dtype=torch.int32), w2b_t=d["w2b_t"])
    want = ref_q(x, W, b, move1=torch.tensor([575, 0, 575, 0, 575]), w2b_t=d["w2b_t"])
    assert torch.equal(q, want)


@pytest.mark.parametrize("scale", [1.0, 16.0])
def test_emulated_reference_is_within_the_bound_of_the_plain_net(scale):
    """ref_q(emulate=True) is one admissible kernel (float64 sums are exact sums), so it lies within bound() of the
    plain net.  The bound is not vacuous: at the default init it is below the fixed tolerance the older tests use."""
    W, b = default_net(0, scale)
    x, m1 = _cpu_inputs(512, 13)
    emu, plain = ref_q(x, W, b), ref_q(x, W, b, emulate=False)
    bnd = bound(x, W, b)
    assert ((emu - plain).abs() <= bnd).all()
    assert bnd.max() < 5e-3 * scale ** 3, bnd.max().item()
    w2b_t = torch.randn(OUT, OUT, generator=_gen(3)) * 0.03 * scale
    emu = ref_q(x, W, b, move1=m1, w2b_t=w2b_t)
    plain = ref_q(x, W, b, move1=m1, w2b_t=w2b_t, emulate=False)
    assert ((emu - plain).abs() <= bound(x, W, b, move1=m1, w2b_t=w2b_t)).all()


def test_bound_scales_with_the_weights():
    """Weights times 4 and biases times 4, 16, 64 scale Q by exactly 64 (ReLU is positively homogeneous): so does
    the bound, unlike a fixed absolute tolerance."""
    W, b = default_net(0, 1.0)
    x, _ = _cpu_inputs(64, 14)
    W4 = tuple(w * 4 for w in W)
    b4 = tuple(v * 4 ** (i + 1) for i, v in enumerate(b))
    assert torch.allclose(ref_q(x, W4, b4, emulate=False), 64 * ref_q(x, W, b, emulate=False), rtol=1e-12, atol=0)
    assert torch.allclose(bound(x, W4, b4), 64 * bound(x, W, b), rtol=1e-12, atol=0)
