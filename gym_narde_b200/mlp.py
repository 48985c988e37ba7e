"""Afterstate-scoring MLP (BASELINE config 5): host side of narde_mlp_forward.

Architecture = the reference's DecomposedDQN with state_size 198 (train_deepq_pytorch.py:184-236):
forward(x) = Linear(198,256)-ReLU-Linear(256,256)-ReLU-Linear(256,576) (move1_head), and
forward(x, selected_move1) = move2_head(cat(features, onehot(move1))), Linear(832,576), whose one-hot half is a
column gather added in the same kernel's epilogue.
The CUDA kernel (csrc/narde_mlp.cu) runs bf16 operands / fp32 accumulation on tcgen05 tensor cores;
weights are re-packed once on the host into the shared-memory operand layout it streams.
"""
from __future__ import annotations

import numpy as np

from . import _cabi

IN, HID, OUT, K1, KC = 198, 256, 576, 208, 32


def _pack_block(w_blk, two_sm=False):
    """w_blk: [nb, K] float32 (K a multiple of 16) -> bf16 stages of 32 K (the last may be 16) in the K-major
    interleave layout: offset(n, k) = (k//8)*(nb*16) + (n//8)*128 + (n%8)*16 + (k%8)*2 within a stage.
    two_sm: every stage is stored as [rows 0..nb/2) | rows nb/2..nb)], each half in that layout on its own
    (the B operand halves of a cta_group::2 MMA, one per CTA of the pair)."""
    import torch

    nb, k = w_blk.shape
    stages = []
    for k0 in range(0, k, KC):
        klen = min(KC, k - k0)
        for rows in ((slice(0, nb // 2), slice(nb // 2, nb)) if two_sm else (slice(0, nb),)):
            s = w_blk[rows, k0:k0 + klen].to(torch.bfloat16)             # [n, klen]
            n = s.shape[0]
            s = s.reshape(n // 8, 8, klen // 8, 8).permute(2, 0, 1, 3)   # [kchunk, rowgroup, row, k]
            stages.append(s.contiguous().view(torch.int16).reshape(-1))
    return torch.cat(stages)


def pack_weights(w1, b1, w2, b2, w3, b3, two_sm=False):
    """torch Linear weights ([out, in]) and biases -> (wpack int16 tensor, bias float32 [1088])."""
    import torch

    assert tuple(w1.shape) == (HID, IN) and tuple(w2.shape) == (HID, HID) and tuple(w3.shape) == (OUT, HID)
    w1p = torch.zeros((HID, K1), dtype=torch.float32, device=w1.device)
    w1p[:, :IN] = w1.float()
    parts = [_pack_block(w1p, two_sm), _pack_block(w2.float(), two_sm)]
    for n0 in range(0, OUT, 256):
        parts.append(_pack_block(w3.float()[n0:min(n0 + 256, OUT)], two_sm))
    wpack = torch.cat(parts).contiguous()
    bias = torch.cat([b1.float(), b2.float(), b3.float()]).contiguous()
    return wpack, bias


class AfterstateMLP:
    """DecomposedDQN.forward(x) with state_size 198 on the tcgen05 tensor cores.

    forward(x)            x float32 [K,198]            -> q float32 [K,576]   (move1 Q-values)
    score(x)              x float32 [K,198]            -> max_a q[:, a]  float32 [K]
    forward_states(lo,hi) packed states [K,16] uint8 x2 -> q   (Box(198) encoded inside the kernel)
    score_states(lo,hi)   packed states                -> max_a q[:, a]       (the afterstate score)
    forward(x, selected_move1) / forward_states(lo, hi, selected_move1)  -> move2 Q-values [K,576] (needs the
                          move2_head weights: from_module(..., move2_head) or set_move2_head(w, b))"""

    def __init__(self, w1, b1, w2, b2, w3, b3, w_move2=None, b_move2=None):
        torch = _cabi.require_cuda()
        _cabi.load()
        self.torch = torch
        self._trunk = (w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda())
        self.wpack, self.bias = pack_weights(*self._trunk, w3.cuda(), b3.cuda())
        self.wpack2, _ = pack_weights(*self._trunk, w3.cuda(), b3.cuda(), two_sm=True)
        self.wpack_m2 = self.bias_m2 = self.w2b_t = None
        if w_move2 is not None:
            self.set_move2_head(w_move2, b_move2)

    def set_move2_head(self, w, b):
        """move2_head = Linear(256 + 576, 576) (train_deepq_pytorch.py:200-201): its first 256 input columns become
        the third GEMM of the chain, the other 576 (one per first-move code) a transposed fp32 gather table."""
        if tuple(w.shape) != (OUT, HID + OUT) or tuple(b.shape) != (OUT,):
            raise ValueError("move2_head must be Linear(%d, %d)" % (HID + OUT, OUT))
        w = w.cuda().float()
        self.wpack_m2, self.bias_m2 = pack_weights(*self._trunk, w[:, :HID].contiguous(), b.cuda())
        self.w2b_t = w[:, HID:].t().contiguous()

    @classmethod
    def from_module(cls, feature_network, move1_head, move2_head=None):
        """feature_network = nn.Sequential(Linear, ReLU, Linear, ReLU), move1_head / move2_head = Linear (the
        reference's attribute names)."""
        l1, l2 = feature_network[0], feature_network[2]
        m2 = (move2_head.weight.data, move2_head.bias.data) if move2_head is not None else (None, None)
        return cls(l1.weight.data, l1.bias.data, l2.weight.data, l2.bias.data, move1_head.weight.data, move1_head.bias.data,
                   *m2)

    @classmethod
    def from_state_dict(cls, sd):
        """Weights from a `DecomposedDQN.state_dict()` (train_deepq_pytorch.py:184-201: keys `feature_network.{0,2}.*`,
        `move1_head.*`, `move2_head.*`) built with state_size=198.  The reference's own scripts construct
        DecomposedDQN(state_size=24) (train_deepq_pytorch.py:831, evaluate_model.py): those checkpoints feed the raw
        24-int board, not the README's Box(198), and are NOT supported by this kernel -- a clear error instead of
        silently wrong scores."""
        w1 = sd["feature_network.0.weight"]
        if tuple(w1.shape) != (HID, IN):
            raise ValueError("AfterstateMLP needs a DecomposedDQN(state_size=198) checkpoint; got first layer %s "
                             "(the reference's state_size=24 checkpoints are unsupported)" % (tuple(w1.shape),))
        m2 = (sd["move2_head.weight"], sd["move2_head.bias"]) if "move2_head.weight" in sd else (None, None)
        return cls(w1, sd["feature_network.0.bias"], sd["feature_network.2.weight"], sd["feature_network.2.bias"],
                   sd["move1_head.weight"], sd["move1_head.bias"], *m2)

    def _move1(self, selected_move1):
        if self.wpack_m2 is None:
            raise _cabi.NardeCudaError("move2_head weights were not given (set_move2_head)")
        return selected_move1.to(self.torch.int32).contiguous()

    def _out(self, out, like, *cols):
        """out, or a new float32 [K, *cols] tensor on like's device (K = len(like))."""
        t = self.torch
        return t.empty((like.shape[0], *cols), dtype=t.float32, device=like.device) if out is None else out

    def forward(self, x, selected_move1=None, out=None):
        """DecomposedDQN.forward (train_deepq_pytorch.py:203-233): move1 Q-values, or, given selected_move1
        (int tensor [K], codes in [0,576)), the move2 Q-values."""
        out = self._out(out, x, OUT)
        if selected_move1 is not None:
            _cabi.mlp_forward_move2(x, self._move1(selected_move1), self.wpack_m2, self.bias_m2, self.w2b_t, out)
        else:
            _cabi.mlp_forward(x, self.wpack, self.bias, out)
        return out

    def score(self, x, out=None):
        out = self._out(out, x)
        _cabi.mlp_score(x, self.wpack, self.bias, out)
        return out

    def forward_states(self, lo, hi, selected_move1=None, out=None):
        out = self._out(out, lo, OUT)
        if selected_move1 is not None:
            _cabi.mlp_forward_move2_states(lo, hi, self._move1(selected_move1), self.wpack_m2, self.bias_m2, self.w2b_t, out)
        else:
            _cabi.mlp_forward_states(lo, hi, self.wpack, self.bias, out)
        return out

    def score_states(self, lo, hi, out=None, rows_dev=None):
        """rows_dev: optional int64 CUDA tensor [1]; only min(rows_dev, len(lo)) rows are scored (no host sync)."""
        out = self._out(out, lo)
        _cabi.mlp_score_states(lo, hi, self.wpack, self.bias, out, rows_dev)
        return out

    def score_states_2sm(self, lo, hi, out=None, rows_dev=None):
        """score_states through the cta_group::2 kernel (clusters of two CTAs, M = 256 per tcgen05.mma)."""
        out = self._out(out, lo)
        _cabi.mlp_score_states(lo, hi, self.wpack2, self.bias, out, rows_dev, two_sm=True)
        return out

    __call__ = forward
