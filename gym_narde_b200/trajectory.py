"""Device-resident trajectory ring + exact checkpoint/resume (SURVEY.md section 8(f) rank 3).

The reference only checkpoints model weights (train_deepq_pytorch.py:1136-1145).  Here a whole run is
resumable bit for bit: the SoA state planes plus the Philox (seed, step) are the complete env state, and
the ring keeps one 48-byte record per env turn in HBM:
    state after the turn (2 x 16 B) | u64 action played | f32 reward | u8 die1 | u8 die2 | u8 done | u8 0
"""
from __future__ import annotations

from . import _cabi

RECORD_BYTES = 48


class TrajectoryRing:
    def __init__(self, env, capacity):
        """env: VecNardeEnv(rules="full"); capacity: number of lock-step turns kept (ring)."""
        t = env.torch
        self.env, self.capacity = env, int(capacity)
        self.records = t.zeros((self.capacity, env.num_envs, RECORD_BYTES), dtype=t.uint8, device=env.device)
        self.initial_lo, self.initial_hi = env.lo.clone(), env.hi.clone()   # s_0 (call after env.reset())
        self.cursor = 0          # total turns appended (slot = cursor % capacity)

    def append(self):
        """Record the turn VecNardeEnv.step() has just played (one kernel, 48 B per env)."""
        env = self.env
        _cabi.trajectory_append(env.lo, env.hi, self.records[self.cursor % self.capacity], dice=env.dice, chosen=env.chosen,
                                reward=env.reward, done=env.done, truncated=env.trunc)
        self.cursor += 1

    def step(self, actions=None, dice=None, fraction=False):
        out = self.env.step(actions, dice=dice, fraction=fraction)
        self.append()
        return out

    def view(self, turn):
        """Fields of the record of absolute turn index `turn` (must still be in the ring), zero-copy views."""
        t = self.env.torch
        if not (max(0, self.cursor - self.capacity) <= turn < self.cursor):
            raise IndexError("turn %d is not in the ring" % turn)
        r = self.records[turn % self.capacity]
        return {"lo": r[:, 0:16], "hi": r[:, 16:32], "action": r[:, 32:40].view(t.int64)[:, 0],
                "reward": r[:, 40:44].view(t.float32)[:, 0], "dice": r[:, 44:46], "done": r[:, 46]}

    # -- checkpoint: env planes + Philox (seed, step) + ring ------------------------------------
    def state_dict(self):
        return {"env": self.env.state_dict(), "records": self.records.clone(), "cursor": self.cursor,
                "initial_lo": self.initial_lo.clone(), "initial_hi": self.initial_hi.clone(),
                "stats": self.env.stats.clone()}

    def load_state_dict(self, sd):
        self.env.load_state_dict(sd["env"])
        self.env.stats.copy_(sd["stats"])
        self.records.copy_(sd["records"])
        self.initial_lo.copy_(sd["initial_lo"])
        self.initial_hi.copy_(sd["initial_hi"])
        self.cursor = sd["cursor"]


def action_codes(env, actions=None, counts=None):
    """The reference trainer's (move1_code, move2_code) pairs for every stored legal turn action of every env
    (train_deepq_pytorch.py:432-437,495-507): int32 [N, cap, 3] = (move1_code, move2_code, half-moves in turn)."""
    t = env.torch
    actions = env.actions if actions is None else actions
    counts = env.counts if counts is None else counts
    n, cap = actions.shape
    codes = t.zeros((n, cap, 3), dtype=t.int32, device=actions.device)
    _cabi.action_codes(actions, counts, codes)
    return codes
