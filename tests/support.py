"""Shared helpers for the test-suite (host simulation harness + position generators)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from gym_narde_b200 import state as S  # noqa: E402

_HS_DIR = os.path.join(ROOT, "tests", "hostsim")
_HS_LIB = os.path.join(_HS_DIR, "_build", "libnarde_hostsim.so")


def build_hostsim():
    csrc = os.path.join(ROOT, "gym_narde_b200", "csrc")
    srcs = [os.path.join(_HS_DIR, "hostsim.cpp"), os.path.join(ROOT, "include", "narde_b200.h")] + sorted(
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh"))
    if (not os.path.exists(_HS_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_HS_LIB) for s in srcs):
        os.makedirs(os.path.dirname(_HS_LIB), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-Wno-unknown-pragmas",
                               "-o", _HS_LIB, srcs[0]])
    return _HS_LIB


def _p(a, t=C.c_void_p):
    return None if a is None else a.ctypes.data_as(t)


class HostSim:
    """The device core compiled for the host (TEST ONLY), same call surface as the C-ABI."""

    def __init__(self):
        self.lib = C.CDLL(build_hostsim())

    def reset(self, n, env_base=0, seed=0, step=0):
        lo = np.zeros((n, 16), np.uint8)
        hi = np.zeros((n, 16), np.uint8)
        self.lib.hs_reset(_p(lo), _p(hi), C.c_int64(n), C.c_int64(env_base), C.c_uint64(seed), C.c_uint64(step), None)
        return lo, hi

    def half_moves(self, lo, hi, dice4, player_override=0):
        n = lo.shape[0]
        dice4 = np.ascontiguousarray(dice4, np.uint8)
        moves = np.zeros((n, 96, 2), np.uint8)
        counts = np.zeros(n, np.int32)
        self.lib.hs_half_moves(_p(lo), _p(hi), _p(dice4), C.c_int64(n), C.c_int(player_override), _p(moves), _p(counts), None)
        return moves, counts

    def step_ref(self, lo, hi, dice, codes, max_episode_steps=0):
        n = lo.shape[0]
        dice = np.ascontiguousarray(dice, np.uint8)
        codes = np.ascontiguousarray(codes, np.int32)
        obs = np.zeros((n, 24), np.int32)
        rew = np.zeros(n, np.int32)
        done = np.zeros(n, np.uint8)
        self.lib.hs_step_ref(_p(lo), _p(hi), _p(dice), _p(codes), C.c_int64(n), C.c_int32(max_episode_steps),
                             _p(obs), _p(rew), _p(done), None, None)
        return obs, rew, done

    enumerate_fast = False  # True: narde_enumerate_fast (fused-step phases, enumerate-only mode)

    def enumerate(self, lo, hi, dice, cap):
        n = lo.shape[0]
        dice = np.ascontiguousarray(dice, np.uint8)
        actions = np.full((n, cap), 0xFFFFFFFFFFFFFFFF, np.uint64)
        counts = np.zeros(n, np.int32)
        overflow = np.zeros(n, np.uint8)
        if self.enumerate_fast:
            lo0, hi0 = lo.copy(), hi.copy()
            ws = np.zeros(n + 8, np.int32)
            self.lib.hs_enumerate_fast(_p(lo), _p(hi), _p(dice), C.c_int64(n), C.c_int32(cap), _p(actions), _p(counts),
                                       _p(overflow), _p(ws), None)
            assert (lo == lo0).all() and (hi == hi0).all()   # states untouched
        else:
            self.lib.hs_enumerate(_p(lo), _p(hi), _p(dice), C.c_int64(n), C.c_int32(cap), _p(actions), _p(counts),
                                  _p(overflow), None)
        return actions, counts, overflow

    def obs198(self, lo, hi):
        n = lo.shape[0]
        obs = np.zeros((n, 198), np.float32)
        self.lib.hs_obs198(_p(lo), _p(hi), C.c_int64(n), _p(obs), None)
        return obs

    def obs24(self, lo, hi):
        n = lo.shape[0]
        obs = np.zeros((n, 24), np.int32)
        self.lib.hs_obs24(_p(lo), _p(hi), C.c_int64(n), _p(obs), None)
        return obs

    per_thread = False  # True: the thread-per-env body (k_step_full); False: the CTA-cooperative phases
    defer = True        # CTA-cooperative path: hand block-rule doubles turns to the CTA-per-env exact phases

    def step_full(self, lo, hi, env_base=0, seed=0, step=0, dice_in=None, action_idx=None, cap=64, flags=0,
                  max_episode_steps=0, want_actions=True, want_obs=True):
        n = lo.shape[0]
        if dice_in is not None:
            dice_in = np.ascontiguousarray(dice_in, np.uint8)
        if action_idx is not None:
            action_idx = np.ascontiguousarray(action_idx, np.int32)
        out = {
            "actions": np.full((n, cap), 0xFFFFFFFFFFFFFFFF, np.uint64) if want_actions else None,
            "counts": np.zeros(n, np.int32),
            "dice": np.zeros((n, 2), np.uint8),
            "chosen": np.zeros(n, np.uint64),
            "obs198": np.zeros((n, 198), np.float32) if want_obs else None,
            "reward": np.zeros(n, np.float32),
            "done": np.zeros(n, np.uint8),
            "trunc": np.zeros(n, np.uint8),
            "stats": np.zeros(9, np.int64),
        }
        v1 = self.per_thread or (flags & 8)
        ws = np.zeros(n + 8, np.int32) if (self.defer and not v1) else None
        fn = self.lib.hs_step_full if v1 else self.lib.hs_step_full_v2
        tail = (None,) if v1 else (_p(ws), None)
        fn(_p(lo), _p(hi), C.c_int64(n), C.c_int64(env_base), C.c_uint64(seed), C.c_uint64(step),
                              _p(dice_in), _p(action_idx), C.c_int32(cap), _p(out["actions"]), _p(out["counts"]),
                              _p(out["dice"]), _p(out["chosen"]), _p(out["obs198"]), _p(out["reward"]),
                              _p(out["done"]), _p(out["trunc"]), _p(out["stats"]), C.c_int32(flags), C.c_int32(max_episode_steps), *tail)
        out["deferred"] = int(ws[0]) if ws is not None else 0
        return out

    def apply_actions(self, lo, hi, acts, flags=0):
        n = lo.shape[0]
        acts = np.ascontiguousarray(acts, np.uint64)
        rew = np.zeros(n, np.float32)
        done = np.zeros(n, np.uint8)
        self.lib.hs_apply_actions(_p(lo), _p(hi), _p(acts), C.c_int64(n), C.c_int32(flags), _p(rew), _p(done), None)
        return rew, done

    def block_irrelevant(self, lo, hi, dice):
        n = lo.shape[0]
        dice = np.ascontiguousarray(dice, np.uint8)
        out = np.zeros(n, np.uint8)
        self.lib.hs_block_irrelevant(_p(lo), _p(hi), _p(dice), C.c_int64(n), _p(out))
        return out


class CudaBackend:
    """The product path: torch CUDA tensors through the C ABI (gym_narde_b200/_cabi.py)."""

    def __init__(self):
        import torch
        from gym_narde_b200 import _cabi
        self.torch, self.cabi = torch, _cabi
        _cabi.require_cuda()
        _cabi.load()
        self.dev = torch.device("cuda")

    def _up(self, a, dtype=None):
        if a is None:
            return None
        t = self.torch.from_numpy(np.ascontiguousarray(a))
        if dtype is not None:
            t = t.to(dtype)
        return t.to(self.dev)

    def _sync_back(self, lo, hi, tlo, thi):
        lo[...] = tlo.cpu().numpy()
        hi[...] = thi.cpu().numpy()

    def reset(self, n, env_base=0, seed=0, step=0):
        t = self.torch
        lo = t.zeros((n, 16), dtype=t.uint8, device=self.dev)
        hi = t.zeros((n, 16), dtype=t.uint8, device=self.dev)
        self.cabi.reset(lo, hi, env_base, seed, step)
        return lo.cpu().numpy(), hi.cpu().numpy()

    def half_moves(self, lo, hi, dice4, player_override=0):
        t = self.torch
        n = lo.shape[0]
        tlo, thi = self._up(lo), self._up(hi)
        moves = t.zeros((n, 96, 2), dtype=t.uint8, device=self.dev)
        counts = t.zeros(n, dtype=t.int32, device=self.dev)
        self.cabi.half_moves(tlo, thi, self._up(np.asarray(dice4, np.uint8)), moves, counts, player_override)
        return moves.cpu().numpy(), counts.cpu().numpy()

    def step_ref(self, lo, hi, dice, codes, max_episode_steps=0):
        t = self.torch
        n = lo.shape[0]
        tlo, thi = self._up(lo), self._up(hi)
        obs = t.zeros((n, 24), dtype=t.int32, device=self.dev)
        rew = t.zeros(n, dtype=t.int32, device=self.dev)
        done = t.zeros(n, dtype=t.uint8, device=self.dev)
        self.cabi.step_ref(tlo, thi, self._up(np.asarray(dice, np.uint8)), self._up(np.asarray(codes, np.int32)),
                           obs, rew, done, max_episode_steps)
        self._sync_back(lo, hi, tlo, thi)
        return obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()

    enumerate_fast = False  # True: narde_enumerate_fast (fused-step kernels, enumerate-only mode)

    def enumerate(self, lo, hi, dice, cap):
        t = self.torch
        n = lo.shape[0]
        tlo, thi = self._up(lo), self._up(hi)
        actions = t.full((n, cap), -1, dtype=t.int64, device=self.dev)
        counts = t.zeros(n, dtype=t.int32, device=self.dev)
        overflow = t.zeros(n, dtype=t.uint8, device=self.dev)
        if self.enumerate_fast:
            ws = t.zeros(n + 8, dtype=t.int32, device=self.dev)
            self.cabi.enumerate_actions_fast(tlo, thi, self._up(np.asarray(dice, np.uint8)), actions, counts, overflow, ws)
            assert t.equal(tlo.cpu(), t.from_numpy(lo)) and t.equal(thi.cpu(), t.from_numpy(hi))   # states untouched
            return actions.cpu().numpy().view(np.uint64), counts.cpu().numpy(), overflow.cpu().numpy()
        self.cabi.enumerate_actions(tlo, thi, self._up(np.asarray(dice, np.uint8)), actions, counts, overflow)
        return actions.cpu().numpy().view(np.uint64), counts.cpu().numpy(), overflow.cpu().numpy()

    def obs198(self, lo, hi):
        t = self.torch
        out = t.zeros((lo.shape[0], 198), dtype=t.float32, device=self.dev)
        self.cabi.obs198(self._up(lo), self._up(hi), out)
        return out.cpu().numpy()

    def obs24(self, lo, hi):
        t = self.torch
        out = t.zeros((lo.shape[0], 24), dtype=t.int32, device=self.dev)
        self.cabi.obs24(self._up(lo), self._up(hi), out)
        return out.cpu().numpy()

    def step_full(self, lo, hi, env_base=0, seed=0, step=0, dice_in=None, action_idx=None, cap=64, flags=0,
                  max_episode_steps=0, want_actions=True, want_obs=True):
        t = self.torch
        n = lo.shape[0]
        tlo, thi = self._up(lo), self._up(hi)
        actions = t.full((n, cap), -1, dtype=t.int64, device=self.dev) if want_actions else None
        counts = t.zeros(n, dtype=t.int32, device=self.dev)
        dice = t.zeros((n, 2), dtype=t.uint8, device=self.dev)
        chosen = t.zeros(n, dtype=t.int64, device=self.dev)
        obs = t.zeros((n, 198), dtype=t.float32, device=self.dev) if want_obs else None
        rew = t.zeros(n, dtype=t.float32, device=self.dev)
        done = t.zeros(n, dtype=t.uint8, device=self.dev)
        stats = t.zeros(9, dtype=t.int64, device=self.dev)
        trunc = t.zeros(n, dtype=t.uint8, device=self.dev)
        ws = t.zeros(n + 8, dtype=t.int32, device=self.dev) if (getattr(self, "defer", True) and not (flags & 8)) else None
        if getattr(self, "per_thread", False):
            flags |= 8  # NARDE_PER_THREAD_KERNEL
        self.cabi.step_full(tlo, thi, env_base, seed, step,
                            dice_in=self._up(None if dice_in is None else np.asarray(dice_in, np.uint8)),
                            action_idx=self._up(None if action_idx is None else np.asarray(action_idx, np.int32)),
                            actions=actions, counts=counts, dice_out=dice, chosen=chosen, obs198=obs, reward=rew,
                            done=done, stats=stats, flags=flags, max_episode_steps=max_episode_steps, truncated=trunc,
                            workspace=ws)  # noqa
        self._sync_back(lo, hi, tlo, thi)
        return {
            "actions": actions.cpu().numpy().view(np.uint64) if want_actions else None,
            "counts": counts.cpu().numpy(), "dice": dice.cpu().numpy(),
            "chosen": chosen.cpu().numpy().view(np.uint64),
            "obs198": obs.cpu().numpy() if want_obs else None, "reward": rew.cpu().numpy(),
            "done": done.cpu().numpy(), "trunc": trunc.cpu().numpy(), "stats": stats.cpu().numpy(),
            "deferred": int(ws[0].item()) if ws is not None else 0,
        }

    def apply_actions(self, lo, hi, acts, flags=0):
        t = self.torch
        n = lo.shape[0]
        tlo, thi = self._up(lo), self._up(hi)
        rew = t.zeros(n, dtype=t.float32, device=self.dev)
        done = t.zeros(n, dtype=t.uint8, device=self.dev)
        self.cabi.apply_actions(tlo, thi, self._up(np.asarray(acts, np.uint64).view(np.int64)), rew, done, flags)
        self._sync_back(lo, hi, tlo, thi)
        return rew.cpu().numpy(), done.cpu().numpy()
