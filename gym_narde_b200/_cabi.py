"""ctypes binding of the C ABI in include/narde_b200.h (device pointers from torch tensors).

This is the only bridge between the Python host side and the CUDA kernels (the single-env facade in
envs/ keeps pointers cached at construction for its per-call latency).  There is no CPU fallback:
`load()` raises if libnarde_b200.so has not been built, and every compute wrapper raises if CUDA is
unavailable or a tensor is not a CUDA tensor.  The wrappers of the actor, trajectory and MLP entry
points also check the length of every buffer the kernel indexes by a size argument, before the launch.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnarde_b200.so")
if os.environ.get("NARDE_B200_DEBUG_HOOKS") == "1":   # measurement tools only (tools/*.py): the -DNARDE_DEBUG_HOOKS build
    LIB_PATH = os.path.join(_HERE, "libnarde_b200_debug.so")

ABI_VERSION = 4
# flags / bits (include/narde_b200.h)
REWARD_MOVER12 = 1
AUTORESET = 2
ACTION_FRACTION = 32
ENUMERATE_ONLY = 64
PACK_RESULT = 128
DEVICE_ADVANCE = 256
HALF_MOVES_ONLY = 4
MAX_HALF_MOVES = 96
NUM_STATS = 9
STAT_NAMES = ("episodes", "white_wins", "black_wins", "mars", "episode_steps", "legal_actions",
              "max_actions", "overflows", "clamped_actions")



def workspace_ints(n):
    """NARDE_WORKSPACE_INTS(n), include/narde_b200.h."""
    return int(n) + 8


_vp, _i64, _u64, _i32, _int = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32, C.c_int

_SIGNATURES = {
    "narde_abi_version": ([], _int),
    "narde_build_arch": ([], C.c_char_p),
    "narde_reset": ([_vp, _vp, _i64, _i64, _u64, _u64, _vp], _int),
    "narde_reset_masked": ([_vp, _vp, _vp, _i64, _i64, _u64, _u64, _vp], _int),
    "narde_half_moves": ([_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp], _int),
    "narde_step_ref": ([_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_enumerate": ([_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp], _int),
    "narde_enumerate_fast": ([_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_step_full": ([_vp, _vp, _i64, _i64, _u64, _u64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                         _vp, _vp, _i32, _i32, _vp, _vp, _vp], _int),
    "narde_step_full_mirror": ([_vp, _vp, _i64, _i64, _u64, _u64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_advance_counter": ([_vp, _vp], _int),
    "narde_mlp_forward": ([_vp, _i64, _vp, _vp, _vp, _vp], _int),
    "narde_mlp_score": ([_vp, _i64, _vp, _vp, _vp, _vp], _int),
    "narde_mlp_forward_states": ([_vp, _vp, _i64, _vp, _vp, _vp, _vp], _int),
    "narde_mlp_score_states": ([_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_mlp_score_states_2sm": ([_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_mlp_use_cluster_pair": ([_int], _int),
    "narde_mlp_forward_move2": ([_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_mlp_forward_move2_states": ([_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_action_codes": ([_vp, _vp, _i64, _i32, _vp, _vp], _int),
    "narde_trajectory_append": ([_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp], _int),
    "narde_afterstates": ([_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp], _int),
    "narde_afterstates_scan": ([_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp], _int),
    "narde_gather_overflow": ([_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_gather_overflow_clear": ([_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_scatter_choice": ([_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_step_chosen": ([_vp, _vp, _i64, _i64, _u64, _u64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                           _i32, _i32, _vp, _vp], _int),
    "narde_segment_argmax": ([_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp], _int),
    "narde_segment_sample": ([_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _i64, _u64, _u64, _vp, _vp, _vp, _vp, _vp], _int),
    "narde_obs198": ([_vp, _vp, _i64, _vp, _vp], _int),
    "narde_obs24": ([_vp, _vp, _i64, _vp, _vp], _int),
    "narde_apply_actions": ([_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp], _int),
    "narde_roll_dice": ([_i64, _i64, _u64, _u64, _vp, _vp], _int),
    "narde_violates_block_rule": ([_vp, _i64, _vp, _vp], _int),
}

_lib = None


class NardeCudaError(RuntimeError):
    pass


def load():
    """Open libnarde_b200.so (built in-tree by gym_narde_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NardeCudaError(
            "gym_narde_b200: CUDA extension %s is missing. Build it with `python -m gym_narde_b200.build` "
            "(needs nvcc; sm_100a only). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (argtypes, restype) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export the symbol
        fn.argtypes = argtypes
        fn.restype = restype
    if lib.narde_abi_version() != ABI_VERSION:
        raise NardeCudaError("libnarde_b200.so ABI version mismatch")
    _lib = lib
    return lib


def exported_symbols():
    return tuple(_SIGNATURES)


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise NardeCudaError("gym_narde_b200 needs a CUDA device (B200 / sm_100a); there is no CPU fallback")
    return torch


def _check(rc, what):
    if rc != 0:
        msg = "bad argument" if rc == -1 else "cudaError %d" % rc
        raise NardeCudaError("%s failed: %s" % (what, msg))


def _device():
    """The current CUDA device, read once per wrapper call: every launch goes to its current stream."""
    import torch

    try:
        return torch.cuda.current_device()
    except (AssertionError, RuntimeError) as e:   # no driver / no CUDA build of torch
        raise NardeCudaError("gym_narde_b200 needs a CUDA device (B200 / sm_100a); there is no CPU fallback") from e


class _Any:
    """Shape entry that matches any extent: the tuple comparison in _ptr falls back to this __eq__ (no Python loop)."""
    __slots__ = ()
    __hash__ = object.__hash__

    def __eq__(self, other):
        return True

    def __repr__(self):
        return "*"


_ANY = _Any()


def _ptr(t, dtype, name, dev, shape=None, min_rows=0):
    """Pointer to `t` (None: NULL) once `t` is what the kernel will index: `dtype`, contiguous, on device `dev`, of
    `shape` (_ANY entries: any extent) and at least `min_rows` long in its first dimension."""
    if t is None:
        return None
    # device memory, or page-locked host memory (mapped into the device address space by CUDA's unified
    # addressing: the kernels read / write it directly over PCIe -- the zero-copy I/O of VecNardeEnv.step_host)
    try:
        usable = t.is_cuda or t.is_pinned()
    except AttributeError:          # not a tensor
        usable = False
    if not usable:
        raise NardeCudaError("%s must be a CUDA tensor or a pinned host tensor (no CPU fallback)" % name)
    if not t.is_contiguous():
        raise NardeCudaError("%s must be contiguous" % name)
    if t.dtype != dtype:
        raise NardeCudaError("%s must have dtype %s, got %s" % (name, dtype, t.dtype))
    # launches go to the CURRENT device's current stream: a tensor of another GPU would be an illegal address there
    if t.is_cuda and t.get_device() != dev:
        raise NardeCudaError("%s lives on %s but the current CUDA device is cuda:%d: call torch.cuda.set_device(...) "
                             "or wrap the call in `with torch.cuda.device(...)`" % (name, t.device, dev))
    if shape is not None and t.shape != shape:
        raise NardeCudaError("%s must have shape %s, got %s" % (name, list(shape), list(t.shape)))
    if min_rows and t.shape[0] < min_rows:
        raise NardeCudaError("%s must have at least %d rows, got %d" % (name, min_rows, t.shape[0]))
    return C.c_void_p(t.data_ptr())


def _stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------------------------------
# thin wrappers (tensors in, tensors mutated in place); all asynchronous on the current stream
# ------------------------------------------------------------------------------------------
def reset(lo, hi, env_base, seed, step, mask=None):
    import torch

    dev = _device()
    n = lo.shape[0]
    rc = load().narde_reset_masked(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev),
                                   _ptr(mask, torch.uint8, "mask", dev), n, env_base, seed, step, _stream())
    _check(rc, "narde_reset")


def half_moves(lo, hi, dice4, moves, counts, player_override=0):
    import torch

    dev = _device()
    rc = load().narde_half_moves(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev),
                                 _ptr(dice4, torch.uint8, "dice", dev), lo.shape[0], player_override,
                                 _ptr(moves, torch.uint8, "moves", dev), _ptr(counts, torch.int32, "counts", dev), _stream())
    _check(rc, "narde_half_moves")


def step_ref(lo, hi, dice, codes, obs24, reward, done, max_episode_steps=0, truncated=None):
    import torch

    dev = _device()
    rc = load().narde_step_ref(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev),
                               _ptr(dice, torch.uint8, "dice", dev), _ptr(codes, torch.int32, "codes", dev), lo.shape[0],
                               max_episode_steps, _ptr(obs24, torch.int32, "obs24", dev),
                               _ptr(reward, torch.int32, "reward", dev), _ptr(done, torch.uint8, "done", dev),
                               _ptr(truncated, torch.uint8, "truncated", dev), _stream())
    _check(rc, "narde_step_ref")


def enumerate_actions(lo, hi, dice, actions, counts, overflow=None):
    import torch

    dev = _device()
    cap = actions.shape[1] if actions is not None else 0
    rc = load().narde_enumerate(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev),
                                _ptr(dice, torch.uint8, "dice", dev), lo.shape[0], cap,
                                _ptr(actions, torch.int64, "actions", dev), _ptr(counts, torch.int32, "counts", dev),
                                _ptr(overflow, torch.uint8, "overflow", dev), _stream())
    _check(rc, "narde_enumerate")


def enumerate_actions_fast(lo, hi, dice, actions, counts, overflow=None, workspace=None):
    import torch

    dev = _device()
    cap = actions.shape[1] if actions is not None else 0
    if workspace is not None and workspace.numel() < workspace_ints(lo.shape[0]):
        raise NardeCudaError("workspace must hold NARDE_WORKSPACE_INTS(n) = n + 8 int32")
    rc = load().narde_enumerate_fast(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev),
                                     _ptr(dice, torch.uint8, "dice", dev), lo.shape[0], cap,
                                     _ptr(actions, torch.int64, "actions", dev), _ptr(counts, torch.int32, "counts", dev),
                                     _ptr(overflow, torch.uint8, "overflow", dev), _ptr(workspace, torch.int32, "workspace", dev),
                                     _stream())
    _check(rc, "narde_enumerate_fast")


def step_full(lo, hi, env_base, seed, step, dice_in=None, action_idx=None, actions=None, counts=None,
              dice_out=None, chosen=None, obs198=None, reward=None, done=None, stats=None, flags=0,
              max_episode_steps=0, truncated=None, workspace=None, step_dev=None, mirror_lo=None, mirror_hi=None):
    import torch

    dev = _device()
    cap = actions.shape[1] if actions is not None else 0
    if workspace is not None and workspace.numel() < workspace_ints(lo.shape[0]):
        raise NardeCudaError("workspace must hold NARDE_WORKSPACE_INTS(n) = n + 8 int32")
    rc = load().narde_step_full_mirror(
        _ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev), lo.shape[0], env_base, seed, step,
        _ptr(dice_in, torch.uint8, "dice_in", dev), _ptr(action_idx, torch.int32, "action_idx", dev), cap,
        _ptr(actions, torch.int64, "actions", dev), _ptr(counts, torch.int32, "counts", dev),
        _ptr(dice_out, torch.uint8, "dice_out", dev), _ptr(chosen, torch.int64, "chosen", dev),
        _ptr(obs198, torch.float32, "obs198", dev), _ptr(reward, torch.float32, "reward", dev),
        _ptr(done, torch.uint8, "done", dev), _ptr(truncated, torch.uint8, "truncated", dev), _ptr(stats, torch.int64, "stats", dev),
        flags, max_episode_steps, _ptr(workspace, torch.int32, "workspace", dev), _ptr(step_dev, torch.int64, "step_dev", dev),
        _ptr(mirror_lo, torch.uint8, "mirror_lo", dev), _ptr(mirror_hi, torch.uint8, "mirror_hi", dev), _stream())
    _check(rc, "narde_step_full")


def advance_counter(counter):
    import torch

    dev = _device()
    _check(load().narde_advance_counter(_ptr(counter, torch.int64, "counter", dev), _stream()), "narde_advance_counter")


def obs198(lo, hi, out):
    import torch

    dev = _device()
    rc = load().narde_obs198(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev), lo.shape[0],
                             _ptr(out, torch.float32, "obs198", dev), _stream())
    _check(rc, "narde_obs198")


def obs24(lo, hi, out):
    import torch

    dev = _device()
    rc = load().narde_obs24(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev), lo.shape[0],
                            _ptr(out, torch.int32, "obs24", dev), _stream())
    _check(rc, "narde_obs24")


def apply_actions(lo, hi, acts, reward=None, done=None, flags=0):
    import torch

    dev = _device()
    rc = load().narde_apply_actions(_ptr(lo, torch.uint8, "lo", dev), _ptr(hi, torch.uint8, "hi", dev),
                                    _ptr(acts, torch.int64, "acts", dev), lo.shape[0], flags,
                                    _ptr(reward, torch.float32, "reward", dev), _ptr(done, torch.uint8, "done", dev), _stream())
    _check(rc, "narde_apply_actions")


def roll_dice(dice, env_base, seed, step):
    import torch

    dev = _device()
    rc = load().narde_roll_dice(dice.shape[0], env_base, seed, step, _ptr(dice, torch.uint8, "dice", dev), _stream())
    _check(rc, "narde_roll_dice")


def violates_block_rule(boards, out):
    import torch

    dev = _device()
    rc = load().narde_violates_block_rule(_ptr(boards, torch.int8, "boards", dev), boards.shape[0],
                                          _ptr(out, torch.uint8, "out", dev), _stream())
    _check(rc, "narde_violates_block_rule")


# -- afterstate-greedy actor (gym_narde_b200/actor.py) -------------------------------------------
def afterstates(lo, hi, actions, counts, offsets, as_lo, as_hi, row_env=None):
    import torch

    dev, n = _device(), lo.shape[0]
    acts = _ptr(actions, torch.int64, "actions", dev, (n, _ANY))
    rows = _ptr(as_lo, torch.uint8, "as_lo", dev, (_ANY, 16))    # the caller's offsets say how many rows are written
    rc = load().narde_afterstates(_ptr(lo, torch.uint8, "lo", dev, (n, 16)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)), acts,
                                  _ptr(counts, torch.int32, "counts", dev, (n,)), _ptr(offsets, torch.int64, "offsets", dev, (n,)),
                                  n, actions.shape[1], rows, _ptr(as_hi, torch.uint8, "as_hi", dev, tuple(as_lo.shape)),
                                  _ptr(row_env, torch.int32, "row_env", dev, (as_lo.shape[0],)), _stream())
    _check(rc, "narde_afterstates")


def afterstates_scan(lo, hi, actions, counts, as_lo, as_hi, scratch, offsets=None, rows_out=None, rows_cap=0,
                     counts_eff=None, row_env=None):
    """Rows of every env's first min(counts, cap) actions; rows_cap > 0 bounds them, else there may be n * cap."""
    import torch

    dev, n = _device(), lo.shape[0]
    acts = _ptr(actions, torch.int64, "actions", dev, (n, _ANY))
    cap = actions.shape[1]
    rows = rows_cap if rows_cap > 0 else n * cap
    rc = load().narde_afterstates_scan(
        _ptr(lo, torch.uint8, "lo", dev, (n, 16)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)), acts,
        _ptr(counts, torch.int32, "counts", dev, (n,)), n, cap, _ptr(offsets, torch.int64, "offsets", dev, (n,)),
        _ptr(rows_out, torch.int64, "rows_out", dev, (1,)), _ptr(as_lo, torch.uint8, "as_lo", dev, (_ANY, 16), rows),
        _ptr(as_hi, torch.uint8, "as_hi", dev, (_ANY, 16), rows), _ptr(row_env, torch.int32, "row_env", dev, (_ANY,), rows),
        _ptr(scratch, torch.int64, "scratch", dev, (_ANY,), (n + 127) // 128 + 4), rows_cap,   # NARDE_AFTERSTATE_SCRATCH_WORDS
        _ptr(counts_eff, torch.int32, "counts_eff", dev, (n,)), _stream())
    _check(rc, "narde_afterstates_scan")


def gather_overflow(lo, hi, dice, overflow, sub_lo, sub_hi, sub_dice, sub_idx, ctrl, act_override=None):
    """act_override ([n] int64, optional) is zeroed for every env: the turn starts with no stale override."""
    import torch

    dev, n, m = _device(), lo.shape[0], sub_lo.shape[0]
    if m % 32:
        raise NardeCudaError("the side batch must have a multiple of 32 slots, got %d" % m)
    rc = load().narde_gather_overflow_clear(
        _ptr(lo, torch.uint8, "lo", dev, (n, 16)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)),
        _ptr(dice, torch.uint8, "dice", dev, (n, 2)), _ptr(overflow, torch.uint8, "overflow", dev, (n,)), n, m,
        _ptr(sub_lo, torch.uint8, "sub_lo", dev, (m, 16)), _ptr(sub_hi, torch.uint8, "sub_hi", dev, (m, 16)),
        _ptr(sub_dice, torch.uint8, "sub_dice", dev, (m, 2)), _ptr(sub_idx, torch.int32, "sub_idx", dev, (m,)),
        _ptr(ctrl, torch.int32, "ctrl", dev, (_ANY,), 4), _ptr(act_override, torch.int64, "act_override", dev, (n,)),
        _stream())
    _check(rc, "narde_gather_overflow")


def scatter_choice(sub_choice, sub_value, sub_idx, sub_counts_eff, sub_counts, cap, choice, value, ctrl, sub_actions=None,
                   act_out=None):
    import torch

    dev, m, n = _device(), sub_choice.shape[0], choice.shape[0]
    rc = load().narde_scatter_choice(
        _ptr(sub_choice, torch.int32, "sub_choice", dev, (m,)), _ptr(sub_value, torch.float32, "sub_value", dev, (m,)),
        _ptr(sub_idx, torch.int32, "sub_idx", dev, (m,)), _ptr(sub_counts_eff, torch.int32, "sub_counts_eff", dev, (m,)),
        _ptr(sub_counts, torch.int32, "sub_counts", dev, (m,)), m, cap, _ptr(choice, torch.int32, "choice", dev, (n,)),
        _ptr(value, torch.float32, "value", dev, (n,)), _ptr(ctrl, torch.int32, "ctrl", dev, (_ANY,), 4),
        _ptr(sub_actions, torch.int64, "sub_actions", dev, (m, cap)), _ptr(act_out, torch.int64, "act_out", dev, (n,)),
        _stream())
    _check(rc, "narde_scatter_choice")


def segment_argmax(score, offsets, counts, hi, cap, mode, idx_out, best_out=None):
    """idx_out[i] = arg-max (mode 1: BLACK to move takes the arg-min) of score[offsets[i] : offsets[i] + min(counts[i], cap)]."""
    import torch

    dev, n = _device(), hi.shape[0]
    rc = load().narde_segment_argmax(
        _ptr(score, torch.float32, "score", dev, (_ANY,)), _ptr(offsets, torch.int64, "offsets", dev, (n,)),
        _ptr(counts, torch.int32, "counts", dev, (n,)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)), n, cap, mode,
        _ptr(idx_out, torch.int32, "idx_out", dev, (n,)), _ptr(best_out, torch.float32, "best_out", dev, (n,)), _stream())
    _check(rc, "narde_segment_argmax")


def segment_sample(score, offsets, counts, hi, cap, mode, env_base, seed, step, params, idx_out, value_out=None,
                   env_idx=None, step_dev=None):
    """narde_segment_sample: segment_argmax with epsilon-greedy / softmax exploration, params = float32 [2] on the device
    {epsilon, 1 / temperature}; env_idx ([n] int32, optional) maps slot i to its env (env_base + env_idx[i]); step_dev
    (int64 [1], optional) overrides `step` with the device-resident turn number."""
    import torch

    dev, n = _device(), hi.shape[0]
    rc = load().narde_segment_sample(
        _ptr(score, torch.float32, "score", dev, (_ANY,)), _ptr(offsets, torch.int64, "offsets", dev, (n,)),
        _ptr(counts, torch.int32, "counts", dev, (n,)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)), n, cap, mode,
        _ptr(env_idx, torch.int32, "env_idx", dev, (n,)), env_base, seed & 0xFFFFFFFFFFFFFFFF, step,
        _ptr(step_dev, torch.int64, "step_dev", dev, (1,)), _ptr(params, torch.float32, "params", dev, (2,)),
        _ptr(idx_out, torch.int32, "idx_out", dev, (n,)), _ptr(value_out, torch.float32, "value_out", dev, (n,)), _stream())
    _check(rc, "narde_segment_sample")


def step_chosen(lo, hi, env_base, seed, step, dice, choice, actions, counts, act_override=None, chosen=None, obs198=None,
                reward=None, done=None, truncated=None, stats=None, flags=0, max_episode_steps=0, step_dev=None):
    import torch

    dev, n = _device(), lo.shape[0]
    acts = _ptr(actions, torch.int64, "actions", dev, (n, _ANY))
    rc = load().narde_step_chosen(
        _ptr(lo, torch.uint8, "lo", dev, (n, 16)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)), n, env_base, seed, step,
        _ptr(dice, torch.uint8, "dice", dev, (n, 2)), _ptr(choice, torch.int32, "choice", dev, (n,)), acts, actions.shape[1],
        _ptr(counts, torch.int32, "counts", dev, (n,)), _ptr(act_override, torch.int64, "act_override", dev, (n,)),
        _ptr(chosen, torch.int64, "chosen", dev, (n,)), _ptr(obs198, torch.float32, "obs198", dev, (n, 198)),
        _ptr(reward, torch.float32, "reward", dev, (n,)), _ptr(done, torch.uint8, "done", dev, (n,)),
        _ptr(truncated, torch.uint8, "truncated", dev, (n,)), _ptr(stats, torch.int64, "stats", dev, (NUM_STATS,)), flags,
        max_episode_steps, _ptr(step_dev, torch.int64, "step_dev", dev, (1,)), _stream())
    _check(rc, "narde_step_chosen")


# -- trajectory ring and trainer action codes (gym_narde_b200/trajectory.py) ---------------------
def action_codes(actions, counts, codes):
    import torch

    dev, n = _device(), actions.shape[0]
    acts = _ptr(actions, torch.int64, "actions", dev, (n, _ANY))
    cap = actions.shape[1]
    rc = load().narde_action_codes(acts, _ptr(counts, torch.int32, "counts", dev, (n,)), n, cap,
                                   _ptr(codes, torch.int32, "codes", dev, (n, cap, 3)), _stream())
    _check(rc, "narde_action_codes")


def trajectory_append(lo, hi, records, dice=None, chosen=None, reward=None, done=None, truncated=None):
    import torch

    dev, n = _device(), lo.shape[0]
    rc = load().narde_trajectory_append(
        _ptr(lo, torch.uint8, "lo", dev, (n, 16)), _ptr(hi, torch.uint8, "hi", dev, (n, 16)),
        _ptr(dice, torch.uint8, "dice", dev, (n, 2)), _ptr(chosen, torch.int64, "chosen", dev, (n,)),
        _ptr(reward, torch.float32, "reward", dev, (n,)), _ptr(done, torch.uint8, "done", dev, (n,)),
        _ptr(truncated, torch.uint8, "truncated", dev, (n,)), n, _ptr(records, torch.uint8, "records", dev, (n, 48)),
        _stream())
    _check(rc, "narde_trajectory_append")


# -- afterstate-scoring MLP (gym_narde_b200/mlp.py): x [K,198] f32 rows or packed states [K,16] x2 in; q [K,576] or
#    score [K] f32 out; wpack int16 / bias f32 / w2b_t f32 as mlp.pack_weights and AfterstateMLP.set_move2_head make them
def mlp_forward(x, wpack, bias, out):
    import torch

    dev, k = _device(), x.shape[0]
    rc = load().narde_mlp_forward(_ptr(x, torch.float32, "x", dev, (k, 198)), k, _ptr(wpack, torch.int16, "wpack", dev),
                                  _ptr(bias, torch.float32, "bias", dev), _ptr(out, torch.float32, "out", dev, (k, 576)),
                                  _stream())
    _check(rc, "narde_mlp_forward")


def mlp_score(x, wpack, bias, out):
    import torch

    dev, k = _device(), x.shape[0]
    rc = load().narde_mlp_score(_ptr(x, torch.float32, "x", dev, (k, 198)), k, _ptr(wpack, torch.int16, "wpack", dev),
                                _ptr(bias, torch.float32, "bias", dev), _ptr(out, torch.float32, "out", dev, (k,)), _stream())
    _check(rc, "narde_mlp_score")


def mlp_forward_states(lo, hi, wpack, bias, out):
    import torch

    dev, k = _device(), lo.shape[0]
    rc = load().narde_mlp_forward_states(_ptr(lo, torch.uint8, "lo", dev, (k, 16)), _ptr(hi, torch.uint8, "hi", dev, (k, 16)), k,
                                         _ptr(wpack, torch.int16, "wpack", dev), _ptr(bias, torch.float32, "bias", dev),
                                         _ptr(out, torch.float32, "out", dev, (k, 576)), _stream())
    _check(rc, "narde_mlp_forward_states")


def mlp_score_states(lo, hi, wpack, bias, out, rows_dev=None, two_sm=False):
    """rows_dev: int64 [1] on the device; only min(rows_dev, K) rows are scored.  two_sm: the cta_group::2 kernel
    (wpack packed with pack_weights(two_sm=True))."""
    import torch

    dev, k = _device(), lo.shape[0]
    name = "narde_mlp_score_states_2sm" if two_sm else "narde_mlp_score_states"
    rc = getattr(load(), name)(
        _ptr(lo, torch.uint8, "lo", dev, (k, 16)), _ptr(hi, torch.uint8, "hi", dev, (k, 16)), k,
        _ptr(rows_dev, torch.int64, "rows_dev", dev, (1,)), _ptr(wpack, torch.int16, "wpack", dev),
        _ptr(bias, torch.float32, "bias", dev), _ptr(out, torch.float32, "out", dev, (k,)), _stream())
    _check(rc, name)


def mlp_forward_move2(x, move1, wpack, bias, w2b_t, out):
    import torch

    dev, k = _device(), x.shape[0]
    rc = load().narde_mlp_forward_move2(_ptr(x, torch.float32, "x", dev, (k, 198)), k,
                                        _ptr(move1, torch.int32, "selected_move1", dev, (k,)),
                                        _ptr(wpack, torch.int16, "wpack", dev), _ptr(bias, torch.float32, "bias", dev),
                                        _ptr(w2b_t, torch.float32, "w2b_t", dev, (576, 576)),
                                        _ptr(out, torch.float32, "out", dev, (k, 576)), _stream())
    _check(rc, "narde_mlp_forward_move2")


def mlp_forward_move2_states(lo, hi, move1, wpack, bias, w2b_t, out):
    import torch

    dev, k = _device(), lo.shape[0]
    rc = load().narde_mlp_forward_move2_states(
        _ptr(lo, torch.uint8, "lo", dev, (k, 16)), _ptr(hi, torch.uint8, "hi", dev, (k, 16)), k,
        _ptr(move1, torch.int32, "selected_move1", dev, (k,)), _ptr(wpack, torch.int16, "wpack", dev),
        _ptr(bias, torch.float32, "bias", dev), _ptr(w2b_t, torch.float32, "w2b_t", dev, (576, 576)),
        _ptr(out, torch.float32, "out", dev, (k, 576)), _stream())
    _check(rc, "narde_mlp_forward_move2_states")
