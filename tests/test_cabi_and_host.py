"""CPU: the C-ABI library loads and exports every symbol include/narde_b200.h declares; the host
side fails loudly without CUDA; the product never touches the oracle."""
import os
import re

import numpy as np
import pytest

from gym_narde_b200 import _cabi
from gym_narde_b200 import state as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "narde_b200.h")).read()
    declared = set(re.findall(r"\b(narde_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 13
    lib = _cabi.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_cabi.exported_symbols())
    # and the other way round: every narde_* symbol the product library exports is declared (no debug hooks, no
    # undeclared entry points)
    import subprocess
    nm = subprocess.run(["nm", "-D", "--defined-only", _cabi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (narde_[A-Za-z0-9_]+)$", nm, flags=re.M))
    assert exported == declared, exported ^ declared
    assert lib.narde_abi_version() == _cabi.ABI_VERSION == 4 and lib.narde_build_arch() == b"sm_100a"


def test_bad_arguments_are_rejected_without_a_gpu():
    lib = _cabi.load()
    assert lib.narde_reset(None, None, 4, 0, 0, 0, None) == -1
    assert lib.narde_enumerate(None, None, None, 4, 8, None, None, None, None) == -1
    assert lib.narde_reset(None, None, -1, 0, 0, 0, None) == -1
    # empty batches are a no-op for every entry point (n == 0 / rows == 0 returns before any CUDA call)
    assert lib.narde_reset(None, None, 0, 0, 0, 0, None) == 0
    assert lib.narde_enumerate(None, None, None, 0, 8, None, None, None, None) == 0
    assert lib.narde_enumerate_fast(None, None, None, 0, 8, None, None, None, None, None) == 0
    assert lib.narde_step_full(None, None, 0, 0, 0, 0, None, None, 8, None, None, None, None, None, None, None, None,
                               None, 0, 0, None, None, None) == 0
    assert lib.narde_mlp_forward(None, 0, None, None, None, None) == 0
    assert lib.narde_afterstates(None, None, None, None, None, 0, 8, None, None, None, None) == 0
    # null / misaligned buffers and negative sizes are rejected with -1, nothing is launched
    assert lib.narde_step_full(None, None, 4, 0, 0, 0, None, None, 8, None, None, None, None, None, None, None, None,
                               None, 0, 0, None, None, None) == -1
    assert lib.narde_enumerate_fast(None, None, None, 4, 8, None, None, None, None, None) == -1
    assert lib.narde_mlp_forward(None, 4, None, None, None, None) == -1
    assert lib.narde_mlp_score(None, 4, None, None, None, None) == -1
    assert lib.narde_mlp_forward_states(None, None, 4, None, None, None, None) == -1
    assert lib.narde_mlp_score_states(None, None, 4, None, None, None, None, None) == -1
    assert lib.narde_afterstates(None, None, None, None, None, 4, 8, None, None, None, None) == -1
    assert lib.narde_afterstates_scan(None, None, None, None, 0, 8, None, None, None, None, None, None, 0, None, None) == 0
    assert lib.narde_afterstates_scan(None, None, None, None, 4, 8, None, None, None, None, None, None, 0, None, None) == -1
    assert lib.narde_segment_argmax(None, None, None, None, 4, 8, 0, None, None, None) == -1
    assert lib.narde_mlp_forward(None, -3, None, None, None, None) == -1
    assert lib.narde_mlp_forward_move2(None, 0, None, None, None, None, None, None) == 0
    assert lib.narde_mlp_forward_move2(None, 4, None, None, None, None, None, None) == -1
    assert lib.narde_mlp_forward_move2_states(None, None, 4, None, None, None, None, None, None) == -1
    import ctypes as C
    buf = C.create_string_buffer(256)
    base = C.addressof(buf)
    mis = C.c_void_p(base + 8 if base % 16 == 0 else base)          # 8-byte aligned, not 16
    assert lib.narde_reset(mis, mis, 2, 0, 0, 0, None) == -1


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import gym_narde_b200
    with pytest.raises(_cabi.NardeCudaError):
        gym_narde_b200.make("narde-v0")
    with pytest.raises(_cabi.NardeCudaError):
        gym_narde_b200.VecNardeEnv(4)
    with pytest.raises(_cabi.NardeCudaError):
        _cabi.reset(torch.zeros((1, 16), dtype=torch.uint8), torch.zeros((1, 16), dtype=torch.uint8), 0, 0, 0)


def test_actor_trajectory_and_mlp_wrappers_have_no_cpu_fallback():
    """Every C-ABI wrapper of the actor, trajectory and MLP entry points raises NardeCudaError for CPU tensors (with or
    without a CUDA device present)."""
    import torch
    u8, i16, i32, i64, f32 = torch.uint8, torch.int16, torch.int32, torch.int64, torch.float32
    z = lambda dt, *shape: torch.zeros(shape, dtype=dt)
    n, cap, m = 4, 8, 32
    lo, hi, acts, counts = z(u8, n, 16), z(u8, n, 16), z(i64, n, cap), z(i32, n)
    x, wpack, bias, w2b_t, move1 = z(f32, n, 198), z(i16, 64), z(f32, 1088), z(f32, 576, 576), z(i32, n)
    calls = [
        ("afterstates", (lo, hi, acts, counts, z(i64, n), z(u8, n * cap, 16), z(u8, n * cap, 16))),
        ("afterstates_scan", (lo, hi, acts, counts, z(u8, n * cap, 16), z(u8, n * cap, 16), z(i64, 5))),
        ("gather_overflow", (lo, hi, z(u8, n, 2), z(u8, n), z(u8, m, 16), z(u8, m, 16), z(u8, m, 2), z(i32, m), z(i32, 4))),
        ("scatter_choice", (z(i32, m), z(f32, m), z(i32, m), z(i32, m), z(i32, m), cap, z(i32, n), z(f32, n), z(i32, 4))),
        ("segment_argmax", (z(f32, n * cap), z(i64, n), counts, hi, cap, 0, z(i32, n))),
        ("step_chosen", (lo, hi, 0, 0, 0, z(u8, n, 2), z(i32, n), acts, counts)),
        ("action_codes", (acts, counts, z(i32, n, cap, 3))),
        ("trajectory_append", (lo, hi, z(u8, n, 48))),
        ("mlp_forward", (x, wpack, bias, z(f32, n, 576))),
        ("mlp_score", (x, wpack, bias, z(f32, n))),
        ("mlp_forward_states", (lo, hi, wpack, bias, z(f32, n, 576))),
        ("mlp_score_states", (lo, hi, wpack, bias, z(f32, n))),
        ("mlp_score_states", (lo, hi, wpack, bias, z(f32, n), None, True)),
        ("mlp_forward_move2", (x, move1, wpack, bias, w2b_t, z(f32, n, 576))),
        ("mlp_forward_move2_states", (lo, hi, move1, wpack, bias, w2b_t, z(f32, n, 576))),
    ]
    for name, args in calls:
        with pytest.raises(_cabi.NardeCudaError):
            getattr(_cabi, name)(*args)


def test_only_cabi_calls_the_library():
    """_cabi.py is the package's one bridge to the C ABI: no other module builds ctypes pointers or calls a narde_*
    symbol itself.  (envs/, the single-env facade, keeps pointers cached at construction: its per-call latency is its
    point.)"""
    pkg = os.path.join(ROOT, "gym_narde_b200")
    for dp, _, files in os.walk(pkg):
        if os.path.relpath(dp, pkg).split(os.sep)[0] == "envs":
            continue
        for f in files:
            if f.endswith(".py") and f != "_cabi.py":
                src = open(os.path.join(dp, f)).read()
                assert "c_void_p" not in src and not re.search(r"\.narde_\w+\s*\(", src), (dp, f)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gym_narde_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("the oracle computes", "").replace("against the oracle", "") \
                    .replace("oracle/narde_oracle.c", "") or f in ("narde_core.cuh",), (dp, f)
                assert "hostsim" not in src or "test-only" in src or "tests/hostsim" in src, (dp, f)


def test_state_pack_roundtrip():
    rng = np.random.RandomState(0)
    b = rng.randint(-15, 16, size=(50, 24))
    lo, hi = S.pack_states(b, rng.randint(0, 16, 50), rng.randint(0, 16, 50), rng.choice([1, -1], 50),
                           rng.rand(50) < .5, rng.rand(50) < .5, steps=rng.randint(0, 60000, 50))
    u = S.unpack_states(lo, hi)
    assert (u["board"] == b).all()
    acts = [[(23, 17), (17, 11)], [(3, 'off')], [], [(5, 4), (4, 3), (3, 2), (2, 'off')]]
    for a in acts:
        assert S.decode_action(S.encode_action(a)) == a


def test_expand_obs198_on_the_host_equals_the_oracle():
    """gym_narde_b200.expand_obs198 (decoder of the packed observation a host consumer of step_host(obs="packed")
    receives) against o_obs198 (README.md:44-102), bit for bit."""
    import gym_narde_b200
    import parity as P
    from oracle import oracle as O
    lo, hi = P.pack_corpus(P.selfplay_corpus(12, 3))
    got = gym_narde_b200.expand_obs198(lo, hi)
    u = S.unpack_states(lo, hi)
    for i in range(lo.shape[0]):
        ref = O.obs198(u["board"][i], int(u["off_w"][i]), int(u["off_b"][i]), int(u["turn"][i]))
        assert (ref == got[i]).all(), i


def test_compact_record_decoder_round_trip():
    """gym_narde_b200.state.unpack_compact against a numpy restatement of the packing the kernels do
    (narde_env.cuh pack_compact; layout in include/narde_b200.h): random legal-range states survive the round trip."""
    import numpy as np
    from gym_narde_b200 import state as S
    rng = np.random.default_rng(5)
    n = 4000
    boards = rng.integers(-15, 16, (n, 24))
    off_w, off_b = rng.integers(0, 16, n), rng.integers(0, 16, n)
    turn = rng.choice([-1, 1], n)
    fw, fb, dn = rng.integers(0, 2, n).astype(bool), rng.integers(0, 2, n).astype(bool), rng.integers(0, 2, n).astype(bool)
    steps = rng.integers(0, 1 << 16, n)
    result = rng.integers(0, 12, n)
    lo, hi = S.pack_states(boards, off_w, off_b, turn, fw, fb, dn, steps)
    a = np.zeros(n, np.uint64)
    b = np.zeros(n, np.uint64)
    for p in range(12):
        a |= (boards[:, p].astype(np.int64) & 31).astype(np.uint64) << np.uint64(5 * p)
        b |= (boards[:, p + 12].astype(np.int64) & 31).astype(np.uint64) << np.uint64(5 * p)
    x0 = a | (b << np.uint64(60))
    x1 = (b >> np.uint64(4)) | (off_w.astype(np.uint64) << np.uint64(56)) | (off_b.astype(np.uint64) << np.uint64(60))
    w4 = ((turn == 1).astype(np.uint32) | (hi[:, 11].astype(np.uint32) << 1) | (result.astype(np.uint32) << 4)
          | (steps.astype(np.uint32) << 8))
    rec = np.zeros((n, 20), np.uint8)
    rec[:, 0:8] = x0.view(np.uint8).reshape(n, 8)
    rec[:, 8:16] = x1.view(np.uint8).reshape(n, 8)
    rec[:, 16:20] = w4.astype("<u4").view(np.uint8).reshape(n, 4)
    lo2, hi2, res = S.unpack_compact(rec)
    assert (lo2 == lo).all() and (hi2 == hi).all() and (res == result).all()
