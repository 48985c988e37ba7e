"""Loads the REAL Python reference (the original gym-narde) -- TEST INFRASTRUCTURE ONLY.

The original is not part of this repository: it is read from NARDE_REFERENCE_ROOT, or else from
baseline/_ref (vendored there by baseline/fetch_ref.py).  Where neither holds it, callers must
check `available()` and skip.
The reference needs `gymnasium`; when the real package is absent, a minimal stub of the few names
it touches (Env, spaces.Box/Discrete/Tuple, envs.registration.register) is injected into sys.modules.

`injected_dice(stream)` replays an explicit dice stream through the reference by patching
numpy.random.randint, which is the only RNG call the reference env makes
(gym_narde/envs/narde_env.py:29,112-113).
"""
from __future__ import annotations

import contextlib
import importlib
import os
import sys
from unittest import mock

import numpy as np

REF_ROOT = os.environ.get("NARDE_REFERENCE_ROOT") or os.path.join(
    os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "baseline", "_ref")


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "gym_narde", "envs", "narde.py"))


def _install_gymnasium_stub():
    """tests/gymnasium_stub.py (one stub for the whole test-suite)."""
    tests = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests")
    if tests not in sys.path:
        sys.path.insert(0, tests)
    import gymnasium_stub
    gymnasium_stub.install()


_cache = {}


def load():
    """Returns (narde_module, narde_env_module) of the real reference."""
    if "mods" in _cache:
        return _cache["mods"]
    if not available():
        raise RuntimeError("reference not present at %s" % REF_ROOT)
    _install_gymnasium_stub()
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    narde = importlib.import_module("gym_narde.envs.narde")
    narde_env = importlib.import_module("gym_narde.envs.narde_env")
    _cache["mods"] = (narde, narde_env)
    return _cache["mods"]


@contextlib.contextmanager
def injected_dice(stream):
    """Patch numpy.random.randint so the reference env consumes `stream` (ints 1..6) verbatim."""
    it = iter(stream)

    def fake_randint(low, high=None, size=None, dtype=int):
        assert size is None
        return int(next(it))

    with mock.patch("numpy.random.randint", side_effect=fake_randint):
        yield
