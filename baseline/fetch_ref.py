"""Vendor the UNMODIFIED original gym-narde files into baseline/_ref/ (git-ignored: nothing of the original enters
this repository's history).  The original is not part of this repository; point the script at a checkout of it:

    NARDE_REFERENCE_ROOT=<gym-narde checkout> python baseline/fetch_ref.py
    python baseline/fetch_ref.py <gym-narde checkout>

__graft_entry__.build() runs it when NARDE_REFERENCE_ROOT is set.

What is copied: the env path (`gym_narde/`), the two wrappers its tests need (`web/narde_patched.py`,
`my_game/narde_game_manager.py`), the original's own runnable tests, and the two caller scripts of
SURVEY.md 8(f)-2 (`evaluate_model.py`, `train_deepq_pytorch.py`) with the checkpoint `evaluate` loads.
Used by: tests/test_gpu_reference_suite.py (the original's tests and scripts run against the facade),
tests/test_oracle.py::test_oracle_vs_live_reference_short (through oracle/ref_loader.py), bench.py's
python_reference rates.  Those skip (or leave the rates out) when baseline/_ref is absent.
"""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")

FILES = [
    "gym_narde/__init__.py", "gym_narde/envs/__init__.py", "gym_narde/envs/narde.py", "gym_narde/envs/narde_env.py",
    "gym_narde/envs/rendering.py",
    "web/narde_patched.py", "my_game/__init__.py", "my_game/narde_game_manager.py",
    "tests/test_move_validation.py", "tests/test_doubles_sequence.py", "tests/test_narde_game_manager.py",
    "evaluate_model.py", "train_deepq_pytorch.py", "saved_models/narde_model_final.pt", "LICENSE",
]


def available() -> bool:
    return os.path.isfile(os.path.join(DEST, "gym_narde", "envs", "narde.py"))


def fetch(src: str, verbose: bool = True) -> bool:
    if not os.path.isfile(os.path.join(src, "gym_narde", "envs", "narde.py")):
        raise SystemExit("fetch_ref: %s is not a gym-narde checkout (no gym_narde/envs/narde.py)" % src)
    os.makedirs(DEST, exist_ok=True)
    for rel in FILES:
        s, d = os.path.join(src, rel), os.path.join(DEST, rel)
        if not os.path.isfile(s):
            continue
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
    with open(os.path.join(DEST, "FETCHED.txt"), "w") as f:
        f.write("unmodified files of %s\n" % os.path.abspath(src))
    if verbose:
        print("fetch_ref: %d files -> %s" % (len(FILES), DEST))
    return available()


if __name__ == "__main__":
    src = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("NARDE_REFERENCE_ROOT")
    if not src:
        raise SystemExit(__doc__)
    sys.exit(0 if fetch(src) else 1)
