"""GPU (-m gpu): the reference's OWN tests and caller scripts, unmodified, against this repo's env.

The original is not part of this repository: baseline/fetch_ref.py vendors its untouched files from a checkout into
baseline/_ref (git-ignored), and these tests skip without them.  tests/refsuite_runner.py runs them in a fresh
process twice: on the real reference env, and with
`gym_narde` aliased to the GPU facade (gym_narde_b200.envs.NardeEnv / Narde through the C ABI).

  * north star: tests/test_move_validation.py and tests/test_doubles_sequence.py pass against the new env
    (the latter through the reference's own web/narde_patched.py + my_game/narde_game_manager.py wrapping env.game);
  * tests/test_narde_game_manager.py: the same per-test outcome as on the reference itself (its
    test_enhance_valid_moves_for_doubles fails on the reference too, SURVEY.md A.3);
  * SURVEY 8(f)-2: evaluate_model.evaluate and train_deepq_pytorch.main run unmodified on the facade and print
    exactly what they print on the reference under the same seeds (the facade consumes the global numpy RNG like
    narde_env.py:29,107-115, so dice, observations, rewards and episode lengths are identical).
"""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "tests", "refsuite_runner.py")
HAVE_REF = os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "gym_narde", "envs", "narde.py"))
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="the original gym-narde is not in the repository: vendor it into "
                                                    "baseline/_ref (build() with NARDE_REFERENCE_ROOT set, or "
                                                    "baseline/fetch_ref.py)")


def _run(impl, what, n=3):
    p = subprocess.run([sys.executable, RUNNER, "--impl", impl, "--what", what, "-n", str(n)], capture_output=True,
                       text=True, timeout=1500, cwd=ROOT)
    lines = [l for l in p.stdout.splitlines() if l.startswith("REFSUITE ")]
    assert p.returncode == 0 and lines, (p.returncode, p.stdout[-2000:], p.stderr[-4000:])
    out = json.loads(lines[-1][len("REFSUITE "):])
    assert out["env_module"].startswith("gym_narde_b200 @" if impl == "facade" else "gym_narde @"), out["env_module"]
    return out["result"]


@needs_ref
def test_reference_unit_tests_run_unmodified_on_the_facade():
    fac, ref = _run("facade", "tests"), _run("reference", "tests")
    for f in ("test_move_validation.py", "test_doubles_sequence.py"):      # named by north_star: all must pass
        assert fac[f] and all(v == "ok" for v in fac[f].values()), (f, fac[f])
    assert len(fac["test_move_validation.py"]) == 2 and len(fac["test_doubles_sequence.py"]) == 3
    assert fac == ref, (fac, ref)                                           # incl. test_narde_game_manager.py, test by test


@needs_ref
def test_evaluate_model_runs_unmodified_and_prints_the_reference_report():
    fac, ref = _run("facade", "evaluate", 4), _run("reference", "evaluate", 4)
    assert any("Games played: 4" in l for l in fac) and any("Average game length" in l for l in fac)
    assert fac == ref, (fac, ref)


@needs_ref
def test_train_deepq_main_runs_unmodified_for_three_episodes():
    fac, ref = _run("facade", "train", 3), _run("reference", "train", 3)
    eps = [l for l in fac if l.startswith("Episode: ")]
    assert len(eps) == 3 and any("Total episodes: 3" in l for l in fac)
    # identical dice / observations / rewards => identical episode lengths and scores, episode by episode
    strip = lambda ls: [l.split(", Epsilon")[0] for l in ls if l.startswith("Episode: ")]
    assert strip(fac) == strip(ref), (fac, ref)
