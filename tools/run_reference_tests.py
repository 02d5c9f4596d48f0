"""Run the REFERENCE's own hot-path test files against the GPU adapter (SURVEY section 4, plan step 2).

    python tools/run_reference_tests.py [--reference /path/to/RL_brain_trainer] [-k pattern]

The reference's tests construct ``ArmKinematicEnv`` / ``Phase1EnvConfig`` from ``hrl_trainer.kinematic_phase1.envs.arm_kinematic_env``.
This runner imports the reference package from the given checkout (read-only, nothing is copied), replaces those two names -- in that
module and in the package namespaces that re-export them -- with this repository's drop-in classes, then loads
``tests/test_kinematic_phase1_{env,eval,reward,approach_reward,split}.py`` and runs them with unittest.  Tests that never touch the env
class (pure reward-function tests) run against the reference's own functions and pass trivially; the ones that step the env exercise
``libkin_b200.so``.

It needs a machine with BOTH a B200 and a checkout of the reference, and reference sources must not be copied into the repository,
so the test suite does not run it; ``tests/test_gpu_rollout.py::test_single_env_adapter_conformance`` restates the env-facing
assertions of those files.
"""
from __future__ import annotations

import argparse
import importlib
import importlib.util
import sys
import unittest
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
FILES = ("test_kinematic_phase1_env.py", "test_kinematic_phase1_eval.py", "test_kinematic_phase1_reward.py",
         "test_kinematic_phase1_approach_reward.py", "test_kinematic_phase1_split.py")


def patch_reference(reference_root: Path):
    """Import the reference package and swap its env class / config for the drop-in ones.  Returns the patched module."""
    pkg = reference_root / "hrl_ws" / "src" / "hrl_trainer"
    if not (pkg / "hrl_trainer" / "kinematic_phase1").exists():
        raise FileNotFoundError(f"no reference checkout under {reference_root}")
    sys.dont_write_bytecode = True
    for p in (str(ROOT), str(pkg)):
        if p not in sys.path:
            sys.path.insert(0, p)
    from rl_brain_trainer_b200.config import Phase1EnvConfig
    from rl_brain_trainer_b200.env import ArmKinematicEnv

    mod = importlib.import_module("hrl_trainer.kinematic_phase1.envs.arm_kinematic_env")
    mod.ArmKinematicEnv, mod.Phase1EnvConfig = ArmKinematicEnv, Phase1EnvConfig
    for name in ("hrl_trainer.kinematic_phase1", "hrl_trainer.kinematic_phase1.envs"):
        ns = importlib.import_module(name)
        for attr, val in (("ArmKinematicEnv", ArmKinematicEnv), ("Phase1EnvConfig", Phase1EnvConfig)):
            if hasattr(ns, attr):
                setattr(ns, attr, val)
    return mod


def load_suite(reference_root: Path, pattern: str | None = None) -> unittest.TestSuite:
    tests_dir = reference_root / "hrl_ws" / "src" / "hrl_trainer" / "tests"
    suite = unittest.TestSuite()
    loader = unittest.TestLoader()
    if pattern:
        loader.testNamePatterns = [f"*{pattern}*"]
    for f in FILES:
        spec = importlib.util.spec_from_file_location(f"_ref_{f[:-3]}", tests_dir / f)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        suite.addTests(loader.loadTestsFromModule(m))
    return suite


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    ap.add_argument("-k", default=None)
    a = ap.parse_args()
    patch_reference(Path(a.reference))
    result = unittest.TextTestRunner(verbosity=2).run(load_suite(Path(a.reference), a.k))
    sys.exit(0 if result.wasSuccessful() else 1)
