"""The K2-TC variant matrix: the tensor-core rollout's launch-time switches, each in its own process (the kernel reads them once,
as function statics), on the same Stage-5 suites.

Default, KIN_TC16_SMEM_A=1 (activations through shared memory: the AT = false instantiation), KIN_TC16_NO_ISSUER_WARPS=1 (the
last-arriving warp issues the MMAs), KIN_TC_WARPS=8 (another CTA shape) must give bitwise the same result rows; KIN_TC16_EXACT_SINCOS=1
(the polynomial sine / cosine, FAST = 1) may flip a success flag only on an episode whose fp64 oracle outcome is threshold-sensitive,
and takes the same number of approach steps.
"""

from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from ._util import env_config, oracle_policy, threshold_sensitive_episodes

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
SIZES = (8192, 100)   # a multi-CTA batch and a ragged one (partial tile, partial CTA)
VARIANTS = {
    "default": {},
    "smem_a": {"KIN_TC16_SMEM_A": "1"},
    "no_issuer": {"KIN_TC16_NO_ISSUER_WARPS": "1"},
    "warps8": {"KIN_TC_WARPS": "8"},
    "exact_sincos": {"KIN_TC16_EXACT_SINCOS": "1"},
}
SWITCHES = ("KIN_TC16_SMEM_A", "KIN_TC16_NO_ISSUER_WARPS", "KIN_TC_WARPS", "KIN_TC16_EXACT_SINCOS", "KIN_TC16_POLL_HINT")

CHILD = r"""
import sys
import numpy as np
import torch
from rl_brain_trainer_b200 import config as kcfg
from rl_brain_trainer_b200.policy import PolicyWeights
from rl_brain_trainer_b200.rollout import VARIANT_TC, ApproachFinisherRollout
from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

out = sys.argv[1]
acfg, fcfg = kcfg.load_preset("approach_dynamic_scale_big"), kcfg.load_preset("finisher_noop_ft")
ro = ApproachFinisherRollout(acfg, PolicyWeights.preset("approach_stage8_11", "cuda"), fcfg, PolicyWeights.preset("finisher", "cuda"),
                             variant=VARIANT_TC)
rows = {}
for n in (%s):
    suite = build_curriculum_local_eval_suite(acfg, seed=700001 + 5 * 1009, stage_index=5, n_episodes=n)
    res = ro.evaluate_suite(suite)
    torch.cuda.synchronize()
    rows[f"raw_{n}"] = res.raw[:, :n].cpu().numpy()
    for k, v in res.to_numpy().items():
        rows[f"{k}_{n}"] = v
np.savez(out, **rows)
""" % ", ".join(str(n) for n in SIZES)


def _run_variant(name: str, tmp_path: Path) -> dict[str, np.ndarray]:
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env.update(VARIANTS[name])
    out = tmp_path / f"{name}.npz"
    cmd = [sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", CHILD, str(out)]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"variant {name} failed:\n{r.stdout[-4000:]}\n{r.stderr[-4000:]}"
    with np.load(out) as z:
        return {k: z[k] for k in z.files}


def test_tc16_variants_agree(tmp_path):
    res = {name: _run_variant(name, tmp_path) for name in VARIANTS}
    base = res["default"]
    for name in ("smem_a", "no_issuer", "warps8"):
        for n in SIZES:
            same = base[f"raw_{n}"] == res[name][f"raw_{n}"]
            assert same.all(), f"{name}: result rows differ from the default at n = {n} ({int((~same).sum())} words, rows {np.unique(np.nonzero(~same)[0])})"
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    acfg, fcfg = env_config("approach_dynamic_scale_big"), env_config("finisher_noop_ft")
    ex = res["exact_sincos"]
    for n in SIZES:
        assert np.array_equal(ex[f"approach_steps_{n}"], base[f"approach_steps_{n}"]), n
        flips = ex[f"success_{n}"] != base[f"success_{n}"]
        if flips.any():
            suite = build_curriculum_local_eval_suite(acfg, seed=700001 + 5 * 1009, stage_index=5, n_episodes=n)
            _, sensitive = threshold_sensitive_episodes(acfg, fcfg, oracle_policy("approach_stage8_11"), oracle_policy("finisher"), suite, 0.01,
                                                        n_threads=8)
            assert not (flips & ~sensitive).any(), f"EXACT_SINCOS flips {int((flips & ~sensitive).sum())} episodes that are not threshold-sensitive"
        print(f"n = {n}: EXACT_SINCOS flips {int(flips.sum())} success flags against the MUFU default")
