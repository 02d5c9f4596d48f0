"""Adaptive frontier curriculum costs on the GPU (CUDA events / host clock after a device synchronise; the GPU's name and power limit
are read in the same run).

    python tools/frontier_bench.py [--envs 65536] [--steps 128] [--rounds 5] [--collects 10] [--parent-tree DIR] [--out FILE]

A. K4 cost: ``PPOTrainer.collect()`` (one fused ``kin_ppo_collect`` launch + bootstrap + GAE) on the randomstart preset at Stage 8,
   the bundled ``randomstart`` policy.  Variants: the new library with the frontier branch unarmed, the same library armed at p = 0.5
   (a training-map table of the preset's coverage sizes), and -- with ``--parent-tree`` (a checkout of the previous commit with its
   library built) -- the previous library, which has no branch.  Each variant runs in a child process per round, the order alternating
   round by round; inside the new library's process the unarmed and armed collections alternate.  Reported: the median over rounds of
   each round's median collect time, and the spread of the round medians.
B. Refresh cost: ``FrontierCurriculum.maybe_refresh`` (coverage eval with the Finisher, priorities, table build, upload) at the preset's
   sizes (2 048 pairs, 96 episodes per split) and at 10^6 pairs with no split limit (the stress split runs every pair).
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]


def gpu_identity() -> dict:
    import torch

    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        out["nvidia_smi"] = f"unavailable: {exc}"
    return out


def collect_worker(tree: Path, arms: list[str], envs: int, steps: int, collects: int) -> dict:
    """Runs in a child process against the package of ``tree``: per arm, ``collects`` timed collections (alternating arms)."""
    sys.path.insert(0, str(tree))
    import torch

    from rl_brain_trainer_b200 import config as kcfg, ppo
    from rl_brain_trainer_b200.policy import PolicyWeights

    torch.cuda.set_device(0)
    cfg = kcfg.load_preset("randomstart_overnight")
    hp = ppo.PPOHyper(n_steps=steps, batch_size=envs * steps // 4, n_epochs=1, learning_rate=0.0)
    tr = ppo.PPOTrainer(cfg, PolicyWeights.preset("randomstart", "cuda"), num_envs=envs, hyper=hp, seed=3, stage_index=8)
    table = None
    if "armed" in arms:
        from rl_brain_trainer_b200 import coverage as cov, workspace as ws

        tm = ws.generate_workspace_target_map(cfg, seed=940001 + 104729, stage_samples_per_stage=192, random_samples=768)
        tb = cov.target_buckets(tm)
        rng = np.random.default_rng(0)
        table = cov.FrontierTable.build(tm, tb, {b: float(rng.uniform(0.05, 1.1)) for b in tb.ids}, device="cuda")

    def arm(name: str) -> None:
        if table is not None:
            tr.env.set_frontier_targets(table if name == "armed" else None, 0.5)
        tr.env._ensure_sampler()          # the (synchronous) sampler upload stays outside the timed window

    for name in arms * 2:                 # warm-up
        arm(name)
        tr.collect()
    out: dict[str, list[float]] = {a: [] for a in arms}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(collects):
        for name in arms:
            arm(name)
            torch.cuda.synchronize()
            ev0.record()
            tr.collect()
            ev1.record()
            torch.cuda.synchronize()
            out[name].append(ev0.elapsed_time(ev1))
    return out


def refresh_cost(pairs: int, episodes_per_split: int, repeats: int) -> dict:
    sys.path.insert(0, str(ROOT))
    import torch

    from rl_brain_trainer_b200 import config as kcfg, coverage as cov
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv
    from rl_brain_trainer_b200.policy import PolicyWeights

    preset = kcfg.preset_dict("randomstart_overnight")
    acfg, fcfg = kcfg.to_env_config(preset), kcfg.load_preset("finisher_noop_ft")
    cur = cov.FrontierCurriculum.from_config(preset, acfg, fcfg, PolicyWeights.preset("finisher", "cuda"), pair_count=pairs,
                                             episodes_per_split=episodes_per_split)
    env = BatchedArmKinematicEnv(acfg, 1024, "cuda", host_sampler=False)
    pol = PolicyWeights.preset("randomstart", "cuda")
    cur.maybe_refresh(0, pol, env, force=True)          # warm-up: module loads, allocator
    times, recs = [], []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rec = cur.maybe_refresh(0, pol, env, force=True)
        env._ensure_sampler()                           # the upload of the new table belongs to the refresh
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
        recs.append(rec)
    last = recs[-1]
    episodes = sum(cur.last_summary[k]["episode_count"] for k in ("random_start_known_workspace", "random_start_frontier", "full_reachable_stress"))
    return {"pairs": pairs, "episodes_per_split": episodes_per_split, "episodes": int(episodes), "env_steps": int(cur.last_summary["env_steps"]),
            "refresh_ms": times, "median_ms": float(np.median(times)), "table_buckets": last["table_bucket_count"],
            "table_targets": cur.table.target_count, "defaulted_buckets": last["defaulted_bucket_count"], "checksum": last["table_checksum"]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--collects", type=int, default=10)
    ap.add_argument("--parent-tree", type=Path, default=None)
    ap.add_argument("--skip-collect", action="store_true")
    ap.add_argument("--skip-refresh", action="store_true")
    ap.add_argument("--out", type=Path, default=None)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)     # internal: "<tree>|<arm,arm>"
    a = ap.parse_args()
    if a.worker:
        tree, arms = a.worker.split("|")
        print(json.dumps(collect_worker(Path(tree), arms.split(","), a.envs, a.steps, a.collects)))
        return
    result: dict = {}
    if not a.skip_collect:
        jobs = [("new", str(ROOT), "unarmed,armed")]
        if a.parent_tree is not None:
            jobs.append(("parent", str(a.parent_tree.resolve()), "unarmed"))
        rounds: dict[str, list[float]] = {}
        for r in range(a.rounds):
            for label, tree, arms in (jobs if r % 2 == 0 else jobs[::-1]):
                cmd = [sys.executable, str(Path(__file__).resolve()), "--worker", f"{tree}|{arms}", "--envs", str(a.envs), "--steps", str(a.steps),
                       "--collects", str(a.collects)]
                p = subprocess.run(cmd, capture_output=True, text=True, cwd=tree)
                if p.returncode != 0:
                    raise RuntimeError(f"{label} worker failed:\n{p.stdout}\n{p.stderr}")
                for arm, ms in json.loads(p.stdout.strip().splitlines()[-1]).items():
                    rounds.setdefault(f"{label}_{arm}", []).append(float(np.median(ms)))
            print(f"round {r}: " + ", ".join(f"{k} {v[-1]:.3f} ms" for k, v in rounds.items()), flush=True)
        result["collect"] = {"envs": a.envs, "steps": a.steps, "collects_per_round": a.collects,
                             **{k: {"median_ms": float(np.median(v)), "round_medians_ms": v, "spread_ms": float(max(v) - min(v))} for k, v in rounds.items()}}
    if not a.skip_refresh:
        result["refresh_preset"] = refresh_cost(2048, 96, 5)
        result["refresh_1m"] = refresh_cost(1_000_000, 1_000_000, 3)
    result["gpu"] = gpu_identity()
    line = json.dumps(result)
    print(line)
    if a.out is not None:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
