"""Route env auto-reset and VecEnv timings (CUDA events; the GPU's name and power limit are read in the same run).

    python tools/route_vec_env_bench.py [--replicas 1048576] [--rounds 5] [--launches 20] [--out FILE]

A. 1 M replicas of the synthetic 483-waypoint route: ``kin_route_step`` vs ``kin_route_step_autoreset`` alternated round by round, with
   no slot finishing (no time limit within the run, no success termination) and with every slot finishing every 4 steps
   (``max_episode_steps`` 4); in the second regime also the three-launch form the fused kernel replaces (``kin_route_step``, the masked
   terminal-observation copy, ``kin_route_reset_sampled``).  Per-launch device time, median over rounds.
B. ``BatchedRouteKinematicEnv.step`` (auto-reset) per call at 65 536 and 4 096 envs, eager vs ``graph_step``: host clock over many
   calls ending in a device synchronise; next to it the device time of the step launch alone (events around back-to-back launches).
C. ``KinRouteVecEnv.step`` per call at 1 024 envs (SB3's loop: numpy actions in, numpy observations and per-env infos out).
"""

from __future__ import annotations

import argparse
import dataclasses
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from rl_brain_trainer_b200 import _lib, config as kcfg  # noqa: E402
from rl_brain_trainer_b200.route import BatchedRouteKinematicEnv, synthetic_route  # noqa: E402
from rl_brain_trainer_b200.vec_env import make_route_vec_env  # noqa: E402

D = _lib.define


def gpu_identity() -> dict:
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        out["nvidia_smi"] = f"unavailable: {exc}"
    return out


def route_config(route, max_steps: int, terminate_on_success: bool):
    renv, _ = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    base = renv.base_env_config
    base = dataclasses.replace(base, episode_length=max_steps,
                               termination_config=dataclasses.replace(base.termination_config, max_episode_steps=max_steps,
                                                                      terminate_on_success=terminate_on_success))
    return dataclasses.replace(renv, base_env_config=base)


def device_ms(fn, launches: int) -> float:
    """Mean device milliseconds per call of ``fn`` over ``launches`` back-to-back calls (events around the whole batch)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(launches):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / launches


def part_a(route, n: int, rounds: int, launches: int) -> dict:
    g = torch.Generator(device="cuda").manual_seed(2)
    actions = ((torch.rand((n, 7), device="cuda", generator=g) * 2 - 1) * 0.1).contiguous()
    out = {}
    for regime, max_steps in (("no_slot_finishes", 60000), ("every_slot_finishes_every_4_steps", 4)):
        cfg = route_config(route, max_steps, terminate_on_success=max_steps < 60000)
        plain = BatchedRouteKinematicEnv(route, cfg, n)
        fused = BatchedRouteKinematicEnv(route, cfg, n, auto_reset=True, seed=5)
        three = BatchedRouteKinematicEnv(route, cfg, n)
        for e in (plain, fused, three):
            e.set_route_window(max_route_index=120)
        fused.reset()
        plain.state.copy_(fused.state)
        three.state.copy_(fused.state)
        terminal = torch.zeros_like(three.obs)
        counter = [0]

        def three_launch():
            three.step_raw(actions)
            finished = ((three.done & (D("KIN_DONE_TERMINATED") | D("KIN_DONE_TRUNCATED"))) != 0).unsqueeze(1)
            torch.where(finished, three.obs, terminal, out=terminal)
            counter[0] += 1
            three.reset_done(seed=5, counter=counter[0])

        variants = {"kin_route_step": lambda: plain.step_raw(actions), "kin_route_step_autoreset": lambda: fused.step_raw(actions)}
        if max_steps < 60000:
            variants["three_launch_step_copy_reset"] = three_launch
        for fn in variants.values():        # warm-up: module load, smem attribute, first resets
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(rounds):
            for k, fn in variants.items():
                times[k].append(device_ms(fn, launches))
        done_frac = float(((fused.done & D("KIN_DONE_AUTORESET")) != 0).float().mean())
        out[regime] = {k: {"ms_median": float(np.median(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v))} for k, v in times.items()}
        out[regime]["autoreset_fraction_last_step"] = done_frac
        del plain, fused, three, terminal
        torch.cuda.empty_cache()
    return out


def per_call_us(fn, calls: int) -> float:
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / calls * 1e6


def part_b(route, sizes, calls: int) -> dict:
    cfg = route_config(route, 40, terminate_on_success=True)
    out = {}
    for n in sizes:
        g = torch.Generator(device="cuda").manual_seed(3)
        actions = ((torch.rand((n, 7), device="cuda", generator=g) * 2 - 1) * 0.1).contiguous()
        row = {}
        for name, graph in (("eager", False), ("graph_step", True)):
            env = BatchedRouteKinematicEnv(route, cfg, n, auto_reset=True, seed=9, graph_step=graph)
            env.set_route_window(max_route_index=120)
            env.reset()
            row[name + "_us_per_call"] = per_call_us(lambda: env.step(actions), calls)
        row["kernel_us_device"] = device_ms(lambda: env.step_raw(actions), calls) * 1e3      # the step launch alone, back to back
        out[str(n)] = row
    return out


def part_c(route, n: int, calls: int) -> dict:
    cfg = route_config(route, 40, terminate_on_success=True)
    venv = make_route_vec_env(route, cfg, n, seed=4)
    venv.env_method("set_route_window", max_route_index=120)
    venv.reset()
    rng = np.random.default_rng(0)
    acts = (rng.uniform(-1, 1, (calls + 5, n, 7)) * 0.1).astype(np.float32)
    it = iter(acts)
    return {"us_per_call": per_call_us(lambda: venv.step(next(it)), calls), "num_envs": n}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicas", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--out", type=Path, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("route_vec_env_bench needs a CUDA device")
    route = synthetic_route(483, seed=7)
    res = {"gpu": gpu_identity(), "route_waypoints": len(route)}
    res["A_step_kernels"] = {"replicas": a.replicas, "rounds": a.rounds, "launches_per_round": a.launches, **part_a(route, a.replicas, a.rounds, a.launches)}
    res["B_batched_env_step"] = part_b(route, (65536, 4096), 2000)
    res["C_vec_env_step"] = part_c(route, 1024, 300)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out is not None:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
