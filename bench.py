#!/usr/bin/env python
"""Headline benchmark: kinematic env-steps/s with the policy in the loop (BASELINE.json `metric`).

Workload (BASELINE.json configs[1]): Stage 5 Approach -> Finisher evaluation, 65,536 parallel episodes per GPU,
official approach config (128 steps) + finisher config (36 steps), bundled checkpoints, suite built like
`build_curriculum_local_eval_suite(seed=700001+5*1009, stage_index=5)`.  One "step" = one full pass of the hot path
over the suite = 65,536 episodes x 164 env-steps, each with a policy forward.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); episodes shard by index with no data-path collective
(weak scaling: 65,536 episodes per GPU), one all-reduce of the eval statistics after the timed region.
`--impl reference` times the CPU implementation of the same path (the oracle port of the reference's pure-Python
env, all host threads) on a bounded sample of the same workload.

Keys beyond the base contract: `roofline` (fused rollout kernel), `step_kernel_roofline` (the standalone fused
env-step kernel K1 measured at an HBM-resident size), `cpu_baseline`, `e2e`, `clocks`, `gpu_launches`, `parity`.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "kinematic_env_steps_per_sec_policy_in_loop"
UNIT = "env-steps/s"
EPISODES_PER_GPU = 65536
STAGE = 5
SUITE_SEED = 700001 + STAGE * 1009
# algorithmic work per env-step (DESIGN.md / SURVEY 8d)
STEP_BYTES_APPROACH = 532
# measured DRAM traffic per launch (ncu --set full captures committed under profiles/): read + write bytes
NCU_TRAFFIC_STEP_KERNEL = 369_136_896 + 690_771_968     # kin_step_kernel<approach>, 2 097 152 envs: 1 060 MB vs 1 116 MB algorithmic
NCU_TRAFFIC_ROLLOUT_TC = 4_111_360 + 0                  # kin_rollout_tc16_kernel, 65 536 episodes (profiles/r2_rollout_tc16_raw.csv): inputs only, the 6 MB of result rows stay in L2
ACTOR_FLOPS = 2 * (56 * 64 + 64 * 64 + 64 * 7)   # 16256
ENV_FLOPS = 1800
XU_OPS_PER_ENV_STEP = 160     # MUFU-class instructions per env-step of the tensor-core rollout: 128 tanh + 12 sin/cos + ~20 rcp / sqrt / conversions (SASS count)
THRESHOLD_BAND = 0.01         # parity: an episode is "within tolerance of a threshold" if scaling the decision thresholds by 1 -+ 1 % flips the ORACLE
DUMP_LIMIT_BYTES = 64_000_000


def peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        d["source"] = "measured"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int) -> None:
        self.gpu = gpu_index
        self.rows: list[list[str]] = []
        self._stop = threading.Event()
        self._t: threading.Thread | None = None

    def _run_nvml(self) -> bool:
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        except Exception:
            return False
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        while not self._stop.is_set():
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                reasons = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                flags = ["Active" if reasons & bits[k] else "Not Active" for k in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")]
                self.rows.append([str(sm), str(mx), f"{pw:.1f}", *flags])
            except Exception:
                pass
            self._stop.wait(0.02)
        return True

    def _run(self) -> None:
        if self._run_nvml():
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)

    def summary(self) -> dict:
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) >= 7 and r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def _oracle_setup():
    from oracle import kin_oracle as ko
    from rl_brain_trainer_b200 import config as kcfg

    acfg, fcfg = kcfg.load_preset("approach_dynamic_scale_big"), kcfg.load_preset("finisher_noop_ft")
    w = lambda name: dict(np.load(kcfg.PRESET_DIR / "policies" / f"{name}.npz"))  # noqa: E731
    return ko, acfg, fcfg, ko.params_from_config(acfg), ko.params_from_config(fcfg), ko.OracleMlp(w("approach_stage8_11")), ko.OracleMlp(w("finisher"))


def bench_config(episodes_per_gpu: int, world: int) -> dict:
    """The `config` object of the JSON line -- the same dict on both arms (b200 and --impl reference)."""
    return {"workload": "stage5_approach_finisher_eval_65536env", "episodes_per_gpu": episodes_per_gpu, "env_steps_per_episode": 164,
            "approach_config": "workspace_expansion_dynamic_scale_big", "finisher_config": "dock_workspace_handoff_noop_ft_12env",
            "policies": "bundled approach stage8-11 + finisher checkpoints", "parallelism": f"env-sharded x{world}",
            "l2": "256 MB flush between timed iterations"}


def dump_outputs(out_dir: Path, arrays: dict[str, np.ndarray]) -> None:
    """Per-episode results as ``out_dir/<name>.npy``: float32 stays float32, flags and counters become (exact) float64, so two builds
    can be compared output for output.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of episodes is written, the same rows
    of every array; ``episode_index.npy`` holds their indices into the suite."""
    out_dir.mkdir(parents=True, exist_ok=True)
    arrays = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    n = len(arrays["success"])
    arrays["episode_index"] = np.arange(n, dtype=np.float64)
    row_bytes = sum(a.nbytes for a in arrays.values()) // n
    keep = min(n, (DUMP_LIMIT_BYTES - 4096 * len(arrays)) // row_bytes)     # 4 KB per file covers the .npy header
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    for k, a in arrays.items():
        np.save(out_dir / f"{k}.npy", a[rows])


def cpu_config1(threads_all: int) -> dict:
    """BASELINE.json configs[0]: Stage-0 Approach env, random-init 56-64-64-7 tanh MLP in the loop, auto-reset, >= 1 000 env-steps on
    the reference CPU path -- here the C port (fp64 env + fp32 MLP) on ONE host thread, then one independent env per host core."""
    from oracle import kin_oracle as ko
    from rl_brain_trainer_b200 import config as kcfg
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    cfg = kcfg.load_preset("approach_dynamic_scale_big")
    params = ko.params_from_config(cfg)
    rng = np.random.default_rng(0)
    K = ko.OracleMlp.KEYS
    w = {K["pi_w0"]: rng.standard_normal((64, 56)) * 0.1, K["pi_b0"]: np.zeros(64), K["pi_w1"]: rng.standard_normal((64, 64)) * 0.1,
         K["pi_b1"]: np.zeros(64), K["act_w"]: rng.standard_normal((7, 64)) * 0.01, K["act_b"]: np.zeros(7)}
    mlp = ko.OracleMlp({k: v.astype(np.float32) for k, v in w.items()})
    ep_len = cfg.termination_config.max_episode_steps
    out = {}
    for label, threads, episodes in (("single_thread", 1, -(-1000 // ep_len)), ("all_cores", threads_all, threads_all * 8 * -(-1000 // ep_len))):
        suite = build_curriculum_local_eval_suite(cfg, seed=0, stage_index=0, n_episodes=episodes)
        t0 = time.perf_counter()
        _, steps = ko.eval_approach_finisher(params, None, mlp, None, initial_q=suite.initial_q, goal_q=suite.goal_q, n_threads=threads)
        dt = time.perf_counter() - t0
        out[label] = {"env_steps_per_s": steps / dt, "env_steps": steps, "seconds": dt, "threads": threads}
    out["what"] = ("Stage-0 approach env, random-init MLP policy in the loop, episodes run back to back (auto-reset), C port of the reference's "
                   "Python env; os.cpu_count() = %d" % threads_all)
    rec = ROOT / "profiles" / "r2_config1_reference_python.json"
    if rec.exists():
        out["python_reference_recorded"] = json.loads(rec.read_text())   # the reference itself, timed where /root/reference exists (build container)
    return out


def cpu_reference_steps_per_sec(n_episodes: int, threads: int, offset: int = 0):
    """Oracle port of the reference CPU path on `n_episodes` of the same suite -> (env-steps/s, env_steps, seconds, success_rate)."""
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    ko, acfg, fcfg, pa, pf, A, F = _oracle_setup()
    suite = build_curriculum_local_eval_suite(acfg, seed=SUITE_SEED + offset, stage_index=STAGE, n_episodes=n_episodes)
    t0 = time.perf_counter()
    res, steps = ko.eval_approach_finisher(pa, pf, A, F, initial_q=suite.initial_q, goal_q=suite.goal_q, n_threads=threads)
    dt = time.perf_counter() - t0
    return steps / dt, steps, dt, float(res["success"].mean())


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import kin_oracle as ko

    ko.build()
    threads = os.cpu_count() or 1
    pilot_rate, _, _, _ = cpu_reference_steps_per_sec(256, threads)
    budget_s = 90.0 / max(args.steps + args.warmup, 1)
    n_ep = int(np.clip(pilot_rate * budget_s / 164.0, 256, 8192)) // 64 * 64
    for w in range(args.warmup):
        cpu_reference_steps_per_sec(n_ep, threads, offset=w + 1)
    total_steps, total_s, succ = 0, 0.0, []
    for k in range(args.steps):
        _, steps, dt, sr = cpu_reference_steps_per_sec(n_ep, threads, offset=100 + k)
        total_steps += steps
        total_s += dt
        succ.append(sr)
    value = total_steps / total_s
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_s / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": bench_config(EPISODES_PER_GPU, max(args.gpus, 1)),
        "reference_arm": {"episodes_per_step_sampled": n_ep,
                          "note": "each step is a bounded sample of the same 65,536-episode suite; CPU port (C, fp64) of the reference's pure-Python "
                                  "env + fp32 MLP on all host threads (the Python reference itself runs ~1,000 env-steps/s per core)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} x {n_ep} episodes x 164 env-steps, {threads} host threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "success_rate": float(np.mean(succ)) if succ else None,
    }
    print(json.dumps(line))


def measure_step_kernel(torch, device, pk, n_envs: int = 1 << 21, launches: int = 20) -> dict:
    """K1 standalone at an HBM-resident size (working set >> 126 MB L2): achieved GB/s = 532 B x n_envs / event time."""
    from rl_brain_trainer_b200 import config as kcfg
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv

    acfg = kcfg.load_preset("approach_dynamic_scale_big")
    env = BatchedArmKinematicEnv(acfg, n_envs, device, with_aux=False, seed=3, host_sampler=False)
    env.set_curriculum_stage(STAGE)
    env.reset()
    g = torch.Generator(device=device)
    g.manual_seed(1)
    actions = torch.rand((n_envs, 7), device=device, generator=g) * 2 - 1
    for _ in range(3):
        env.step_raw(actions)
    torch.cuda.synchronize(device)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    for a, b in ev:
        a.record()
        env.step_raw(actions)   # exactly one kin_step_kernel launch between the events
        b.record()
    torch.cuda.synchronize(device)
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    t = float(np.mean(ms)) * 1e-3
    gbs = STEP_BYTES_APPROACH * n_envs / t / 1e9
    del env
    return {"kernel": "kin_step_kernel<approach>", "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": gbs / pk["hbm_gbs"], "traffic": NCU_TRAFFIC_STEP_KERNEL if n_envs == 2_097_152 else None,
            "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch, profiles/r1_step_v3_raw.csv (ncu --set full, same size)",
            "peak_source": pk["source"], "n_envs": n_envs, "launches": launches,
            "us_per_launch": t * 1e6, "env_steps_per_sec": n_envs / t, "bytes_per_env_step": STEP_BYTES_APPROACH,
            "note": "working set %.0f MB per launch (> L2), CUDA events on the launching stream" % (STEP_BYTES_APPROACH * n_envs / 1e6)}


def _time_launches(torch, device, fn, launches: int) -> float:
    """Mean seconds per call of `fn` (CUDA events on the launching stream, after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize(device)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize(device)
    return float(np.mean([a.elapsed_time(b) for a, b in ev])) * 1e-3


def measure_step_variants(torch, device, pk, n_envs: int = 1 << 21, launches: int = 10) -> dict:
    """The other instances of the step kernel family at an HBM-resident size, each against its own algorithmic bytes (SURVEY 8d:
    dock 548 B, approach with in-kernel auto-reset 532 B, route step 644 B), plus the documented per-step API (`env.step`, lazy
    info) at the same size and at 65 536 envs where launch overhead shows."""
    from rl_brain_trainer_b200 import config as kcfg
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv
    from rl_brain_trainer_b200.route import BatchedRouteKinematicEnv, synthetic_route

    out = {}
    g = torch.Generator(device=device)
    g.manual_seed(2)
    actions = torch.rand((n_envs, 7), device=device, generator=g) * 2 - 1

    def entry(kernel, bytes_per_step, t, n):
        gbs = bytes_per_step * n / t / 1e9
        return {"kernel": kernel, "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                "bytes_per_env_step": bytes_per_step, "n_envs": n, "us_per_launch": t * 1e6, "env_steps_per_sec": n / t, "peak_source": pk["source"]}

    acfg, fcfg = kcfg.load_preset("approach_dynamic_scale_big"), kcfg.load_preset("finisher_noop_ft")
    env = BatchedArmKinematicEnv(fcfg, n_envs, device, with_aux=False, seed=3, host_sampler=False)
    env.reset()
    out["dock"] = entry("kin_step_kernel<dock>", 548, _time_launches(torch, device, lambda: env.step_raw(actions), launches), n_envs)
    del env
    env = BatchedArmKinematicEnv(acfg, n_envs, device, with_aux=False, seed=3, host_sampler=False, auto_reset=True)
    env.set_curriculum_stage(STAGE)
    env.reset()
    out["approach_autoreset"] = entry("kin_step_kernel<approach, AUTORESET>", 532, _time_launches(torch, device, lambda: env.step_raw(actions), launches), n_envs)
    # the public per-step API on the same env: kernel + lazily decoded info (only the two done-bit tests run per call)
    t_api = _time_launches(torch, device, lambda: env.step(actions), launches)
    out["step_api"] = {"call": "BatchedArmKinematicEnv.step (auto-reset, lazy info)", "n_envs": n_envs, "us_per_call": t_api * 1e6,
                       "env_steps_per_sec": n_envs / t_api, "frac_of_hbm_peak": 532 * n_envs / t_api / 1e9 / pk["hbm_gbs"]}
    del env
    small = BatchedArmKinematicEnv(acfg, 65536, device, with_aux=False, seed=3, host_sampler=False, auto_reset=True)
    small.set_curriculum_stage(STAGE)
    small.reset()
    a_small = actions[:65536].contiguous()
    t_small = _time_launches(torch, device, lambda: small.step(a_small), 50)
    out["step_api_65536"] = {"call": "BatchedArmKinematicEnv.step (auto-reset, lazy info)", "n_envs": 65536, "us_per_call": t_small * 1e6,
                             "env_steps_per_sec": 65536 / t_small, "note": "35 MB working set: L2-resident, launch-latency bound"}
    del small
    gsmall = BatchedArmKinematicEnv(acfg, 65536, device, with_aux=False, seed=3, host_sampler=False, auto_reset=True, graph_step=True)
    gsmall.set_curriculum_stage(STAGE)
    gsmall.reset()
    for _ in range(3):
        gsmall.step(a_small)
    t_graph = _time_launches(torch, device, lambda: gsmall.step(a_small), 50)
    out["step_api_65536_graph"] = {"call": "BatchedArmKinematicEnv.step(graph_step=True): CUDA graph of the step kernel + done-bit ops", "n_envs": 65536,
                                   "us_per_call": t_graph * 1e6, "env_steps_per_sec": 65536 / t_graph}
    del gsmall
    route = synthetic_route(483, seed=7)
    renv, _ = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    n_route = n_envs // 2
    # two regimes of the route reward's nearest-waypoint term: replicas tracking the route (small actions, as under a trained policy:
    # pruned walk over a few waypoints) and replicas driven off it by uniform +-1 actions (the plain scan over all 483 waypoints)
    for key, scale in (("route_step", 0.1), ("route_step_random_actions", 1.0)):
        renv_b = BatchedRouteKinematicEnv(route, renv, n_route, device)
        renv_b.reset(seed=5)
        a_route = (actions[:n_route] * scale).contiguous()
        out[key] = entry("kin_route_step_kernel", 644, _time_launches(torch, device, lambda: renv_b.step_raw(a_route), launches), n_route)
        out[key]["action_scale"] = scale
    del renv_b
    torch.cuda.empty_cache()
    return out


def measure_training(torch, dist, device, world: int, envs: int = 65536, n_steps: int = 128, iters: int = 2, grad_exchange: str = "peer") -> dict:
    """BASELINE config 5: Stage-10 stress-shell PPO (fused collection K4 + tensor-core update K3-TC, 8 epochs x 16 minibatches,
    one gradient sum over ranks per minibatch when world > 1: NVLink peer-memory push (csrc/kin_peer.cu) or NCCL all-reduce).
    CUDA events, max over ranks; whole-job env-steps/s."""
    from rl_brain_trainer_b200 import config as kcfg, ppo

    cfg = kcfg.load_preset("approach_dynamic_scale_big")
    pol = ppo.random_policy(56, seed=0, log_std_init=-1.0, device=device)
    S = envs * n_steps
    hp = ppo.PPOHyper(learning_rate=4e-6, n_steps=n_steps, batch_size=S // 16, n_epochs=8, gamma=0.995, gae_lambda=0.95, clip_range=0.1, ent_coef=0.0003)
    tr = ppo.PPOTrainer(cfg, pol, num_envs=envs, hyper=hp, device=device, seed=1, stage_index=10,
                        process_group=dist.group.WORLD if world > 1 else None, grad_exchange=grad_exchange if world > 1 else "nccl")
    tr.collect()
    tr.update()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    t_roll = t_upd = 0.0
    for _ in range(iters):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        tr.collect()
        e1.record()
        stats = tr.update()
        e2.record()
        torch.cuda.synchronize(device)
        t_roll += e0.elapsed_time(e1) * 1e-3
        t_upd += e1.elapsed_time(e2) * 1e-3
    t = torch.tensor([t_roll, t_upd], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    steps = S * iters * world
    # multi-rank correctness in the same line: every rank must hold bitwise the same parameters after the timed updates, and the
    # peer-memory exchange must reproduce the NCCL all-reduce (small side run from identical seeds, both exchanges)
    check = {"param_checksum": float(tr.params.double().sum())}
    if world > 1:
        mine = tr.params.clone()
        allp = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allp, mine)
        check["params_bitwise_identical_across_ranks"] = all(bool(torch.equal(allp[0], q)) for q in allp)
        check["param_checksums"] = [float(q.double().sum()) for q in allp]
    fused_update = bool(tr.fused_update)
    tr.close()
    if world > 1:
        side = {}
        hp2 = ppo.PPOHyper(learning_rate=3e-4, n_steps=32, batch_size=4096 * 32 // 4, n_epochs=2, gamma=0.995, gae_lambda=0.95, clip_range=0.1, ent_coef=0.0003)
        for ex in ("nccl", "peer"):
            t2 = ppo.PPOTrainer(cfg, ppo.random_policy(56, seed=0, log_std_init=-1.0, device=device), num_envs=4096, hyper=hp2, device=device, seed=1,
                                stage_index=10, process_group=dist.group.WORLD, grad_exchange=ex)
            t2.collect()
            t2.update()
            torch.cuda.synchronize(device)
            side[ex] = t2.params.clone()
            t2.close()
        check["peer_vs_nccl_rel_diff"] = float((side["peer"] - side["nccl"]).norm() / side["nccl"].norm())
    return {"workload": "stage10_ppo_train", "exchange_check": check, "envs_per_gpu": envs, "n_steps": n_steps, "epochs": 8, "minibatches_per_epoch": 16, "iters": iters,
            "rollout_env_steps_per_s": steps / float(t[0]), "update_env_steps_per_s": steps / float(t[1]),
            "e2e_env_steps_per_s": steps / float(t[0] + t[1]), "collect": "kin_ppo_collect (fused, tcgen05 bf16)",
            "update": "kin_ppo_grad_tc_update (tcgen05 bf16; gradient + exchange + clip + Adam in one launch)" if fused_update else "kin_ppo_grad_tc (tcgen05 bf16) + kin_ppo_adam",
            "grad_exchange": (grad_exchange if world > 1 else "none"), "approx_kl": stats["approx_kl"], "value_loss": stats["value_loss"]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--episodes", type=int, default=EPISODES_PER_GPU, help="episodes per GPU (default: the BASELINE config)")
    ap.add_argument("--variant", default=os.environ.get("KIN_ROLLOUT_VARIANT", "auto"), choices=["auto", "ffma", "tc"])
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-step-kernel", action="store_true")
    ap.add_argument("--grad-exchange", default="peer", choices=["peer", "nccl"], help="training leg, N > 1: gradient sum over NVLink peer buffers or NCCL")
    ap.add_argument("--skip-train", action="store_true", help="skip the BASELINE config-5 leg (Stage-10 PPO training, extra key `train`)")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="write the per-episode results of the last timed step (all ranks' shards) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU path; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    from rl_brain_trainer_b200 import config as kcfg
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.rollout import VARIANT_FFMA, VARIANT_TC, ApproachFinisherRollout, RolloutResult
    from rl_brain_trainer_b200.samplers import EvalSuite, build_curriculum_local_eval_suite

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # stdout carries exactly ONE JSON line: native libraries that write to fd 1 (NCCL prints its version banner there when the
    # first communicator comes up) are pointed at stderr; the line itself goes to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "INFO")     # an inherited setting wins; INFO prints the rank / channel lines the driver greps
        dist.init_process_group("nccl", device_id=device)
    pk = peaks()

    acfg, fcfg = kcfg.load_preset("approach_dynamic_scale_big"), kcfg.load_preset("finisher_noop_ft")
    pol_a, pol_f = PolicyWeights.preset("approach_stage8_11", device), PolicyWeights.preset("finisher", device)
    n = int(args.episodes)
    # every rank evaluates its own shard of one long suite: episodes [rank*n, (rank+1)*n)
    full = build_curriculum_local_eval_suite(acfg, seed=SUITE_SEED, stage_index=STAGE, n_episodes=n * world)
    sl = slice(rank * n, (rank + 1) * n)
    suite = EvalSuite(initial_q=full.initial_q[sl], goal_q=full.goal_q[sl])

    variant = {"ffma": VARIANT_FFMA, "tc": VARIANT_TC}.get(args.variant)
    if variant is None:
        variant = VARIANT_TC
        try:
            probe = ApproachFinisherRollout(acfg, pol_a, fcfg, pol_f, device=device, variant=VARIANT_TC)
            probe.evaluate_suite(EvalSuite(initial_q=suite.initial_q[:128], goal_q=suite.goal_q[:128]))
            torch.cuda.synchronize(device)
        except Exception:
            variant = VARIANT_FFMA
    ro = ApproachFinisherRollout(acfg, pol_a, fcfg, pol_f, device=device, variant=variant)
    dev_in = ro.upload(suite)
    stride = (n + 31) // 32 * 32
    out = RolloutResult(raw=torch.zeros((24, stride), dtype=torch.int32, device=device), n=n, env_steps=torch.zeros(1, dtype=torch.int64, device=device))
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- device-resident leg ----------------------------------------------------------------------
    for _ in range(args.warmup):
        ro.run(dev_in, out=out)
    barrier()
    out.env_steps.zero_()
    events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    clocks = ClockSampler(local_rank)   # samples through the device leg, the e2e leg and the step-kernel measurement
    clocks.__enter__()
    barrier()
    t_wall0 = time.perf_counter()
    for a, b in events:
        flush.fill_(0.0)          # L2 flush between timed iterations (outside the event pair)
        a.record()
        ro.run(dev_in, out=out)
        b.record()
        launches += 1
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms = np.array([a.elapsed_time(b) for a, b in events])
    dev_s = float(ms.sum()) * 1e-3
    env_steps = int(out.env_steps.item())
    res = out.to_numpy()
    success = float(res["success"].mean())
    dumped = res
    if args.dump_outputs is not None and world > 1:     # the whole suite in episode order: every rank's shard
        mine = out.raw[:, :n].contiguous()
        shards = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(shards, mine)
        dumped = RolloutResult(raw=torch.cat(shards, dim=1), n=n * world, env_steps=out.env_steps).to_numpy()

    # ---- end-to-end leg: host buffers, pinned H2D + D2H inside the timed region ----------------------
    pinned = {k: torch.as_tensor(np.ascontiguousarray(getattr(suite, k), dtype=np.float32)).pin_memory() for k in ("initial_q", "goal_q")}
    host_out = torch.empty((24, stride), dtype=torch.int32).pin_memory()
    h2d = sum(v.numel() * 4 for v in pinned.values())
    d2h = host_out.numel() * 4

    # all K steps go through the public pipelined API: per step one pinned H2D copy of the suite and one D2H copy of the
    # result rows, overlapped with the neighbouring steps' kernels on separate streams
    host_ins = [{**pinned, "initial_dq": None, "initial_prev_action": None, "goal_pose6": None} for _ in range(args.steps)]
    host_outs = [host_out for _ in range(args.steps)]
    for _ in range(2):
        ro.evaluate_stream(host_ins[: args.warmup], host_outs[: args.warmup])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    counters = ro.evaluate_stream(host_ins, host_outs)
    e1.record()
    barrier()
    e2e_s = e0.elapsed_time(e1) * 1e-3
    e2e_steps = int(sum(int(c.item()) for c in counters))
    e2e_success = float((host_out[0, :n] != 0).float().mean())

    # ---- reductions over ranks (the only collective: eval statistics) --------------------------------
    stats = torch.tensor([dev_s, e2e_s], dtype=torch.float64, device=device)
    sums = torch.tensor([env_steps, e2e_steps, success * n, n], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    dev_s_max, e2e_s_max = float(stats[0]), float(stats[1])
    value = float(sums[0]) / dev_s_max
    e2e_value = float(sums[1]) / e2e_s_max
    success_all = float(sums[2] / sums[3])

    # ---- BASELINE config 5 (extra key, every rank takes part: NCCL gradient all-reduce per minibatch) ------------------
    train = None
    if not args.skip_train:
        del flush
        torch.cuda.empty_cache()
        train = measure_training(torch, dist, device, world, grad_exchange=args.grad_exchange)
        # the update kernel against the tensor peak (a long step: the sustained figure) -- its binder is the shared-memory data pipe, not the
        # tensor pipe (DESIGN.md K3-TC): 95.2 kFLOP per sample and epoch (forward, data gradients, weight gradients of both nets)
        upd_tf = 95.2e3 * 8 * train["update_env_steps_per_s"] / world / 1e12
        train["update_roofline"] = {"kernel": "kin_ppo_grad_tc_kernel (+ reduction, Adam, exchange: the whole update is timed)", "bound": "tensor",
                                    "achieved": upd_tf, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": upd_tf / pk["bf16_tflops_sustained"],
                                    "peak_kind": "sustained (bf16_tflops_sustained): 128 back-to-back launches per update", "peak_source": pk["source"],
                                    "limiter": "shared-memory data pipe (tensor-core operand fetch 29 % + epilogue LDS/STS 24 % of its peak) and the 11-phase "
                                               "per-tile dependency chain at two chains per SM; ncu: profiles/r2_ppo_tc_atmem_raw.csv"}

    # ---- the strict-fp32 variant of the same rollout, timed the same way (rank 0, a few launches): the parity path beside the headline
    strict = None
    res_strict = None
    if rank == 0 and variant == VARIANT_TC:
        ro_s = ApproachFinisherRollout(acfg, pol_a, fcfg, pol_f, device=device, variant=VARIANT_FFMA)
        out_s = RolloutResult(raw=torch.zeros((24, stride), dtype=torch.int32, device=device), n=n, env_steps=torch.zeros(1, dtype=torch.int64, device=device))
        ro_s.run(dev_in, out=out_s)
        torch.cuda.synchronize(device)
        out_s.env_steps.zero_()
        ev_s = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(3)]
        for a, b in ev_s:
            a.record()
            ro_s.run(dev_in, out=out_s)
            b.record()
        torch.cuda.synchronize(device)
        s_sec = sum(a.elapsed_time(b) for a, b in ev_s) * 1e-3
        res_strict = out_s.to_numpy()
        strict = {"kernel": "kin_rollout_ffma_kernel", "value": int(out_s.env_steps.item()) / s_sec, "unit": UNIT, "launches": 3,
                  "success_rate": float(res_strict["success"].mean())}

    step_roof = None
    cpu_base = None
    parity = None
    step_variants = None
    if rank == 0 and not args.skip_step_kernel:
        step_roof = measure_step_kernel(torch, device, pk)
        step_variants = measure_step_variants(torch, device, pk)
    clocks.__exit__(None, None, None)
    if rank == 0:
        if world == 1 and not args.skip_cpu_baseline:
            from oracle.parity import threshold_sensitive_episodes

            threads = os.cpu_count() or 1
            n_cpu = 4096
            rate, steps_cpu, dt, sr = cpu_reference_steps_per_sec(n_cpu, threads)
            cpu_base = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"first {n_cpu} episodes of the same suite x 164 env-steps ({steps_cpu} env-steps in {dt:.2f} s), "
                                  f"C port (fp64) of the reference's Python env + fp32 MLP, {threads} host threads",
                        "config1": cpu_config1(threads)}
            # parity of EVERY episode of the timed suite against the fp64 oracle; a differing success flag is "explained" only if the
            # oracle's own verdict for that episode changes when the decision thresholds are scaled by 1 -+ THRESHOLD_BAND
            ko, _, _, _, _, A, F = _oracle_setup()
            t0 = time.perf_counter()
            ref, sensitive = threshold_sensitive_episodes(acfg, fcfg, A, F, suite, THRESHOLD_BAND, n_threads=threads)
            flips = res["success"].astype(int) != ref["success"]
            parity = {"episodes_checked": n, "threshold_band": THRESHOLD_BAND, "threshold_sensitive_episodes": int(sensitive.sum()),
                      "success_flag_mismatches": int(flips.sum()), "unexplained_mismatches": int((flips & ~sensitive).sum()),
                      "gpu_success_rate": float(res["success"].mean()), "oracle_success_rate": float(ref["success"].mean()),
                      "mean_final_pos_err_gpu": float(res["final_position_error"].mean()),
                      "mean_final_pos_err_oracle": float(ref["final_position_error"].mean()), "oracle_seconds": time.perf_counter() - t0}
            if res_strict is not None:
                f_s = res_strict["success"].astype(int) != ref["success"]
                strict["flips"] = int(f_s.sum())
                strict["unexplained_flips"] = int((f_s & ~sensitive).sum())

    if rank == 0:
        steps_per_launch = env_steps / max(args.steps, 1)
        t_launch = dev_s / max(args.steps, 1)
        tc = variant == VARIANT_TC
        flops = (ACTOR_FLOPS + (0 if tc else ENV_FLOPS)) * steps_per_launch
        if tc:
            # each launch is a sub-millisecond kernel timed alone between L2 flushes: the BURST fp16/bf16 peak applies (kind::f16 runs at the bf16 rate)
            peak_tf = pk["bf16_tflops"]
            xu_ceiling = 148 * 16 * pk["sm_max_mhz"] * 1e6 / XU_OPS_PER_ENV_STEP      # 16 MUFU lanes / clk / SM
            roof = {"kernel": "kin_rollout_tc16_kernel", "bound": "tensor", "achieved": flops / t_launch / 1e12, "peak": peak_tf,
                    "unit": "TFLOP/s", "frac": flops / t_launch / 1e12 / peak_tf,
                    "traffic": NCU_TRAFFIC_ROLLOUT_TC if n == EPISODES_PER_GPU else None,
                    "traffic_source": "dram bytes per launch, profiles/r2_rollout_tc16_raw.csv (ncu --set full, 65 536 episodes)", "peak_source": pk["source"],
                    "peak_kind": "burst (bf16_tflops): the kernel is timed in isolation",
                    "note": "actor MLP 16,256 FLOP/env-step on tcgen05 kind::f16 (fp16 operands, fp32 accumulate)",
                    "limiter": {"pipe": "xu (MUFU)", "ops_per_env_step": XU_OPS_PER_ENV_STEP, "ceiling_env_steps_per_s": xu_ceiling,
                                "frac": (steps_per_launch / t_launch) / xu_ceiling,
                                "note": "128 tanh + the FK's sin/cos per env-step go through the 16-lane/clk/SM special-function pipe; with the "
                                        "issue slots (ncu: profiles/r2_rollout_tc16_raw.csv) it, not the tensor pipe, bounds this kernel"}}
        else:
            fp32_peak = 148 * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12
            roof = {"kernel": "kin_rollout_ffma_kernel", "bound": "fp32", "achieved": flops / t_launch / 1e12, "peak": fp32_peak,
                    "unit": "TFLOP/s", "frac": flops / t_launch / 1e12 / fp32_peak, "traffic": None, "peak_source": "148 SM x 128 lanes x 2 x sm_max_mhz",
                    "note": "strict-fp32 variant: 16,256 (MLP) + 1,800 (env) FP32 FLOP per env-step on the FP32 pipe"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dev_s_max / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if not tc else "f32 env + f16 MLP operands (f32 accumulate)", "data": "synthetic",
            "config": bench_config(n, world), "rollout_variant": "tc" if tc else "ffma",
            "env_steps_per_step": env_steps / max(args.steps, 1), "success_rate": success_all, "wall_s_timed_region": t_wall,
            "roofline": roof, "step_kernel_roofline": step_roof, "step_kernel_variants": step_variants, "cpu_baseline": cpu_base, "parity": parity, "strict_fp32": strict,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "success_rate": e2e_success},
            "clocks": clocks.summary(), "gpu_launches": launches, "train": train,
        }
        if args.dump_outputs is not None:
            dump_outputs(args.dump_outputs, dumped)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
