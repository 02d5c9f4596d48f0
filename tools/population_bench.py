"""Population vs standalone PPO training at the reference's own small-batch shape.

  python tools/population_bench.py [--members 1 8 32] [--iters 5]

Every member: 128 envs x 256 steps (the 32 768 samples of 16 x 2048), batch_size 512, 8 epochs, approach_dynamic_scale_big's
learning rate / clip / entropy / gamma / lambda, Stage 10.  For each K it times, per iteration (collect + update):
  (a) a PPOPopulation of K members, (b) one standalone PPOTrainer with a member's arguments, (c) K members one after another = K x (b).
Device work is timed with CUDA events and a synchronise; one warm-up iteration of each is excluded; population and standalone
iterations alternate in the same process and the median over --iters is reported.  Prints one JSON line.
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch

from rl_brain_trainer_b200 import config as kcfg, ppo
from rl_brain_trainer_b200.population import PPOPopulation

ap = argparse.ArgumentParser()
ap.add_argument("--members", type=int, nargs="+", default=[1, 8, 32])
ap.add_argument("--iters", type=int, default=5)
ap.add_argument("--envs", type=int, default=128)
ap.add_argument("--n-steps", type=int, default=256)
ap.add_argument("--stage", type=int, default=10)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("population_bench needs a CUDA device")
dev = torch.device("cuda", 0)


def device_info() -> dict:
    info = {"device": torch.cuda.get_device_name(dev)}
    try:      # read-only query
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        _, power, clock = [s.strip() for s in out.split(",")]
        info.update(power_limit=power, max_sm_clock=clock)
    except Exception as exc:  # noqa: BLE001
        info.update(power_limit=f"unknown ({exc})", max_sm_clock="unknown")
    return info


cfg = kcfg.load_preset("approach_dynamic_scale_big")
ref = kcfg.preset_dict("approach_dynamic_scale_big")["algorithms"]["ppo"]
hp = dict(learning_rate=ref["learning_rate"], n_steps=a.n_steps, batch_size=ref["batch_size"], n_epochs=ref["n_epochs"], gamma=ref["gamma"],
          gae_lambda=ref["gae_lambda"], clip_range=ref["clip_range"], ent_coef=ref["ent_coef"])


def trainer(seed: int) -> ppo.PPOTrainer:
    return ppo.PPOTrainer(cfg, ppo.random_policy(56, seed=seed, log_std_init=-1.0, device=dev), num_envs=a.envs, hyper=ppo.PPOHyper(**hp), device=dev,
                          seed=seed, stage_index=a.stage)


def timed(collect, update) -> tuple[float, float]:
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize(dev)
    e[0].record()
    collect()
    e[1].record()
    update()
    e[2].record()
    torch.cuda.synchronize(dev)
    return e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])


S = a.envs * a.n_steps
result = {"bench": "population", **device_info(), "envs_per_member": a.envs, "n_steps": a.n_steps, "batch_size": hp["batch_size"],
          "n_epochs": hp["n_epochs"], "stage": a.stage, "iters": a.iters, "results": []}
for K in a.members:
    pop = PPOPopulation([trainer(1000 + k) for k in range(K)])
    alone = trainer(1000)
    timed(pop.collect, pop.update)          # warm-up
    timed(alone.collect, alone.update)
    tp, ts = [], []
    for _ in range(a.iters):
        tp.append(timed(pop.collect, pop.update))
        ts.append(timed(alone.collect, alone.update))
    med = lambda xs, i: statistics.median(x[i] for x in xs)  # noqa: E731
    pc, pu, sc, su = med(tp, 0), med(tp, 1), med(ts, 0), med(ts, 1)
    ptot, stot = statistics.median(x[0] + x[1] for x in tp), statistics.median(x[0] + x[1] for x in ts)
    result["results"].append({
        "members": K,
        "population_ms": {"collect": round(pc, 3), "update": round(pu, 3), "total": round(ptot, 3)},
        "standalone_ms": {"collect": round(sc, 3), "update": round(su, 3), "total": round(stot, 3),
                          "total_min": round(min(x[0] + x[1] for x in ts), 3), "total_max": round(max(x[0] + x[1] for x in ts), 3)},
        "sequential_ms": {"collect": round(K * sc, 3), "update": round(K * su, 3), "total": round(K * stot, 3)},
        "env_steps_per_s": {"population": round(K * S / (ptot * 1e-3)), "standalone": round(S / (stot * 1e-3)),
                            "sequential": round(K * S / (K * stot * 1e-3))},
        "sequential_over_population": round(K * stot / ptot, 3),
    })
    del pop, alone
    torch.cuda.empty_cache()
print(json.dumps(result))
