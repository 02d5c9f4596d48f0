"""Full-workspace coverage evaluation and adaptive bucket priorities at scale.

Mirrors ``kinematic_phase1/eval/eval_full_workspace_coverage.py:75-308`` (``_summarize``, ``_bucket_metrics``,
``evaluate_full_workspace_coverage``), the bucket ids of ``workspace/workspace_target_map.py:51-121`` and
``workspace/adaptive_frontier_sampler.py`` (``classify_bucket``, ``priority_for_category``, ``update_bucket_priorities``).  The
reference walks Python dict rows one episode at a time; here the episodes of all three splits run in fused rollout launches and the
per-bucket / per-source / per-reason statistics are device segment reductions (``torch.bincount``), so a 10^6-pair sweep costs
milliseconds and can feed the adaptive frontier curriculum every few updates.
"""

from __future__ import annotations

import hashlib
import time
from dataclasses import asdict, dataclass
from typing import Any, Sequence

import numpy as np
import torch

from . import workspace as ws
from .config import Phase1EnvConfig
from .kinematics import fk_pose6_folded
from .policy import PolicyWeights
from .rollout import FAILURE_REASONS, VARIANT_FFMA, ApproachFinisherRollout, RolloutResult, failure_reason_codes


# ------------------------------------------------------------------------------------------------
# buckets (workspace_target_map.py:51-121)
# ------------------------------------------------------------------------------------------------
@dataclass
class TargetBuckets:
    code: np.ndarray          # [T] dense bucket index (order of first appearance)
    ids: list[str]            # bucket_id string of every dense index: "x{}_y{}_z{}_o{}_q{}"
    pose6: np.ndarray         # [T,6] FK(q_target), fp64
    lo: np.ndarray | None = None    # [3] the xyz box the bins span
    hi: np.ndarray | None = None

    @property
    def count(self) -> int:
        return len(self.ids)


def target_buckets(targets: ws.TargetMap, *, xyz_bins: int = 8, ori_bins: int = 6, q_l2_bins: int = 6,
                   bounds: tuple[np.ndarray, np.ndarray] | None = None) -> TargetBuckets:
    """Bucket id of every target: xyz bins span the map's own bounding box (+-1e-6), orientation = |rpy| / pi, joint = |q| / 4.5.
    ``bounds=(lo, hi)`` spans the xyz bins over that box instead (targets outside it fall into the edge bins), so another map -- a
    training map -- gets the bucket ids of the map the box came from (``TargetBuckets.lo`` / ``hi`` of an eval map)."""
    pose = np.array([fk_pose6_folded(q) for q in targets.q]).reshape(-1, 6)
    if bounds is None:
        lo, hi = pose[:, :3].min(axis=0) - 1e-6, pose[:, :3].max(axis=0) + 1e-6
    else:
        lo, hi = np.asarray(bounds[0], dtype=np.float64).reshape(3), np.asarray(bounds[1], dtype=np.float64).reshape(3)
    xyz = np.clip(np.floor((pose[:, :3] - lo) / np.maximum(hi - lo, 1e-9) * xyz_bins), 0, xyz_bins - 1).astype(int)
    ori = np.clip(np.floor(np.linalg.norm(pose[:, 3:], axis=1) / np.pi * ori_bins), 0, ori_bins - 1).astype(int)
    qb = np.clip(np.floor(np.linalg.norm(targets.q, axis=1) / 4.5 * q_l2_bins), 0, q_l2_bins - 1).astype(int)
    ids_per_target = [f"x{a}_y{b}_z{c}_o{o}_q{q}" for (a, b, c), o, q in zip(xyz, ori, qb)]
    index: dict[str, int] = {}
    code = np.array([index.setdefault(s, len(index)) for s in ids_per_target], dtype=np.int64)
    return TargetBuckets(code=code, ids=list(index), pose6=pose, lo=lo, hi=hi)


# ------------------------------------------------------------------------------------------------
# adaptive priorities (adaptive_frontier_sampler.py)
# ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class BucketPriority:
    bucket_id: str
    success_rate: float
    mean_min_error: float
    mean_final_error: float
    previous_success_rate: float | None
    failure_count: int
    category: str
    sampling_priority: float


_PRIORITY = {"mastered": 0.15, "frontier": 1.00, "hard_but_promising": 0.95, "forgetting_risk": 1.10, "stress": 0.25, "too_hard": 0.05}


def classify_bucket(*, success_rate: float, mean_min_error: float, mean_final_error: float, previous_success_rate: float | None = None) -> str:
    if previous_success_rate is not None and previous_success_rate >= 0.75 and success_rate < previous_success_rate - 0.20:
        return "forgetting_risk"
    if success_rate >= 0.85:
        return "mastered"
    if 0.35 <= success_rate < 0.85:
        return "frontier"
    if success_rate < 0.20 and mean_min_error > 0.025:
        return "too_hard"
    if mean_min_error <= 0.012 and mean_final_error > mean_min_error + 0.006:
        return "hard_but_promising"
    return "stress"


def priority_for_category(category: str) -> float:
    return _PRIORITY.get(category, 0.20)


def update_bucket_priorities(bucket_metrics: dict[str, dict[str, Any]]) -> list[BucketPriority]:
    out = []
    for bucket_id, m in bucket_metrics.items():
        sr = float(m.get("success_rate", 0.0))
        mn = float(m.get("mean_min_position_error", m.get("mean_min_error", 999.0)))
        fin = float(m.get("mean_final_position_error", m.get("mean_final_error", 999.0)))
        prev = m.get("previous_success_rate")
        prev = float(prev) if prev is not None else None
        cat = classify_bucket(success_rate=sr, mean_min_error=mn, mean_final_error=fin, previous_success_rate=prev)
        fails = int(m.get("failure_count", 0))
        out.append(BucketPriority(bucket_id, sr, mn, fin, prev, fails, cat, float(priority_for_category(cat) * (1.0 + min(fails, 20) / 40.0))))
    return sorted(out, key=lambda p: p.sampling_priority, reverse=True)      # stable, like the reference's sorted()


# ------------------------------------------------------------------------------------------------
# device reductions
# ------------------------------------------------------------------------------------------------
def _seg_mean(idx: torch.Tensor, values: torch.Tensor, n: int) -> tuple[np.ndarray, np.ndarray]:
    count = torch.bincount(idx, minlength=n)
    total = torch.bincount(idx, weights=values.double(), minlength=n)
    return (total / count.clamp_min(1).double()).cpu().numpy(), count.cpu().numpy()


def bucket_metrics(result: RolloutResult, bucket_code: torch.Tensor, buckets: TargetBuckets,
                   previous: dict[str, dict[str, Any]] | None = None) -> dict[str, dict[str, Any]]:
    """``_bucket_metrics`` (:110-124) for every bucket that received an episode; ``previous`` (an earlier call's output) fills
    ``previous_success_rate`` so :func:`update_bucket_priorities` can flag forgetting."""
    idx, nb = bucket_code.long(), buckets.count
    sr, count = _seg_mean(idx, result.success, nb)
    fin, _ = _seg_mean(idx, result.final_position_error, nb)
    mn, _ = _seg_mean(idx, result.min_position_error, nb)
    fails = torch.bincount(idx, weights=(~result.success).double(), minlength=nb).cpu().numpy()
    out: dict[str, dict[str, Any]] = {}
    for b in np.nonzero(count)[0]:
        bid = buckets.ids[b]
        out[bid] = {"episode_count": int(count[b]), "success_rate": float(sr[b]), "failure_count": int(round(fails[b])),
                    "mean_final_position_error": float(fin[b]), "mean_min_position_error": float(mn[b])}
        if previous is not None and bid in previous:
            out[bid]["previous_success_rate"] = float(previous[bid]["success_rate"])
    return out


def summarize_split(result: RolloutResult, approach_config: Phase1EnvConfig, *, start_source: torch.Tensor, joint_distance_l2: torch.Tensor,
                    ee_position_distance: torch.Tensor, handoff_confirm_steps: int = 2) -> dict[str, Any]:
    """``_summarize`` (:75-107): rates, mean errors, pair distances, failure reasons, success by start source."""
    f = lambda t: float(t.double().mean().item()) if t.numel() else 0.0  # noqa: E731
    reason = failure_reason_codes(result, approach_config, handoff_confirm_steps)
    counts = torch.bincount(reason, minlength=len(FAILURE_REASONS)).cpu().numpy()
    ok = result.success
    by_src, n_src = _seg_mean(start_source.long(), ok, len(ws.START_SOURCES))
    okd = joint_distance_l2[ok]
    return {
        "episode_count": result.n, "success_rate": f(ok), "ready_rate": f(result.ready_hit), "dwell_success_rate": f(result.ready_dwell),
        "mean_final_position_error": f(result.final_position_error), "mean_final_orientation_error": f(result.final_orientation_error),
        "mean_final_action_magnitude": f(result.final_action_magnitude), "mean_final_dq_norm": f(result.final_dq_norm),
        "average_start_target_joint_distance": f(joint_distance_l2), "average_start_target_ee_distance": f(ee_position_distance),
        "max_successful_joint_l2": float(okd.max().item()) if okd.numel() else 0.0,
        "failure_reason_counts": {FAILURE_REASONS[i]: int(c) for i, c in enumerate(counts) if c},
        "success_by_start_source": {ws.START_SOURCES[s]: {"episode_count": int(n_src[s]), "success_rate": float(by_src[s])}
                                    for s in range(len(ws.START_SOURCES)) if n_src[s]},
    }


def evaluate_full_workspace_coverage(approach_config: Phase1EnvConfig, approach_policy: PolicyWeights, finisher_config: Phase1EnvConfig | None = None,
                                     finisher_policy: PolicyWeights | None = None, *, seed: int = 940001, episodes_per_split: int = 96,
                                     stage_samples_per_stage: int = 96, random_target_samples: int = 384, random_start_samples: int = 384,
                                     pair_count: int = 2048, handoff_confirm_steps: int = 2, variant: int = VARIANT_FFMA,
                                     previous_bucket_metrics: dict[str, dict[str, Any]] | None = None,
                                     device: str | torch.device = "cuda") -> dict[str, Any]:
    """``evaluate_full_workspace_coverage`` (:193-291) without the file writing: maps -> pairs -> the three splits (seed schedule
    seed+1/+2/+3 and the split-selection stream of ``seed``) -> one fused rollout per split -> split summaries, bucket metrics,
    covered / stable / partial / stress bucket fractions and the top sampling priorities."""
    rng = np.random.default_rng(seed)
    targets = ws.generate_workspace_target_map(approach_config, seed=seed + 1, stage_samples_per_stage=stage_samples_per_stage, random_samples=random_target_samples)
    starts = ws.generate_workspace_start_state_map(approach_config, seed=seed + 2, stage_samples_per_stage=max(stage_samples_per_stage // 2, 1),
                                                   random_samples=random_start_samples)
    pairs = ws.build_pair_table(starts, targets, seed=seed + 3, pair_count=pair_count)
    buckets = target_buckets(targets)
    start_pos = np.array([fk_pose6_folded(q)[:3] for q in starts.q]).reshape(-1, 3)
    ro = ApproachFinisherRollout(approach_config, approach_policy, finisher_config, finisher_policy, device=device,
                                 handoff_confirm_steps=handoff_confirm_steps, variant=variant)
    dev = torch.device(device)
    names = {"known": "random_start_known_workspace", "frontier": "random_start_frontier", "stress": "full_reachable_stress"}
    out: dict[str, Any] = {}
    results, codes = [], []
    env_steps = 0
    for split in ("known", "frontier", "stress"):
        sel = ws.select_pairs(pairs, targets, mode=split, limit=episodes_per_split, rng=rng)
        res = ro.evaluate_suite(ws.pairs_to_suite(starts, targets, pairs, sel))
        si, ti = pairs.start[sel], pairs.target[sel]
        ee_dist = np.linalg.norm(buckets.pose6[ti, :3] - start_pos[si], axis=1)
        out[names[split]] = summarize_split(res, approach_config, start_source=torch.as_tensor(starts.source[si], device=dev),
                                            joint_distance_l2=torch.as_tensor(pairs.q_l2[sel], device=dev),
                                            ee_position_distance=torch.as_tensor(ee_dist, device=dev), handoff_confirm_steps=handoff_confirm_steps)
        results.append(res)
        codes.append(torch.as_tensor(buckets.code[ti], device=dev))
        env_steps += int(res.env_steps.item())
    n_all = sum(r.n for r in results)
    merged = RolloutResult(raw=torch.cat([r.raw[:, : r.n] for r in results], dim=1).contiguous(), n=n_all,
                           env_steps=torch.tensor([env_steps], dtype=torch.int64, device=dev))
    metrics = bucket_metrics(merged, torch.cat(codes), buckets, previous_bucket_metrics)
    priorities = update_bucket_priorities(metrics)
    stable = sum(1 for m in metrics.values() if m["success_rate"] >= 0.85)
    partial = sum(1 for m in metrics.values() if 0.35 <= m["success_rate"] < 0.85)
    stress = sum(1 for m in metrics.values() if m["success_rate"] < 0.35)
    nb = max(len(metrics), 1)
    out.update({
        "target_map_summary": {"seed": seed + 1, "total_target_count": int(targets.q.shape[0]), "bucket_count": buckets.count},
        "start_state_map_summary": {"seed": seed + 2, "total_start_count": int(starts.q.shape[0])},
        "pair_sampler_summary": {"seed": seed + 3, "pair_count": int(pairs.start.shape[0]),
                                 "difficulty_class_counts": {ws.DIFFICULTY_CLASSES[k]: int(c) for k, c in enumerate(np.bincount(pairs.klass, minlength=5)) if c}},
        "covered_bucket_fraction": float((stable + partial) / nb), "stable_bucket_fraction": float(stable / nb),
        "partial_bucket_fraction": float(partial / nb), "stress_bucket_fraction": float(stress / nb),
        "covered_bucket_count": int(stable + partial), "total_eval_bucket_count": len(metrics),
        "top_sampling_priorities": [asdict(p) for p in priorities[:30]], "bucket_metrics": metrics, "env_steps": env_steps,
    })
    return out


# ------------------------------------------------------------------------------------------------
# adaptive frontier curriculum (this project's extension: the reference stops at the priorities above)
# ------------------------------------------------------------------------------------------------
def alias_table(weights: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Walker / Vose alias table of ``weights`` (fp64): bucket k is drawn as ``u < prob[k] ? k : alias[k]`` with k uniform."""
    w = np.asarray(weights, dtype=np.float64)
    n = w.size
    scaled = w / w.sum() * n
    prob, alias = np.ones(n, dtype=np.float64), np.arange(n, dtype=np.int64)
    small = [i for i in range(n) if scaled[i] < 1.0]
    large = [i for i in range(n) if scaled[i] >= 1.0]
    while small and large:
        s, g = small.pop(), large.pop()
        prob[s], alias[s] = scaled[s], g
        scaled[g] = (scaled[g] + scaled[s]) - 1.0
        (small if scaled[g] < 1.0 else large).append(g)
    return prob, alias          # what is left in either list keeps probability 1 (rounding residue of weights that sum to n)


def alias_probabilities(prob: np.ndarray, alias: np.ndarray) -> np.ndarray:
    """Per-bucket probability an alias table encodes: (prob[k] + sum over j with alias[j] = k of (1 - prob[j])) / n, in fp64."""
    p = np.asarray(prob, dtype=np.float64)
    return (p + np.bincount(np.asarray(alias), weights=1.0 - p, minlength=p.size)) / p.size


@dataclass
class FrontierTable:
    """Device image of the adaptive frontier targets (``KinSamplerParams.frontier_*``): training-map targets grouped by bucket (CSR),
    and an alias table over the buckets weighted by their coverage-eval ``sampling_priority``."""
    bucket_ids: list[str]          # [B] bucket of each table slot
    weights: np.ndarray            # [B] fp64 sampling weight (priority, or the default for buckets the eval did not see)
    probabilities: np.ndarray      # [B] fp64 bucket probabilities the fp32 alias table encodes
    target_index: np.ndarray       # [T] training-map row of each table row
    offsets: torch.Tensor          # [B + 1] int32
    alias_prob: torch.Tensor       # [B] float32
    alias_index: torch.Tensor      # [B] int32
    targets: torch.Tensor          # [T, KIN_FRONTIER_TARGET_FLOATS] float32: goal_q 7 | stage (-1: uniform-valid)
    dropped_bucket_count: int      # buckets with a priority but no training target
    defaulted_bucket_count: int    # buckets with training targets but no priority
    checksum: str

    @property
    def bucket_count(self) -> int:
        return len(self.bucket_ids)

    @property
    def target_count(self) -> int:
        return int(self.target_index.size)

    @classmethod
    def build(cls, train_targets: ws.TargetMap, train_buckets: TargetBuckets, priorities: Sequence[BucketPriority] | dict[str, float], *,
              default_priority: float = priority_for_category("unknown"), device: str | torch.device = "cuda") -> "FrontierTable":
        prio = {p.bucket_id: float(p.sampling_priority) for p in priorities} if not isinstance(priorities, dict) else {k: float(v) for k, v in priorities.items()}
        if not all(np.isfinite(v) for v in prio.values()) or not np.isfinite(default_priority):
            raise ValueError("FrontierTable: non-finite sampling priority")
        n_t = int(train_targets.q.shape[0])
        code = np.asarray(train_buckets.code, dtype=np.int64)
        if n_t == 0 or code.size != n_t:
            raise ValueError("FrontierTable: the training map is empty or does not match its buckets")
        counts = np.bincount(code, minlength=train_buckets.count)
        keep = np.nonzero(counts)[0]                         # buckets without a training target cannot be drawn: dropped
        ids = [train_buckets.ids[b] for b in keep]
        weights = np.array([prio.get(b, float(default_priority)) for b in ids], dtype=np.float64)
        if not (np.isfinite(weights).all() and (weights >= 0.0).all() and weights.sum() > 0.0):
            raise ValueError("FrontierTable: bucket weights must be finite, >= 0 and not all zero")
        slot = np.full(train_buckets.count, -1, dtype=np.int64)
        slot[keep] = np.arange(keep.size)
        order = np.argsort(slot[code], kind="stable")        # targets grouped by table slot, map order inside a slot
        offsets = np.concatenate([[0], np.cumsum(counts[keep])]).astype(np.int32)
        prob, alias = alias_table(weights)
        prob32, alias32 = prob.astype(np.float32), alias.astype(np.int32)
        rows = np.zeros((n_t, 8), dtype=np.float32)
        rows[:, :7] = train_targets.q[order]
        rows[:, 7] = train_targets.stage[order]
        if not (np.all(np.diff(offsets) > 0) and offsets[-1] == n_t and np.all((alias32 >= 0) & (alias32 < keep.size))
                and np.all((prob32 >= 0.0) & (prob32 <= 1.0)) and np.isfinite(rows).all()):
            raise AssertionError("FrontierTable: inconsistent table")      # a defect of the builder, not of its input
        h = hashlib.sha256()
        for a in (offsets, prob32, alias32, rows):
            h.update(np.ascontiguousarray(a).tobytes())
        dev = torch.device(device)
        return cls(bucket_ids=ids, weights=weights, probabilities=alias_probabilities(prob32, alias32), target_index=order,
                   offsets=torch.as_tensor(offsets, device=dev), alias_prob=torch.as_tensor(prob32, device=dev),
                   alias_index=torch.as_tensor(alias32, device=dev), targets=torch.as_tensor(rows, device=dev).contiguous(),
                   dropped_bucket_count=len(set(prio) - set(ids)), defaulted_bucket_count=sum(1 for b in ids if b not in prio),
                   checksum=h.hexdigest()[:16])


class FrontierCurriculum:
    """Adaptive frontier curriculum for random-start training, modelled on ``gate.EvalGate``: every ``refresh_interval`` timesteps run
    the full-workspace coverage eval (with the previous eval's bucket metrics, so ``forgetting_risk`` can fire), turn its bucket
    priorities into a ``FrontierTable`` over a TRAINING target map and arm it on the env: with ``probability`` a random-start reset
    takes its goal from the table.  The training map has its own seed and is larger than the eval map, so training never draws the
    exact eval targets; it is bucketed on the eval map's bin edges so the eval's bucket ids apply to it."""

    def __init__(self, approach_config: Phase1EnvConfig, finisher_config: Phase1EnvConfig | None = None, finisher_policy: PolicyWeights | None = None, *,
                 refresh_interval: int, probability: float = 0.5, seed: int = 940001, episodes_per_split: int = 96, stage_samples_per_stage: int = 96,
                 random_target_samples: int = 384, random_start_samples: int = 384, pair_count: int = 2048, train_seed: int | None = None,
                 train_stage_samples_per_stage: int | None = None, train_random_samples: int | None = None,
                 default_priority: float = priority_for_category("unknown"), variant: int = VARIANT_FFMA, handoff_confirm_steps: int = 2) -> None:
        if not 0.0 <= float(probability) <= 1.0:
            raise ValueError("probability must be in [0, 1]")
        self.acfg, self.fcfg, self.fpol = approach_config, finisher_config, finisher_policy
        self.refresh_interval, self.probability = max(int(refresh_interval), 1), float(probability)
        self.eval_kwargs = dict(seed=int(seed), episodes_per_split=int(episodes_per_split), stage_samples_per_stage=int(stage_samples_per_stage),
                                random_target_samples=int(random_target_samples), random_start_samples=int(random_start_samples),
                                pair_count=int(pair_count), handoff_confirm_steps=int(handoff_confirm_steps), variant=int(variant))
        self.train_seed = int(seed) + 104729 if train_seed is None else int(train_seed)
        if self.train_seed == int(seed) + 1:
            raise ValueError("the training target map must not be the eval target map (seed + 1)")
        eval_map = ws.generate_workspace_target_map(approach_config, seed=int(seed) + 1, stage_samples_per_stage=int(stage_samples_per_stage),
                                                    random_samples=int(random_target_samples))
        eval_buckets = target_buckets(eval_map)
        self.train_targets = ws.generate_workspace_target_map(
            approach_config, seed=self.train_seed,
            stage_samples_per_stage=2 * int(stage_samples_per_stage) if train_stage_samples_per_stage is None else int(train_stage_samples_per_stage),
            random_samples=2 * int(random_target_samples) if train_random_samples is None else int(train_random_samples))
        self.train_buckets = target_buckets(self.train_targets, bounds=(eval_buckets.lo, eval_buckets.hi))
        self.default_priority = float(default_priority)
        self.next_refresh = self.refresh_interval
        self.previous_metrics: dict[str, dict[str, Any]] | None = None
        self.table: FrontierTable | None = None
        self.last_summary: dict[str, Any] | None = None
        self.history: list[dict[str, Any]] = []

    @classmethod
    def from_config(cls, preset: dict[str, Any], approach_config: Phase1EnvConfig | None = None, finisher_config: Phase1EnvConfig | None = None,
                    finisher_policy: PolicyWeights | None = None, **overrides: Any) -> "FrontierCurriculum":
        """Eval sizes from the preset's ``full_workspace_randomstart`` section, the refresh interval from ``workspace_expansion.eval_interval``
        (``presets/randomstart_overnight.json``); keyword arguments override them."""
        from .config import to_env_config

        fw, we = dict(preset.get("full_workspace_randomstart", {})), dict(preset.get("workspace_expansion", {}))
        kw: dict[str, Any] = dict(seed=int(fw.get("seed", 940001)), pair_count=int(fw.get("pair_count", 2048)),
                                  episodes_per_split=int(fw.get("eval_episodes_per_split", 96)),
                                  stage_samples_per_stage=int(fw.get("target_stage_samples_per_stage", 96)),
                                  random_target_samples=int(fw.get("target_random_samples", 384)),
                                  random_start_samples=int(fw.get("start_random_samples", 384)),
                                  refresh_interval=int(we.get("eval_interval", 200000)))
        kw.update(overrides)
        return cls(approach_config or to_env_config(preset), finisher_config, finisher_policy, **kw)

    def maybe_refresh(self, num_timesteps: int, policy: PolicyWeights, env: Any, *, force: bool = False) -> dict[str, Any] | None:
        """Evaluate ``policy`` and re-arm ``env`` (``BatchedArmKinematicEnv.set_frontier_targets``) when the interval has passed (or
        ``force``).  Returns the refresh record, or None when nothing ran."""
        if num_timesteps < self.next_refresh and not force:
            return None
        while self.next_refresh <= num_timesteps:
            self.next_refresh += self.refresh_interval
        t0 = time.perf_counter()
        summary = evaluate_full_workspace_coverage(self.acfg, policy, self.fcfg, self.fpol, previous_bucket_metrics=self.previous_metrics,
                                                   device=env.device, **self.eval_kwargs)
        metrics = summary["bucket_metrics"]
        priorities = update_bucket_priorities(metrics)
        table = FrontierTable.build(self.train_targets, self.train_buckets, priorities, default_priority=self.default_priority, device=env.device)
        env.set_frontier_targets(table, self.probability)
        self.previous_metrics, self.table, self.last_summary = metrics, table, summary
        rec: dict[str, Any] = {
            "timesteps": int(num_timesteps),
            "known_success_rate": float(summary["random_start_known_workspace"]["success_rate"]),
            "frontier_success_rate": float(summary["random_start_frontier"]["success_rate"]),
            "stress_success_rate": float(summary["full_reachable_stress"]["success_rate"]),
            **{k: float(summary[k]) for k in ("covered_bucket_fraction", "stable_bucket_fraction", "partial_bucket_fraction", "stress_bucket_fraction")},
            "eval_bucket_count": len(metrics), "previous_rate_bucket_count": sum(1 for m in metrics.values() if "previous_success_rate" in m),
            "table_bucket_count": table.bucket_count, "dropped_bucket_count": table.dropped_bucket_count,
            "defaulted_bucket_count": table.defaulted_bucket_count, "refresh_seconds": time.perf_counter() - t0,
            "top_priorities": [(p.bucket_id, p.category, p.sampling_priority) for p in priorities[:5]], "table_checksum": table.checksum,
        }
        self.history.append(rec)
        return rec


__all__ = ["BucketPriority", "FrontierCurriculum", "FrontierTable", "TargetBuckets", "alias_probabilities", "alias_table", "bucket_metrics",
           "classify_bucket", "evaluate_full_workspace_coverage", "priority_for_category", "summarize_split", "target_buckets", "update_bucket_priorities"]
