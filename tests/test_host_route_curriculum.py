"""CPU tests: host port of the route reset sampler vs draws of the live reference; prefix-curriculum promotion logic."""

from __future__ import annotations

import json

import numpy as np
import pytest

from rl_brain_trainer_b200 import config as kcfg
from rl_brain_trainer_b200.route import ROUTE_RESET_MODES, RouteCurriculumStage, RouteDataset, RoutePrefixCurriculum, sample_route_reset

from ._util import env_config, golden


def test_route_reset_sampler_matches_reference_stream():
    g = golden("route_reset.npz")
    route = RouteDataset.from_q(g["route_q"])
    specs = env_config("approach_default").joint_specs
    for name in ("mixed", "recovery", "prefix_nonoise"):
        cfg = kcfg.RouteResetSamplerConfig(**json.loads(str(g[f"{name}_config"])))
        rng = np.random.default_rng(123)
        for i in range(200):
            s = sample_route_reset(rng, route, specs, cfg)
            assert s["route_index"] == g[f"{name}_route_index"][i] and s["start_route_index"] == g[f"{name}_start_route_index"][i], (name, i)
            assert ROUTE_RESET_MODES.index(s["reset_mode"]) == g[f"{name}_mode"][i]
            for k in ("initial_q", "initial_dq", "initial_prev_action", "goal_q"):
                assert np.array_equal(s[k], g[f"{name}_{k}"][i]), (name, i, k)
    assert len(set(g["mixed_mode"].tolist())) == 5            # every branch was exercised


def _curriculum(**kw):
    stages = [RouteCurriculumStage("p20", 20), RouteCurriculumStage("p60", 60), RouteCurriculumStage("p120", 120)]
    args = dict(promotion_success_rate=0.8, promotion_route_ready_hit_rate=0.7, promotion_orientation_hit_rate=0.6, promotion_max_regression_rate=0.2,
                window_episodes=10, min_episodes_per_stage=12)
    args.update(kw)
    return RoutePrefixCurriculum(stages, **args)


def test_prefix_curriculum_promotion_rules():
    c = _curriculum()
    assert c.prefix_end_index == 20
    ok = lambda n: (np.ones(n), np.ones(n), np.ones(n), np.zeros(n))  # noqa: E731
    assert not c.record(*ok(11))                      # window full (10) but fewer than min_episodes_per_stage (12)
    assert c.record(*ok(1), total_timesteps=999)      # 12th episode promotes
    assert c.prefix_end_index == 60 and c.stage_episode_count == 0 and c.metrics()["recent_success_rate"] == 0.0
    assert c.history[0]["from_prefix_end_index"] == 20 and c.history[0]["to_prefix_end_index"] == 60 and c.history[0]["total_timesteps"] == 999
    # one failing criterion blocks the promotion: regression rate above the bound
    assert not c.record(np.ones(20), np.ones(20), np.ones(20), np.r_[np.ones(3), np.zeros(17)][::-1].copy() * 0 + np.tile([1, 0, 0], 7)[:20])
    assert c.prefix_end_index == 60
    # ... until the window holds good episodes only
    assert c.record(*ok(10)) and c.prefix_end_index == 120
    # last stage: nothing to promote to
    assert not c.record(*ok(40)) and c.summary()["stage_name"] == "p120" and len(c.history) == 2
    # orientation-hit criterion
    c2 = _curriculum(min_episodes_per_stage=1)
    assert not c2.record(np.ones(10), np.ones(10), np.r_[np.ones(5), np.zeros(5)], np.zeros(10))
    with pytest.raises(ValueError):
        RoutePrefixCurriculum([], promotion_success_rate=1, promotion_route_ready_hit_rate=1, promotion_orientation_hit_rate=1,
                              promotion_max_regression_rate=0, window_episodes=1)


def test_route_eval_summaries_reproduce_the_reference_on_its_own_rows():
    """summarize_route_rows / route_chunk_metrics / route_failure_reason (eval_route_curriculum.py:127-186) fed with the per-waypoint
    rows the live reference produced (tests/golden/route_eval.json) must give the reference's own summary, chunk table and reasons."""
    import json
    from pathlib import Path

    import numpy as np

    from rl_brain_trainer_b200.route import RouteDataset, route_chunk_metrics, route_failure_reason, summarize_route_rows

    gold = Path(__file__).resolve().parent / "golden"
    ref = json.loads((gold / "route_eval.json").read_text())
    route = RouteDataset.from_q(np.load(gold / "trace_route.npz")["route_q"])
    got = summarize_route_rows(ref["rows"], route)
    for k, v in ref["summary"].items():
        if isinstance(v, float):
            assert abs(got[k] - v) < 1e-9, k
        else:
            assert got[k] == v, k
    assert route_chunk_metrics(ref["rows"]) == ref["chunk_metrics"]
    assert [None if r["success"] else route_failure_reason(r) for r in ref["rows"]] == ref["failure_reasons"]
    assert summarize_route_rows([], route) == {"target_count": 0}


def test_prefix_curriculum_matches_the_reference_callback_on_random_streams():
    """``RoutePrefixCurriculum.record`` against the reference's ``RoutePrefixCurriculumCallback._on_step`` (route/route_curriculum.py:85-111)
    on random episode streams cut into random per-step groups: same stage after every step, same promotion history (stage names, prefix
    ends, timesteps, the four windowed rates), checked against a sequential restatement of the same lines."""
    from collections import deque

    class Restated:
        def __init__(self, stages, thr, window, min_ep):
            self.stages, self.thr, self.window, self.min_ep = stages, thr, window, min_ep
            self.idx, self.count, self.history = 0, 0, []
            self.w = [deque(maxlen=window) for _ in range(4)]

        def step(self, dones, infos, t):
            for done, info in zip(dones, infos):
                if not done:
                    continue
                self.count += 1
                for d, k in zip(self.w, ("success", "route_ready", "route_orientation_hit", "route_regression")):
                    d.append(1 if info.get(k, False) else 0)
                if self.count < self.min_ep or len(self.w[0]) < self.window:
                    continue
                m = [sum(d) / len(d) for d in self.w]
                if m[0] >= self.thr[0] and m[1] >= self.thr[1] and m[2] >= self.thr[2] and m[3] <= self.thr[3] and self.idx < len(self.stages) - 1:
                    self.history.append((self.stages[self.idx].name, self.stages[self.idx + 1].name, t, *m))
                    self.idx += 1
                    self.count = 0
                    for d in self.w:
                        d.clear()

    rng = np.random.default_rng(42)
    for case in range(12):
        n_stage = int(rng.integers(1, 5))
        stages = [RouteCurriculumStage(name=f"prefix_{20 * (i + 1)}", prefix_end_index=20 * (i + 1)) for i in range(n_stage)]
        thr = (float(rng.choice([0.5, 0.7, 0.9])), float(rng.choice([0.4, 0.8])), float(rng.choice([0.3, 0.6])), float(rng.choice([0.05, 0.3])))
        window, min_ep = int(rng.integers(1, 24)), int(rng.integers(1, 40))
        mine = RoutePrefixCurriculum(stages, promotion_success_rate=thr[0], promotion_route_ready_hit_rate=thr[1], promotion_orientation_hit_rate=thr[2],
                                     promotion_max_regression_rate=thr[3], window_episodes=window, min_episodes_per_stage=min_ep)
        rest = Restated(stages, thr, window, min_ep)
        p_good = float(rng.choice([0.6, 0.85, 0.97]))
        t = 0
        for _ in range(int(rng.integers(50, 400))):
            n_env = int(rng.integers(1, 9))
            t += n_env
            dones = rng.random(n_env) < 0.4
            infos = [{"success": bool(rng.random() < p_good), "route_ready": bool(rng.random() < p_good), "route_orientation_hit": bool(rng.random() < p_good),
                      "route_regression": bool(rng.random() < 0.1)} for _ in range(n_env)]
            fin = [i for i in range(n_env) if dones[i]]
            mine.record([infos[i]["success"] for i in fin], [infos[i]["route_ready"] for i in fin], [infos[i]["route_orientation_hit"] for i in fin],
                        [infos[i]["route_regression"] for i in fin], total_timesteps=t)
            rest.step(dones, infos, t)
            assert mine.current_stage_index == rest.idx and mine.stage_episode_count == rest.count
        assert [(h["from_stage"], h["to_stage"], h["total_timesteps"], h["recent_success_rate"], h["recent_route_ready_hit_rate"],
                 h["recent_orientation_hit_rate"], h["recent_regression_rate"]) for h in mine.history] == rest.history


def test_nearest_scan_bounds_equal_their_definition():
    """``nearest_scan_bounds`` (diagonal sweep) against the definition ``lb[i, k] = min_{|j - i| >= k} |q_j - q_i|`` evaluated by brute force,
    rounded down to fp32 -- the pruned nearest-waypoint scan of the route kernels is exact only if these are true lower bounds."""
    from rl_brain_trainer_b200.route import nearest_scan_bounds, synthetic_route

    def brute(q, k_max=64):
        q = np.asarray(q, dtype=np.float64)
        n = q.shape[0]
        k_max = int(min(k_max, max(n, 2)))
        out = np.full((n, k_max), np.inf)
        for i in range(n):
            for k in range(k_max):
                js = [j for j in range(n) if abs(j - i) >= k]
                if js:
                    out[i, k] = min(float(np.linalg.norm(q[j] - q[i])) for j in js)
        return out

    rng = np.random.default_rng(3)
    for n in (1, 2, 3, 9, 40):
        q = rng.normal(size=(n, 7))
        got, want = nearest_scan_bounds(q), brute(q)
        assert got.dtype == np.float32 and got.shape == want.shape
        assert np.all(got.astype(np.float64) <= want) and np.allclose(got, want, rtol=2e-7, atol=0.0, equal_nan=True)
    route = synthetic_route(120, seed=7)
    lb = nearest_scan_bounds(route.q_goal)
    assert lb.shape == (120, 64) and np.all(lb[:, 0] == 0.0) and np.all(lb[:, 1:] >= lb[:, :-1])      # k = 0 includes j = i; monotone in k

