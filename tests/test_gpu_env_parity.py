"""GPU parity tests: the CUDA env (through the C ABI) against the CPU fp64 oracle on identical inputs.

Tolerances (north_star): poses within 1e-5 m / 1e-5 rad in fp32; flags and counters identical except for steps whose
fp64 error norms sit within EPS_BAND of a threshold (there the fp32 rounding may legitimately flip a predicate; the
rest of that episode's counters/flags/rewards are then excluded, the kinematic state is still compared).
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import kin_oracle as ko

from ._util import GOLD, _geodesic, _near, _thresholds, env_config, env_config_from_json, golden, oracle_params

pytestmark = pytest.mark.gpu

POS_TOL = 1e-5
ANG_TOL = 1e-5
EPS_BAND = 3e-6


class BatchOracle:
    """n oracle envs stepped in lock-step (fp64)."""

    def __init__(self, cfg, n):
        self.params = oracle_params(cfg)
        self.states = ko.state_array(n)
        self.n = n

    def reset(self, mode, iq, gq, gp=None, idq=None, ipa=None):
        L = ko.lib()
        import ctypes

        for e in range(self.n):
            L.kor_reset(ctypes.byref(self.params), ctypes.byref(self.states[e]), mode, ko._dptr(ko._f64(iq[e])),
                        None if idq is None else ko._dptr(ko._f64(idq[e])), None if ipa is None else ko._dptr(ko._f64(ipa[e])),
                        ko._dptr(ko._f64(gq[e])), None if gp is None else ko._dptr(ko._f64(gp[e])))

    def step(self, actions):
        return ko.step_batch(self.params, self.states, actions)

    def field(self, name, k=None):
        if k is None:
            return np.array([getattr(s, name) for s in self.states])
        return np.array([[getattr(s, name)[i] for i in range(k)] for s in self.states])


def _make_env(cfg, n, **kw):
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv

    return BatchedArmKinematicEnv(cfg, n, "cuda", with_aux=True, with_components=True, **kw)


def test_library_is_sm100_and_loaded():
    from rl_brain_trainer_b200 import _lib

    L = _lib.lib()
    import ctypes

    sm, major, minor = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    name = ctypes.create_string_buffer(128)
    _lib.check(L.kin_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor), name, 128))
    assert major.value == 10, f"expected a Blackwell sm_100 device, got {major.value}.{minor.value} ({name.value})"


def test_fk_matches_oracle():
    g = golden("fk.npz")
    env = _make_env(env_config("approach_dynamic_scale_big"), 1)
    pose = env.fk_pose6(torch.as_tensor(g["q"], dtype=torch.float32)).cpu().numpy().astype(float)
    ref = ko.fk_pose6(g["q"].astype(np.float32).astype(float))  # oracle on the same fp32-rounded inputs
    assert np.abs(pose[:, :3] - ref[:, :3]).max() < POS_TOL
    d = np.abs((pose[:, 3:] - ref[:, 3:] + np.pi) % (2 * np.pi) - np.pi)
    # inside the curriculum shells the Euler extraction is well conditioned
    shell = slice(2, 130)
    assert d[shell].max() < 2e-6
    assert np.median(d) < 5e-7
    # EVERY pose, the gimbal-lock neighbourhood included (SURVEY F11): the orientation itself agrees to 1e-5 rad (geodesic angle between
    # the two rotations), and each Euler component to 1e-5 rad scaled by its conditioning 1 / cos(pitch) -- a bound, not a mask
    assert _geodesic(pose[:, 3:], ref[:, 3:]).max() < ANG_TOL
    assert (d * np.maximum(np.abs(np.cos(ref[:, 4:5])), 1e-4)).max() < ANG_TOL


def _compare_rollout(cfg, mode, iq, gq, actions, gp=None, idq=None, ipa=None, names=ko.APPROACH_COMPONENT_NAMES, mode_hint_mixed=False):
    """Open-loop parity over T steps for n envs: actions [T,n,7]."""
    n = iq.shape[0]
    T = actions.shape[0]
    env = _make_env(cfg, n)
    mode_name = "approach" if mode == 0 else "dock"
    opts = {"initial_q": iq, "goal_q": gq, "policy_mode": mode_name}
    if gp is not None:
        opts["goal_pose6"] = gp
    if idq is not None:
        opts["initial_dq"] = idq
    if ipa is not None:
        opts["initial_prev_action"] = ipa
    obs, info = env.reset(options=opts)
    if mode_hint_mixed:
        env._mode_all = None  # force the per-env-mode kernel
    orc = BatchOracle(cfg, n)
    f32 = lambda a: None if a is None else np.asarray(a, dtype=np.float32).astype(float)  # noqa: E731
    orc.reset(mode, f32(iq), f32(gq), f32(gp), f32(idq), f32(ipa))
    ref_obs0 = np.stack([_obs_of(orc, e) for e in range(min(n, 64))])
    assert np.abs(obs[: ref_obs0.shape[0]].cpu().numpy() - ref_obs0).max() < 2e-5
    pos_thr, ori_thr, act_thr, dq_thr = _thresholds(cfg)
    clean = np.ones(n, dtype=bool)   # episodes with no epsilon-band event so far
    prev_pos = np.array([st.entry_position_error_norm for st in orc.states])
    prev_ori = np.array([st.entry_orientation_error_norm for st in orc.states])
    stats = {"max_pos": 0.0, "max_ang": 0.0, "max_q": 0.0, "max_reward": 0.0, "max_obs": 0.0, "banded": 0, "checked_flags": 0}
    for t in range(T):
        a = np.asarray(actions[t], dtype=np.float32)
        obs, reward, term, trunc, info = env.step(torch.as_tensor(a))
        robs, routs = orc.step(a.astype(float))
        rq, rdq = orc.field("q", 7), orc.field("dq", 7)
        ree = orc.field("ee_pose6", 6)
        q = env.q.cpu().numpy().astype(float)
        dq = env.dq.cpu().numpy().astype(float)
        ee = env.ee_pose6.cpu().numpy().astype(float)
        stats["max_q"] = max(stats["max_q"], np.abs(q - rq).max(), np.abs(dq - rdq).max())
        stats["max_pos"] = max(stats["max_pos"], np.abs(ee[:, :3] - ree[:, :3]).max())
        ang = np.abs((ee[:, 3:] - ree[:, 3:] + np.pi) % (2 * np.pi) - np.pi)
        # no pose is skipped: Euler components are bounded with their conditioning (1 / cos(pitch) near gimbal lock), and the
        # rotation itself (geodesic angle) with the plain tolerance
        stats["max_ang"] = max(stats["max_ang"], (ang * np.maximum(np.abs(np.cos(ree[:, 4:5])), 1e-4)).max(), _geodesic(ee[:, 3:], ree[:, 3:]).max())
        r_pos = np.array([o.position_error_norm for o in routs])
        r_ori = np.array([o.orientation_error_norm for o in routs])
        r_an = np.array([o.action_l2 for o in routs])
        r_dq = np.array([o.executed_delta_q_l2 for o in routs])
        # previous-step norms matter too (prev_in_* predicates): approximate by also banding on the previous values
        band = _near(r_pos, pos_thr, EPS_BAND) | _near(r_ori, ori_thr, 4 * EPS_BAND) | _near(r_an, act_thr, EPS_BAND) | _near(r_dq, dq_thr, EPS_BAND / 3)
        # predicates of the form curr < prev (drift counter, alignment / tiny-correction / no-progress terms) are
        # undecidable in fp32 when the two norms agree to ~1e-7
        band |= (np.abs(r_pos - prev_pos) < EPS_BAND / 3) | (np.abs(r_ori - prev_ori) < EPS_BAND)
        prev_pos, prev_ori = r_pos, r_ori
        clean &= ~band
        stats["banded"] = int((~clean).sum())
        gpos = info["position_error_norm"].cpu().numpy().astype(float)
        gori = info["orientation_error_norm"].cpu().numpy().astype(float)
        assert np.abs(gpos - r_pos).max() < POS_TOL
        # the orientation-error norm is what every predicate consumes: bounded for EVERY pose, with the Euler conditioning of the
        # current and the goal pose (1 / cos(pitch); 1 inside the curriculum shells) -- no pose is masked out
        cond = np.maximum(np.minimum(np.abs(np.cos(ree[:, 4])), np.abs(np.cos(orc.field("goal_pose6", 6)[:, 4]))), 1e-4)
        assert (np.abs(gori - r_ori) * cond).max() < 2 * ANG_TOL
        sel = clean
        if sel.any():
            r_flags = np.array([[o.terminated, o.truncated, o.success, o.curr_in_pre_near_goal, o.curr_in_near_goal, o.reason] for o in routs])
            g_flags = np.stack([term.cpu().numpy(), trunc.cpu().numpy(), info["success"].cpu().numpy(), info["curr_in_pre_near_goal"].cpu().numpy(),
                                info["curr_in_near_goal"].cpu().numpy(), info["reason_code"].cpu().numpy()], axis=1).astype(int)
            assert np.array_equal(g_flags[sel], r_flags[sel]), f"flags differ at step {t}"
            r_cnt = np.stack([orc.field("episode_step"), orc.field("dwell_count"), orc.field("near_goal_entry_count"),
                              orc.field("near_goal_drift_count"), orc.field("pre_near_goal_hit"), orc.field("near_goal_hit")], axis=1)
            g_cnt = np.stack([info[k].cpu().numpy().astype(int) for k in ("step_count", "dwell_count", "near_goal_entry_count",
                                                                         "near_goal_drift_count", "pre_near_goal_hit", "near_goal_hit")], axis=1)
            assert np.array_equal(g_cnt[sel], r_cnt[sel]), f"counters differ at step {t}"
            r_rew = np.array([o.reward for o in routs])
            g_rew = reward.cpu().numpy().astype(float)
            err = np.abs(g_rew - r_rew)[sel] / np.maximum(1.0, np.abs(r_rew[sel]))
            if err.max() > 2e-4:
                e = np.nonzero(sel)[0][int(np.argmax(err))]
                comps = info["reward_components"][: len(names), e].cpu().numpy()
                rc = np.array(routs[e].components[: len(names)])
                bad = [(names[i], float(comps[i]), float(rc[i])) for i in np.nonzero(np.abs(comps - rc) > 1e-4 * np.maximum(1, np.abs(rc)))[0]]
                raise AssertionError(f"reward differs at step {t} env {e}: {g_rew[e]} vs {r_rew[e]}; components {bad}")
            stats["max_reward"] = max(stats["max_reward"], float(err.max()))
            stats["checked_flags"] += int(sel.sum())
            stats["max_obs"] = max(stats["max_obs"], float(np.abs(obs.cpu().numpy()[sel] - robs[sel]).max()))
    assert stats["max_pos"] < POS_TOL and stats["max_ang"] < ANG_TOL and stats["max_q"] < 5e-6, stats
    assert stats["max_obs"] < 5e-5, stats
    return stats


def _obs_of(orc, e):
    import ctypes

    obs = np.zeros(56, dtype=np.float32)
    ko.lib().kor_observation(ctypes.byref(orc.params), ctypes.byref(orc.states[e]), ko._fptr(obs))
    return obs


def _trace_inputs(trace):
    """Golden trace episodes -> lock-step batch [T,n,7] (zero actions after an episode's end)."""
    starts = trace["episode_start"]
    n = len(starts) - 1
    T = int(np.max(np.diff(starts)))
    actions = np.zeros((T, n, 7))
    for e in range(n):
        seg = trace["action"][starts[e]:starts[e + 1]]
        actions[: len(seg), e] = seg
    return n, T, actions


@pytest.mark.parametrize("fixture,preset,mode,names", [
    ("trace_approach.npz", "approach_dynamic_scale_big", 0, ko.APPROACH_COMPONENT_NAMES),
    ("trace_dock.npz", "finisher_noop_ft", 1, ko.DOCK_COMPONENT_NAMES),
    ("trace_dock_alt.npz", "trace_dock_alt_config.json", 1, ko.DOCK_COMPONENT_NAMES),
    ("trace_approach_alt.npz", "trace_approach_alt_config.json", 0, ko.APPROACH_COMPONENT_NAMES),
])
def test_golden_traces_open_loop(fixture, preset, mode, names):
    trace = golden(fixture)
    cfg = env_config_from_json(GOLD / preset) if preset.endswith(".json") else env_config(preset)
    n, T, actions = _trace_inputs(trace)
    has_gp = trace["reset_has_goal_pose6"].astype(bool)
    gp = trace["reset_goal_pose6"] if has_gp.all() else None
    stats = _compare_rollout(cfg, mode, trace["reset_initial_q"], trace["reset_goal_q"], actions, gp=gp, idq=trace["reset_initial_dq"],
                             ipa=trace["reset_initial_prev_action"], names=names)
    assert stats["checked_flags"] > 0.5 * n * T * 0.2


@pytest.mark.parametrize("preset,mode,names,scale", [
    ("approach_dynamic_scale_big", 0, ko.APPROACH_COMPONENT_NAMES, 1.0),
    ("finisher_noop_ft", 1, ko.DOCK_COMPONENT_NAMES, 0.05),
])
def test_random_batch_open_loop(preset, mode, names, scale):
    cfg = env_config(preset)
    rng = np.random.default_rng(11 + mode)
    n, T = 2048, 48
    stages = env_config("approach_dynamic_scale_big").curriculum_config.stages
    st = [stages[i % len(stages)] for i in range(n)]
    gq = np.array([np.asarray(s.goal_q) + rng.uniform(-1, 1, 7) * np.asarray(s.goal_noise) for s in st])
    if mode == 0:
        iq = np.array([np.asarray(s.start_q) + rng.uniform(-1, 1, 7) * np.asarray(s.start_noise) for s in st])
        # a proportional controller with noise: reaches the near-goal zones so the reward families fire
        actions = np.zeros((T, n, 7))
        q = iq.copy()
        dl = np.array([sp.delta_limit for sp in cfg.joint_specs]) * cfg.action_delta_scale
        for t in range(T):
            a = np.clip((gq - q) / dl * 0.6 + rng.normal(0, 0.05, (n, 7)) * (rng.random((n, 1)) < 0.5), -1.3, 1.3)
            actions[t] = a
            q = q + np.clip(a, -1, 1) * dl
    else:
        iq = gq + rng.uniform(-0.003, 0.003, (n, 7))
        actions = rng.normal(0, 1.0, (T, n, 7)) * scale * rng.choice([0.1, 1.0, 4.0], size=(1, n, 1))
    stats = _compare_rollout(cfg, mode, iq, gq, actions, idq=rng.uniform(-0.001, 0.001, (n, 7)), ipa=rng.uniform(-0.05, 0.05, (n, 7)), names=names)
    assert stats["checked_flags"] > 0.5 * n * T


def test_per_env_mode_kernel_matches_uniform_kernels():
    cfg = env_config("finisher_noop_ft")
    rng = np.random.default_rng(5)
    n, T = 256, 12
    gq = rng.uniform(-0.4, 0.4, (n, 7))
    iq = gq + rng.uniform(-0.004, 0.004, (n, 7))
    acts = rng.normal(0, 0.2, (T, n, 7)).astype(np.float32)
    outs = []
    for mixed in (False, True):
        env = _make_env(cfg, n)
        env.reset(options={"initial_q": iq, "goal_q": gq, "policy_mode": "dock"})
        if mixed:
            env._mode_all = None
        rew = []
        for t in range(T):
            obs, r, te, tr, info = env.step(torch.as_tensor(acts[t]))
            rew.append(r.clone())
        outs.append((obs.clone(), torch.stack(rew), env.state.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])


def test_mixed_mode_batch():
    """Half the batch in approach mode, half in dock mode, one launch (per-env mode bits)."""
    cfg = env_config("finisher_noop_ft")
    rng = np.random.default_rng(6)
    n = 128
    gq = rng.uniform(-0.4, 0.4, (n, 7))
    iq = gq + rng.uniform(-0.004, 0.004, (n, 7))
    a = rng.normal(0, 0.3, (n, 7)).astype(np.float32)
    ref = {}
    for mode in ("approach", "dock"):
        env = _make_env(cfg, n)
        env.reset(options={"initial_q": iq, "goal_q": gq, "policy_mode": mode})
        obs, r, *_ = env.step(torch.as_tensor(a))
        ref[mode] = (obs.clone(), r.clone())
    env = _make_env(cfg, n)
    env.reset(options={"initial_q": iq, "goal_q": gq, "policy_mode": "approach"})
    mask = torch.arange(n) % 2 == 1
    env.set_policy_mode("dock", env_mask=mask)
    # dock entries need their entry metrics: they equal the reset-time ones, which reset already captured
    obs, r, *_ = env.step(torch.as_tensor(a))
    m = mask.cuda()
    assert torch.equal(obs[~m], ref["approach"][0][~m]) and torch.equal(r[~m], ref["approach"][1][~m])
    assert torch.equal(obs[m], ref["dock"][0][m]) and torch.equal(r[m], ref["dock"][1][m])


def test_reset_paths_and_ragged_sizes():
    cfg = env_config("approach_dynamic_scale_big")
    rng = np.random.default_rng(9)
    for n in (1, 31, 33, 100):   # warp-tail handling of the smem-staged tiles
        env = _make_env(cfg, n)
        iq = rng.uniform(-0.5, 0.5, (n, 7))
        gq = rng.uniform(-0.5, 0.5, (n, 7))
        obs, info = env.reset(options={"initial_q": iq, "goal_q": gq})
        orc = BatchOracle(cfg, n)
        orc.reset(0, iq.astype(np.float32).astype(float), gq.astype(np.float32).astype(float))
        ref = np.stack([_obs_of(orc, e) for e in range(n)])
        assert np.abs(obs.cpu().numpy() - ref).max() < 2e-5
        assert np.abs(env.current_observation().cpu().numpy() - ref).max() < 2e-5
        a = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        obs2, *_ = env.step(torch.as_tensor(a))
        robs, _ = orc.step(a.astype(float))
        assert np.abs(obs2.cpu().numpy() - robs).max() < 3e-5
    # partial reset by env_ids leaves the other slots untouched; explicit goal_pose6 wins over goal_q
    env = _make_env(cfg, 64)
    env.reset(options={"initial_q": rng.uniform(-0.3, 0.3, (64, 7)), "goal_q": rng.uniform(-0.3, 0.3, (64, 7))})
    before = env.state.clone()
    ids = [3, 40, 63]
    gp = rng.uniform(-0.5, 0.5, (3, 6))
    env.reset(options={"initial_q": np.zeros((3, 7)), "goal_q": np.ones((3, 7)) * 0.1, "goal_pose6": gp}, env_ids=ids)
    after = env.state
    other = [i for i in range(64) if i not in ids]
    assert torch.equal(before[:, other], after[:, other])
    assert np.allclose(env.goal_pose6[ids].cpu().numpy(), gp.astype(np.float32))
    assert np.allclose(env.goal_q[ids].cpu().numpy(), 0.1)   # stored unclipped, as given (AKE:190-192)
    with pytest.raises(ValueError):
        env.step(torch.zeros(63, 7))
    with pytest.raises(ValueError):
        env.set_policy_mode("nonsense")


def test_invalid_state_terminates():
    cfg = env_config("approach_dynamic_scale_big")
    env = _make_env(cfg, 32)
    gp = np.zeros((32, 6))
    gp[5, 0] = np.nan
    env.reset(options={"initial_q": np.zeros((32, 7)), "goal_q": np.zeros((32, 7)), "goal_pose6": gp})
    _, _, term, trunc, info = env.step(torch.zeros(32, 7))
    assert bool(term[5]) and int(info["reason_code"][5]) == 3 and not bool(term[4])


def test_graph_step_replays_the_eager_step():
    """``graph_step=True`` (a CUDA graph of the step kernel + the done-bit ops) gives bit for bit the eager ``step()``: observations,
    rewards, flags, lazily decoded info, through auto-resets, a curriculum-stage change and a policy-mode change (the graph is re-captured
    when a baked-in argument changes)."""
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv

    cfg = env_config("approach_dynamic_scale_big")
    n = 2048
    envs = [BatchedArmKinematicEnv(cfg, n, "cuda", auto_reset=True, seed=11, host_sampler=False, graph_step=g) for g in (False, True)]
    gen = torch.Generator(device="cuda").manual_seed(3)
    for e in envs:
        e.set_curriculum_stage(3)
        e.reset()
    for t in range(150):
        a = torch.rand((n, 7), device="cuda", generator=gen) * 2 - 1
        if t == 60:
            for e in envs:
                e.set_curriculum_stage(7)
        outs = [e.step(a.clone()) for e in envs]
        (o0, r0, te0, tr0, i0), (o1, r1, te1, tr1, i1) = outs
        assert torch.equal(o0, o1) and torch.equal(r0, r1) and torch.equal(te0, te1) and torch.equal(tr0, tr1)
        if t % 37 == 0:
            for k in ("success", "position_error_norm", "step_count", "reason_code"):
                assert torch.equal(i0[k], i1[k]), k
    assert envs[1]._graph is not None and int((envs[0].state != envs[1].state).sum()) == 0
    assert bool(te0.any() or tr0.any() or (envs[0].state[48] > 0).any())      # episodes did end and were reset inside the kernel

