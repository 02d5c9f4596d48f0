"""Flatten the reference-shaped config objects into the POD structs of the C ABI."""

from __future__ import annotations

import ctypes
from typing import Any

import numpy as np

from . import _lib, kinematics
from .config import Phase1EnvConfig

MAX_STAGES = 16


def env_params(cfg: Phase1EnvConfig, route_reward: Any | None = None):
    """``Phase1EnvConfig`` -> ``KinEnvParams`` (field names of include/kin_b200.h map 1:1 to config attributes)."""
    if len(cfg.joint_specs) != cfg.n_joints or cfg.n_joints != 7:
        raise ValueError("joint_specs length must match n_joints")  # arm_kinematic_env.py:76-77
    cls = _lib.c_struct("KinEnvParams")
    p = cls()
    for i, spec in enumerate(cfg.joint_specs):
        p.joint_lower[i], p.joint_upper[i], p.joint_delta_limit[i] = spec.lower, spec.upper, spec.delta_limit
    k = kinematics.fold_chain()
    for name, arr in (("fk_pbase", k["pbase"]), ("fk_pq0", k["pq0"]), ("fk_C", k["C"]), ("fk_t", k["t"]), ("fk_AT", k["AT"])):
        flat = np.asarray(arr, dtype=np.float64).reshape(-1)
        dst = getattr(p, name)
        for i, v in enumerate(flat):
            dst[i] = float(v)
    groups = {"ar_": cfg.reward_config, "dr_": cfg.dock_reward_config, "term_": cfg.termination_config,
              "obs_": cfg.observation_config, "rr_": route_reward}
    skip = {"ar_n_milestones", "ar_orientation_milestone_thresholds_rad", "ar_orientation_milestone_bonuses"}
    for fname, ftype in cls._fields_:
        if fname.startswith(("joint_", "fk_", "k_")) or fname in skip:
            continue
        src, key = cfg, fname
        for prefix, sub in groups.items():
            if fname.startswith(prefix):
                src, key = sub, fname[len(prefix):]
                break
        if src is None:  # route reward not supplied
            continue
        value = getattr(src, key)
        setattr(p, fname, int(value) if ftype is ctypes.c_int else float(value))
    for i, spec in enumerate(cfg.joint_specs):
        p.k_inv_span[i] = 1.0 / max(spec.upper - spec.lower, 1e-9)
        p.k_inv_delta_limit[i] = 1.0 / max(spec.delta_limit, 1e-9)
    p.k_inv_pos_err_scale = 1.0 / cfg.observation_config.pos_err_scale_m
    p.k_inv_ori_err_scale = 1.0 / cfg.observation_config.ori_err_scale_rad
    p.k_inv_episode_length = 1.0 / max(cfg.episode_length, 1)
    p.k_inv_dwell_steps_target = 1.0 / max(cfg.dwell_steps_target, 1)
    thr = tuple(cfg.reward_config.orientation_milestone_thresholds_rad or ())
    bon = tuple(cfg.reward_config.orientation_milestone_bonuses or ())
    n = min(len(thr), len(bon))  # zip(strict=False), reward_approach.py:111
    if n > 4:
        raise ValueError("at most 4 orientation milestones are supported")
    p.ar_n_milestones = n
    for i in range(n):
        p.ar_orientation_milestone_thresholds_rad[i] = float(thr[i])
        p.ar_orientation_milestone_bonuses[i] = float(bon[i])
    return p


def sampler_params(cfg: Phase1EnvConfig, stage_index: int = 0):
    """Curriculum shells + workspace_stage_sampling + dock reset -> ``KinSamplerParams``.

    Default values of the optional keys are the reference's (``reset_samplers.py:213-389``).
    """
    cls = _lib.c_struct("KinSamplerParams")
    s = cls()
    cur = cfg.curriculum_config
    stages = cur.stages
    if len(stages) > MAX_STAGES:
        raise ValueError(f"at most {MAX_STAGES} curriculum stages are supported on the device")
    n = len(stages)
    s.n_stages = n
    s.curriculum_enabled = int(bool(cur.enabled))
    current = int(np.clip(stage_index, 0, max(n - 1, 0)))
    s.current_stage = current
    for i, st in enumerate(stages):
        for j in range(7):
            s.start_q[i * 7 + j] = st.start_q[j]
            s.start_noise[i * 7 + j] = st.start_noise[j]
            s.goal_q[i * 7 + j] = st.goal_q[j]
            s.goal_noise[i * 7 + j] = st.goal_noise[j]
    s.start_sample_margin_fraction = cfg.start_sample_margin_fraction
    s.goal_sample_margin_fraction = cfg.goal_sample_margin_fraction
    w = dict(cfg.workspace_stage_sampling or {})
    s.stage_mix_enabled = int(bool(w.get("enabled", False)))
    s.current_stage_ratio = float(w.get("current_stage_ratio", 0.50))
    s.previous_stage_ratio = float(w.get("previous_stage_ratio", 0.25))
    s.old_workspace_replay_ratio = float(w.get("old_workspace_replay_ratio", 0.20))
    s.failure_replay_ratio = float(w.get("failure_replay_ratio", 0.05))
    s.previous_stage_min_index = int(w.get("previous_stage_min_index", 0))
    s.old_workspace_max_stage_index = int(w.get("old_workspace_max_stage_index", min(5, current)))
    r = dict(w.get("random_start_pair_sampling", {}))
    s.random_start_enabled = int(bool(r.get("enabled", False)))
    ratios = (r.get("home_start_ratio", 0.15), r.get("old_successful_start_ratio", 0.25), r.get("random_valid_q_start_ratio", 0.25),
              r.get("frontier_pair_ratio", 0.20), r.get("failure_recovery_start_ratio", 0.10), r.get("stress_start_ratio", 0.05))
    for i, v in enumerate(ratios):
        s.source_ratio[i] = float(v)
    s.home_stage_index = int(r.get("home_stage_index", 0))
    s.known_target_max_stage_index = int(r.get("known_target_max_stage_index", min(7, current)))
    s.mixed_target_max_stage_index = int(r.get("mixed_target_max_stage_index", current))
    s.frontier_min_stage_index = int(r.get("frontier_min_stage_index", min(8, current)))
    s.frontier_max_stage_index = int(r.get("frontier_max_stage_index", current))
    s.frontier_target_min_stage_index = int(r.get("frontier_target_min_stage_index", min(8, current)))
    s.frontier_target_max_stage_index = int(r.get("frontier_target_max_stage_index", current))
    s.stress_target_min_stage_index = int(r.get("stress_target_min_stage_index", min(8, current)))
    s.stress_target_max_stage_index = int(r.get("stress_target_max_stage_index", max(n - 1, 0)))
    s.old_success_max_stage_index = int(r.get("old_success_max_stage_index", min(7, current)))
    s.random_valid_start_margin_fraction = float(r.get("random_valid_start_margin_fraction", cfg.start_sample_margin_fraction))
    s.stress_start_margin_fraction = float(r.get("stress_start_margin_fraction", cfg.start_sample_margin_fraction))
    for i in range(7):
        s.failure_recovery_q_noise[i] = float(r.get("failure_recovery_q_noise", [0.04] * 7)[i])
        s.initial_dq_noise[i] = float(r.get("initial_dq_noise", [0.0] * 7)[i])
        s.initial_prev_action_noise[i] = float(r.get("initial_prev_action_noise", [0.0] * 7)[i])
    s.min_pair_joint_l2 = float(r.get("min_pair_joint_l2", 0.0))
    d = cfg.dock_reset_config
    s.dock_use_stage_goal = int(bool(cur.enabled and n > 0))
    for i in range(7):
        s.dock_goal_q[i] = d.goal_q[i]
        s.dock_goal_noise[i] = d.goal_noise[i]
        s.dock_init_q_noise[i] = d.init_q_noise[i]
        s.dock_close_init_q_noise[i] = d.close_init_q_noise[i]
    s.dock_close_bucket_probability = float(d.close_bucket_probability)
    s.dock_close_bucket_min_pos_error_m = float(d.close_bucket_min_pos_error_m)
    s.dock_close_bucket_max_pos_error_m = float(d.close_bucket_max_pos_error_m)
    s.dock_close_bucket_min_ori_error_rad = float(d.close_bucket_min_ori_error_rad)
    s.dock_close_bucket_max_ori_error_rad = float(d.close_bucket_max_ori_error_rad)
    s.dock_close_bucket_max_attempts = int(d.close_bucket_max_attempts)
    s.dock_handoff_state_probability = 0.0      # set together with the device buffer (ParamsHandle.set_sampler(handoff_states=...))
    s.dock_handoff_state_count = 0
    s.dock_handoff_states = None
    s.frontier_probability = 0.0                # set together with the device table (ParamsHandle.set_sampler(frontier=...))
    s.frontier_bucket_count = 0
    s.frontier_target_count = 0
    return s
