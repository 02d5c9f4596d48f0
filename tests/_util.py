"""Shared helpers for the test-suite (oracle construction from presets, fixtures)."""

from __future__ import annotations

import json
from pathlib import Path

import numpy as np

from oracle import kin_oracle as ko
from rl_brain_trainer_b200 import config as kcfg

GOLD = Path(__file__).resolve().parent / "golden"
POLICY_DIR = kcfg.PRESET_DIR / "policies"


def golden(name: str):
    return np.load(GOLD / name, allow_pickle=False)


def env_config(preset: str) -> kcfg.Phase1EnvConfig:
    return kcfg.load_preset(preset)


def env_config_from_json(path: Path) -> kcfg.Phase1EnvConfig:
    return kcfg.to_env_config(json.loads(Path(path).read_text()))


def oracle_params(cfg, route_reward=None):
    return ko.params_from_config(cfg, route_reward)


def policy_weights(name: str) -> dict[str, np.ndarray]:
    with np.load(POLICY_DIR / f"{name}.npz") as z:
        return {k: z[k] for k in z.files}


def oracle_policy(name: str) -> ko.OracleMlp:
    return ko.OracleMlp(policy_weights(name))


# ---- per-step parity helpers shared by the env parity tests ---------------------------------------------------------------
def _thresholds(cfg):
    rc, dr, tc = cfg.reward_config, cfg.dock_reward_config, cfg.termination_config
    pos = [rc.pre_near_goal_pos_threshold_m, rc.near_goal_pos_threshold_m, rc.handover_pos_threshold_m, rc.dock_coarse_ready_pos_threshold_m,
           rc.finisher_ready_pos_threshold_m, rc.near_handoff_pos_threshold_m, tc.success_pos_threshold_m, dr.tight_pose_pos_threshold_m,
           dr.near_strict_pos_threshold_m or 2 * dr.tight_pose_pos_threshold_m, dr.convergence_position_radius_m,
           dr.position_first_orientation_pos_threshold_m, dr.basin_outer_radius_m, dr.basin_inner_radius_m, dr.basin_dwell_radius_m,
           dr.tight_position_shaping_radius_m, dr.strict_center_small_action_pos_radius_m,
           cfg.dynamic_action_delta_scale_near_pos_threshold_m, cfg.dynamic_action_delta_scale_far_pos_threshold_m,
           dr.entry_action_penalty_near_pos_threshold_m, dr.entry_action_penalty_far_pos_threshold_m]
    ori = [rc.near_goal_ori_threshold_rad, rc.coarse_orientation_bonus_threshold_rad, rc.handover_ori_threshold_rad,
           rc.dock_coarse_ready_ori_threshold_rad, rc.finisher_ready_ori_threshold_rad, rc.near_handoff_ori_threshold_rad,
           tc.success_ori_threshold_rad, dr.tight_pose_ori_threshold_rad, dr.near_strict_ori_threshold_rad or 3 * dr.tight_pose_ori_threshold_rad,
           dr.convergence_orientation_radius_rad, dr.tight_orientation_shaping_radius_rad, *rc.orientation_milestone_thresholds_rad]
    act = [rc.dock_coarse_ready_action_threshold, rc.finisher_ready_action_threshold, dr.low_motion_action_threshold,
           dr.tiny_correction_action_threshold, dr.aggressive_action_threshold]
    dq = [rc.dock_coarse_ready_dq_threshold, rc.finisher_ready_dq_threshold, dr.low_motion_dq_threshold, dr.dq_penalty_threshold]
    f = lambda xs: np.array(sorted({float(x) for x in xs if x and x > 0}))  # noqa: E731
    return f(pos), f(ori), f(act), f(dq)


def _near(values, thresholds, band):
    if thresholds.size == 0:
        return np.zeros(np.shape(values), dtype=bool)
    return (np.abs(np.asarray(values)[..., None] - thresholds) < band).any(-1)


def _rot(rpy: np.ndarray) -> np.ndarray:
    """Rz(yaw) Ry(pitch) Rx(roll) for rows of (roll, pitch, yaw) -- the reference's Euler convention (ee_fk.py:64-71)."""
    cr, sr, cp, sp, cy, sy = np.cos(rpy[:, 0]), np.sin(rpy[:, 0]), np.cos(rpy[:, 1]), np.sin(rpy[:, 1]), np.cos(rpy[:, 2]), np.sin(rpy[:, 2])
    return np.stack([np.stack([cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr], -1),
                     np.stack([sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr], -1),
                     np.stack([-sp, cp * sr, cp * cr], -1)], -2)


def _geodesic(rpy_a: np.ndarray, rpy_b: np.ndarray) -> np.ndarray:
    """Angle of the rotation taking orientation a to orientation b (singularity-free, unlike Euler differences)."""
    rel = np.einsum("nij,nkj->nik", _rot(rpy_a), _rot(rpy_b))
    skew = np.stack([rel[:, 2, 1] - rel[:, 1, 2], rel[:, 0, 2] - rel[:, 2, 0], rel[:, 1, 0] - rel[:, 0, 1]], -1)
    return np.arctan2(0.5 * np.linalg.norm(skew, axis=1), 0.5 * (np.trace(rel, axis1=1, axis2=2) - 1.0))


from oracle.parity import scale_decision_thresholds, threshold_sensitive_episodes  # noqa: E402,F401  (re-exported for the tests)
