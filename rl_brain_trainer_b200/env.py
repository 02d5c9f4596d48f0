"""Host-side mirror of the reference env API on top of the C ABI (include/kin_b200.h).

``BatchedArmKinematicEnv``  N envs on one GPU, torch CUDA tensors in/out, one fused kernel per step.
``ArmKinematicEnv``         1-env adapter with the reference's exact signature (numpy in/out, dict
                            observation, the same ``info`` keys, the same ``ValueError``s), so the
                            reference's eval loops and its own tests run against the GPU path unchanged
                            (``kinematic_phase1/envs/arm_kinematic_env.py:69-557``, "AKE" below).

PyTorch is used for device memory and streams only; all arithmetic happens in csrc/*.cu.
"""

from __future__ import annotations

import ctypes
from dataclasses import replace
from typing import Any, Mapping, Sequence

import numpy as np
import torch

from . import _lib, params as _params, samplers
from .config import Phase1EnvConfig

OBS_DIM = 56
MODE_INDEX = {"approach": 0, "dock": 1}
MODE_NAME = {0: "approach", 1: "dock"}
REASONS = ("running", "success", "max_steps", "invalid_state")

# slices of the flat 56-vector == SB3's alphabetical flattening of the 13-key dict observation
OBS_SLICES: dict[str, slice] = {
    "dq": slice(0, 7), "goal_ori_err": slice(7, 10), "goal_pos_err": slice(10, 13), "joint_limit_margin": slice(13, 20),
    "mode_flag": slice(20, 24), "next_wp_ori_err": slice(24, 27), "next_wp_pos_err": slice(27, 30), "prev_action": slice(30, 37),
    "progress": slice(37, 40), "q": slice(40, 47), "task_type": slice(47, 50), "wp_ori_err": slice(50, 53), "wp_pos_err": slice(53, 56),
}
# key order of the reference's dict observation (observation_builder.py:73-93)
OBS_KEYS = ("q", "dq", "prev_action", "goal_pos_err", "goal_ori_err", "wp_pos_err", "wp_ori_err", "next_wp_pos_err",
            "next_wp_ori_err", "task_type", "mode_flag", "progress", "joint_limit_margin")

APPROACH_COMPONENT_NAMES = (
    "position_progress", "global_orientation_progress", "near_field_orientation_progress", "orientation_progress",
    "orientation_milestone_bonus", "near_field_orientation_center", "pre_near_goal_bonus", "near_goal_bonus",
    "pre_near_to_near_progress", "near_goal_bonus_scale", "coarse_orientation_bonus", "handover_bonus",
    "handover_retention_bonus", "handover_dwell_bonus", "handover_leave_penalty", "handover_regression_penalty",
    "dock_coarse_ready_bonus", "dock_coarse_ready_retention_bonus", "dock_coarse_ready_dwell_bonus",
    "dock_coarse_ready_leave_penalty", "dock_coarse_ready_regression_penalty", "finisher_ready_bonus",
    "finisher_ready_retention_bonus", "finisher_ready_dwell_bonus", "finisher_ready_leave_penalty",
    "finisher_ready_regression_penalty", "near_handoff_action_penalty", "near_handoff_dq_penalty",
    "near_handoff_motion_bonus", "near_handoff_settle_bonus", "same_step_alignment_bonus", "dwell_bonus",
    "drift_penalty", "near_goal_leave_penalty", "drift_penalty_scale", "near_goal_entry_count",
    "near_goal_drift_count", "smoothness_penalty", "smoothness_multiplier", "joint_limit_penalty", "success_bonus",
    "curr_pos_error", "curr_ori_error", "curr_action_norm", "curr_dq_norm", "dwell_count", "in_pre_near_goal",
    "in_near_goal", "in_handover_zone", "in_dock_coarse_ready", "in_dock_coarse_ready_pose", "in_finisher_ready",
    "in_finisher_ready_pose", "in_near_handoff_zone",
)
DOCK_COMPONENT_NAMES = (
    "position_progress", "orientation_progress", "stay_in_zone_bonus", "dwell_bonus", "working_range_bonus",
    "working_range_dwell_bonus", "tight_pose_bonus", "tight_pose_dwell_bonus", "strict_pose_leave_penalty",
    "strict_center_reward", "strict_center_position_penalty", "strict_center_orientation_penalty",
    "strict_center_small_action_bonus", "strict_center_dwell_bonus", "tight_position_shaping",
    "tight_orientation_shaping", "convergence_position_progress", "convergence_orientation_progress",
    "orientation_position_gate_scale", "entry_action_penalty_scale", "leave_zone_penalty",
    "working_range_exit_penalty", "drift_penalty", "smoothness_penalty", "action_delta_violation_penalty",
    "delta_q_change_penalty", "preserve_state_bonus", "strict_hold_bonus", "low_motion_bonus",
    "tiny_correction_bonus", "worse_than_entry_penalty", "near_strict_regression_penalty",
    "aggressive_action_penalty", "dq_penalty", "joint_limit_penalty", "success_bonus", "basin_outer_bonus",
    "basin_inner_bonus", "basin_dwell_bonus", "basin_outer_exit_penalty", "basin_inner_exit_penalty",
    "basin_dwell_break_penalty", "basin_drift_penalty", "basin_zone_index", "curr_pos_error", "curr_ori_error",
    "dwell_count", "in_tight_pose", "in_near_strict", "entry_pos_error", "entry_ori_error", "entry_action_l2",
    "entry_dq_norm", "entry_to_curr_delta_position_error", "entry_to_curr_delta_orientation_error",
    "entry_to_curr_delta_action_l2", "entry_to_curr_delta_dq_norm", "near_goal_entry_count",
    "near_goal_drift_count", "in_near_goal",
)


def _D(name: str) -> int:
    return _lib.define(name)


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def obs_dict(obs: torch.Tensor | np.ndarray) -> dict[str, Any]:
    """Split a flat ``[..., 56]`` observation into the reference's 13-key dict (views, no copy)."""
    return {k: obs[..., OBS_SLICES[k]] for k in OBS_KEYS}


class ParamsHandle:
    """Owns one ``kin_params_create`` handle (the device-side image of a ``Phase1EnvConfig``)."""

    def __init__(self, config: Phase1EnvConfig, route_reward: Any | None = None) -> None:
        self.config = config
        self.c_params = _params.env_params(config, route_reward)
        self._h = ctypes.c_void_p()
        _lib.check(_lib.lib().kin_params_create(ctypes.byref(self.c_params), ctypes.byref(self._h)))
        self._sampler = None

    @property
    def handle(self) -> ctypes.c_void_p:
        return self._h

    def set_sampler(self, stage_index: int, handoff_states: torch.Tensor | None = None, frontier: Any = None) -> None:
        """Upload the reset sampler tables; ``handoff_states`` ([M, 34] float32 on the device, ``handoff.HandoffBuffer.device_rows``)
        arms the dock reset's handoff-state replay with ``dock_reset_config.handoff_state_probability``; ``frontier`` (a
        ``coverage.FrontierTable`` and a probability, ``(table, p)``) arms the random-start sampler's adaptive frontier targets."""
        self._sampler = _params.sampler_params(self.config, stage_index)
        if frontier is not None:
            table, probability = frontier
            if not self._sampler.random_start_enabled:
                raise _lib.KinError("frontier targets are drawn by the random-start pair sampler: the config has random_start_pair_sampling disabled")
            self._sampler.frontier_probability = float(probability)
            self._sampler.frontier_bucket_count = int(table.bucket_count)
            self._sampler.frontier_target_count = int(table.target_count)
            self._sampler.frontier_bucket_offset = table.offsets.data_ptr()
            self._sampler.frontier_alias_prob = table.alias_prob.data_ptr()
            self._sampler.frontier_alias_index = table.alias_index.data_ptr()
            self._sampler.frontier_targets = table.targets.data_ptr()
        if handoff_states is not None and handoff_states.numel() > 0:
            if handoff_states.dtype != torch.float32 or handoff_states.dim() != 2 or handoff_states.shape[1] != _D("KIN_HANDOFF_STATE_FLOATS") \
                    or not handoff_states.is_cuda or not handoff_states.is_contiguous():
                raise ValueError("handoff_states must be a contiguous CUDA float32 [M, 34] tensor")
            self._sampler.dock_handoff_state_probability = float(self.config.dock_reset_config.handoff_state_probability)
            self._sampler.dock_handoff_state_count = int(handoff_states.shape[0])
            self._sampler.dock_handoff_states = handoff_states.data_ptr()
        _lib.check(_lib.lib().kin_params_set_sampler(self._h, ctypes.byref(self._sampler)))
        # keep the device buffers alive as long as the sampler points at them; the ones replaced are released only now, after the
        # synchronous upload has ordered them behind every kernel that could still read them
        self._handoff_states, self._frontier = handoff_states, frontier

    def __del__(self) -> None:  # pragma: no cover - interpreter teardown order
        try:
            if self._h:
                _lib.lib().kin_params_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass


class LazyInfo(Mapping):
    """Read-only ``info`` mapping whose values are produced on first access (and then cached).  Behaves like the dict the reference
    returns for every reader (``info[key]``, ``key in info``, ``info.get``, iteration, ``dict(info)``)."""

    __slots__ = ("_thunks", "_cache")

    def __init__(self, thunks: dict[str, Any]) -> None:
        self._thunks = thunks
        self._cache: dict[str, Any] = {}

    def __getitem__(self, key: str) -> Any:
        if key not in self._cache:
            self._cache[key] = self._thunks[key]()
        return self._cache[key]

    def __iter__(self):
        return iter(self._thunks)

    def __len__(self) -> int:
        return len(self._thunks)

    def __contains__(self, key: object) -> bool:
        return key in self._thunks


class BatchedArmKinematicEnv:
    """``num_envs`` independent kinematic envs resident on one GPU.

    Semantics per env are ``ArmKinematicEnv``'s (AKE:102-365); tensors replace scalars:

    * ``reset(seed=, options={initial_q [M,7], initial_dq, initial_prev_action, goal_q, goal_pose6 [M,6],
      policy_mode}, env_ids=None)`` -> ``(obs [N,56], info)``.  Without ``initial_q`` the starts are drawn by the
      device sampler (Philox) -- or, with ``host_sampler=True``, by the numpy port that consumes the reference's
      PCG64 stream in the reference's order (bit-identical starts, O(N) host work).
    * ``step(actions [N,7])`` -> ``(obs [N,56], reward [N], terminated [N] bool, truncated [N] bool, info)``;
      no auto-reset unless ``auto_reset=True`` (then VecEnv semantics, see ``kin_env_step``).
    """

    def __init__(self, config: Phase1EnvConfig | None = None, num_envs: int = 1, device: str | torch.device = "cuda", *,
                 auto_reset: bool = False, seed: int = 0, host_sampler: bool | None = None, with_aux: bool = True,
                 with_components: bool = False, route_reward: Any | None = None, graph_step: bool = False) -> None:
        self.config = config or Phase1EnvConfig()
        # graph_step: ``step()`` replays a CUDA graph of [kin_env_step, the two done-bit ops] instead of launching them from Python -- for
        # callers that drive the env step by step at sizes where the launch path, not the kernel, is the cost (65 536 envs: 57 us per
        # call eager).  The graph bakes the config / mode / seed in and is re-captured when one of them changes.
        self.graph_step = bool(graph_step)
        self._graph: Any = None
        self._graph_key: Any = None
        if len(self.config.joint_specs) != self.config.n_joints:
            raise ValueError("joint_specs length must match n_joints")
        if num_envs <= 0:
            raise ValueError("num_envs must be positive")
        if not torch.cuda.is_available():
            raise _lib.KinError("BatchedArmKinematicEnv needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.KinError("BatchedArmKinematicEnv only runs on CUDA devices")
        self.num_envs = int(num_envs)
        self.stride = (self.num_envs + 31) // 32 * 32
        self.auto_reset = bool(auto_reset)
        self.host_sampler = (self.num_envs == 1) if host_sampler is None else bool(host_sampler)
        self._L = _lib.lib()
        with torch.cuda.device(self.device):
            self._params = ParamsHandle(self.config, route_reward)
            rows = _D("KIN_STATE_ROWS")
            self.state = torch.zeros((rows, self.stride), dtype=torch.float32, device=self.device)
            self.state[_D("KIN_ROW_MIN_POS")].fill_(float("inf"))
            self.obs = torch.zeros((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
            self.reward = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
            self.done = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
            self.aux = torch.zeros((_D("KIN_AUX_ROWS"), self.stride), dtype=torch.float32, device=self.device) if (with_aux or with_components) else None
            self.components = torch.zeros((_D("KIN_MAX_COMPONENTS"), self.stride), dtype=torch.float32, device=self.device) if with_components else None
            self.terminal_obs = torch.zeros_like(self.obs) if self.auto_reset else None
        self._rng = np.random.default_rng(0)  # AKE:80
        self._seed = int(seed)
        self._mode_all: int | None = MODE_INDEX.get(self.config.mode_name, 0)
        self._default_mode = self._mode_all
        self._stage = 0
        self._sampler_stage: int | None = None
        self._step_calls = 0

    # ------------------------------------------------------------------ curriculum / mode
    def set_curriculum_stage(self, stage_index: int) -> None:
        if not self.config.curriculum_config.enabled:  # AKE:446-449
            return
        self._stage = int(np.clip(stage_index, 0, len(self.config.curriculum_config.stages) - 1))

    def get_curriculum_stage(self) -> int:
        return int(self._stage)

    def set_policy_mode(self, mode_name: str, env_mask: torch.Tensor | None = None) -> None:
        if mode_name not in {"approach", "bridge", "dock", "dock_coarse"}:
            raise ValueError(f"Unsupported policy mode '{mode_name}'")  # AKE:454-457
        if mode_name not in MODE_INDEX:
            raise _lib.KinError(f"policy mode '{mode_name}' belongs to the pipeline stages the reference removed; not built (DESIGN.md)")
        m = MODE_INDEX[mode_name]
        flags = self.state[_D("KIN_ROW_FLAGS")].view(torch.int32)
        shift = _D("KIN_FLAG_MODE_SHIFT")
        new = (flags & ~(3 << shift)) | (m << shift)
        if env_mask is None:
            flags.copy_(new)
            self._mode_all = m
        else:
            mask = torch.zeros(self.stride, dtype=torch.bool, device=self.device)
            mask[: self.num_envs] = env_mask.to(self.device, torch.bool)
            flags.copy_(torch.where(mask, new, flags))
            self._mode_all = None

    def _ensure_sampler(self) -> None:
        if self._sampler_stage != self._stage:
            self._params.set_sampler(self._stage, getattr(self, "_handoff_rows", None), getattr(self, "_frontier", None))
            self._sampler_stage = self._stage

    def set_handoff_states(self, rows: torch.Tensor | None) -> None:
        """Arm (or clear) the dock reset's handoff-state replay (reset_samplers.py:434-446): ``rows`` is ``[M, 34]`` float32
        (initial_q | initial_dq | initial_prev_action | goal_q | goal_pose6), e.g. ``HandoffBuffer.device_rows(device)``."""
        self._handoff_rows = None if rows is None else rows.to(self.device, torch.float32).contiguous()
        self._sampler_stage = None

    def set_frontier_targets(self, table: Any, probability: float = 0.5) -> None:
        """Arm (or, with ``None``, clear) the adaptive frontier targets of the random-start sampler: with ``probability`` an approach
        reset draws its goal from ``table`` (a ``coverage.FrontierTable`` on this device: alias-table bucket, uniform target in it)
        instead of the stage shell.  Uploaded with the next reset / rollout; the env keeps the table alive while the sampler uses it."""
        if table is not None:
            if not _params.sampler_params(self.config, self._stage).random_start_enabled:
                raise _lib.KinError("frontier targets are drawn by the random-start pair sampler: the config has random_start_pair_sampling disabled")
            if not (0.0 <= float(probability) <= 1.0):
                raise ValueError("frontier probability must be in [0, 1]")
            here = self.device.index if self.device.index is not None else torch.cuda.current_device()
            if not table.offsets.is_cuda or table.offsets.device.index != here:
                raise ValueError(f"the frontier table lives on {table.offsets.device}, the env on {self.device}")
        self._frontier = None if table is None else (table, float(probability))
        self._sampler_stage = None

    # ------------------------------------------------------------------ reset
    def _as_dev(self, x: Any, cols: int, m: int) -> torch.Tensor | None:
        if x is None:
            return None
        t = torch.as_tensor(x, dtype=torch.float32, device=self.device).reshape(-1, cols)
        if t.shape[0] == 1 and m > 1:
            t = t.expand(m, cols)
        if t.shape[0] != m:
            raise ValueError(f"expected {m} rows of {cols}, got {tuple(t.shape)}")
        return t.contiguous()

    def reset(self, *, seed: int | None = None, options: Mapping[str, Any] | None = None,
              env_ids: torch.Tensor | Sequence[int] | None = None) -> tuple[torch.Tensor, dict[str, Any]]:
        if seed is not None:
            self._rng = np.random.default_rng(seed)
            self._seed = int(seed)
        opts = dict(options or {})
        mode_name = str(opts.get("policy_mode", self.config.mode_name))
        if mode_name not in MODE_INDEX:
            raise _lib.KinError(f"policy mode '{mode_name}' is not built (only approach / dock are on the hot path)")
        mode = MODE_INDEX[mode_name]
        ids = None
        m = self.num_envs
        if env_ids is not None:
            ids = torch.as_tensor(env_ids, dtype=torch.int32, device=self.device).contiguous()
            m = int(ids.numel())
        with torch.cuda.device(self.device):
            if opts.get("initial_q") is None and not self.host_sampler:
                # device sampler (Philox); explicit goals are not combined with sampled starts on this path
                self._ensure_sampler()
                mask = None
                if ids is not None:
                    mask = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
                    mask[ids.long()] = 1
                _lib.check(self._L.kin_env_reset_sampled(self._params.handle, _ptr(self.state), self.stride, self.num_envs, _ptr(mask), mode,
                                                         self._seed, _ptr(self.obs), _stream()))
            else:
                if opts.get("initial_q") is None:
                    draws = [samplers.sample_reset(self._rng, self.config, mode_name, self._stage, fk=self.fk_pose6_host) for _ in range(m)]
                    opts.update({
                        "initial_q": np.stack([d.initial_q for d in draws]), "goal_q": np.stack([d.goal_q for d in draws]),
                        "initial_dq": np.stack([d.initial_dq if d.initial_dq is not None else np.zeros(7) for d in draws]),
                        "initial_prev_action": np.stack([d.initial_prev_action if d.initial_prev_action is not None else np.zeros(7) for d in draws]),
                    })
                    gp = [d.goal_pose6 for d in draws]
                    if all(g is not None for g in gp):
                        opts["goal_pose6"] = np.stack(gp)
                elif opts.get("goal_q") is None and opts.get("goal_pose6") is None:
                    # AKE:199-206: explicit start, sampled reachable goal
                    goals = [samplers.sample_joint_configuration(self._rng, self.config.joint_specs, self.config.goal_sample_margin_fraction)
                             for _ in range(m)]
                    opts["goal_q"] = np.stack(goals)
                iq = self._as_dev(opts["initial_q"], 7, m)
                idq = self._as_dev(opts.get("initial_dq"), 7, m)
                ipa = self._as_dev(opts.get("initial_prev_action"), 7, m)
                gq = self._as_dev(opts.get("goal_q"), 7, m)
                gp = self._as_dev(opts.get("goal_pose6"), 6, m)
                obs_out = self.obs if ids is None else torch.empty((m, OBS_DIM), dtype=torch.float32, device=self.device)
                _lib.check(self._L.kin_env_reset(self._params.handle, _ptr(self.state), self.stride, self.num_envs, _ptr(ids), m, mode, _ptr(iq),
                                                 _ptr(idq), _ptr(ipa), _ptr(gq), _ptr(gp), _ptr(obs_out), _stream()))
                if ids is not None:
                    self.obs[ids.long()] = obs_out
        if ids is None:
            self._mode_all = mode
        elif self._mode_all != mode:
            self._mode_all = None
        return self.obs, self._info(reset=True)

    # ------------------------------------------------------------------ step
    def step(self, actions: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, dict[str, Any]]:
        a = torch.as_tensor(actions, dtype=torch.float32, device=self.device)
        if a.shape != (self.num_envs, 7):
            raise ValueError(f"Expected action shape {(self.num_envs, 7)}, got {tuple(a.shape)}")
        a = a.contiguous()
        hint = _D("KIN_MODE_PER_ENV") if self._mode_all is None else self._mode_all
        if self.auto_reset:
            self._ensure_sampler()
        self._step_calls += 1
        masks = getattr(self, "_done_masks", None)
        if masks is None:
            masks = self._done_masks = torch.tensor([[_D("KIN_DONE_TERMINATED")], [_D("KIN_DONE_TRUNCATED")]], dtype=self.done.dtype, device=self.device)
        if self.graph_step and self._step_calls > 1:       # (the first call runs eagerly: one-off attribute / sampler set-up happens there)
            key = (id(self._params), hint, self._seed, bool(self.auto_reset))
            if self._graph is None or self._graph_key != key:
                self._g_act = torch.empty_like(a)
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.device(self.device), torch.cuda.graph(g):
                    _lib.check(self._L.kin_env_step(self._params.handle, _ptr(self.state), self.stride, self.num_envs, hint, _ptr(self._g_act),
                                                    _ptr(self.obs), _ptr(self.reward), _ptr(self.done), _ptr(self.aux), _ptr(self.components),
                                                    int(self.auto_reset), self._seed, _ptr(self.terminal_obs), _stream()))
                    self._g_tt = (self.done.unsqueeze(0) & masks) != 0
                self._graph, self._graph_key = g, key
            self._g_act.copy_(a, non_blocking=True)
            self._graph.replay()
            return self.obs, self.reward, self._g_tt[0], self._g_tt[1], self._info(reset=False)
        with torch.cuda.device(self.device):
            _lib.check(self._L.kin_env_step(self._params.handle, _ptr(self.state), self.stride, self.num_envs, hint, _ptr(a), _ptr(self.obs),
                                            _ptr(self.reward), _ptr(self.done), _ptr(self.aux), _ptr(self.components), int(self.auto_reset),
                                            self._seed, _ptr(self.terminal_obs), _stream()))
        tt = (self.done.unsqueeze(0) & masks) != 0          # both done-bit tests in two launches: [2, n]
        return self.obs, self.reward, tt[0], tt[1], self._info(reset=False)

    def step_raw(self, actions: torch.Tensor) -> None:
        """One fused-kernel step with no host-side post-processing: results land in ``self.obs / reward / done / aux``.

        ``actions`` must already be a contiguous float32 ``[num_envs, 7]`` tensor on this device.  This is the call a
        device-resident rollout loop makes (policy kernel -> step_raw -> policy kernel ...).
        """
        hint = _D("KIN_MODE_PER_ENV") if self._mode_all is None else self._mode_all
        _lib.check(self._L.kin_env_step(self._params.handle, self.state.data_ptr(), self.stride, self.num_envs, hint, actions.data_ptr(),
                                        self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(), _ptr(self.aux), _ptr(self.components),
                                        int(self.auto_reset), self._seed, _ptr(self.terminal_obs), _stream()))

    def current_observation(self) -> torch.Tensor:
        out = torch.empty_like(self.obs)
        with torch.cuda.device(self.device):
            _lib.check(self._L.kin_env_observe(self._params.handle, _ptr(self.state), self.stride, self.num_envs, _ptr(out), _stream()))
        return out

    # ------------------------------------------------------------------ views of the SoA state
    def _rows(self, name: str, count: int) -> torch.Tensor:
        r = _D(name)
        return self.state[r:r + count, : self.num_envs].t()

    @property
    def q(self) -> torch.Tensor:
        return self._rows("KIN_ROW_Q", 7)

    @property
    def dq(self) -> torch.Tensor:
        return self._rows("KIN_ROW_DQ", 7)

    @property
    def prev_action(self) -> torch.Tensor:
        return self._rows("KIN_ROW_PREV_ACTION", 7)

    @property
    def goal_q(self) -> torch.Tensor:
        return self._rows("KIN_ROW_GOAL_Q", 7)

    @property
    def goal_pose6(self) -> torch.Tensor:
        return self._rows("KIN_ROW_GOAL_POSE", 6)

    @property
    def ee_pose6(self) -> torch.Tensor:
        return self._rows("KIN_ROW_EE_POSE", 6)

    def counters(self) -> dict[str, torch.Tensor]:
        c0 = self.state[_D("KIN_ROW_CNT0"), : self.num_envs].view(torch.int32)
        c1 = self.state[_D("KIN_ROW_CNT1"), : self.num_envs].view(torch.int32)
        fl = self.state[_D("KIN_ROW_FLAGS"), : self.num_envs].view(torch.int32)
        return {"step_count": c0 & 0xFFFF, "dwell_count": (c0 >> 16) & 0xFFFF, "near_goal_entry_count": c1 & 0xFFFF,
                "near_goal_drift_count": (c1 >> 16) & 0xFFFF, "pre_near_goal_hit": (fl & 1) != 0, "near_goal_hit": (fl & 2) != 0,
                "mode": (fl >> _D("KIN_FLAG_MODE_SHIFT")) & 3, "stage": (fl >> _D("KIN_FLAG_STAGE_SHIFT")) & 15}

    def _info(self, *, reset: bool) -> "LazyInfo":
        """Batched ``info`` keyed like the reference's ``_base_info`` (AKE:384-423), decoded LAZILY: ``step()`` is the kernel launch
        plus the two done-bit tests; a key costs its one or two elementwise ops only when somebody reads it.  Values are views of
        (or derived from) the env's buffers as they are at first access, valid until the next ``step`` / ``reset``."""
        n, st, d = self.num_envs, self.state, self.done
        # the thunks only close over the env's buffers: built once per (reset, buffer set), shared by every LazyInfo (each has its own cache)
        key_ = (bool(reset), id(st), id(d), id(self.aux), id(self.components), id(self.terminal_obs))
        cached = getattr(self, "_info_thunks", None)
        if cached is not None and cached[0] == key_:
            return LazyInfo(cached[1])
        e = _D("KIN_ROW_ENTRY")
        t: dict[str, Any] = {
            "q": lambda: self.q, "dq": lambda: self.dq, "goal_q": lambda: self.goal_q, "goal_pose6": lambda: self.goal_pose6,
            "ee_pose6": lambda: self.ee_pose6, "min_position_error": lambda: st[_D("KIN_ROW_MIN_POS"), :n],
            "entry_position_error_norm": lambda: st[e, :n], "entry_orientation_error_norm": lambda: st[e + 1, :n],
            "entry_action_l2": lambda: st[e + 2, :n], "entry_dq_norm": lambda: st[e + 3, :n],
        }
        if reset:
            t["position_error_norm"] = t["entry_position_error_norm"]
            t["orientation_error_norm"] = t["entry_orientation_error_norm"]
            t["success"] = lambda: torch.zeros(n, dtype=torch.bool, device=self.device)
        else:
            t["success"] = lambda: (d & _D("KIN_DONE_SUCCESS")) != 0
            t["curr_in_pre_near_goal"] = lambda: (d & _D("KIN_DONE_PRE_NEAR")) != 0
            t["curr_in_near_goal"] = lambda: (d & _D("KIN_DONE_NEAR")) != 0
            t["reason_code"] = lambda: (d >> _D("KIN_DONE_REASON_SHIFT")) & 3
            t["auto_reset"] = lambda: (d & _D("KIN_DONE_AUTORESET")) != 0
            if self.aux is not None:
                ax = self.aux
                for key, row in (("position_error_norm", "KIN_AUX_POS_ERR"), ("orientation_error_norm", "KIN_AUX_ORI_ERR"),
                                 ("action_l2", "KIN_AUX_ACTION_L2"), ("executed_delta_q_l2", "KIN_AUX_DQ_L2"),
                                 ("delta_q_change_l2", "KIN_AUX_DQ_CHANGE_L2"), ("dock_action_limit", "KIN_AUX_DOCK_LIMIT"),
                                 ("dock_delta_q_change_limit_scale", "KIN_AUX_DQC_SCALE"), ("joint_limit_margin_min", "KIN_AUX_MARGIN_MIN")):
                    t[key] = (lambda r: (lambda: ax[_D(r), :n]))(row)
            if self.components is not None:
                t["reward_components"] = lambda: self.components[:, :n]
            if self.terminal_obs is not None:
                t["terminal_observation"] = lambda: self.terminal_obs
        for key in ("step_count", "dwell_count", "near_goal_entry_count", "near_goal_drift_count", "pre_near_goal_hit", "near_goal_hit", "mode", "stage"):
            t[key] = (lambda k: (lambda: self.counters()[k]))(key)
        self._info_thunks = (key_, t)
        return LazyInfo(t)

    # ------------------------------------------------------------------ helpers
    def fk_pose6(self, q: torch.Tensor) -> torch.Tensor:
        """``compute_ee_pose6`` for a batch (fk_interface.py:21): q [M,7] -> pose6 [M,6], on the device."""
        qd = torch.as_tensor(q, dtype=torch.float32, device=self.device).reshape(-1, 7).contiguous()
        out = torch.empty((qd.shape[0], 6), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._L.kin_fk_pose6(self._params.handle, _ptr(qd), _ptr(out), qd.shape[0], _stream()))
        return out

    def fk_pose6_host(self, q: np.ndarray) -> np.ndarray:
        return self.fk_pose6(torch.as_tensor(np.asarray(q, dtype=np.float32))).cpu().numpy().astype(float).reshape(np.shape(q)[:-1] + (6,))

    def apply_dock_training_stage(self, stage_updates: Mapping[str, Any]) -> None:
        """AKE:459-487: swap dock control knobs mid-training (rebuilds the device params)."""
        if self.config.mode_name != "dock":
            return
        cfg = self.config
        dr = dict(stage_updates.get("dock_reset", {}))
        if dr:
            cfg = replace(cfg, dock_reset_config=replace(cfg.dock_reset_config, **dr))
        keys = ("action_delta_scale", "dock_action_delta_scale", "dock_residual_action_limit", "dock_delta_q_change_limit_scale",
                "dock_dynamic_action_limit_near_pos_threshold_m", "dock_dynamic_action_limit_far_pos_threshold_m",
                "dock_dynamic_residual_action_limit_near", "dock_dynamic_residual_action_limit_far",
                "dock_dynamic_delta_q_change_limit_scale_near", "dock_dynamic_delta_q_change_limit_scale_far")
        upd = {k: float(stage_updates[k]) for k in keys if k in stage_updates}
        if upd:
            cfg = replace(cfg, **upd)
        self.config = cfg
        with torch.cuda.device(self.device):
            self._params = ParamsHandle(cfg)
        self._sampler_stage = None

    def close(self) -> None:
        return None


class _Box:
    def __init__(self, low: float, high: float, shape: tuple[int, ...]) -> None:
        self.low = np.full(shape, low, dtype=np.float32)
        self.high = np.full(shape, high, dtype=np.float32)
        self.shape = shape
        self.dtype = np.float32


class _DictSpace:
    def __init__(self, spaces: dict[str, _Box]) -> None:
        self.spaces = spaces


def build_action_space(n_joints: int) -> _Box:
    return _Box(-1.0, 1.0, (n_joints,))


def build_observation_space(n_joints: int) -> _DictSpace:
    """Same keys / bounds / shapes as ``spaces.py:73-90``."""
    unit = ("q", "dq", "prev_action")
    err = ("goal_pos_err", "goal_ori_err", "wp_pos_err", "wp_ori_err", "next_wp_pos_err", "next_wp_ori_err")
    sp: dict[str, _Box] = {k: _Box(-1.0, 1.0, (n_joints,)) for k in unit}
    sp.update({k: _Box(-1.0, 1.0, (3,)) for k in err})
    sp.update({"task_type": _Box(0.0, 1.0, (3,)), "mode_flag": _Box(0.0, 1.0, (4,)), "progress": _Box(0.0, 1.0, (3,)),
               "joint_limit_margin": _Box(0.0, 1.0, (n_joints,))})
    return _DictSpace(sp)


class ArmKinematicEnv:
    """Drop-in for the reference's single env: same constructor, ``reset``/``step``/``current_observation`` and ``info``.

    Every call runs the CUDA kernels on a 1-env batch and copies the result to numpy, so it is for conformance
    (the reference's own tests, eval scripts) rather than throughput -- throughput is ``BatchedArmKinematicEnv``.
    Private attributes the reference's evaluators reach into (``_q, _dq, _prev_action, _goal_q, _goal_pose6``,
    AKE users listed in SURVEY 8b) are exposed as numpy properties with setters.
    """

    metadata = {"render_modes": []}

    def __init__(self, config: Phase1EnvConfig | None = None, device: str | torch.device = "cuda") -> None:
        self.config = config or Phase1EnvConfig()
        if len(self.config.joint_specs) != self.config.n_joints:
            raise ValueError("joint_specs length must match n_joints")
        self.action_space = build_action_space(self.config.n_joints)
        self.observation_space = build_observation_space(self.config.n_joints)
        self._b = BatchedArmKinematicEnv(self.config, 1, device, host_sampler=True, with_components=True)
        self._policy_mode_name = self.config.mode_name
        # AKE:86-97: a fresh env sits at q = 0 with goal pose 0 and cached FK(0)
        self._b.reset(options={"initial_q": np.zeros(7), "goal_q": np.zeros(7), "goal_pose6": np.zeros(6), "policy_mode": self._safe_mode()})

    def _safe_mode(self) -> str:
        return self._policy_mode_name if self._policy_mode_name in MODE_INDEX else "approach"

    # --- reference API ---------------------------------------------------------------------------
    def reset(self, *, seed: int | None = None, options: dict[str, Any] | None = None):
        opts = dict(options or {})
        self._policy_mode_name = str(opts.get("policy_mode", self.config.mode_name))
        opts["policy_mode"] = self._policy_mode_name
        obs, _ = self._b.reset(seed=seed, options=opts)
        return self._obs_np(obs), self._info_np(reset=True)

    def step(self, action: Sequence[float]):
        action_arr = np.asarray(action, dtype=float)
        if action_arr.shape != (self.config.n_joints,):
            raise ValueError(f"Expected action shape {(self.config.n_joints,)}, got {action_arr.shape}")
        obs, reward, terminated, truncated, _ = self._b.step(torch.as_tensor(action_arr[None], dtype=torch.float32))
        info = self._info_np(reset=False)
        return self._obs_np(obs), float(reward[0].item()), bool(terminated[0].item()), bool(truncated[0].item()), info

    def current_observation(self) -> dict[str, np.ndarray]:
        return self._obs_np(self._b.current_observation())

    def set_curriculum_stage(self, stage_index: int) -> None:
        self._b.set_curriculum_stage(stage_index)

    def get_curriculum_stage(self) -> int:
        return self._b.get_curriculum_stage()

    def set_policy_mode(self, mode_name: str) -> None:
        self._b.set_policy_mode(mode_name)
        self._policy_mode_name = mode_name

    def apply_dock_training_stage(self, stage_updates: dict[str, Any]) -> None:
        self._b.apply_dock_training_stage(stage_updates)
        self.config = self._b.config

    def render(self) -> None:
        return None

    def close(self) -> None:
        return None

    # --- private state the reference's evaluators touch --------------------------------------------
    def _get(self, t: torch.Tensor) -> np.ndarray:
        return t[0].detach().cpu().numpy().astype(float)

    def _set_rows(self, name: str, value: Sequence[float]) -> None:
        r = _D(name)
        v = torch.as_tensor(np.asarray(value, dtype=np.float32), device=self._b.device)
        self._b.state[r:r + v.numel(), 0] = v

    _q = property(lambda self: self._get(self._b.q), lambda self, v: self._set_rows("KIN_ROW_Q", v))
    _dq = property(lambda self: self._get(self._b.dq), lambda self, v: self._set_rows("KIN_ROW_DQ", v))
    _prev_action = property(lambda self: self._get(self._b.prev_action), lambda self, v: self._set_rows("KIN_ROW_PREV_ACTION", v))
    _goal_q = property(lambda self: self._get(self._b.goal_q), lambda self, v: self._set_rows("KIN_ROW_GOAL_Q", v))
    _goal_pose6 = property(lambda self: self._get(self._b.goal_pose6), lambda self, v: self._set_rows("KIN_ROW_GOAL_POSE", v))
    _ee_pose6 = property(lambda self: self._get(self._b.ee_pose6))

    def _capture_entry_metrics(self) -> None:
        """AKE:425-430 after a caller rewrote the goal in place (route_sequence_env.py:253-257)."""
        st = self._b.state[:, 0].detach().cpu().numpy().astype(float)
        ee, goal = st[_D("KIN_ROW_EE_POSE"):][:6], st[_D("KIN_ROW_GOAL_POSE"):][:6]
        pos = goal[:3] - ee[:3]
        ori = (goal[3:] - ee[3:] + np.pi) % (2 * np.pi) - np.pi
        pa, dq = st[_D("KIN_ROW_PREV_ACTION"):][:7], st[_D("KIN_ROW_DQ"):][:7]
        self._set_rows("KIN_ROW_ENTRY", [np.linalg.norm(pos), np.linalg.norm(ori), np.linalg.norm(pa), np.linalg.norm(dq)])

    # --- conversions -------------------------------------------------------------------------------
    @staticmethod
    def _obs_np(obs: torch.Tensor) -> dict[str, np.ndarray]:
        flat = obs[0].detach().cpu().numpy().astype(np.float32)
        return {k: flat[OBS_SLICES[k]].copy() for k in OBS_KEYS}

    def _info_np(self, *, reset: bool) -> dict[str, Any]:
        b = self._b
        st = b.state[:, 0].detach().cpu().numpy()
        f = lambda name, n: st[_D(name):_D(name) + n].astype(float)  # noqa: E731
        goal, ee, q = f("KIN_ROW_GOAL_POSE", 6), f("KIN_ROW_EE_POSE", 6), f("KIN_ROW_Q", 7)
        pos_vec = goal[:3] - ee[:3]
        ori_vec = (goal[3:] - ee[3:] + np.pi) % (2 * np.pi) - np.pi
        words = st.view(np.uint32)
        c0, c1, fl = int(words[_D("KIN_ROW_CNT0")]), int(words[_D("KIN_ROW_CNT1")]), int(words[_D("KIN_ROW_FLAGS")])
        entry = f("KIN_ROW_ENTRY", 4)
        specs = self.config.joint_specs
        lo, hi = np.array([s.lower for s in specs]), np.array([s.upper for s in specs])
        margin = np.clip(2.0 * np.minimum((q - lo) / np.maximum(hi - lo, 1e-9), (hi - q) / np.maximum(hi - lo, 1e-9)), 0.0, 1.0)
        if reset:
            pos_norm, ori_norm = float(entry[0]), float(entry[1])
            done = 0
        else:
            ax = b.aux[:, 0].detach().cpu().numpy().astype(float)
            pos_norm, ori_norm = float(ax[_D("KIN_AUX_POS_ERR")]), float(ax[_D("KIN_AUX_ORI_ERR")])
            done = int(b.done[0].item())
        rc = self.config.reward_config
        gate = bool(rc.use_orientation_gate)
        in_pre = pos_norm <= rc.pre_near_goal_pos_threshold_m and not (gate and ori_norm > rc.near_goal_ori_threshold_rad)
        in_near = pos_norm <= rc.near_goal_pos_threshold_m and not (gate and ori_norm > rc.near_goal_ori_threshold_rad)
        stage = b.get_curriculum_stage()
        cur = self.config.curriculum_config
        info: dict[str, Any] = {
            "goal_pose6": goal, "goal_q": f("KIN_ROW_GOAL_Q", 7), "q": q, "dq": f("KIN_ROW_DQ", 7), "ee_pose6": ee,
            "position_error_norm": pos_norm, "orientation_error_norm": ori_norm, "position_error_vec": pos_vec, "orientation_error_vec": ori_vec,
            "curr_in_pre_near_goal": bool(in_pre) if reset else bool(done & _D("KIN_DONE_PRE_NEAR")),
            "curr_in_near_goal": bool(in_near) if reset else bool(done & _D("KIN_DONE_NEAR")),
            "pre_near_goal_hit": bool(fl & 1), "near_goal_hit": bool(fl & 2), "dwell_count": (c0 >> 16) & 0xFFFF,
            "near_goal_entry_count": c1 & 0xFFFF, "near_goal_drift_count": (c1 >> 16) & 0xFFFF,
            "min_position_error": float(st[_D("KIN_ROW_MIN_POS")]), "entry_position_error_norm": float(entry[0]),
            "entry_orientation_error_norm": float(entry[1]), "entry_action_l2": float(entry[2]), "entry_dq_norm": float(entry[3]),
            "joint_limit_margin_min": float(margin.min()), "success": bool(done & _D("KIN_DONE_SUCCESS")),
            "terminated": bool(done & _D("KIN_DONE_TERMINATED")), "truncated": bool(done & _D("KIN_DONE_TRUNCATED")),
            "reason": "reset" if reset else REASONS[(done >> _D("KIN_DONE_REASON_SHIFT")) & 3], "mode_name": self._policy_mode_name,
            "curriculum_stage_index": int(stage), "step_count": c0 & 0xFFFF,
            "curriculum_stage_name": cur.stages[stage].name if cur.enabled else "random_goal",
        }
        if not reset:
            names = DOCK_COMPONENT_NAMES if self._policy_mode_name == "dock" else APPROACH_COMPONENT_NAMES
            comps = b.components[: len(names), 0].detach().cpu().numpy().astype(float)
            info["reward_components"] = {k: float(v) for k, v in zip(names, comps)}
            info["action_l2"] = float(ax[_D("KIN_AUX_ACTION_L2")])
            info["executed_delta_q_l2"] = float(ax[_D("KIN_AUX_DQ_L2")])
            info["delta_q_change_l2"] = float(ax[_D("KIN_AUX_DQ_CHANGE_L2")])
            info["dock_action_limit"] = float(ax[_D("KIN_AUX_DOCK_LIMIT")])
            info["dock_delta_q_change_limit_scale"] = float(ax[_D("KIN_AUX_DQC_SCALE")])
        return info


__all__ = ["APPROACH_COMPONENT_NAMES", "ArmKinematicEnv", "BatchedArmKinematicEnv", "DOCK_COMPONENT_NAMES", "OBS_DIM", "OBS_KEYS",
           "OBS_SLICES", "ParamsHandle", "build_action_space", "build_observation_space", "obs_dict"]
