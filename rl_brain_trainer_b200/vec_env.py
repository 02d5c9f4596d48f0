"""A stable-baselines3 ``VecEnv`` over the batched GPU env, so the reference's training CLIs run on it unchanged.

The reference builds ``SubprocVecEnv([lambda: ArmKinematicEnv(cfg)] * n)`` and hands it to ``PPO("MultiInputPolicy", env)``
(``kinematic_phase1/train_workspace_expansion.py:180-199``, ``training/train_approach_policy.py:99-114``); its callbacks talk to
the envs through ``training_env.env_method("set_curriculum_stage", i)`` / ``env_method("apply_dock_training_stage", payload)``
(``training/callbacks.py:55,69,151``) and read ``infos[i]["success"]`` on ``dones`` (:73-82).  :class:`KinVecEnv` implements that
protocol -- ``reset / step_async / step_wait / step / close / seed / env_method / get_attr / set_attr / env_is_wrapped`` with
SB3's semantics (auto-reset, ``infos[i]["terminal_observation"]``, ``infos[i]["TimeLimit.truncated"]``) -- on ONE
``BatchedArmKinematicEnv`` (one ``kin_env_step`` launch per step for all envs).  If stable-baselines3 is importable the class
derives from its ``VecEnv`` (and uses gymnasium spaces); otherwise it is a duck-typed stand-in with the same methods, which is
what the tests exercise in this image (SB3 is not installed here, SURVEY 8c).

This adapter is for *compatibility*: SB3's own rollout loop stays on the host (numpy observations, one policy call per step).
The fast path is :class:`rl_brain_trainer_b200.ppo.PPOTrainer` (fused on-device collection and update).

:class:`KinRouteVecEnv` is the same protocol over one auto-reset ``BatchedRouteKinematicEnv`` for the route training CLI
(``kinematic_phase1/train_route_curriculum.py``): ``env_method("set_route_window", ...)`` and the route ``infos`` on ``dones``.
"""

from __future__ import annotations

from typing import Any, Sequence

import numpy as np
import torch

from . import _lib
from .config import Phase1EnvConfig, RouteEnvConfig, RouteSequenceConfig
from .env import OBS_KEYS, OBS_SLICES, BatchedArmKinematicEnv, build_action_space, build_observation_space
from .route import ROUTE_OBS_SLICES, BatchedRouteKinematicEnv, RouteDataset, build_route_observation_space, route_obs_keys

try:  # pragma: no cover - stable-baselines3 / gymnasium are absent from the build image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase
    import gymnasium as _gym

    _HAVE_SB3 = True
except Exception:  # noqa: BLE001
    _VecEnvBase = object
    _gym = None
    _HAVE_SB3 = False

_D = _lib.define
_INFO_SCALARS = ("position_error_norm", "orientation_error_norm", "min_position_error", "action_l2", "executed_delta_q_l2", "delta_q_change_l2")
_REASONS = ("running", "success", "max_steps", "invalid_state")        # termination.py:20-57


def _spaces(obs_shim: Any, n_joints: int):
    """The env's dict observation space (``env._DictSpace`` of ``env._Box``) and the action box, as gymnasium spaces under SB3."""
    if _HAVE_SB3:  # pragma: no cover
        obs = _gym.spaces.Dict({k: _gym.spaces.Box(low=float(np.min(b.low)), high=float(np.max(b.high)), shape=b.shape, dtype=np.float32)
                                for k, b in obs_shim.spaces.items()})
        return obs, _gym.spaces.Box(low=-1.0, high=1.0, shape=(n_joints,), dtype=np.float32)
    return obs_shim, build_action_space(n_joints)


class _KinVecEnvProtocol(_VecEnvBase):
    """What :class:`KinVecEnv` and :class:`KinRouteVecEnv` share: one batched env ``self.env`` with an ``_seed`` and a ``device``,
    SB3's action hand-over (``step_async`` / ``step``) and the attribute / wrapper queries.  Subclasses provide ``reset``,
    ``step_wait`` and ``env_method``."""

    def _init_protocol(self, num_envs: int, obs_space: Any, act_space: Any) -> None:
        if _HAVE_SB3:  # pragma: no cover
            super().__init__(int(num_envs), obs_space, act_space)
        else:
            self.num_envs, self.observation_space, self.action_space = int(num_envs), obs_space, act_space
        self.render_mode = None
        self.metadata = {"render_modes": []}
        self._actions: torch.Tensor | None = None
        self._attrs: dict[str, Any] = {}

    def step_async(self, actions: np.ndarray) -> None:
        a = np.asarray(actions, dtype=np.float32)
        if a.shape != (self.num_envs, 7):
            raise ValueError(f"Expected action shape {(self.num_envs, 7)}, got {a.shape}")
        self._actions = torch.as_tensor(a, device=self.env.device)

    def _take_actions(self) -> torch.Tensor:
        if self._actions is None:
            raise RuntimeError("step_wait() without step_async()")
        a, self._actions = self._actions, None
        return a

    def step(self, actions: np.ndarray):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        self.env.close()

    def seed(self, seed: int | None = None) -> list[int | None]:
        if seed is not None:
            self.env._seed = int(seed)
        return [None if seed is None else int(seed) + i for i in range(self.num_envs)]

    def _indices(self, indices: Any) -> list[int]:
        if indices is None:
            return list(range(self.num_envs))
        return [int(indices)] if isinstance(indices, (int, np.integer)) else [int(i) for i in indices]

    def get_attr(self, attr_name: str, indices: Any = None) -> list[Any]:
        n = len(self._indices(indices))
        if attr_name in self._attrs:
            return [self._attrs[attr_name]] * n
        if attr_name in ("config", "metadata", "render_mode", "action_space", "observation_space"):
            return [getattr(self.env, attr_name, getattr(self, attr_name, None))] * n
        raise AttributeError(attr_name)

    def set_attr(self, attr_name: str, value: Any, indices: Any = None) -> None:
        self._attrs[attr_name] = value

    def env_is_wrapped(self, wrapper_class: Any, indices: Any = None) -> list[bool]:
        return [False] * len(self._indices(indices))

    def get_images(self) -> list[None]:
        return [None] * self.num_envs

    def render(self, mode: str | None = None) -> None:
        return None


class KinVecEnv(_KinVecEnvProtocol):
    """``num_envs`` kinematic envs behind SB3's ``VecEnv`` interface (see the module docstring)."""

    def __init__(self, config: Phase1EnvConfig | None = None, num_envs: int = 1, device: str | torch.device = "cuda", *, seed: int = 0,
                 stage_index: int = 0, handoff_states: torch.Tensor | None = None, info_keys: Sequence[str] = _INFO_SCALARS,
                 graph_step: bool = False) -> None:
        self.env = BatchedArmKinematicEnv(config, num_envs, device, auto_reset=True, seed=seed, host_sampler=False, with_aux=True,
                                          graph_step=graph_step)
        self.env.set_curriculum_stage(stage_index)
        if handoff_states is not None:
            self.env.set_handoff_states(handoff_states)
        n_joints = self.env.config.n_joints
        self._init_protocol(num_envs, *_spaces(build_observation_space(n_joints), n_joints))
        self._info_keys = tuple(info_keys)

    # ------------------------------------------------------------------ VecEnv protocol
    def _obs_dict(self, flat: np.ndarray) -> dict[str, np.ndarray]:
        return {k: np.ascontiguousarray(flat[:, OBS_SLICES[k]]) for k in OBS_KEYS}

    def reset(self) -> dict[str, np.ndarray]:
        obs, _ = self.env.reset()
        return self._obs_dict(obs.cpu().numpy())

    def step_wait(self) -> tuple[dict[str, np.ndarray], np.ndarray, np.ndarray, list[dict[str, Any]]]:
        obs, reward, terminated, truncated, info = self.env.step(self._take_actions())
        flat = obs.cpu().numpy()
        term, trunc = terminated.cpu().numpy(), truncated.cpu().numpy()
        dones = term | trunc
        host = {k: info[k].cpu().numpy() for k in self._info_keys if k in info}
        success, reason, stage = info["success"].cpu().numpy(), info["reason_code"].cpu().numpy(), info["stage"].cpu().numpy()
        terminal = info["terminal_observation"].cpu().numpy() if dones.any() else None
        infos: list[dict[str, Any]] = []
        for i in range(self.num_envs):
            d: dict[str, Any] = {k: float(v[i]) for k, v in host.items()}
            d["success"] = bool(success[i])
            d["reason"] = _REASONS[int(reason[i])]
            d["curriculum_stage"] = int(stage[i])
            d["TimeLimit.truncated"] = bool(trunc[i] and not term[i])
            if dones[i]:
                d["terminal_observation"] = {k: terminal[i, OBS_SLICES[k]].copy() for k in OBS_KEYS}
            infos.append(d)
        return self._obs_dict(flat), reward.cpu().numpy().astype(np.float32), dones, infos

    def env_method(self, method_name: str, *method_args: Any, indices: Any = None, **method_kwargs: Any) -> list[Any]:
        """The calls the reference's callbacks make; they address all envs at once (one shared device config / sampler)."""
        n = len(self._indices(indices))
        if method_name in ("set_curriculum_stage", "get_curriculum_stage", "set_policy_mode", "apply_dock_training_stage", "current_observation"):
            out = getattr(self.env, method_name)(*method_args, **method_kwargs)
            if method_name == "current_observation":
                flat = out.cpu().numpy()
                return [{k: flat[i, OBS_SLICES[k]].copy() for k in OBS_KEYS} for i in self._indices(indices)]
            return [out] * n
        raise AttributeError(f"KinVecEnv.env_method: '{method_name}' is not part of the kinematic env's interface")


def make_vec_env(config: Phase1EnvConfig, n_envs: int, *, seed: int = 0, device: str | torch.device = "cuda", **kwargs: Any) -> KinVecEnv:
    """Drop-in for the reference's ``_make_env`` + ``SubprocVecEnv`` construction (train_workspace_expansion.py:176-183)."""
    return KinVecEnv(config, n_envs, device, seed=seed, **kwargs)


class KinRouteVecEnv(_KinVecEnvProtocol):
    """``num_envs`` route envs -- ``RouteKinematicEnv``, or ``RouteSequenceKinematicEnv`` when ``sequence_config.enabled`` -- behind SB3's
    ``VecEnv`` interface, on ONE auto-reset ``BatchedRouteKinematicEnv`` (one ``kin_route_step_autoreset`` launch per step).

    This is the env ``train_route_curriculum.py`` builds with ``SubprocVecEnv``: the observations are the route wrappers' dicts (the
    four route keys only when ``config.observation_config.include_route_keys``), ``infos[i]`` carries the keys its
    ``RoutePrefixCurriculumCallback`` reads on ``dones`` (``success``, ``route_ready``, ``route_orientation_hit``, ``route_regression``,
    ...) for the step that ended the episode, and ``env_method("set_route_window", max_route_index=, min_route_index=)`` moves the
    waypoint window the following auto-resets draw from.  Resets draw from the device sampler (Philox), not the numpy stream."""

    def __init__(self, route: RouteDataset, config: RouteEnvConfig, num_envs: int = 1, device: str | torch.device = "cuda", *,
                 sequence_config: RouteSequenceConfig | None = None, seed: int = 0, graph_step: bool = False) -> None:
        self.env = BatchedRouteKinematicEnv(route, config, num_envs, device, sequence_config=sequence_config, auto_reset=True, seed=seed,
                                            graph_step=graph_step)
        self._keys = route_obs_keys(config.observation_config.include_route_keys)
        n_joints = config.base_env_config.n_joints
        self._init_protocol(num_envs, *_spaces(build_route_observation_space(n_joints, config.observation_config.include_route_keys), n_joints))

    def _obs_dict(self, flat: np.ndarray) -> dict[str, np.ndarray]:
        return {k: np.ascontiguousarray(flat[:, ROUTE_OBS_SLICES[k]]) for k in self._keys}

    def reset(self) -> dict[str, np.ndarray]:
        return self._obs_dict(self.env.reset().cpu().numpy())

    def step_wait(self) -> tuple[dict[str, np.ndarray], np.ndarray, np.ndarray, list[dict[str, Any]]]:
        obs, reward, _, _, _ = self.env.step(self._take_actions())
        n, D = self.num_envs, _D
        flat, rew, done = obs.cpu().numpy(), reward.cpu().numpy().astype(np.float32), self.env.done.cpu().numpy()
        raux = self.env.raux[:, :n].cpu().numpy()
        term, trunc = (done & D("KIN_DONE_TERMINATED")) != 0, (done & D("KIN_DONE_TRUNCATED")) != 0
        success = (done & D("KIN_DONE_SUCCESS")) != 0
        dones = term | trunc
        words = raux.view(np.int32)
        flags, index = words[D("KIN_RAUX_FLAGS")], words[D("KIN_RAUX_ROUTE_INDEX")]
        streak, completed = words[D("KIN_RAUX_STREAK")], words[D("KIN_RAUX_COMPLETED")]
        q_err, pos, ori = raux[D("KIN_RAUX_Q_ERR")], raux[D("KIN_RAUX_POS_ERR")], raux[D("KIN_RAUX_ORI_ERR")]
        sequence = self.env.sequence is not None
        terminal = self.env.terminal_obs.cpu().numpy() if dones.any() else None
        infos: list[dict[str, Any]] = []
        for i in range(n):
            d: dict[str, Any] = {
                "success": bool(success[i]), "route_ready": bool(flags[i] & 1), "route_ready_streak": int(streak[i]),
                "route_q_error_norm": float(q_err[i]), "route_orientation_hit": bool(flags[i] & 4), "route_regression": bool(flags[i] & 2),
                "route_index": int(index[i]), "position_error_norm": float(pos[i]), "orientation_error_norm": float(ori[i]),
                "TimeLimit.truncated": bool(trunc[i] and not term[i]),
            }
            if sequence:
                d["route_waypoint_success"] = bool(flags[i] & 8)
                d["route_completed_waypoints"] = int(completed[i])
            if dones[i]:
                d["terminal_observation"] = {k: terminal[i, ROUTE_OBS_SLICES[k]].copy() for k in self._keys}
            infos.append(d)
        return self._obs_dict(flat), rew, dones, infos

    def env_method(self, method_name: str, *method_args: Any, indices: Any = None, **method_kwargs: Any) -> list[Any]:
        """``set_route_window`` (the call of ``RoutePrefixCurriculumCallback``); it addresses all envs at once (one shared window)."""
        n = len(self._indices(indices))
        if method_name == "set_route_window":
            return [self.env.set_route_window(*method_args, **method_kwargs)] * n
        raise AttributeError(f"KinRouteVecEnv.env_method: '{method_name}' is not part of the route env's interface")


def make_route_vec_env(route: RouteDataset, config: RouteEnvConfig, n_envs: int, *, sequence_config: RouteSequenceConfig | None = None,
                       seed: int = 0, device: str | torch.device = "cuda", **kwargs: Any) -> KinRouteVecEnv:
    """Drop-in for the ``SubprocVecEnv`` of route wrappers that train_route_curriculum.py builds."""
    return KinRouteVecEnv(route, config, n_envs, device, sequence_config=sequence_config, seed=seed, **kwargs)
