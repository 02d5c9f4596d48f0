"""Dense holder-route wrappers on the GPU: route dataset, batched Route(Sequence)KinematicEnv, sequential probe.

Mirrors ``kinematic_phase1/route/route_dataset.py:16-99``, ``route/route_env.py:27-212``,
``route/route_sequence_env.py:29-278`` and ``eval/eval_route_curriculum.py:55-246``.  The 483-waypoint route file of
the reference (``tray1_holder1_to_8_route_q_dense.json``) is not in its snapshot (SURVEY F9): ``load_route_dataset``
reads that JSON format when a user supplies the file, ``synthetic_route`` builds a seeded stand-in with similar
statistics for tests and benchmarks.
"""

from __future__ import annotations

import ctypes
import json
from dataclasses import dataclass
from pathlib import Path
from typing import Any, Sequence

import numpy as np
import torch

from . import _lib, kinematics
from .config import RouteEnvConfig, RouteSequenceConfig
from .env import LazyInfo, ParamsHandle, _D, _ptr, _stream
from .policy import PolicyWeights

ROUTE_OBS_DIM = 80
ROUTE_OBS_SLICES: dict[str, slice] = {
    "dq": slice(0, 7), "goal_ori_err": slice(7, 10), "goal_pos_err": slice(10, 13), "joint_limit_margin": slice(13, 20),
    "mode_flag": slice(20, 24), "next_wp_ori_err": slice(24, 27), "next_wp_pos_err": slice(27, 30), "prev_action": slice(30, 37),
    "progress": slice(37, 40), "q": slice(40, 47), "route_q_error": slice(47, 54), "route_q_goal": slice(54, 61),
    "route_scalar": slice(61, 64), "route_tangent": slice(64, 71), "task_type": slice(71, 74), "wp_ori_err": slice(74, 77),
    "wp_pos_err": slice(77, 80),
}


def default_chunk_bounds(max_index: int) -> tuple[tuple[int, int], ...]:
    """route_dataset.py:60-70."""
    edges = ((1, 40), (41, 80), (81, 120), (121, 180), (181, 260), (261, 360))
    return tuple((lo, min(hi, max_index)) for lo, hi in edges) + ((361, max_index),)


@dataclass
class RouteDataset:
    """Waypoint table: ``q_goal [n,7]``, FK ``pose6 [n,6]``, ``next_q_delta [n,7]``, cumulative EE path ``progress_m [n]``, chunk ids."""

    q_goal: np.ndarray
    pose6: np.ndarray
    next_q_delta: np.ndarray
    progress_m: np.ndarray
    chunk_id: np.ndarray
    path: Path | None = None

    def __len__(self) -> int:
        return int(self.q_goal.shape[0])

    @classmethod
    def from_q(cls, q_goals: np.ndarray, path: Path | None = None, chunk_bounds: Sequence[tuple[int, int]] | None = None) -> "RouteDataset":
        q = np.asarray(q_goals, dtype=float).reshape(-1, 7)
        if q.shape[0] < 1:
            raise ValueError("Route dataset must contain a non-empty list")
        pose = np.array([kinematics.fk_pose6_folded(x) for x in q])
        steps = np.linalg.norm(np.diff(pose[:, :3], axis=0), axis=1) if len(q) > 1 else np.zeros(0)
        progress = np.concatenate([[0.0], np.cumsum(steps)])
        nxt = q[np.minimum(np.arange(len(q)) + 1, len(q) - 1)] - q
        bounds = tuple(chunk_bounds) if chunk_bounds is not None else default_chunk_bounds(len(q) - 1)
        chunk = np.full(len(q), len(bounds) - 1, dtype=np.int64)
        for i in range(len(q)):
            for c, (lo, hi) in enumerate(bounds):
                if lo <= i <= hi:
                    chunk[i] = c
                    break
        return cls(q_goal=q, pose6=pose, next_q_delta=nxt, progress_m=progress, chunk_id=chunk, path=path)


def load_route_dataset(path: str | Path, *, chunk_bounds: Sequence[tuple[int, int]] | None = None) -> RouteDataset:
    """Reference JSON format: ``{"route_q": [...]}`` or a bare list; entries are 7-vectors or dicts with ``q`` / ``q_goal``."""
    p = Path(path)
    payload = json.loads(p.read_text(encoding="utf-8"))
    entries = payload.get("route_q") if isinstance(payload, dict) else payload
    if not isinstance(entries, list) or not entries:
        raise ValueError(f"Route dataset must contain a non-empty list: {p}")

    def q_of(e: Any) -> Any:
        if isinstance(e, dict):
            return e["q"] if "q" in e else e["q_goal"]
        return e

    return RouteDataset.from_q(np.asarray([q_of(e) for e in entries], dtype=float), path=p, chunk_bounds=chunk_bounds)


def synthetic_route(n_waypoints: int = 483, *, seed: int = 7, n_knots: int = 9, knot_sigma: float = 0.22, target_spacing_m: float = 0.012) -> RouteDataset:
    """Seeded dense q-route: smooth-step interpolation through random-walk joint knots inside the Stage-<=8 envelope.

    The knot spread is rescaled so the mean EE spacing is ~``target_spacing_m`` (the reference route: 483 waypoints, ~5.8 m).
    """
    rng = np.random.default_rng(seed)
    knots = np.cumsum(rng.normal(0.0, knot_sigma, size=(n_knots, 7)), axis=0) * np.array([0.2, 1, 1, 1, 1, 1, 1])
    knots = np.clip(knots, [-0.30, -1.2, -1.2, -1.2, -1.0, -1.0, -1.0], [0.30, 1.2, 1.2, 1.2, 1.0, 1.0, 1.0])

    def sample(k: np.ndarray) -> np.ndarray:
        t = np.linspace(0, len(k) - 1, n_waypoints)
        i0 = np.clip(np.floor(t).astype(int), 0, len(k) - 2)
        w = (t - i0)[:, None]
        w = w * w * (3 - 2 * w)
        return k[i0] * (1 - w) + k[i0 + 1] * w

    ds = RouteDataset.from_q(sample(knots))
    spacing = ds.progress_m[-1] / max(n_waypoints - 1, 1)
    if spacing > 0:
        ds = RouteDataset.from_q(sample(knots * min(target_spacing_m / spacing, 1.0)))
    return ds


class DeviceRoute:
    """Route table resident on one GPU + the ``KinRouteTable`` view."""

    def __init__(self, route: RouteDataset, device: str | torch.device = "cuda") -> None:
        self.route = route
        self.device = torch.device(device)
        f = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(self.device)  # noqa: E731
        self.q, self.pose, self.tan, self.prog = f(route.q_goal), f(route.pose6), f(route.next_q_delta), f(route.progress_m)
        t = _lib.c_struct("KinRouteTable")()
        t.n_waypoints = len(route)
        t.q_goal, t.pose6, t.next_q_delta, t.progress_m = self.q.data_ptr(), self.pose.data_ptr(), self.tan.data_ptr(), self.prog.data_ptr()
        # pruning bounds of the nearest-waypoint scan: a property of the route, computed once per RouteDataset object
        lb = getattr(route, "_nearest_lb_cache", None)
        if lb is None:
            lb = nearest_scan_bounds(route.q_goal)
            try:
                object.__setattr__(route, "_nearest_lb_cache", lb)
            except (AttributeError, TypeError):
                pass
        self.nearest_lb = f(lb)
        t.nearest_lb, t.nearest_lb_k = self.nearest_lb.data_ptr(), int(self.nearest_lb.shape[1])
        self.c = t


def nearest_scan_bounds(q_goal: np.ndarray, k_max: int = 64) -> np.ndarray:
    """``KinRouteTable.nearest_lb``: ``lb[i, k] = min_{|j - i| >= k} |q_goal[j] - q_goal[i]|`` (``+inf`` where no such j), fp64 -> fp32
    rounded DOWN.  The route reward's off-route term scans the whole route for the nearest waypoint every step (route_env.py:135); with
    these bounds the step kernel walks outward from the env's current target and stops when the triangle inequality
    ``|q_j - q| >= |q_j - q_i| - |q_i - q|`` excludes everything further along -- the same minimum from ~10 candidates instead of 483."""
    q = np.asarray(q_goal, dtype=np.float64)
    n = q.shape[0]
    k_max = int(min(k_max, max(n, 2)))
    d = np.linalg.norm(q[:, None, :] - q[None, :, :], axis=2)
    off = np.abs(np.arange(n)[:, None] - np.arange(n)[None, :])
    lb = np.full((n, k_max), np.inf)
    # min over offsets >= k  =  min(min over offsets >= k + 1, the two waypoints at offset exactly k): one masked pass for the last
    # column, then a backwards sweep over the diagonals (min is exact, so this equals the masked minimum per column)
    lb[:, k_max - 1] = np.where(off >= k_max - 1, d, np.inf).min(axis=1)
    idx = np.arange(n)
    for k in range(k_max - 2, -1, -1):
        at_k = np.full(n, np.inf)
        lo, hi = idx - k, idx + k
        at_k[lo >= 0] = d[idx[lo >= 0], lo[lo >= 0]]
        at_k[hi < n] = np.minimum(at_k[hi < n], d[idx[hi < n], hi[hi < n]])
        lb[:, k] = np.minimum(lb[:, k + 1], at_k)
    lb32 = lb.astype(np.float32)
    lb32 = np.where(lb32.astype(np.float64) > lb, np.nextafter(lb32, np.float32(-np.inf)), lb32)
    return lb32


class BatchedRouteKinematicEnv:
    """``num_envs`` route replicas: ``RouteKinematicEnv`` (sequence disabled) or ``RouteSequenceKinematicEnv`` semantics.

    ``reset(route_index=[M], start_route_index=None, initial_q=None, ...)`` -> obs [N,80]
    ``step(actions [N,7])`` -> (obs [N,80], reward [N], terminated, truncated, info) with the route info keys.
    """

    def __init__(self, route: RouteDataset, config: RouteEnvConfig, num_envs: int, device: str | torch.device = "cuda", *,
                 sequence_config: RouteSequenceConfig | None = None, with_components: bool = False, auto_reset: bool = False, seed: int = 0,
                 graph_step: bool = False) -> None:
        if not torch.cuda.is_available():
            raise _lib.KinError("BatchedRouteKinematicEnv needs a CUDA device; there is no CPU fallback")
        self.config, self.route = config, route
        self.sequence = sequence_config if (sequence_config is not None and sequence_config.enabled) else None
        self.device = torch.device(device)
        self.num_envs = int(num_envs)
        # auto_reset: a slot whose episode ends is re-seeded inside the step launch (kin_route_step_autoreset) with the draw
        # reset_done(seed=seed, counter=<episodes the slot has finished>) would make; terminal_obs keeps the last observation.
        # graph_step: step() replays a CUDA graph of [step kernel, the two done-bit ops], re-captured when the params handle, the
        # reset window, the seed or the sequence flag changes (as BatchedArmKinematicEnv does).
        self.auto_reset, self._seed, self.graph_step = bool(auto_reset), int(seed), bool(graph_step)
        self._graph: Any = None
        self._graph_key: Any = None
        self._step_calls = 0
        self.stride = (self.num_envs + 31) // 32 * 32
        self._L = _lib.lib()
        with torch.cuda.device(self.device):
            self._params = ParamsHandle(config.base_env_config, config.reward_config)
            self.table = DeviceRoute(route, self.device)
            self.state = torch.zeros((_D("KIN_STATE_ROWS"), self.stride), dtype=torch.float32, device=self.device)
            self.obs = torch.zeros((self.num_envs, ROUTE_OBS_DIM), dtype=torch.float32, device=self.device)
            self.reward = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
            self.done = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
            self.raux = torch.zeros((_D("KIN_RAUX_ROWS"), self.stride), dtype=torch.float32, device=self.device)
            self.rcomp = torch.zeros((17, self.stride), dtype=torch.float32, device=self.device) if with_components else None
            self.terminal_obs = torch.zeros_like(self.obs) if self.auto_reset else None

    def set_route_window(self, *, max_route_index: int, min_route_index: int = 1) -> None:
        """``RouteKinematicEnv.set_route_window`` (route_env.py:99-121): the waypoint range sampled resets draw from."""
        import dataclasses

        self.config = dataclasses.replace(self.config, reset_config=dataclasses.replace(self.config.reset_config, min_route_index=int(min_route_index),
                                                                                         max_route_index=int(max_route_index)))

    def reset(self, *, route_index: Any = None, start_route_index: Any = None, initial_q: Any = None, initial_dq: Any = None,
              initial_prev_action: Any = None, env_ids: Any = None, seed: int | None = None) -> torch.Tensor:
        ids = None if env_ids is None else torch.as_tensor(env_ids, dtype=torch.int32, device=self.device).contiguous()
        m = self.num_envs if ids is None else int(ids.numel())
        self.last_reset: dict[str, torch.Tensor] | None = None
        if route_index is None and self.auto_reset:
            # the draws the in-step resets continue: counter 0 here, then 1, 2, ... per slot (state row KIN_ROW_EPISODE)
            if seed is not None:
                self._seed = int(seed)
            mask = None
            if ids is not None:
                mask = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
                mask[ids.long()] = _D("KIN_DONE_TERMINATED")
            with torch.cuda.device(self.device):
                _lib.check(self._L.kin_route_reset_sampled(self._params.handle, ctypes.byref(self.table.c), ctypes.byref(self._reset_params()),
                                                           _ptr(self.state), self.stride, self.num_envs, _ptr(mask), self._seed, 0, _ptr(self.obs),
                                                           _stream()))
                episode = self.state[_D("KIN_ROW_EPISODE"), :self.num_envs]
                if ids is None:
                    episode.zero_()
                else:
                    episode[ids.long()] = 0.0
            return self.obs
        if route_index is None:      # route_env.py:60-73: no explicit waypoint -> sample_route_reset
            if seed is not None or not hasattr(self, "_gen"):
                self._gen = torch.Generator(device=self.device)
                self._gen.manual_seed(0 if seed is None else int(seed))
            smp = sample_route_reset_batch(self.table, self.config.base_env_config.joint_specs, self.config.reset_config, m, self._gen)
            route_index, start_route_index = smp["route_index"], smp["start_route_index"]
            initial_q, initial_dq, initial_prev_action = smp["initial_q"], smp["initial_dq"], smp["initial_prev_action"]
            self.last_reset = smp
        ri = torch.as_tensor(route_index, dtype=torch.int32, device=self.device).reshape(-1)
        if ri.numel() == 1 and m > 1:
            ri = ri.expand(m)
        ri = ri.contiguous()
        last = None
        if self.sequence is not None:  # route_sequence_env.py:120-124
            max_index = min(self.config.reset_config.max_route_index, len(self.route) - 1)
            ri = ri.clamp(1, max_index).contiguous()
            last = torch.clamp(ri + max(int(self.sequence.sequence_length), 1) - 1, max=max_index).to(torch.int32).contiguous()
        st = None if start_route_index is None else torch.as_tensor(start_route_index, dtype=torch.int32, device=self.device).reshape(-1).expand(m).contiguous()
        f = lambda x: None if x is None else torch.as_tensor(x, dtype=torch.float32, device=self.device).reshape(-1, 7).expand(m, 7).contiguous()  # noqa: E731
        iq, idq, ipa = f(initial_q), f(initial_dq), f(initial_prev_action)
        out = self.obs if ids is None else torch.empty((m, ROUTE_OBS_DIM), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._L.kin_route_reset(self._params.handle, ctypes.byref(self.table.c), _ptr(self.state), self.stride, self.num_envs,
                                               _ptr(ids), m, _ptr(ri), _ptr(st), _ptr(last), _ptr(iq), _ptr(idq), _ptr(ipa), _ptr(out), _stream()))
        if ids is not None:
            self.obs[ids.long()] = out
        return self.obs

    def _reset_params(self) -> Any:
        """``KinRouteResetParams`` of the current reset config / route window (rebuilt after ``set_route_window``)."""
        cfg = self.config.reset_config
        key = (cfg, self.sequence is not None)
        if getattr(self, "_reset_params_key", None) != key:
            c = _lib.c_struct("KinRouteResetParams")()
            max_index = len(self.route) - 1
            cdf = np.cumsum(_reset_mode_ratios(cfg))
            cdf[-1] = 1.0
            rng_tab = _reset_index_ranges(cfg, max_index)
            c.forced_mode = int(_FORCED_MODE.get(cfg.mode, -1))
            for m in range(5):
                lo_m, hi_m = int(rng_tab[m, 0]), int(rng_tab[m, 1])
                if hi_m < lo_m:       # a segment / replay range that starts beyond the current prefix window: the reference's
                    lo_m = hi_m       # rng.integers would raise when that mode is drawn; like sample_route_reset_batch, pin the
                                      # target to the window's upper end instead
                c.mode_cdf[m] = float(cdf[m])
                c.index_lo[m], c.index_hi[m] = lo_m, hi_m
            c.q_noise_std, c.dq_noise_std, c.prev_action_noise_std = float(cfg.q_noise_std), float(cfg.dq_noise_std), float(cfg.prev_action_noise_std)
            c.sequence_length = max(int(self.sequence.sequence_length), 1) if self.sequence is not None else 0
            c.max_route_index = int(min(cfg.max_route_index, max_index))
            self._reset_params_c, self._reset_params_key = c, key
        return self._reset_params_c

    def refresh_observation(self) -> torch.Tensor:
        """Recompute ``self.obs`` from the device state (after the state was written from outside, e.g. a route index override)."""
        n = self.num_envs
        ri = (self.state[_D("KIN_ROW_ROUTE"), :n].view(torch.int32) & 0xFFFF).to(torch.int32)
        r2 = self.state[_D("KIN_ROW_ROUTE2"), :n].view(torch.int32)
        streak = (self.state[_D("KIN_ROW_ROUTE"), :n].view(torch.int32) >> 16) & 0xFFFF
        q = self.state[_D("KIN_ROW_Q"):_D("KIN_ROW_Q") + 7, :n].t().contiguous()
        dq = self.state[_D("KIN_ROW_DQ"):_D("KIN_ROW_DQ") + 7, :n].t().contiguous()
        pa = self.state[_D("KIN_ROW_PREV_ACTION"):_D("KIN_ROW_PREV_ACTION") + 7, :n].t().contiguous()
        keep = self.state[[_D("KIN_ROW_MIN_POS"), _D("KIN_ROW_CNT0"), _D("KIN_ROW_CNT1"), _D("KIN_ROW_FLAGS")], :n].clone()
        last = (r2 & 0xFFFF).to(torch.int32).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self._L.kin_route_reset(self._params.handle, ctypes.byref(self.table.c), _ptr(self.state), self.stride, n, None, n,
                                               _ptr(ri.contiguous()), None, _ptr(last), _ptr(q), _ptr(dq), _ptr(pa), _ptr(self.obs), _stream()))
        # the reset kernel re-derives the cached pose / entry metrics; the episode counters and the bookkeeping words are put back
        self.state[[_D("KIN_ROW_MIN_POS"), _D("KIN_ROW_CNT0"), _D("KIN_ROW_CNT1"), _D("KIN_ROW_FLAGS")], :n] = keep
        self.state[_D("KIN_ROW_ROUTE"), :n] = (ri | (streak << 16)).to(torch.int32).view(torch.float32)
        self.state[_D("KIN_ROW_ROUTE2"), :n] = r2.view(torch.float32)
        return self.obs

    def reset_done(self, *, seed: int, counter: int, done: torch.Tensor | None = None) -> torch.Tensor:
        """The route env's auto-reset in one launch (``kin_route_reset_sampled``): every slot whose ``done`` byte (default: the last
        step's) says terminated / truncated draws a fresh ``sample_route_reset`` start on the device (Philox(seed, env, counter));
        state and observation rows of the other slots are untouched.  No host round trip."""
        d = self.done if done is None else done
        with torch.cuda.device(self.device):
            _lib.check(self._L.kin_route_reset_sampled(self._params.handle, ctypes.byref(self.table.c), ctypes.byref(self._reset_params()), _ptr(self.state),
                                                       self.stride, self.num_envs, _ptr(d), int(seed), int(counter) & 0xFFFFFFFF, _ptr(self.obs), _stream()))
        return self.obs

    def _launch(self, actions: int) -> None:
        """One step launch on the current stream: ``kin_route_step``, or ``kin_route_step_autoreset`` for an auto-reset env."""
        seq = self.sequence is not None
        streak = int(bool(self.sequence.reset_ready_streak_on_advance)) if seq else 1
        if self.auto_reset:
            _lib.check(self._L.kin_route_step_autoreset(self._params.handle, ctypes.byref(self.table.c), ctypes.byref(self._reset_params()),
                                                        _ptr(self.state), self.stride, self.num_envs, actions, _ptr(self.obs), _ptr(self.reward),
                                                        _ptr(self.done), _ptr(self.raux), _ptr(self.rcomp), int(seq), streak, self._seed,
                                                        _ptr(self.terminal_obs), _stream()))
        else:
            _lib.check(self._L.kin_route_step(self._params.handle, ctypes.byref(self.table.c), _ptr(self.state), self.stride, self.num_envs,
                                              actions, _ptr(self.obs), _ptr(self.reward), _ptr(self.done), _ptr(self.raux), _ptr(self.rcomp),
                                              int(seq), streak, _stream()))

    def step_raw(self, actions: torch.Tensor) -> None:
        """One step launch with no host-side post-processing: results land in ``self.obs / reward / done / raux`` (which
        a rollout loop may point at slices of its own buffers).  ``actions``: contiguous float32 ``[num_envs, 7]`` on this device."""
        self._launch(actions.data_ptr())

    def step(self, actions: torch.Tensor):
        a = torch.as_tensor(actions, dtype=torch.float32, device=self.device)
        if a.shape != (self.num_envs, 7):
            raise ValueError(f"Expected action shape {(self.num_envs, 7)}, got {tuple(a.shape)}")
        a = a.contiguous()
        self._step_calls += 1
        masks = getattr(self, "_done_masks", None)
        if masks is None:
            masks = self._done_masks = torch.tensor([[_D("KIN_DONE_TERMINATED")], [_D("KIN_DONE_TRUNCATED")]], dtype=self.done.dtype, device=self.device)
        if self.graph_step and self._step_calls > 1:       # (the first call runs eagerly: the smem attribute is set there)
            if self.auto_reset:
                self._reset_params()
            key = (id(self._params), self._reset_params_key if self.auto_reset else None, self._seed, self.sequence is not None)
            if self._graph is None or self._graph_key != key:
                self._g_act = torch.empty_like(a)
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.device(self.device), torch.cuda.graph(g):
                    self._launch(self._g_act.data_ptr())
                    self._g_tt = (self.done.unsqueeze(0) & masks) != 0
                self._graph, self._graph_key = g, key
            self._g_act.copy_(a, non_blocking=True)
            self._graph.replay()
            tt = self._g_tt
        else:
            with torch.cuda.device(self.device):
                self._launch(a.data_ptr())
            tt = (self.done.unsqueeze(0) & masks) != 0
        d = self.done
        n = self.num_envs
        raux, st = self.raux, self.state
        flags = lambda: raux[_D("KIN_RAUX_FLAGS"), :n].view(torch.int32)  # noqa: E731
        thunks = {      # decoded lazily (env.LazyInfo): step() = the kernel launch + the two done-bit tests
            "success": lambda: (d & _D("KIN_DONE_SUCCESS")) != 0, "route_ready": lambda: (flags() & 1) != 0,
            "route_regression": lambda: (flags() & 2) != 0, "route_orientation_hit": lambda: (flags() & 4) != 0,
            "route_waypoint_success": lambda: (flags() & 8) != 0,
            "route_ready_streak": lambda: raux[_D("KIN_RAUX_STREAK"), :n].view(torch.int32),
            "route_index": lambda: raux[_D("KIN_RAUX_ROUTE_INDEX"), :n].view(torch.int32),
            "route_completed_waypoints": lambda: raux[_D("KIN_RAUX_COMPLETED"), :n].view(torch.int32),
            "route_q_error_norm": lambda: raux[_D("KIN_RAUX_Q_ERR"), :n], "nearest_route_q_distance": lambda: raux[_D("KIN_RAUX_NEAREST"), :n],
            "position_error_norm": lambda: raux[_D("KIN_RAUX_POS_ERR"), :n], "orientation_error_norm": lambda: raux[_D("KIN_RAUX_ORI_ERR"), :n],
            "q": lambda: st[_D("KIN_ROW_Q"):_D("KIN_ROW_Q") + 7, :n].t(), "dq": lambda: st[_D("KIN_ROW_DQ"):_D("KIN_ROW_DQ") + 7, :n].t(),
        }
        if self.rcomp is not None:
            thunks["reward_components"] = lambda: self.rcomp[:, :n]
        if self.auto_reset:
            thunks["auto_reset"] = lambda: (d & _D("KIN_DONE_AUTORESET")) != 0
            thunks["terminal_observation"] = lambda: self.terminal_obs
        return self.obs, self.reward, tt[0], tt[1], LazyInfo(thunks)

    def close(self) -> None:
        return None


# SB3 flattens the Dict observation in alphabetical key order (SURVEY 8a row a17): slices of the 80-vector
ROUTE_OBS_SLICES: dict[str, slice] = {
    "dq": slice(0, 7), "goal_ori_err": slice(7, 10), "goal_pos_err": slice(10, 13), "joint_limit_margin": slice(13, 20),
    "mode_flag": slice(20, 24), "next_wp_ori_err": slice(24, 27), "next_wp_pos_err": slice(27, 30), "prev_action": slice(30, 37),
    "progress": slice(37, 40), "q": slice(40, 47), "route_q_error": slice(47, 54), "route_q_goal": slice(54, 61),
    "route_scalar": slice(61, 64), "route_tangent": slice(64, 71), "task_type": slice(71, 74), "wp_ori_err": slice(74, 77),
    "wp_pos_err": slice(77, 80),
}


def build_route_observation_space(n_joints: int, include_route_keys: bool) -> Any:
    """The route wrappers' dict observation space: the base env's keys, plus the four route keys when the observation config
    includes them (route_observation.py:18-28)."""
    from .env import _Box, _DictSpace, build_observation_space

    base = build_observation_space(n_joints)
    if not include_route_keys:
        return base
    sp = dict(base.spaces)
    sp.update({"route_q_goal": _Box(-1.0, 1.0, (n_joints,)), "route_q_error": _Box(-1.0, 1.0, (n_joints,)),
               "route_tangent": _Box(-1.0, 1.0, (n_joints,)), "route_scalar": _Box(0.0, 1.0, (3,))})
    return _DictSpace(sp)


def route_obs_keys(include_route_keys: bool) -> tuple[str, ...]:
    """Keys of the route wrappers' dict observation, in the order of the flat 80-vector (``ROUTE_OBS_SLICES``)."""
    return tuple(k for k in ROUTE_OBS_SLICES if include_route_keys or not k.startswith("route_"))


class _RouteBaseEnvView:
    """What the reference's evaluators reach for through ``env.base_env`` (eval_route_curriculum.py:73-87,134): the wrapped env's
    private joint state and a ``reset(options=...)`` that re-seats the joint state while the route bookkeeping stays."""

    def __init__(self, owner: "_SingleRouteEnv") -> None:
        self._o = owner
        self.config = owner.config.base_env_config
        self.action_space, self.observation_space = owner.action_space, owner._base_observation_space

    def _rows(self, name: str) -> np.ndarray:
        r = _D(name)
        return self._o._b.state[r:r + 7, 0].detach().cpu().numpy().astype(float)

    _q = property(lambda self: self._rows("KIN_ROW_Q"))
    _dq = property(lambda self: self._rows("KIN_ROW_DQ"))
    _prev_action = property(lambda self: self._rows("KIN_ROW_PREV_ACTION"))
    _goal_q = property(lambda self: self._rows("KIN_ROW_GOAL_Q"))

    def reset(self, *, seed: int | None = None, options: dict[str, Any] | None = None):
        o, opts = self._o, dict(options or {})
        if "initial_q" not in opts:
            raise ValueError("base_env.reset needs options['initial_q'] (the route wrappers own the sampled resets)")
        goal = np.asarray(opts.get("goal_q", o.route.q_goal[o._target_index()]), dtype=float)
        if np.abs(goal - o.route.q_goal[o._target_index()]).max() > 1e-9:
            raise ValueError("base_env.reset: goal_q must be the current route waypoint's q_goal")
        o._seat(o._target_index(), o._start_route_index, opts["initial_q"], opts.get("initial_dq"), opts.get("initial_prev_action"))
        obs = o._obs_np()
        return {k: v for k, v in obs.items() if not k.startswith("route_")}, o._base_info()

    def close(self) -> None:
        return None


class _SingleRouteEnv:
    """Shared 1-env plumbing of the two route wrappers (numpy in / out over a 1-replica ``BatchedRouteKinematicEnv``)."""

    metadata = {"render_modes": []}

    def __init__(self, *, route: RouteDataset, config: RouteEnvConfig, sequence_config: RouteSequenceConfig | None, seed: int | None,
                 device: str | torch.device) -> None:
        from .env import build_action_space, build_observation_space

        self.route, self.config = route, config
        n = config.base_env_config.n_joints
        self.action_space = build_action_space(n)
        self._base_observation_space = build_observation_space(n)
        self.observation_space = build_route_observation_space(n, config.observation_config.include_route_keys)
        self._b = BatchedRouteKinematicEnv(route, config, 1, device, sequence_config=sequence_config, with_components=True)
        self._rng = np.random.default_rng(seed)
        self._start_route_index = 0
        self._prev_info: dict[str, Any] | None = None
        self.base_env = _RouteBaseEnvView(self)
        self._seat(1, 0, route.q_goal[0], None, None)

    # ---- device state <-> the reference's private attributes
    def _word(self, row: str) -> int:
        return int(self._b.state[_D(row), 0].view(torch.int32).item()) & 0xFFFFFFFF

    def _set_word(self, row: str, value: int) -> None:
        v = int(value) & 0xFFFFFFFF
        self._b.state[_D(row), 0] = torch.tensor(v if v < 2 ** 31 else v - 2 ** 32, dtype=torch.int32).view(torch.float32)

    def _target_index(self) -> int:
        return self._word("KIN_ROW_ROUTE") & 0xFFFF

    def _set_target_index(self, value: int) -> None:
        self._set_word("KIN_ROW_ROUTE", (self._word("KIN_ROW_ROUTE") & 0xFFFF0000) | (int(value) & 0xFFFF))

    _ready_streak = property(lambda self: self._word("KIN_ROW_ROUTE") >> 16,
                             lambda self, v: self._set_word("KIN_ROW_ROUTE", (self._word("KIN_ROW_ROUTE") & 0xFFFF) | ((int(v) & 0xFFFF) << 16)))

    def _seat(self, route_index: int, start_index: int, initial_q: Any, initial_dq: Any, initial_prev_action: Any) -> None:
        z = np.zeros(7)
        self._b.reset(route_index=[int(route_index)], start_route_index=[int(start_index)], initial_q=np.asarray(initial_q, dtype=float),
                      initial_dq=z if initial_dq is None else np.asarray(initial_dq, dtype=float),
                      initial_prev_action=z if initial_prev_action is None else np.asarray(initial_prev_action, dtype=float))
        self._start_route_index = int(start_index)

    def _obs_np(self) -> dict[str, np.ndarray]:
        flat = self._b.obs[0].detach().cpu().numpy()
        return {k: flat[ROUTE_OBS_SLICES[k]].copy() for k in route_obs_keys(self.config.observation_config.include_route_keys)}

    def _augment_obs(self, obs: dict[str, np.ndarray] | None = None) -> dict[str, np.ndarray]:
        """``_augment_obs`` (route_env.py:194-207): the observation of the current device state including the route keys.  Meant
        for the evaluator's use right after a (base) reset: the observation is rebuilt as an episode-start observation."""
        self._b.refresh_observation()
        return self._obs_np()

    def _base_info(self) -> dict[str, Any]:
        st = self._b.state[:, 0].detach().cpu().numpy()
        f = lambda name, n: st[_D(name):_D(name) + n].astype(float)  # noqa: E731
        goal, ee = f("KIN_ROW_GOAL_POSE", 6), f("KIN_ROW_EE_POSE", 6)
        ori = (goal[3:] - ee[3:] + np.pi) % (2 * np.pi) - np.pi
        return {"q": f("KIN_ROW_Q", 7), "dq": f("KIN_ROW_DQ", 7), "goal_q": f("KIN_ROW_GOAL_Q", 7), "goal_pose6": goal, "ee_pose6": ee,
                "position_error_norm": float(np.linalg.norm(goal[:3] - ee[:3])), "orientation_error_norm": float(np.linalg.norm(ori)),
                "success": False, "reason": "running"}

    def _route_fields(self, index: int) -> dict[str, Any]:
        return {"route_index": int(index), "start_route_index": int(self._start_route_index), "route_progress_m": float(self.route.progress_m[index]),
                "route_chunk_id": int(self.route.chunk_id[index])}

    def set_route_window(self, *, max_route_index: int, min_route_index: int = 1) -> None:
        self._b.set_route_window(max_route_index=max_route_index, min_route_index=min_route_index)
        self.config = self._b.config

    def _step_device(self, action: Any):
        a = np.asarray(action, dtype=float)
        if a.shape != (self.config.base_env_config.n_joints,):
            raise ValueError(f"Expected action shape {(self.config.base_env_config.n_joints,)}, got {a.shape}")
        _, reward, term, trunc, info = self._b.step(torch.as_tensor(a[None], dtype=torch.float32))
        out = self._base_info()
        out.update({
            "position_error_norm": float(info["position_error_norm"][0]), "orientation_error_norm": float(info["orientation_error_norm"][0]),
            "action_l2": float(np.linalg.norm(self.base_env._prev_action)),        # the stored action is the clipped one that was executed
            "executed_delta_q_l2": float(np.linalg.norm(out["dq"])),
            "success": bool(info["success"][0]), "route_ready": bool(info["route_ready"][0]), "route_ready_streak": int(info["route_ready_streak"][0]),
            "route_q_error_norm": float(info["route_q_error_norm"][0]), "route_orientation_hit": bool(info["route_orientation_hit"][0]),
            "route_regression": bool(info["route_regression"][0]), "nearest_route_q_distance": float(info["nearest_route_q_distance"][0]),
            "reward_components": info["reward_components"][:, 0].detach().cpu().numpy().astype(float),
        })
        return float(reward[0]), bool(term[0]), bool(trunc[0]), info, out

    def render(self) -> None:
        return None

    def close(self) -> None:
        return None


class RouteKinematicEnv(_SingleRouteEnv):
    """Drop-in for ``RouteKinematicEnv`` (route/route_env.py:27-212): same constructor keywords, ``reset(seed=, options=)`` /
    ``step(action)`` / ``set_route_window``, dict observations with the four route keys, the ``info`` keys its readers use
    (``eval_route_curriculum.py:88-132``, ``route_curriculum.py:96-99``) and the private attributes the evaluator touches
    (``_route_index``, ``_start_route_index``, ``_ready_streak``, ``_prev_info``, ``_augment_obs``, ``base_env._q / _prev_action /
    reset``).  Sampled resets consume the numpy PCG64 stream in the reference's order (``sample_route_reset``).  Conformance, not
    throughput: every call is a 1-replica kernel launch plus a host copy."""

    def __init__(self, *, route: RouteDataset, config: RouteEnvConfig, seed: int | None = None, device: str | torch.device = "cuda") -> None:
        super().__init__(route=route, config=config, sequence_config=None, seed=seed, device=device)

    _route_index = property(lambda self: self._target_index(), lambda self, v: self._set_target_index(v))

    def reset(self, *, seed: int | None = None, options: dict[str, Any] | None = None):
        if seed is not None:
            self._rng = np.random.default_rng(seed)
        opts = options or {}
        if "route_index" in opts:           # route_env.py:53-59: explicit waypoint, start state = the start waypoint itself
            ri = int(opts["route_index"])
            st = int(opts.get("start_route_index", max(ri - 1, 0)))
            self._seat(ri, st, self.route.q_goal[st], None, None)
            mode = "explicit"
        else:
            smp = sample_route_reset(self._rng, self.route, self.config.base_env_config.joint_specs, self.config.reset_config)
            self._seat(smp["route_index"], smp["start_route_index"], smp["initial_q"], smp["initial_dq"], smp["initial_prev_action"])
            mode = smp["reset_mode"]
        info = self._base_info()
        info.update(self._route_fields(self._route_index))
        info["route_reset_mode"] = mode
        self._prev_info = dict(info)
        return self._obs_np(), info

    def step(self, action: Any):
        reward, term, trunc, _, info = self._step_device(action)
        if info["success"] and self.config.base_env_config.termination_config.terminate_on_success:
            info["termination_reason"] = "route_ready_success"
        info.update(self._route_fields(self._route_index))
        self._prev_info = dict(info)
        return self._obs_np(), reward, term, trunc, info


class RouteSequenceKinematicEnv(_SingleRouteEnv):
    """Drop-in for ``RouteSequenceKinematicEnv`` (route/route_sequence_env.py:27-278): the target advances to the next dense route
    waypoint inside the episode when the current one is reached; ``_current_route_index`` / ``_last_route_index`` /
    ``_completed_waypoints`` mirror the reference's attributes."""

    def __init__(self, *, route: RouteDataset, config: RouteEnvConfig, sequence_config: RouteSequenceConfig | None = None, seed: int | None = None,
                 device: str | torch.device = "cuda") -> None:
        import dataclasses

        self.sequence_config = sequence_config or RouteSequenceConfig()
        super().__init__(route=route, config=config, sequence_config=dataclasses.replace(self.sequence_config, enabled=True), seed=seed, device=device)

    _current_route_index = property(lambda self: self._target_index(), lambda self, v: self._set_target_index(v))
    _last_route_index = property(lambda self: self._word("KIN_ROW_ROUTE2") & 0xFFFF)
    _completed_waypoints = property(lambda self: self._word("KIN_ROW_ROUTE2") >> 16)

    def _sequence_fields(self, *, waypoint_success: bool, sequence_success: bool) -> dict[str, Any]:
        out = self._route_fields(self._current_route_index)
        out.update({"route_last_index": int(self._last_route_index), "route_completed_waypoints": int(self._completed_waypoints),
                    "route_waypoint_success": bool(waypoint_success), "route_sequence_success": bool(sequence_success)})
        return out

    def reset(self, *, seed: int | None = None, options: dict[str, Any] | None = None):
        if seed is not None:
            self._rng = np.random.default_rng(seed)
        opts = options or {}
        if "route_index" in opts:           # route_sequence_env.py:101-107: explicit start state allowed
            ri = int(opts["route_index"])
            st = int(opts.get("start_route_index", max(ri - 1, 0)))
            self._seat(ri, st, opts.get("initial_q", self.route.q_goal[st]), opts.get("initial_dq"), opts.get("initial_prev_action"))
            mode = "explicit_sequence"
        else:
            smp = sample_route_reset(self._rng, self.route, self.config.base_env_config.joint_specs, self.config.reset_config)
            self._seat(smp["route_index"], smp["start_route_index"], smp["initial_q"], smp["initial_dq"], smp["initial_prev_action"])
            mode = smp["reset_mode"]
        info = self._base_info()
        info.update(self._sequence_fields(waypoint_success=False, sequence_success=False))
        info["route_reset_mode"] = mode
        self._prev_info = dict(info)
        return self._obs_np(), info

    def step(self, action: Any):
        reward, term, trunc, dev, info = self._step_device(action)
        wp = bool(dev["route_waypoint_success"][0])
        info.update(self._sequence_fields(waypoint_success=wp, sequence_success=bool(info["success"])))
        self._prev_info = dict(info)
        return self._obs_np(), reward, term, trunc, info


ROUTE_RESET_MODES = ("prefix_start", "random_prefix", "segment", "replay", "recovery")
_FORCED_MODE = {"prefix_start_reset": 0, "random_prefix_reset": 1, "segment_reset": 2, "replay_reset": 3, "recovery_reset": 4}


def _reset_mode_ratios(config: Any) -> np.ndarray:
    r = np.asarray([max(config.prefix_start_reset_ratio, 0.0), max(config.random_prefix_reset_ratio, 0.0), max(config.segment_reset_ratio, 0.0),
                    max(config.replay_reset_ratio, 0.0), max(config.recovery_reset_ratio, 0.0)], dtype=float)
    return r / r.sum() if r.sum() > 0.0 else np.array([0.0, 1.0, 0.0, 0.0, 0.0])


def _reset_index_ranges(config: Any, max_index: int) -> np.ndarray:
    """[5, 2] inclusive (low, high) of the target waypoint per reset mode (route_reset_samplers.py:48-95)."""
    lo = int(np.clip(config.min_route_index, 1, max_index))
    hi = int(np.clip(config.max_route_index, lo, max_index))
    seg_lo = int(np.clip(config.segment_start_index, 1, max_index))
    seg_hi = int(np.clip(config.segment_end_index, seg_lo, max_index))
    rep_lo = int(np.clip(config.replay_start_index, 1, max_index))
    rep_hi = int(np.clip(config.replay_end_index, rep_lo, max_index))
    return np.array([[lo, hi], [lo, hi], [seg_lo, min(seg_hi, hi)], [rep_lo, min(rep_hi, hi)], [lo, hi]], dtype=np.int64)


def sample_route_reset(rng: np.random.Generator, route: RouteDataset, joint_specs: Sequence[Any], config: Any) -> dict[str, Any]:
    """Host port of ``sample_route_reset`` (route_reset_samplers.py:43-117), consuming the numpy stream in the reference's order
    (``rng.choice`` for the mode, ``rng.integers`` for the waypoint, three ``rng.normal`` noise vectors)."""
    max_index = len(route) - 1
    mode = int(rng.choice(5, p=_reset_mode_ratios(config)))          # rng.choice(list_of_5, p=...) draws the same index
    mode = _FORCED_MODE.get(config.mode, mode)
    lo, hi = _reset_index_ranges(config, max_index)[mode]
    route_index = int(rng.integers(lo, hi + 1))
    start_index = 0 if mode == 0 else max(route_index - 1, 0)
    src = route_index if mode == 4 else start_index
    noise = lambda std: rng.normal(0.0, float(std), size=(7,)) if std > 0.0 else np.zeros(7)  # noqa: E731
    lower = np.array([sp.lower for sp in joint_specs]); upper = np.array([sp.upper for sp in joint_specs])
    initial_q = np.clip(route.q_goal[src] + noise(config.q_noise_std), lower, upper)
    initial_dq = noise(config.dq_noise_std)
    initial_prev_action = np.clip(noise(config.prev_action_noise_std), -1.0, 1.0)
    return {"initial_q": initial_q, "initial_dq": initial_dq, "initial_prev_action": initial_prev_action, "goal_q": route.q_goal[route_index].copy(),
            "route_index": route_index, "start_route_index": start_index, "reset_mode": ROUTE_RESET_MODES[mode]}


def sample_route_reset_batch(table: "DeviceRoute", joint_specs: Sequence[Any], config: Any, n: int, generator: torch.Generator) -> dict[str, torch.Tensor]:
    """The same sampler for ``n`` resets at once on the device (torch Philox stream: distributionally, not bitwise, the reference's)."""
    dev = table.device
    max_index = len(table.route) - 1
    if config.mode in _FORCED_MODE:
        mode = torch.full((n,), _FORCED_MODE[config.mode], dtype=torch.int64, device=dev)
    else:
        p = torch.as_tensor(_reset_mode_ratios(config), dtype=torch.float32, device=dev)
        mode = torch.multinomial(p, n, replacement=True, generator=generator)
    rng_tab = torch.as_tensor(_reset_index_ranges(config, max_index), device=dev)
    lo, hi = rng_tab[mode, 0], rng_tab[mode, 1]
    u = torch.rand(n, device=dev, generator=generator)
    route_index = (lo + torch.floor(u * (hi - lo + 1).float()).long()).clamp(max=hi)
    start_index = torch.where(mode == 0, torch.zeros_like(route_index), (route_index - 1).clamp_min(0))
    src = torch.where(mode == 4, route_index, start_index)
    g = lambda std: torch.randn((n, 7), device=dev, generator=generator) * float(std) if std > 0.0 else torch.zeros((n, 7), device=dev)  # noqa: E731
    lower = torch.tensor([sp.lower for sp in joint_specs], dtype=torch.float32, device=dev)
    upper = torch.tensor([sp.upper for sp in joint_specs], dtype=torch.float32, device=dev)
    initial_q = torch.minimum(torch.maximum(table.q[src] + g(config.q_noise_std), lower), upper)
    return {"initial_q": initial_q, "initial_dq": g(config.dq_noise_std), "initial_prev_action": g(config.prev_action_noise_std).clamp(-1.0, 1.0),
            "route_index": route_index.to(torch.int32), "start_route_index": start_index.to(torch.int32), "reset_mode": mode}


@dataclass(frozen=True)
class RouteCurriculumStage:
    name: str
    prefix_end_index: int


class RoutePrefixCurriculum:
    """``RoutePrefixCurriculumCallback`` (route/route_curriculum.py:23-132) without SB3: feed the finished episodes' flags in env
    order, get the prefix window to apply.  Promotion needs all four windowed rates (success, route-ready hit, orientation hit,
    regression) over ``window_episodes`` and at least ``min_episodes_per_stage`` episodes in the stage."""

    def __init__(self, stages: Sequence[RouteCurriculumStage], *, promotion_success_rate: float, promotion_route_ready_hit_rate: float,
                 promotion_orientation_hit_rate: float, promotion_max_regression_rate: float, window_episodes: int, min_episodes_per_stage: int = 128) -> None:
        if not stages:
            raise ValueError("RoutePrefixCurriculumCallback requires at least one stage")
        from collections import deque

        self.stages = list(stages)
        self.thresholds = (float(promotion_success_rate), float(promotion_route_ready_hit_rate), float(promotion_orientation_hit_rate),
                           float(promotion_max_regression_rate))
        self.window_episodes = max(int(window_episodes), 1)
        self.min_episodes_per_stage = max(int(min_episodes_per_stage), 1)
        self.current_stage_index = 0
        self.stage_episode_count = 0
        self._win = [deque(maxlen=self.window_episodes) for _ in range(4)]
        self.history: list[dict[str, Any]] = []

    @property
    def prefix_end_index(self) -> int:
        return int(self.stages[self.current_stage_index].prefix_end_index)

    def metrics(self) -> dict[str, float]:
        m = lambda d: float(sum(d)) / float(len(d)) if d else 0.0  # noqa: E731
        return {"recent_success_rate": m(self._win[0]), "recent_route_ready_hit_rate": m(self._win[1]),
                "recent_orientation_hit_rate": m(self._win[2]), "recent_regression_rate": m(self._win[3])}

    def record(self, success: Any, route_ready: Any, orientation_hit: Any, regression: Any, *, total_timesteps: int = 0) -> bool:
        """One ``_on_step``: the flags of the episodes that finished at this step (env order).  True when a promotion happened."""
        promoted = False
        for flags in zip(np.atleast_1d(success), np.atleast_1d(route_ready), np.atleast_1d(orientation_hit), np.atleast_1d(regression)):
            self.stage_episode_count += 1
            for d, f in zip(self._win, flags):
                d.append(1 if bool(f) else 0)
            if self.stage_episode_count < self.min_episodes_per_stage or len(self._win[0]) < self.window_episodes:
                continue
            m = self.metrics()
            if (m["recent_success_rate"] >= self.thresholds[0] and m["recent_route_ready_hit_rate"] >= self.thresholds[1]
                    and m["recent_orientation_hit_rate"] >= self.thresholds[2] and m["recent_regression_rate"] <= self.thresholds[3]
                    and self.current_stage_index < len(self.stages) - 1):
                prev = self.stages[self.current_stage_index]
                self.current_stage_index += 1
                nxt = self.stages[self.current_stage_index]
                self.history.append({"from_stage": prev.name, "to_stage": nxt.name, "from_prefix_end_index": int(prev.prefix_end_index),
                                     "to_prefix_end_index": int(nxt.prefix_end_index), "total_timesteps": int(total_timesteps), **m})
                self.stage_episode_count = 0
                for d in self._win:
                    d.clear()
                promoted = True
        return promoted

    def summary(self) -> dict[str, Any]:
        st = self.stages[self.current_stage_index]
        return {"stage_index": int(self.current_stage_index), "stage_name": st.name, "prefix_end_index": int(st.prefix_end_index),
                "stage_episode_count": int(self.stage_episode_count), **self.metrics(), "history": list(self.history)}


ROUTE_EVAL_CHUNKS = ((1, 40), (41, 80), (81, 120), (121, 180), (181, 260), (261, 360), (361, 483))


def route_failure_reason(row: dict[str, Any]) -> str:
    """``_failure_reason`` (eval_route_curriculum.py:156-168)."""
    if row["final_position_error"] > 0.010:
        return "position"
    if row["final_orientation_error"] > 0.150:
        return "orientation"
    if row.get("final_action_magnitude", 0.0) > 1.20 or row.get("final_dq_norm", 0.0) > 0.040:
        return "motion_action"
    if row["final_q_error"] > 0.500:
        return "q_error"
    if not row["route_ready_dwell"]:
        return "dwell_or_motion"
    return "unknown"


def summarize_route_rows(rows: Sequence[dict[str, Any]], route: RouteDataset) -> dict[str, Any]:
    """``_summarize_rows`` (eval_route_curriculum.py:127-153): same keys, same arithmetic."""
    if not rows:
        return {"target_count": 0}
    first_failure = next((r for r in rows if not r["success"]), None)
    longest = 0
    for r in rows:
        if not r["success"]:
            break
        longest += 1
    mean = lambda k: float(np.mean([r[k] for r in rows]))  # noqa: E731
    return {
        "target_count": len(rows), "success_rate": mean("success"), "route_ready_hit_rate": mean("route_ready_hit"),
        "route_ready_dwell_rate": mean("route_ready_dwell"), "longest_success_prefix": int(longest),
        "cumulative_successful_route_distance_m": float(route.progress_m[min(longest, len(route) - 1)] - route.progress_m[0]),
        "first_failure_index": None if first_failure is None else int(first_failure["route_index"]),
        "first_failure_reason": None if first_failure is None else route_failure_reason(first_failure),
        "mean_final_position_error": mean("final_position_error"), "mean_final_orientation_error": mean("final_orientation_error"),
        "mean_final_q_error": mean("final_q_error"),
        "max_final_position_error": float(np.max([r["final_position_error"] for r in rows])),
        "max_final_orientation_error": float(np.max([r["final_orientation_error"] for r in rows])),
    }


def route_chunk_metrics(rows: Sequence[dict[str, Any]]) -> dict[str, Any]:
    """``_chunk_metrics`` (eval_route_curriculum.py:171-186)."""
    out: dict[str, Any] = {}
    for idx, (lo, hi) in enumerate(ROUTE_EVAL_CHUNKS):
        sub = [r for r in rows if lo <= r["route_index"] <= hi]
        if not sub:
            continue
        mean = lambda k: float(np.mean([r[k] for r in sub]))  # noqa: E731
        out[f"chunk_{idx}_{lo}_{hi}"] = {"target_count": len(sub), "success_rate": mean("success"), "route_ready_hit_rate": mean("route_ready_hit"),
                                         "mean_final_position_error": mean("final_position_error"),
                                         "mean_final_orientation_error": mean("final_orientation_error"), "mean_final_q_error": mean("final_q_error")}
    return out


def _rows_from_device(block: np.ndarray, start_index: int) -> list[dict[str, Any]]:
    """[waypoints][KIN_ROUTE_ROW_FIELDS] floats of one replica -> the row dicts of ``_roll_one`` (eval_route_curriculum.py:111-128)."""
    F = lambda name: _D("KIN_ROUTE_ROW_" + name)  # noqa: E731
    rows = []
    for k, r in enumerate(block):
        first = int(r[F("FIRST_READY_STEP")])
        rows.append({
            "route_index": int(start_index + k), "success": bool(r[F("SUCCESS")] > 0.5), "route_ready_hit": bool(r[F("READY_HIT")] > 0.5),
            "route_ready_dwell": bool(r[F("READY_DWELL")] > 0.5), "first_ready_step": None if first < 0 else first,
            "max_ready_streak": int(r[F("MAX_READY_STREAK")]), "steps": int(r[F("STEPS")]),
            "final_position_error": float(r[F("FINAL_POS")]), "final_orientation_error": float(r[F("FINAL_ORI")]),
            "final_q_error": float(r[F("FINAL_Q_ERR")]), "min_position_error": float(r[F("MIN_POS")]),
            "min_orientation_error": float(r[F("MIN_ORI")]), "min_q_error": float(r[F("MIN_Q_ERR")]),
            "final_action_magnitude": float(r[F("FINAL_ACTION_L2")]), "final_dq_norm": float(r[F("FINAL_DQ_L2")]),
        })
    return rows


def evaluate_sequential_route(route: RouteDataset, config: RouteEnvConfig, policy: PolicyWeights, *, n_replicas: int = 1, start_index: int = 1,
                              end_index: int | None = None, start_q_noise_std: float = 0.0, seed: int = 0,
                              device: str | torch.device = "cuda", variant: str = "fp32", detail_replicas: int = 0) -> dict[str, Any]:
    """``evaluate_sequential_route`` (eval_route_curriculum.py:188-246) for ``n_replicas`` independent chains in one launch.

    ``variant``: "fp32" = strict-fp32 policy in the loop (the parity path), "tc" = the actor on tcgen05 tensor cores (TF32 operands).

    Replica 0 starts exactly at waypoint ``start_index - 1`` like the reference; the others add N(0, std) joint noise.
    Returns per-replica ``longest_success_prefix``, the success bitmask, the prefix histogram and env-step count.
    ``detail_replicas`` > 0 (strict variant): the first replicas also return the reference's per-waypoint ``rows`` and, for replica 0,
    its ``summary`` / ``chunk_metrics`` / ``failure_report`` dicts (the JSON files ``evaluate_sequential_route`` writes, :222-245).
    """
    if not torch.cuda.is_available():
        raise _lib.KinError("evaluate_sequential_route needs a CUDA device; there is no CPU fallback")
    if variant not in ("fp32", "tc"):
        raise ValueError("variant must be 'fp32' or 'tc'")
    detail_replicas = int(detail_replicas)
    if detail_replicas and (variant != "fp32" or not 0 < detail_replicas <= n_replicas):
        raise ValueError("detail_replicas needs the strict variant and 0 < detail_replicas <= n_replicas")
    device = torch.device(device)
    end = min(len(route) - 1, len(route) - 1 if end_index is None else int(end_index))
    m = end - start_index + 1
    words = (m + 31) // 32
    with torch.cuda.device(device):
        params = ParamsHandle(config.base_env_config, config.reward_config)
        table = DeviceRoute(route, device)
        base = torch.as_tensor(route.q_goal[max(start_index - 1, 0)], dtype=torch.float32, device=device).expand(n_replicas, 7).clone()
        if start_q_noise_std > 0 and n_replicas > 1:
            g = torch.Generator(device=device)
            g.manual_seed(seed)
            noise = torch.randn((n_replicas, 7), device=device, generator=g) * start_q_noise_std
            noise[0] = 0.0
            base = base + noise
        prefix = torch.zeros(n_replicas, dtype=torch.int32, device=device)
        bits = torch.zeros((n_replicas, words), dtype=torch.int32, device=device)
        steps = torch.zeros(1, dtype=torch.int64, device=device)
        rows_dev = None
        if detail_replicas:
            rows_dev = torch.zeros((detail_replicas, m, _D("KIN_ROUTE_ROW_FIELDS")), dtype=torch.float32, device=device)
            _lib.check(_lib.lib().kin_route_probe_rows(params.handle, ctypes.byref(table.c), ctypes.byref(policy.c), base.data_ptr(), int(start_index), end,
                                                       n_replicas, prefix.data_ptr(), bits.data_ptr(), steps.data_ptr(), rows_dev.data_ptr(), detail_replicas,
                                                       _stream()))
        else:
            probe = _lib.lib().kin_route_probe_tc if variant == "tc" else _lib.lib().kin_route_probe
            _lib.check(probe(params.handle, ctypes.byref(table.c), ctypes.byref(policy.c), base.data_ptr(), int(start_index), end,
                             n_replicas, prefix.data_ptr(), bits.data_ptr(), steps.data_ptr(), _stream()))
    hist = torch.bincount(prefix.long(), minlength=m + 1)
    p0 = int(prefix[0].item())
    detail: dict[str, Any] = {}
    if rows_dev is not None:
        blocks = rows_dev.cpu().numpy()
        all_rows = [_rows_from_device(b, int(start_index)) for b in blocks]
        summary = summarize_route_rows(all_rows[0], route)
        summary.update({"schema_version": "v5.route_curriculum.sequential_eval.v1", "mode": "sequential_actual_final_q_to_next_dense_q_goal",
                        "start_index": int(start_index), "end_index": int(end)})
        failure = next((r for r in all_rows[0] if not r["success"]), None)
        detail = {"rows": all_rows, "summary": summary, "chunk_metrics": route_chunk_metrics(all_rows[0]),
                  "failure_report": {"first_failure_index": summary["first_failure_index"], "first_failure_reason": summary["first_failure_reason"],
                                     "first_failure": failure}}
    return {
        **detail,
        "longest_success_prefix": prefix, "success_bits": bits, "prefix_histogram": hist, "env_steps": steps,
        "replica0_longest_success_prefix": p0,
        "replica0_cumulative_successful_route_distance_m": float(route.progress_m[min(p0, len(route) - 1)] - route.progress_m[0]),
        "start_index": int(start_index), "end_index": int(end), "variant": variant,
    }
