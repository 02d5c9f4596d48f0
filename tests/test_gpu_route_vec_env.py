"""The route env as an SB3 VecEnv: kin_route_step_autoreset (step + in-kernel sampled reset of the finished slots), the auto-reset /
graph-step modes of BatchedRouteKinematicEnv and KinRouteVecEnv, against the existing kernels and the fp64 oracle."""

from __future__ import annotations

import dataclasses
import functools

import numpy as np
import pytest
import torch

from oracle import kin_oracle as ko

from ._util import oracle_params

pytestmark = pytest.mark.gpu


@functools.lru_cache(maxsize=None)
def _route(n_waypoints: int):
    from rl_brain_trainer_b200.route import synthetic_route

    return synthetic_route(n_waypoints, seed=7)


def _config(route, *, max_steps: int, include_route_keys: bool = True, terminate_on_success: bool = True):
    from rl_brain_trainer_b200 import config as kcfg

    renv, seq = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    base = renv.base_env_config
    base = dataclasses.replace(base, episode_length=max_steps,
                               termination_config=dataclasses.replace(base.termination_config, max_episode_steps=max_steps,
                                                                      terminate_on_success=terminate_on_success))
    return dataclasses.replace(renv, base_env_config=base, observation_config=kcfg.RouteObservationConfig(include_route_keys=include_route_keys)), seq


def _D(name: str) -> int:
    from rl_brain_trainer_b200 import _lib

    return _lib.define(name)


def _tracking_actions(env, gen: torch.Generator, gain: float = 0.7, noise: float = 0.03) -> torch.Tensor:
    """Proportional steps toward each slot's current target waypoint plus noise (the actions of test_route_batch_vs_oracle_random)."""
    n = env.num_envs
    q = env.state[_D("KIN_ROW_Q"):_D("KIN_ROW_Q") + 7, :n].t()
    gq = env.state[_D("KIN_ROW_GOAL_Q"):_D("KIN_ROW_GOAL_Q") + 7, :n].t()
    dl = torch.tensor([s.delta_limit for s in env.config.base_env_config.joint_specs], dtype=torch.float32, device=env.device)
    dl = dl * env.config.base_env_config.action_delta_scale
    a = (gq - q) / dl * gain + noise * torch.randn((n, 7), generator=gen, device=env.device)
    return a.clamp(-1.0, 1.0).contiguous()


def _restated_step(env, a: torch.Tensor, seed: int) -> torch.Tensor:
    """kin_route_step_autoreset spelled out with the existing kernels on a non-auto-reset env: kin_route_step, the terminal rows, one
    kin_route_reset_sampled per distinct episode counter among the finished slots, the counter row and the AUTORESET bit.  Returns
    the terminal observations (meaningful on the finished rows)."""
    n = env.num_envs
    env.step_raw(a)
    finished = (env.done & (_D("KIN_DONE_TERMINATED") | _D("KIN_DONE_TRUNCATED"))) != 0
    terminal = torch.zeros_like(env.obs)
    terminal[finished] = env.obs[finished]
    row = env.state[_D("KIN_ROW_EPISODE"), :n].view(torch.int32)
    episode = row + 1
    for v in torch.unique(episode[finished]).tolist():
        mask = (finished & (episode == v)).to(torch.uint8) * _D("KIN_DONE_TERMINATED")
        env.reset_done(seed=seed, counter=int(v), done=mask)
    row[finished] = episode[finished]
    env.done[finished] |= _D("KIN_DONE_AUTORESET")
    return terminal


@pytest.mark.parametrize("n_waypoints", [483, 1100])
@pytest.mark.parametrize("n", [1000, 4096])
@pytest.mark.parametrize("with_components", [False, True])
@pytest.mark.parametrize("sequence", [False, True])
def test_fused_autoreset_step_is_the_three_kernel_sequence_bitwise(sequence, with_components, n, n_waypoints):
    """From the same start state and action tape, kin_route_step_autoreset equals kin_route_step + terminal rows +
    kin_route_reset_sampled(seed, episode) + counter write-back, bit for bit, over several episodes per slot, a partial warp, the global
    waypoint table (1100 > ROUTE_MAX_SMEM_WP), terminate-on-success, a short time limit and a set_route_window change mid-tape."""
    from rl_brain_trainer_b200.route import BatchedRouteKinematicEnv

    route = _route(n_waypoints)
    renv, seq = _config(route, max_steps=7)
    seq_cfg = dataclasses.replace(seq, enabled=True, sequence_length=3) if sequence else None
    seed = 1234
    fused = BatchedRouteKinematicEnv(route, renv, n, sequence_config=seq_cfg, with_components=with_components, auto_reset=True, seed=seed)
    plain = BatchedRouteKinematicEnv(route, renv, n, sequence_config=seq_cfg, with_components=with_components)
    fused.set_route_window(max_route_index=min(200, len(route) - 1))
    plain.set_route_window(max_route_index=min(200, len(route) - 1))
    fused.reset()
    plain.state.copy_(fused.state)
    plain.obs.copy_(fused.obs)
    gen = torch.Generator(device="cuda").manual_seed(5)
    finished_total, terminated_total = 0, 0
    for t in range(64):
        if t == 30:                   # RoutePrefixCurriculum promotion: the next resets draw from the new window
            fused.set_route_window(max_route_index=12, min_route_index=3)
            plain.set_route_window(max_route_index=12, min_route_index=3)
        a = _tracking_actions(fused, gen, gain=0.7 if t % 3 else 1.5)
        fused.step(a)
        terminal = _restated_step(plain, a, seed)
        finished = (plain.done & _D("KIN_DONE_AUTORESET")) != 0
        finished_total += int(finished.sum())
        terminated_total += int(((plain.done & _D("KIN_DONE_TERMINATED")) != 0).sum())
        assert torch.equal(fused.done, plain.done), t
        assert torch.equal(fused.reward, plain.reward), t
        assert torch.equal(fused.raux[:, :n], plain.raux[:, :n]), t
        if with_components:
            assert torch.equal(fused.rcomp[:, :n], plain.rcomp[:, :n]), t
        assert torch.equal(fused.state, plain.state), t
        assert torch.equal(fused.obs, plain.obs), t
        assert torch.equal(fused.terminal_obs[finished], terminal[finished]), t
    episodes = fused.state[_D("KIN_ROW_EPISODE"), :n].view(torch.int32)
    assert finished_total >= 4 * n and int(episodes.min()) >= 3, (finished_total, int(episodes.min()))
    assert terminated_total > 0
    late = (fused.state[_D("KIN_ROW_ROUTE"), :n].view(torch.int32) & 0xFFFF)
    assert int(late.max()) <= 12            # every slot was reset after the window change (sequence targets stop at last <= 12)


@pytest.mark.parametrize("sequence", [False, True])
def test_route_vec_env_against_the_oracle_through_auto_resets(sequence):
    """KinRouteVecEnv driven by proportional-plus-noise actions next to one OracleRouteEnv per env; at every auto-reset the oracle is
    re-seated on the state the device sampler drew.  Replicas that flip at a threshold leave the comparison (<= 3 %)."""
    from rl_brain_trainer_b200.route import ROUTE_OBS_SLICES
    from rl_brain_trainer_b200.vec_env import make_route_vec_env

    route = _route(483)
    renv, seq = _config(route, max_steps=12)
    seq_len = 3 if sequence else 0
    seq_cfg = dataclasses.replace(seq, enabled=True, sequence_length=seq_len) if sequence else None
    n, T = 256, 60
    venv = make_route_vec_env(route, renv, n, sequence_config=seq_cfg, seed=21)
    venv.env_method("set_route_window", max_route_index=120)
    params = oracle_params(renv.base_env_config, renv.reward_config)
    oroute = ko.OracleRoute(route.q_goal)
    oenvs = [ko.OracleRouteEnv(params, oroute, sequence_length=seq_len, max_route_index=len(route) - 1) for _ in range(n)]
    env = venv.env
    order = sorted(ROUTE_OBS_SLICES, key=lambda k: ROUTE_OBS_SLICES[k].start)

    def reseat(envs):
        st = env.state[:, :n].cpu().numpy()
        words = st.view(np.int32)
        for e in envs:
            ri, last = int(words[_D("KIN_ROW_ROUTE"), e] & 0xFFFF), int(words[_D("KIN_ROW_ROUTE2"), e] & 0xFFFF)
            rows = lambda name: st[_D(name):_D(name) + 7, e].astype(float)  # noqa: E731
            oenvs[e].reset(route_index=ri, start_route_index=max(ri - 1, 0), initial_q=rows("KIN_ROW_Q"), initial_dq=rows("KIN_ROW_DQ"),
                           initial_prev_action=rows("KIN_ROW_PREV_ACTION"))
            oenvs[e].state.last_route_index = last

    obs = venv.reset()
    reseat(range(n))
    flat = np.concatenate([obs[k] for k in order], axis=1)
    assert np.abs(flat - np.stack([o.observation() for o in oenvs])).max() < 1e-4
    gen = torch.Generator(device="cuda").manual_seed(3)
    alive = np.ones(n, dtype=bool)
    mism = episodes = 0
    for t in range(T):
        a = _tracking_actions(env, gen).cpu().numpy()
        obs, rew, dones, infos = venv.step(a)
        flat = np.concatenate([obs[k] for k in order], axis=1)
        for e in range(n):
            if not alive[e]:
                continue
            robs, ro = oenvs[e].step(a[e].astype(float))
            i = infos[e]
            same = (i["success"] == bool(ro.success) and i["route_index"] == ro.route_index and i["route_ready"] == bool(ro.route_ready)
                    and bool(dones[e]) == bool(ro.terminated or ro.base.truncated) and i["route_regression"] == bool(ro.route_regression)
                    and i["route_orientation_hit"] == bool(ro.route_orientation_hit))
            if not same:              # threshold-adjacent flip: the trajectories diverge from here
                mism += 1
                alive[e] = False
                continue
            assert abs(float(rew[e]) - ro.route_reward) < 1e-3 * max(1.0, abs(ro.route_reward)), (t, e)
            assert i["route_ready_streak"] == ro.route_ready_streak and abs(i["route_q_error_norm"] - ro.route_q_error_norm) < 1e-4, (t, e)
            assert i["TimeLimit.truncated"] == bool(ro.base.truncated and not ro.terminated), (t, e)
            if sequence:
                assert i["route_waypoint_success"] == bool(ro.waypoint_success), (t, e)
            if dones[e]:
                term = np.concatenate([i["terminal_observation"][k] for k in order])
                assert np.abs(term - robs).max() < 1e-4, (t, e)
            else:
                assert "terminal_observation" not in i and np.abs(flat[e] - robs).max() < 1e-4, (t, e)
        done_ids = np.nonzero(dones)[0]
        episodes += len(done_ids)
        reseat([e for e in done_ids if alive[e]])
        for e in done_ids:            # the observation SB3 sees after a done is the next episode's first one
            if alive[e]:
                assert np.abs(flat[e] - oenvs[e].observation()).max() < 1e-4, (t, e)
    assert mism <= 0.03 * n, mism
    assert episodes >= 3 * n


def test_route_vec_env_protocol_window_and_curriculum():
    from rl_brain_trainer_b200.route import ROUTE_OBS_SLICES, BatchedRouteKinematicEnv, RouteKinematicEnv, RouteCurriculumStage, RoutePrefixCurriculum
    from rl_brain_trainer_b200.vec_env import KinRouteVecEnv, make_route_vec_env

    route = _route(483)
    T = 10
    renv, _ = _config(route, max_steps=T, terminate_on_success=False)
    n = 128
    # spaces and keys are the single-env route adapter's, with and without the four route keys
    for include in (True, False):
        cfg = dataclasses.replace(renv, observation_config=dataclasses.replace(renv.observation_config, include_route_keys=include))
        v = make_route_vec_env(route, cfg, 4, seed=1)
        single = RouteKinematicEnv(route=route, config=cfg)
        assert set(v.observation_space.spaces) == set(single.observation_space.spaces)
        for k, b in single.observation_space.spaces.items():
            assert v.observation_space.spaces[k].shape == b.shape and np.array_equal(v.observation_space.spaces[k].low, b.low), k
        assert v.action_space.shape == (7,)
        assert set(v.reset()) == set(single.observation_space.spaces)
        assert any(k.startswith("route_") for k in v.observation_space.spaces) == include
    venv = make_route_vec_env(route, renv, n, seed=3)
    assert isinstance(venv, KinRouteVecEnv) and venv.num_envs == n
    obs = venv.reset()
    assert set(obs) == set(ROUTE_OBS_SLICES) and obs["q"].shape == (n, 7) and obs["route_scalar"].shape == (n, 3) and obs["q"].dtype == np.float32
    assert np.allclose(obs["progress"][:, 0], 0.0)
    # a plain env started from the same state follows the same episode; at the time limit SB3's semantics hold
    plain = BatchedRouteKinematicEnv(route, renv, n)
    plain.state.copy_(venv.env.state)
    gen = torch.Generator(device="cuda").manual_seed(2)
    for t in range(T):
        a = _tracking_actions(venv.env, gen, gain=0.3)
        obs, rew, dones, infos = venv.step(a.cpu().numpy())
        pobs, prew, _, _, pinfo = plain.step(a)
        assert rew.dtype == np.float32 and dones.dtype == bool and len(infos) == n
        assert np.array_equal(rew, prew.cpu().numpy())
        assert {"success", "route_ready", "route_ready_streak", "route_q_error_norm", "route_orientation_hit", "route_regression", "route_index",
                "position_error_norm", "orientation_error_norm", "TimeLimit.truncated"} <= set(infos[0])
        assert "route_waypoint_success" not in infos[0]
        assert [i["route_index"] for i in infos] == pinfo["route_index"].cpu().tolist()
        if t < T - 1:
            assert not dones.any() and not any("terminal_observation" in i or i["TimeLimit.truncated"] for i in infos)
            for k in ROUTE_OBS_SLICES:
                assert np.array_equal(obs[k], pobs[:, ROUTE_OBS_SLICES[k]].cpu().numpy()), (t, k)
    assert dones.all() and all(i["TimeLimit.truncated"] for i in infos)
    last = pobs.cpu().numpy()
    for e in (0, 77, n - 1):
        for k in ROUTE_OBS_SLICES:
            assert np.array_equal(infos[e]["terminal_observation"][k], last[e, ROUTE_OBS_SLICES[k]]), (e, k)
    assert np.allclose(obs["progress"][:, 0], 0.0) and not np.allclose(obs["q"], last[:, ROUTE_OBS_SLICES["q"]])

    def index_after_full_episodes():
        for _ in range(T):
            _, _, dones, _ = venv.step(np.zeros((n, 7), dtype=np.float32))
        assert dones.all()
        return venv.env.state[_D("KIN_ROW_ROUTE"), :n].view(torch.int32).cpu().numpy() & 0xFFFF

    # set_route_window through env_method: every later auto-reset draws inside the window; widening reaches past the old one
    assert venv.env_method("set_route_window", max_route_index=6) == [None] * n
    ri = index_after_full_episodes()
    assert ri.max() <= 6 and ri.min() >= 1
    venv.env_method("set_route_window", max_route_index=60, min_route_index=1)
    ri = np.concatenate([index_after_full_episodes() for _ in range(2)])
    assert ri.max() > 6 and ri.max() <= 60
    # RoutePrefixCurriculumCallback: infos on dones -> promotion -> env_method widens the window
    venv.env_method("set_route_window", max_route_index=5)
    cur = RoutePrefixCurriculum([RouteCurriculumStage("p5", 5), RouteCurriculumStage("p40", 40)], promotion_success_rate=0.0,
                                promotion_route_ready_hit_rate=0.0, promotion_orientation_hit_rate=0.0, promotion_max_regression_rate=1.0,
                                window_episodes=64, min_episodes_per_stage=64)
    promoted_at = None
    for t in range(3 * T):
        _, _, dones, infos = venv.step(np.zeros((n, 7), dtype=np.float32))
        ended = [infos[i] for i in np.nonzero(dones)[0]]
        if ended and cur.record([i["success"] for i in ended], [i["route_ready"] for i in ended], [i["route_orientation_hit"] for i in ended],
                                [i["route_regression"] for i in ended], total_timesteps=(t + 1) * n):
            venv.env_method("set_route_window", max_route_index=cur.prefix_end_index)
            promoted_at = t
    assert promoted_at is not None and cur.current_stage_index == 1
    assert venv.get_attr("config")[0].reset_config.max_route_index == 40
    ri = np.concatenate([index_after_full_episodes() for _ in range(2)])
    assert ri.max() > 5 and ri.max() <= 40
    # the rest of the protocol, and its errors
    with pytest.raises(ValueError):
        venv.step_async(np.zeros((n, 6), dtype=np.float32))
    with pytest.raises(RuntimeError):
        venv.step_wait()
    with pytest.raises(AttributeError):
        venv.env_method("no_such_method")
    venv.set_attr("tag", 3)
    assert venv.get_attr("tag") == [3] * n and venv.seed(9)[1] == 10 and venv.env._seed == 9
    assert venv.env_is_wrapped(object) == [False] * n
    venv.close()


def test_sequence_route_vec_env_reports_the_waypoint_keys():
    from rl_brain_trainer_b200.vec_env import make_route_vec_env

    route = _route(483)
    renv, seq = _config(route, max_steps=5)
    venv = make_route_vec_env(route, renv, 64, sequence_config=dataclasses.replace(seq, enabled=True, sequence_length=3), seed=4)
    venv.reset()
    for _ in range(5):
        _, _, dones, infos = venv.step(np.zeros((64, 7), dtype=np.float32))
        assert all({"route_waypoint_success", "route_completed_waypoints"} <= set(i) for i in infos)
        assert all(("terminal_observation" in i) == bool(d) for i, d in zip(infos, dones))
    assert dones.any()


@pytest.mark.parametrize("sequence", [False, True])
def test_graph_step_is_the_eager_step_bitwise(sequence):
    """graph_step replays [kin_route_step_autoreset, done-bit ops] as a CUDA graph: bitwise the eager path through auto-resets, and
    re-captured when set_route_window changes the reset parameters."""
    from rl_brain_trainer_b200.route import BatchedRouteKinematicEnv

    route = _route(483)
    renv, seq = _config(route, max_steps=6)
    seq_cfg = dataclasses.replace(seq, enabled=True, sequence_length=3) if sequence else None
    n = 3000
    envs = [BatchedRouteKinematicEnv(route, renv, n, sequence_config=seq_cfg, auto_reset=True, seed=77, graph_step=g) for g in (False, True)]
    for e in envs:
        e.set_route_window(max_route_index=150)
        e.reset()
    gen = torch.Generator(device="cuda").manual_seed(8)
    keys = set()
    for t in range(40):
        if t == 20:
            for e in envs:
                e.set_route_window(max_route_index=9, min_route_index=2)
        a = _tracking_actions(envs[0], gen)
        outs = [e.step(a) for e in envs]
        keys.add(envs[1]._graph_key)
        for x, y in zip(outs[0][:4], outs[1][:4]):
            assert torch.equal(x, y), t
        assert torch.equal(outs[0][4]["auto_reset"], outs[1][4]["auto_reset"]), t
        for name in ("done", "terminal_obs", "state", "raux"):
            assert torch.equal(getattr(envs[0], name), getattr(envs[1], name)), (t, name)
    assert len(keys - {None}) == 2              # one capture per reset window
    ri = envs[1].state[_D("KIN_ROW_ROUTE"), :n].view(torch.int32) & 0xFFFF
    assert int(ri.max()) <= 9
