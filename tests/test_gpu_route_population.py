"""GPU tests of route populations: every member of a ``PPOPopulation`` of 80-input route trainers is bitwise the standalone
``PPOTrainer(route=...)`` built with the same arguments (parameters, Adam moments, weight image, observation rows and images, every
rollout buffer, route flags, env state, counters, learn rows, prefix-curriculum stage and route window)."""

from __future__ import annotations

import ctypes
import dataclasses

import pytest
import torch

pytestmark = pytest.mark.gpu


def _route_setup(episode_steps: int = 20, seed: int = 7):
    """The synthetic 160-waypoint route and the ``route_prefix120`` env, with episodes short enough to hit the time limit in a test."""
    from rl_brain_trainer_b200 import config as kcfg
    from rl_brain_trainer_b200.route import synthetic_route

    route = synthetic_route(160, seed=seed)
    renv, seq = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    b = renv.base_env_config
    b = dataclasses.replace(b, episode_length=episode_steps, termination_config=dataclasses.replace(b.termination_config, max_episode_steps=episode_steps))
    return route, dataclasses.replace(renv, base_env_config=b), seq


def _members(k: int, renv):
    """Per-member arguments that differ in everything a route member may own: seed, initial policy, reset window, PPO and Adam
    hyper-parameters."""
    from rl_brain_trainer_b200 import ppo

    out = []
    for i in range(k):
        cfg = dataclasses.replace(renv, reset_config=dataclasses.replace(renv.reset_config, max_route_index=renv.reset_config.max_route_index - 30 * i))
        hp = ppo.PPOHyper(learning_rate=3e-4 * (1 + i), n_steps=16, batch_size=1024, n_epochs=2, gamma=0.98 - 0.01 * i, gae_lambda=0.95 - 0.02 * i,
                          clip_range=0.2 + 0.05 * i, ent_coef=0.001 * i, vf_coef=0.5 + 0.1 * i, max_grad_norm=0.5 + 0.25 * i,
                          normalize_advantage=(i != 2), adam_beta1=0.9 - 0.02 * i, adam_beta2=0.999 - 0.001 * i, adam_eps=1e-5 * (1 + i))
        out.append(dict(cfg=cfg, hp=hp, seed=100 + 7 * i, policy_seed=i))
    return out


def _curriculum(promote: bool):
    from rl_brain_trainer_b200.route import RouteCurriculumStage, RoutePrefixCurriculum

    thr = (0.0, 0.0, 0.0, 1.0) if promote else (2.0, 2.0, 2.0, -1.0)
    return RoutePrefixCurriculum([RouteCurriculumStage("prefix40", 40), RouteCurriculumStage("prefix159", 159)], promotion_success_rate=thr[0],
                                 promotion_route_ready_hit_rate=thr[1], promotion_orientation_hit_rate=thr[2], promotion_max_regression_rate=thr[3],
                                 window_episodes=8, min_episodes_per_stage=8)


def _trainer(a, route, seq, curriculum=None, chunk=None, n=256):
    from rl_brain_trainer_b200 import ppo

    t = ppo.PPOTrainer(a["cfg"], ppo.random_policy(80, seed=a["policy_seed"], log_std_init=-0.5, device="cuda"), num_envs=n,
                       hyper=dataclasses.replace(a["hp"]), seed=a["seed"], route=route, route_sequence_config=seq, route_curriculum=curriculum)
    if chunk is not None:
        t.route_chunk_steps = chunk
    return t


def _assert_same(alone, member, k):
    tensors = ("params", "adam_m", "adam_v", "weight_image", "obs_buf", "obs_img", "act_buf", "logp_buf", "val_buf", "rew_buf", "done_buf",
               "start_buf", "_route_raw", "adv_buf", "ret_buf", "tile_sums", "last_val", "_next_start", "boot_count", "stats_accum")
    for name in tensors:
        assert torch.equal(getattr(alone, name), getattr(member, name)), f"member {k}: {name} differs"
    assert torch.equal(alone.env.state, member.env.state), f"member {k}: env state differs"
    assert (alone.global_step, alone.num_timesteps, alone.update_count) == (member.global_step, member.num_timesteps, member.update_count)
    assert alone.env.config.reset_config == member.env.config.reset_config, f"member {k}: route window differs"


def _run(k, iterations, sequence, curricula=None, chunk=None):
    from rl_brain_trainer_b200.population import PPOPopulation

    route, renv, seq = _route_setup()
    seq = seq if sequence else None
    args = _members(k, renv)
    cur = curricula or (lambda i: None)
    alone = [_trainer(a, route, seq, cur(i), chunk) for i, a in enumerate(args)]
    logs_alone = [t.learn(iterations) for t in alone]
    pop = PPOPopulation([_trainer(a, route, seq, cur(i), chunk) for i, a in enumerate(args)])
    logs_pop = pop.learn(iterations)
    torch.cuda.synchronize()
    for i in range(k):
        _assert_same(alone[i], pop.members[i], i)
        assert [{**r, "member": i} for r in logs_alone[i]] == logs_pop[i]
    return alone, pop


@pytest.mark.parametrize("sequence", [False, True], ids=["plain", "sequence"])
@pytest.mark.parametrize("k", [1, 3])
def test_route_members_are_standalone_trainers(k, sequence):
    """256 envs x 16 steps, 20-step episodes (time-limit episodes inside the run), 2 epochs of 4 minibatches, 3 iterations."""
    _, pop = _run(k, 3, sequence)
    boots = [int(t.boot_count.item()) for t in pop.members]
    assert all(b > 0 for b in boots), boots            # every member bootstrapped time-limit episodes in the last rollout


def test_route_members_with_their_own_prefix_curricula():
    """Per-member prefix curricula, 4-step chunks of a 16-step rollout: member 0 is promoted mid-rollout (its window widens from the
    next chunk on), members 1 and 2 are not."""
    alone, pop = _run(3, 2, True, curricula=lambda i: _curriculum(i == 0), chunk=4)
    stages = [t.route_curriculum.current_stage_index for t in pop.members]
    assert stages == [1, 0, 0], stages
    hist = pop.members[0].route_curriculum.history
    assert len(hist) == 1 and hist[0]["total_timesteps"] % pop.members[0].S != 0, hist        # inside a rollout, not at its end
    assert hist == alone[0].route_curriculum.history
    windows = [t.env.config.reset_config.max_route_index for t in pop.members]
    assert windows[0] == 159 and windows[1] == windows[2] == 40, windows


def test_route_scope_errors_raise_before_any_launch():
    from rl_brain_trainer_b200 import _lib, ppo
    from rl_brain_trainer_b200.population import PPOPopulation

    route, renv, seq = _route_setup()
    a = _members(1, renv)[0]

    def tr(**kw):
        hp = dataclasses.replace(a["hp"], target_kl=kw.pop("target_kl", None))
        return ppo.PPOTrainer(kw.pop("cfg", renv), ppo.random_policy(80, seed=0, device="cuda"), num_envs=256, hyper=hp, route=kw.pop("route", route),
                              route_sequence_config=kw.pop("seq", seq), **kw)

    ok = tr()
    before = ok.params.clone(), ok.env.state.clone(), ok.obs_buf.clone()
    arm = ppo.PPOTrainer(_arm_config(), ppo.random_policy(56, seed=0, device="cuda"), num_envs=256, hyper=ppo.PPOHyper(n_steps=16, batch_size=1024))
    with pytest.raises(ValueError, match="mixed"):
        PPOPopulation([ok, arm])
    with pytest.raises(ValueError, match="same route"):
        PPOPopulation([ok, tr(route=_route_setup(seed=8)[0])])
    with pytest.raises(ValueError, match="env config"):
        PPOPopulation([ok, tr(cfg=_route_setup(episode_steps=24)[1])])
    with pytest.raises(ValueError, match="sequence wrapper"):
        PPOPopulation([ok, tr(seq=None)])
    with pytest.raises(ValueError, match="sequence wrapper"):
        PPOPopulation([ok, tr(seq=dataclasses.replace(seq, reset_ready_streak_on_advance=False))])
    with pytest.raises(ValueError, match="prefix curriculum"):
        PPOPopulation([ok, tr(route_curriculum=_curriculum(False))])
    chunky = tr()
    chunky.route_chunk_steps = 8
    with pytest.raises(ValueError, match="route_chunk_steps"):
        PPOPopulation([ok, chunky])
    with pytest.raises(ValueError, match="collect_variant"):
        PPOPopulation([ok, tr(collect_variant="steps")])
    with pytest.raises(ValueError, match="target_kl"):
        PPOPopulation([ok, tr(target_kl=0.01)])
    with pytest.raises(ValueError, match="per-sample"):
        PPOPopulation([ok, tr(shuffle="sample")])
    torch.cuda.synchronize()
    assert torch.equal(before[0], ok.params) and torch.equal(before[1], ok.env.state) and torch.equal(before[2], ok.obs_buf)
    assert ok.global_step == 0 and ok.update_count == 0

    L = _lib.lib()
    fake = 4096       # never dereferenced: every call below fails its argument checks first
    for call in (lambda: L.kin_pop_route_collect(None, None, fake, fake, 1, 256, 16, 0, 1, 1, None),
                 lambda: L.kin_pop_route_collect(ok.env._params.handle, ctypes.byref(ok.env.table.c), fake, None, 1, 256, 16, 0, 1, 1, None),
                 lambda: L.kin_pop_route_collect(ok.env._params.handle, ctypes.byref(ok.env.table.c), fake, fake, 1, 200, 16, 0, 1, 1, None),
                 lambda: L.kin_pop_route_collect(ok.env._params.handle, ctypes.byref(ok.env.table.c), fake, fake, 1, 256, 16, -1, 1, 1, None),
                 lambda: L.kin_pop_route_bootstrap_list(fake, 65, 256, 128, 0, None),
                 lambda: L.kin_pop_route_bootstrap_list(fake, 1, 256, 128, -4, None),
                 lambda: L.kin_pop_route_obs_images(fake, None, 1, 4096, None),
                 lambda: L.kin_pop_route_obs_images(fake, fake, 1, 100, None),
                 lambda: L.kin_pop_route_logp(fake, 1, None, 64, 148, None),
                 lambda: L.kin_pop_route_logp(fake, 1, fake, 63, 148, None),
                 lambda: L.kin_pop_route_grad_tc(None, 1, 0, 8, 512, 148, None),
                 lambda: L.kin_pop_route_grad_tc(fake, 1, 0, 7, 448, 148, None),
                 lambda: L.kin_pop_route_adam(fake, 0, None, None, None)):
        with pytest.raises(_lib.KinError, match="kin_pop_route_"):
            _lib.check(call())


def _arm_config():
    from ._util import env_config

    return env_config("approach_default")
