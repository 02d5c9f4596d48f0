"""GPU tests of ``PPOPopulation``: every member of a population is bitwise the standalone ``PPOTrainer`` built with the same arguments
(parameters, Adam moments, weight image, env state, every rollout buffer, learn rows, counters, curriculum stage)."""

from __future__ import annotations

import dataclasses

import pytest
import torch

from ._util import env_config

pytestmark = pytest.mark.gpu


def _members(k: int, finisher: bool = False):
    """Per-member arguments that differ in everything a member may own: seed, initial policy, start stage, curriculum settings,
    PPO and Adam hyper-parameters."""
    from rl_brain_trainer_b200 import ppo

    base = env_config("finisher_noop_ft" if finisher else "approach_default")
    out = []
    for i in range(k):
        cfg = base
        if i == 0 and not finisher:     # host-side curriculum settings only: promoted after every 20 episodes, the env params stay identical
            cfg = dataclasses.replace(base, curriculum_config=dataclasses.replace(base.curriculum_config, success_rate_threshold=0.0,
                                                                                   min_episodes_per_stage=1))
        hp = ppo.PPOHyper(learning_rate=3e-4 * (1 + i), n_steps=16 if not finisher else 48, batch_size=1024, n_epochs=2, gamma=0.98 - 0.01 * i,
                          gae_lambda=0.95 - 0.02 * i, clip_range=0.2 + 0.05 * i, ent_coef=0.001 * i, vf_coef=0.5 + 0.1 * i,
                          max_grad_norm=0.5 + 0.25 * i, normalize_advantage=(i != 2), adam_beta1=0.9 - 0.02 * i, adam_eps=1e-5 * (1 + i))
        out.append(dict(cfg=cfg, hp=hp, seed=100 + 7 * i, stage=(0 if finisher else 1 + i), policy_seed=i))
    return out


def _policy(a, finisher):
    from rl_brain_trainer_b200 import ppo
    from rl_brain_trainer_b200.policy import PolicyWeights

    if finisher and a["policy_seed"] == 0:
        return PolicyWeights.preset("finisher", "cuda")
    return ppo.random_policy(56, seed=a["policy_seed"], log_std_init=-0.5, device="cuda")


def _trainer(a, n, finisher, handoff_rows):
    from rl_brain_trainer_b200 import ppo

    return ppo.PPOTrainer(a["cfg"], _policy(a, finisher), num_envs=n, hyper=dataclasses.replace(a["hp"]), seed=a["seed"], stage_index=a["stage"],
                          handoff_states=handoff_rows)


def _assert_same(alone, member, k):
    tensors = ("params", "adam_m", "adam_v", "weight_image", "obs_img", "act_buf", "logp_buf", "val_buf", "rew_buf", "done_buf", "start_buf",
               "adv_buf", "ret_buf", "tile_sums", "last_val", "_next_start", "boot_count", "stats_accum")
    for name in tensors:
        assert torch.equal(getattr(alone, name), getattr(member, name)), f"member {k}: {name} differs"
    assert torch.equal(alone.env.state, member.env.state), f"member {k}: env state differs"
    assert (alone.global_step, alone.num_timesteps, alone.update_count) == (member.global_step, member.num_timesteps, member.update_count)
    assert alone.env.get_curriculum_stage() == member.env.get_curriculum_stage()


def _run(k, n, iterations, finisher=False, handoff_rows=None):
    from rl_brain_trainer_b200.population import PPOPopulation

    args = _members(k, finisher)
    alone = [_trainer(a, n, finisher, handoff_rows) for a in args]
    logs_alone = [t.learn(iterations) for t in alone]
    pop = PPOPopulation([_trainer(a, n, finisher, handoff_rows) for a in args])
    logs_pop = pop.learn(iterations)
    torch.cuda.synchronize()
    for i in range(k):
        _assert_same(alone[i], pop.members[i], i)
        assert [{**r, "member": i} for r in logs_alone[i]] == logs_pop[i]
    return alone, pop


@pytest.mark.parametrize("k", [1, 3])
def test_members_are_standalone_trainers(k):
    """256 envs x 16 steps, 20-step episodes (finished and truncated inside the run), 2 epochs of 4 minibatches, 3 iterations."""
    alone, pop = _run(k, 256, 3)
    boots = [int(t.boot_count.item()) for t in pop.members]
    assert all(b > 0 for b in boots), boots            # every member bootstrapped time-limit episodes in the last rollout
    if k == 3:
        stages = [t.env.get_curriculum_stage() for t in pop.members]
        assert stages[0] > 1 and stages[1] == 2 and stages[2] == 3, stages       # member 0 was promoted, the others were not
        assert len({t.curriculum.stage_index for t in pop.members}) == 3


def test_finisher_members_with_shared_handoff_states():
    """Dock mode (Finisher training): resets replay Approach handoff states from one shared buffer; 48 steps > the 36-step limit."""
    from rl_brain_trainer_b200 import handoff
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    acfg = env_config("approach_dynamic_scale_big")
    buf, _ = handoff.build_finisher_handoff_state_buffer(acfg, PolicyWeights.preset("approach_stage8_11", "cuda"), stage_index=5,
                                                         suite=build_curriculum_local_eval_suite(acfg, seed=3, stage_index=5, n_episodes=256))
    rows = buf.device_rows("cuda")
    _, pop = _run(2, 256, 2, finisher=True, handoff_rows=rows)
    assert all(int(t.boot_count.item()) > 0 for t in pop.members)


def test_scope_errors_raise_before_any_launch():
    from rl_brain_trainer_b200 import _lib, ppo
    from rl_brain_trainer_b200.population import PPOPopulation

    cfg = env_config("approach_default")

    def tr(**kw):
        hp = ppo.PPOHyper(n_steps=16, batch_size=1024, n_epochs=1, target_kl=kw.pop("target_kl", None))
        return ppo.PPOTrainer(kw.pop("cfg", cfg), ppo.random_policy(56, seed=0, device="cuda"), num_envs=kw.pop("n", 256), hyper=hp, **kw)

    ok = tr()
    before = ok.params.clone(), ok.env.state.clone()
    with pytest.raises(ValueError, match="at least one"):
        PPOPopulation([])
    with pytest.raises(ValueError, match="target_kl"):
        PPOPopulation([ok, tr(target_kl=0.01)])
    with pytest.raises(ValueError, match="per-sample"):
        PPOPopulation([ok, tr(shuffle="sample")])
    with pytest.raises(ValueError, match="collect_variant"):
        PPOPopulation([ok, tr(collect_variant="steps")])
    with pytest.raises(ValueError, match="collect_variant"):
        PPOPopulation([ok, tr(update_variant="fp32", collect_variant="steps")])
    with pytest.raises(ValueError, match="one rank"):
        PPOPopulation([ok, tr(fused_update=True)])
    with pytest.raises(ValueError, match="lockstep"):
        PPOPopulation([ok, tr(n=384)])
    with pytest.raises(ValueError, match="env config"):
        PPOPopulation([ok, tr(cfg=env_config("approach_dynamic_scale_big"))])
    with pytest.raises(ValueError, match="twice"):
        PPOPopulation([ok, ok])
    frontier = tr()
    frontier.env._frontier = object()     # what set_frontier_targets leaves behind
    with pytest.raises(ValueError, match="frontier"):
        PPOPopulation([ok, frontier])
    with pytest.raises(TypeError):
        PPOPopulation([ok, "not a trainer"])
    torch.cuda.synchronize()
    assert torch.equal(before[0], ok.params) and torch.equal(before[1], ok.env.state) and ok.global_step == 0
    with pytest.raises(_lib.KinError, match="kin_pop_gae"):
        _lib.check(_lib.lib().kin_pop_gae(None, 1, 256, 16, None))
