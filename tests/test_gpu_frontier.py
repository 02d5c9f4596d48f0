"""GPU tests of the adaptive frontier curriculum: the device sampler's frontier branch (distribution, unarmed invariance, K4 / K1
agreement) and the PPO training loop that refreshes the table from coverage evals."""

from __future__ import annotations

import dataclasses

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import kin_oracle as ko

from ._util import env_config, oracle_params

pytestmark = pytest.mark.gpu

STAGE = 8


def _cfg(*, min_pair=None, sources=None, episode_steps=None):
    cfg = env_config("randomstart_overnight")
    w = dict(cfg.workspace_stage_sampling)
    r = dict(w["random_start_pair_sampling"])
    if min_pair is not None:
        r["min_pair_joint_l2"] = min_pair
    if sources is not None:
        keys = ("home_start_ratio", "old_successful_start_ratio", "random_valid_q_start_ratio", "frontier_pair_ratio",
                "failure_recovery_start_ratio", "stress_start_ratio")
        r.update(dict(zip(keys, sources)))
    w["random_start_pair_sampling"] = r
    cfg = dataclasses.replace(cfg, workspace_stage_sampling=w)
    if episode_steps is not None:
        cfg = dataclasses.replace(cfg, episode_length=episode_steps,
                                  termination_config=dataclasses.replace(cfg.termination_config, max_episode_steps=episode_steps))
    return cfg


def _synthetic_table(cfg, n_buckets=40, seed=0):
    """~40 buckets of unequal sizes and priorities; targets uniform inside the joint limits, stages in {-1, 0 .. 11}."""
    from rl_brain_trainer_b200 import coverage as cov, workspace as ws

    rng = np.random.default_rng(seed)
    sizes = rng.integers(1, 60, n_buckets)
    code = np.repeat(np.arange(n_buckets), sizes)
    rng.shuffle(code)
    lo, hi = np.array([s.lower for s in cfg.joint_specs]), np.array([s.upper for s in cfg.joint_specs])
    lo, hi = lo + 0.05 * (hi - lo), hi - 0.05 * (hi - lo)
    q = rng.uniform(lo, hi, (code.size, 7))
    stage = rng.integers(-1, 12, code.size)
    targets = ws.TargetMap(q=q, stage=stage)
    buckets = cov.TargetBuckets(code=code, ids=[f"b{k}" for k in range(n_buckets)], pose6=np.zeros((code.size, 6)))
    prio = {f"b{k}": float(v) for k, v in enumerate(rng.uniform(0.05, 1.1, n_buckets))}
    return cov.FrontierTable.build(targets, buckets, prio, device="cuda")


def _match(table, goal_q: torch.Tensor) -> np.ndarray:
    """Table row of every goal (-1: not a table target), by exact fp32 equality."""
    rows = table.targets[:, :7].cpu().numpy()
    index = {r.tobytes(): i for i, r in enumerate(rows)}
    g = np.ascontiguousarray(goal_q.cpu().numpy().astype(np.float32))
    return np.array([index.get(r.tobytes(), -1) for r in g])


def _env(cfg, n, seed=17, **kw):
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv

    env = BatchedArmKinematicEnv(cfg, n, "cuda", seed=seed, host_sampler=False, **kw)
    env.set_curriculum_stage(STAGE)
    return env


def test_frontier_resets_follow_the_table():
    n, p = 262144, 0.5
    cfg = _cfg(min_pair=0.0)           # no retries: the bucket draw is the table's distribution exactly
    table = _synthetic_table(cfg)
    env = _env(cfg, n)
    env.set_frontier_targets(table, p)
    obs, _ = env.reset()
    torch.cuda.synchronize()
    row = _match(table, env.goal_q)
    hit = row >= 0
    m = int(hit.sum())
    assert abs(m / n - p) < 4 * np.sqrt(p * (1 - p) / n), m / n
    # buckets: chi-square against the probabilities the alias table encodes
    slot = np.searchsorted(table.offsets.cpu().numpy(), row[hit], side="right") - 1
    counts = np.bincount(slot, minlength=table.bucket_count)
    chi = stats.chisquare(counts, table.probabilities * m / table.probabilities.sum())
    assert chi.pvalue > 1e-4, chi
    # targets inside a bucket: uniform (pooled chi-square over the buckets with more than one target)
    per_row = np.bincount(row[hit], minlength=table.target_count)
    off = table.offsets.cpu().numpy()
    x2, dof = 0.0, 0
    for k in range(table.bucket_count):
        c = per_row[off[k]:off[k + 1]]
        if c.size > 1:
            e = c.sum() / c.size
            x2 += float(((c - e) ** 2 / e).sum())
            dof += c.size - 1
    assert stats.chi2.sf(x2, dof) > 1e-4, (x2, dof)
    # stage flag: the table's stage, the current stage for uniform-valid (-1) targets
    tstage = table.targets[:, 7].cpu().numpy().astype(int)
    flag = env.counters()["stage"].cpu().numpy()
    want = np.where(tstage[row[hit]] < 0, STAGE, tstage[row[hit]])
    assert np.array_equal(flag[hit], want) and (tstage[row[hit]] < 0).any()
    # observations of frontier-reset envs == the oracle's observation of the same state
    idx = np.nonzero(hit)[0][:256]
    orc = ko.OracleEnv(oracle_params(cfg))
    f64 = lambda t: t[idx].cpu().numpy().astype(np.float64)  # noqa: E731
    iq, gq, dq, pa = f64(env.q), f64(env.goal_q), f64(env.dq), f64(env.prev_action)
    ref = np.stack([orc.reset(mode=0, initial_q=iq[i], goal_q=gq[i], initial_dq=dq[i], initial_prev_action=pa[i]) for i in range(idx.size)])
    assert np.abs(obs[idx].cpu().numpy() - ref).max() < 2e-5


def test_failure_recovery_starts_jitter_their_frontier_goal_and_pairs_keep_their_distance():
    cfg = _cfg(min_pair=0.0, sources=(0, 0, 0, 0, 1.0, 0))      # every start is a failure-recovery start
    table = _synthetic_table(cfg, seed=1)
    n = 65536
    env = _env(cfg, n, seed=3)
    env.set_frontier_targets(table, 0.5)
    env.reset()
    hit = _match(table, env.goal_q) >= 0
    assert 0.45 < hit.mean() < 0.55
    noise = np.array(cfg.workspace_stage_sampling["random_start_pair_sampling"]["failure_recovery_q_noise"], dtype=np.float32)
    d = (env.q - env.goal_q).abs().cpu().numpy()[hit]
    inside = (d <= noise * (1 + 1e-5) + 1e-6).all(axis=1)
    assert inside.mean() > 1 - 1e-4, inside.mean()       # (a source draw of exactly 0 picks "home": probability 2^-24 per reset)
    # the preset's min_pair_joint_l2 with its own source mix: every pair keeps the distance unless the 12 retries ran out
    cfg2 = _cfg()
    l2 = cfg2.workspace_stage_sampling["random_start_pair_sampling"]["min_pair_joint_l2"]
    env2 = _env(cfg2, 262144, seed=5)
    env2.set_frontier_targets(_synthetic_table(cfg2, seed=2), 0.5)
    env2.reset()
    dist = (env2.q - env2.goal_q).norm(dim=1).cpu().numpy()
    rate = float((dist < l2 * (1 - 1e-5)).mean())
    print(f"min_pair_joint_l2 {l2}: retry cap exhausted for {rate:.2e} of 262144 resets")
    assert rate < 1e-3


def test_unarmed_sampler_is_the_plain_sampler():
    """Never armed, armed at p = 0, and armed-uploaded-then-cleared give bitwise the same resets and auto-resets."""
    cfg = _cfg(episode_steps=12)
    n = 4096
    table = _synthetic_table(cfg, seed=4)
    envs = [_env(cfg, n, seed=9, auto_reset=True) for _ in range(4)]
    envs[1].set_frontier_targets(table, 0.0)
    envs[2].set_frontier_targets(table, 0.5)
    envs[2]._ensure_sampler()                      # the armed table reaches the device ...
    envs[2].set_frontier_targets(None)             # ... and is cleared again before the first reset
    envs[3].set_frontier_targets(table, 0.5)       # armed: must differ
    for e in envs:
        e.reset()
    torch.cuda.synchronize()
    for e in envs[1:3]:
        assert torch.equal(e.state, envs[0].state)
    assert not torch.equal(envs[3].goal_q, envs[0].goal_q)
    g = torch.Generator(device="cuda").manual_seed(0)
    resets = 0
    for _ in range(3 * 12):                        # three episodes of K1 auto-resets
        a = torch.rand((n, 7), generator=g, device="cuda") * 2 - 1
        for e in envs:
            e.step(a)
        resets += int(((envs[0].done & 3) != 0).sum())
        for e in envs[1:3]:
            assert torch.equal(e.state, envs[0].state) and torch.equal(e.obs, envs[0].obs) and torch.equal(e.done, envs[0].done)
    assert resets >= 3 * n


def test_fused_collection_replays_through_the_step_kernel_with_frontier_targets():
    """K4 (kin_ppo_collect, in-register auto-reset) against K1 (kin_env_step with auto-reset) with the frontier branch armed at
    p = 0.7: replaying the recorded actions reproduces done bytes, rewards and the final SoA state bit for bit."""
    from rl_brain_trainer_b200 import ppo

    from .test_gpu_ppo import _torch_forward

    cfg = _cfg(episode_steps=24)
    T, n = 60, 512
    pol = ppo.random_policy(56, seed=2, log_std_init=-1.5, device="cuda")
    pol.tensors["act_w"].mul_(40.0)
    hp = ppo.PPOHyper(n_steps=T, batch_size=n * T // 4, n_epochs=1, gamma=0.97, learning_rate=0.0)
    tr = ppo.PPOTrainer(cfg, pol, num_envs=n, hyper=hp, seed=11, stage_index=STAGE, update_variant="tc", collect_variant="fused")
    tr.tiles_per_cta = 2
    table = _synthetic_table(cfg, seed=6)
    tr.env.set_frontier_targets(table, 0.7)
    replay = _env(cfg, n, seed=tr.env._seed, auto_reset=True, with_aux=False)
    replay.set_frontier_targets(table, 0.7)
    replay._ensure_sampler()
    replay.state.copy_(tr.env.state)
    tr.collect()
    torch.cuda.synchronize()
    from_table = resets = 0
    for t in range(T):
        replay.step_raw(tr.act_buf[t].contiguous())
        torch.cuda.synchronize()
        assert torch.equal(replay.done, tr.done_buf[t]), t
        trunc = ((replay.done & 2) != 0) & ((replay.done & 1) == 0)
        plain = ~trunc
        assert torch.equal(tr.rew_buf[t][plain], replay.reward[plain]), (t, float((tr.rew_buf[t] - replay.reward)[plain].abs().max()))
        if bool(trunc.any()):        # TimeLimit bootstrap: r + gamma * V(terminal observation)
            _, tv = _torch_forward(pol, replay.terminal_obs)
            assert torch.allclose(tr.rew_buf[t][trunc], (replay.reward + hp.gamma * tv)[trunc], atol=2e-5)
        fin = ((replay.done & 3) != 0).cpu().numpy()
        if fin.any():
            resets += int(fin.sum())
            from_table += int((_match(table, replay.goal_q[torch.as_tensor(fin, device="cuda")]) >= 0).sum())
    assert torch.equal(replay.state[:, :n], tr.env.state[:, :n])
    assert resets > 0 and 0.5 * resets < from_table < 0.9 * resets, (from_table, resets)


def test_training_loop_refreshes_the_frontier_table():
    from rl_brain_trainer_b200 import coverage as cov, ppo
    from rl_brain_trainer_b200.policy import PolicyWeights

    cfg = _cfg(episode_steps=16)
    N, T = 1024, 32
    hp = ppo.PPOHyper(learning_rate=1e-6, n_steps=T, batch_size=N * T // 4, n_epochs=1, gamma=0.995, clip_range=0.08)
    cur = cov.FrontierCurriculum(cfg, refresh_interval=N * T, probability=0.5, pair_count=512, episodes_per_split=48,
                                 stage_samples_per_stage=16, random_target_samples=64, random_start_samples=64)
    tr = ppo.PPOTrainer(cfg, PolicyWeights.preset("randomstart", "cuda"), num_envs=N, hyper=hp, seed=4, stage_index=STAGE)
    log = tr.learn(2, frontier=cur)
    assert len(cur.history) >= 2
    assert cur.history[0]["previous_rate_bucket_count"] == 0 and cur.history[1]["previous_rate_bucket_count"] > 0
    assert any("previous_success_rate" in m for m in cur.last_summary["bucket_metrics"].values())
    for row in log:
        for k in ("frontier_known_success_rate", "frontier_covered_bucket_fraction", "frontier_table_bucket_count", "frontier_timesteps"):
            assert k in row and np.isfinite(row[k]), (k, row)
    assert log[1]["frontier_timesteps"] == 2 * N * T
    # the next rollout's resets draw from the newest table: the buckets holding the upper half of its probability mass get their share
    table = cur.table
    before = tr.env.goal_q.clone()
    tr.collect()
    changed = (tr.env.goal_q != before).any(dim=1)
    row = _match(table, tr.env.goal_q[changed])
    hit = row[row >= 0]
    assert hit.size > 200, hit.size
    slot = np.searchsorted(table.offsets.cpu().numpy(), hit, side="right") - 1
    top = table.probabilities >= np.median(table.probabilities)
    e = float(table.probabilities[top].sum())
    o = float(top[slot].mean())
    assert abs(o - e) < 5 * np.sqrt(e * (1 - e) / hit.size) + 0.02, (o, e, hit.size)
    # without a curriculum the rows keep today's keys
    plain = ppo.PPOTrainer(cfg, PolicyWeights.preset("randomstart", "cuda"), num_envs=N, hyper=hp, seed=4, stage_index=STAGE)
    keys = set(plain.learn(1)[0])
    assert not any(k.startswith("frontier_") for k in keys)
    assert keys == {"episodes", "successes", "mean_reward", "policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction", "grad_norm",
                    "minibatches", "stage", "timesteps"}


def test_frontier_targets_need_random_start_sampling():
    from rl_brain_trainer_b200 import _lib

    cfg = env_config("approach_dynamic_scale_big")        # no random-start pair sampling
    env = _env(cfg, 64)
    with pytest.raises(_lib.KinError):
        env.set_frontier_targets(_synthetic_table(_cfg(), seed=7), 0.5)
