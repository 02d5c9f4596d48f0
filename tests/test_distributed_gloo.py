"""world_size-2 gloo tests (CPU) of the multi-rank host logic: sharding, gradient / statistics all-reduce, curriculum agreement."""

from __future__ import annotations

import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, out_dir: str) -> None:
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from rl_brain_trainer_b200 import distributed as kd

    # 1. episode sharding: every unit owned exactly once, contiguous
    n_total = 1001
    sl = kd.shard_slice(n_total, rank, world)
    owned = torch.zeros(n_total)
    owned[sl] = 1
    kd.allreduce_sum_(owned)
    assert torch.equal(owned, torch.ones(n_total))
    # 2. gradient all-reduce: each rank holds the sum over ITS samples of per-sample grads / global batch
    g = torch.Generator().manual_seed(0)
    per_sample = torch.randn(64, 16143, generator=g)              # same on both ranks
    mine = per_sample[rank::world]
    grad = mine.sum(0) / 64.0
    kd.allreduce_sum_(grad)
    assert torch.allclose(grad, per_sample.mean(0), atol=1e-6)
    # 3. eval statistics: success rate over the union of the shards
    success = (torch.arange(n_total) % 3 == 0)[sl]
    pos = torch.full((success.numel(),), 0.002 * (rank + 1))
    stats = kd.reduce_eval_stats(success, pos, pos * 2, env_steps=int(success.numel()) * 164)
    assert stats["episodes"] == n_total and abs(stats["success_rate"] - float((torch.arange(n_total) % 3 == 0).double().mean())) < 1e-12
    assert stats["env_steps"] == n_total * 164
    # 4. curriculum: ranks see different local outcomes but promote together
    tr = kd.CurriculumTracker(n_stages=4, success_rate_threshold=0.68, window_episodes=32, min_episodes_per_stage=64, stage_index=0)
    single = kd.CurriculumTracker(n_stages=4, success_rate_threshold=0.68, window_episodes=32, min_episodes_per_stage=64, stage_index=0)
    promoted = []
    g2 = torch.Generator().manual_seed(5)
    for it in range(6):          # both ranks draw the same GLOBAL rollout [T=8, N=24], each keeps its env shard; rates rise with `it`
        fin = torch.rand((8, 24), generator=g2) < 0.5
        suc = (torch.rand((8, 24), generator=g2) < 0.45 + 0.1 * it) & fin
        mine = slice(rank * 12, (rank + 1) * 12)
        promoted.append(tr.record_rollout(fin[:, mine], suc[:, mine]))
        single.record_stream(suc[fin].to(torch.int32))        # the single-process order: time step, then env index
        assert tr.history == single.history and tr.stage_index == single.stage_index and tr.stage_episode_count == single.stage_episode_count
        assert np.array_equal(tr.recent, single.recent)
    np.save(os.path.join(out_dir, f"promoted_{rank}.npy"), np.array(promoted))
    mx = torch.tensor([float(rank)])
    kd.allreduce_max_(mx)
    assert float(mx) == world - 1
    dist.destroy_process_group()


def test_two_rank_gloo(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a, b = np.load(tmp_path / "promoted_0.npy"), np.load(tmp_path / "promoted_1.npy")
    assert np.array_equal(a, b)            # identical decisions on both ranks ...
    assert a.sum() >= 1                    # ... and the stream does promote (each rank also checked itself against the single-process replay)


def test_single_process_helpers():
    from rl_brain_trainer_b200 import distributed as kd

    assert kd.world() == (0, 1)
    parts = [kd.shard_slice(10, r, 4) for r in range(4)]
    assert [p.stop - p.start for p in parts] == [3, 3, 2, 2] and parts[0].start == 0 and parts[-1].stop == 10
    t = torch.ones(3)
    assert kd.allreduce_sum_(t) is t
    tr = kd.CurriculumTracker(3, 0.8, 20, 30)
    assert tr.record_stream([1] * 10 + [0] * 10) == 0            # below min_episodes_per_stage
    assert tr.record_stream([1] * 19 + [0]) == 1 and tr.stage_index == 1 and tr.stage_episode_count == 4   # promoted at the 16th success of the window
    assert tr.history[0]["trigger_success_rate"] == 0.8


def test_curriculum_tracker_matches_sequential_restatement_of_the_reference():
    """``CurriculumTracker.record_stream`` (vectorised replay) against a plain per-episode restatement of ``PointCurriculumTracker.
    record_episode`` (envs/curriculum.py:117-142) on random outcome streams cut into random chunks."""
    from collections import deque

    from rl_brain_trainer_b200 import distributed as kd

    rng = np.random.default_rng(12)
    for case in range(40):
        n_stages, W, M = int(rng.integers(2, 6)), int(rng.integers(1, 40)), int(rng.integers(1, 90))
        thr = float(rng.choice([0.5, 0.68, 0.8, 0.9, 1.0]))
        stream = (rng.random(int(rng.integers(50, 1500))) < rng.uniform(0.4, 0.98)).astype(int)
        # sequential restatement
        stage, count, dq, hist = 0, 0, deque(maxlen=W), []
        for s_ in stream:
            count += 1
            dq.append(int(s_))
            if stage >= n_stages - 1 or count < M or len(dq) < W:
                continue
            rate = float(sum(dq)) / float(len(dq))
            if rate >= thr:
                hist.append((stage, stage + 1, rate))
                stage, count = stage + 1, 0
                dq.clear()
        tr = kd.CurriculumTracker(n_stages, thr, W, M)
        pos = 0
        while pos < stream.size:
            step = int(rng.integers(1, 400))
            tr.record_stream(stream[pos:pos + step])
            pos += step
        assert tr.stage_index == stage and tr.stage_episode_count == count and tr.recent.tolist() == list(dq), case
        assert [(h["from_stage_index"], h["to_stage_index"], h["trigger_success_rate"]) for h in tr.history] == hist, case
