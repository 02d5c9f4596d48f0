"""CPU tests of the adaptive frontier curriculum's host side: alias table, CSR grouping of the training map, builder validation,
the C ABI of the frontier sampler fields and the multi-rank table-checksum check."""

from __future__ import annotations

import ctypes
import os

import numpy as np
import pytest
import torch

from rl_brain_trainer_b200 import _lib, coverage as cov, workspace as ws
from rl_brain_trainer_b200.kinematics import fk_pose6_folded

from ._util import env_config


def _encoded(prob: np.ndarray, alias: np.ndarray) -> np.ndarray:
    """The issue's formula written out: (prob[k] + sum_{j: alias[j] = k} (1 - prob[j])) / B."""
    B = prob.size
    return np.array([(prob[k] + sum(1.0 - prob[j] for j in range(B) if alias[j] == k)) / B for k in range(B)])


@pytest.mark.parametrize("weights", [
    [0.7],                                                           # one bucket
    [0.2] * 9,                                                       # equal weights
    list(np.random.default_rng(3).uniform(0.05, 1.1, 41)),           # the priority range of update_bucket_priorities
    [0.0, 1.1, 0.05, 0.0, 0.95, 0.15, 0.0, 0.25, 1.0, 0.0],          # zero-weight buckets
])
def test_alias_table_encodes_the_normalised_weights(weights):
    w = np.asarray(weights, dtype=np.float64)
    prob, alias = cov.alias_table(w)
    want = w / w.sum()
    for p, a in ((prob, alias), (prob.astype(np.float32).astype(np.float64), alias)):      # fp64 build and its fp32 image
        assert np.abs(_encoded(p, a) - want).max() < 1e-6
        assert np.abs(cov.alias_probabilities(p, a) - want).max() < 1e-6
    assert np.all((prob >= 0) & (prob <= 1)) and np.all((alias >= 0) & (alias < w.size))
    assert np.all(prob[w == 0] == 0.0)              # a zero-weight bucket is never drawn as itself ...
    assert not np.isin(np.nonzero(w == 0)[0], alias[prob < 1]).any()     # ... nor as anyone's alias


def _maps():
    cfg = env_config("approach_dynamic_scale_big")
    ev = ws.generate_workspace_target_map(cfg, seed=11, stage_samples_per_stage=8, random_samples=40)
    tr = ws.generate_workspace_target_map(cfg, seed=12, stage_samples_per_stage=16, random_samples=80)
    return ev, tr


def test_target_buckets_without_bounds_is_unchanged():
    ev, _ = _maps()
    b = cov.target_buckets(ev)
    # restatement of the parent's function body
    pose = np.array([fk_pose6_folded(q) for q in ev.q]).reshape(-1, 6)
    lo, hi = pose[:, :3].min(axis=0) - 1e-6, pose[:, :3].max(axis=0) + 1e-6
    xyz = np.clip(np.floor((pose[:, :3] - lo) / np.maximum(hi - lo, 1e-9) * 8), 0, 7).astype(int)
    ori = np.clip(np.floor(np.linalg.norm(pose[:, 3:], axis=1) / np.pi * 6), 0, 5).astype(int)
    qb = np.clip(np.floor(np.linalg.norm(ev.q, axis=1) / 4.5 * 6), 0, 5).astype(int)
    ids = [f"x{a}_y{b_}_z{c}_o{o}_q{q}" for (a, b_, c), o, q in zip(xyz, ori, qb)]
    index: dict[str, int] = {}
    code = np.array([index.setdefault(s, len(index)) for s in ids], dtype=np.int64)
    assert np.array_equal(b.code, code) and b.ids == list(index) and np.array_equal(b.pose6, pose)
    assert np.array_equal(b.lo, lo) and np.array_equal(b.hi, hi)
    same = cov.target_buckets(ev, bounds=(b.lo, b.hi))
    assert np.array_equal(same.code, b.code) and same.ids == b.ids


def test_target_buckets_with_bounds_clip_to_the_edge_bins():
    ev, tr = _maps()
    eb = cov.target_buckets(ev)
    mid = 0.5 * (eb.lo + eb.hi)
    lo, hi = mid - 0.25 * (eb.hi - eb.lo), mid + 0.25 * (eb.hi - eb.lo)      # a box smaller than the map: many targets outside
    b = cov.target_buckets(tr, bounds=(lo, hi))
    assert np.array_equal(b.lo, lo) and np.array_equal(b.hi, hi)
    bins = np.array([[int(s.split("_")[k][1:]) for k in range(3)] for s in np.asarray(b.ids)[b.code]])
    pos = b.pose6[:, :3]
    below, above = pos < lo, pos >= hi
    assert below.any() and above.any()
    assert np.all(bins[below] == 0) and np.all(bins[above] == 7)
    inside = ~below & ~above
    assert np.array_equal(bins[inside], np.floor((pos - lo) / (hi - lo) * 8).astype(int)[inside])


def test_frontier_table_groups_every_target_once_in_its_bucket():
    ev, tr = _maps()
    eb = cov.target_buckets(ev)
    tb = cov.target_buckets(tr, bounds=(eb.lo, eb.hi))
    rng = np.random.default_rng(5)
    seen = [b for b in tb.ids if rng.random() < 0.6]
    prio = {b: float(rng.uniform(0.05, 1.1)) for b in seen}
    prio.update({"x9_y9_z9_o9_q9": 1.0, "x8_y8_z8_o8_q8": 0.5})      # buckets the training map does not have: dropped
    t = cov.FrontierTable.build(tr, tb, prio, default_priority=0.2, device="cpu")
    assert t.dropped_bucket_count == 2 and t.defaulted_bucket_count == len(tb.ids) - len(seen)
    assert t.bucket_count == tb.count and t.target_count == tr.q.shape[0]
    off = t.offsets.numpy()
    assert off[0] == 0 and off[-1] == t.target_count and np.all(np.diff(off) > 0)
    assert np.array_equal(np.sort(t.target_index), np.arange(tr.q.shape[0]))           # every training target exactly once
    rows = t.targets.numpy()
    for k, bid in enumerate(t.bucket_ids):
        members = t.target_index[off[k]:off[k + 1]]
        assert all(tb.ids[c] == bid for c in tb.code[members])                         # ... in a bucket with its own code
        assert np.array_equal(rows[off[k]:off[k + 1], :7], tr.q[members].astype(np.float32))
        assert np.array_equal(rows[off[k]:off[k + 1], 7], tr.stage[members].astype(np.float32))
        assert t.weights[k] == prio.get(bid, 0.2)
    assert np.abs(t.probabilities - t.weights / t.weights.sum()).max() < 1e-6
    assert t.alias_prob.dtype == torch.float32 and t.alias_index.dtype == torch.int32 and t.offsets.dtype == torch.int32
    # BucketPriority rows (update_bucket_priorities' output) build the same table
    rows_in = [cov.BucketPriority(b, 0.0, 0.0, 0.0, None, 0, "x", p) for b, p in prio.items()]
    assert cov.FrontierTable.build(tr, tb, rows_in, default_priority=0.2, device="cpu").checksum == t.checksum


def test_frontier_table_rejects_bad_input():
    ev, tr = _maps()
    tb = cov.target_buckets(tr)
    empty = ws.TargetMap(q=np.zeros((0, 7)), stage=np.zeros(0, dtype=np.int64))
    with pytest.raises(ValueError, match="empty"):
        cov.FrontierTable.build(empty, cov.TargetBuckets(code=np.zeros(0, dtype=np.int64), ids=[], pose6=np.zeros((0, 6))), {}, device="cpu")
    with pytest.raises(ValueError, match="not all zero"):
        cov.FrontierTable.build(tr, tb, {b: 0.0 for b in tb.ids}, default_priority=0.0, device="cpu")
    with pytest.raises(ValueError, match="non-finite"):
        cov.FrontierTable.build(tr, tb, {tb.ids[0]: float("nan")}, device="cpu")
    with pytest.raises(ValueError, match="non-finite"):
        cov.FrontierTable.build(tr, tb, {}, default_priority=float("inf"), device="cpu")


def test_sampler_struct_has_the_frontier_fields_and_abi_4():
    S = _lib.c_struct("KinSamplerParams")
    names = [f for f, _ in S._fields_]
    tail = ["frontier_probability", "frontier_bucket_count", "frontier_target_count", "frontier_bucket_offset", "frontier_alias_prob",
            "frontier_alias_index", "frontier_targets"]
    assert names[-len(tail):] == tail and names[-len(tail) - 1] == "dock_handoff_states"      # appended: no existing offset moved
    assert S.frontier_probability.offset == S.dock_handoff_states.offset + ctypes.sizeof(ctypes.c_void_p)
    assert _lib.define("KIN_ABI_VERSION") == 4 and _lib.define("KIN_FRONTIER_TARGET_FLOATS") == 8
    assert _lib.lib().kin_abi_version() == 4


def test_set_sampler_rejects_bad_frontier_fields():
    """Validation happens before the device copy, so the rejections are checkable without a GPU."""
    from rl_brain_trainer_b200 import params as kparams

    cfg = env_config("approach_dynamic_scale_big")
    L = _lib.lib()
    p = kparams.env_params(cfg)
    h = ctypes.c_void_p()
    _lib.check(L.kin_params_create(ctypes.byref(p), ctypes.byref(h)))
    dummy = ctypes.c_void_p(4096)
    try:
        def attempt(**fields):
            s = kparams.sampler_params(cfg, 3)
            s.random_start_enabled = 1
            s.frontier_probability, s.frontier_bucket_count, s.frontier_target_count = 0.5, 4, 10
            s.frontier_bucket_offset = s.frontier_alias_prob = s.frontier_alias_index = s.frontier_targets = dummy.value
            for k, v in fields.items():
                setattr(s, k, v)
            code = L.kin_params_set_sampler(h, ctypes.byref(s))
            return code, L.kin_last_error_string().decode()

        for bad in (float("nan"), float("inf"), -0.1, 1.5):
            code, msg = attempt(frontier_probability=bad)
            assert code == _lib.define("KIN_ERR_INVALID_ARG") and "frontier_probability" in msg, bad
        for fields, word in (({"frontier_bucket_count": 0}, "counts"), ({"frontier_target_count": 0}, "counts"),
                             ({"frontier_alias_prob": None}, "pointers"), ({"frontier_targets": None}, "pointers"),
                             ({"random_start_enabled": 0}, "random_start")):
            code, msg = attempt(**fields)
            assert code == _lib.define("KIN_ERR_INVALID_ARG") and word in msg, fields
    finally:
        L.kin_params_destroy(h)


def test_curriculum_reads_the_preset_and_keeps_the_training_map_apart():
    from rl_brain_trainer_b200 import config as kcfg

    preset = kcfg.preset_dict("randomstart_overnight")
    fw = preset["full_workspace_randomstart"]
    cur = cov.FrontierCurriculum.from_config(preset, train_stage_samples_per_stage=8, train_random_samples=32)
    kw = cur.eval_kwargs
    assert kw["pair_count"] == fw["pair_count"] and kw["episodes_per_split"] == fw["eval_episodes_per_split"]
    assert kw["stage_samples_per_stage"] == fw["target_stage_samples_per_stage"] and kw["random_target_samples"] == fw["target_random_samples"]
    assert kw["random_start_samples"] == fw["start_random_samples"] and kw["variant"] == cov.VARIANT_FFMA
    assert cur.refresh_interval == preset["workspace_expansion"]["eval_interval"] and cur.probability == 0.5
    assert cur.train_seed != kw["seed"] + 1 and cur.train_targets.q.shape[0] == 12 * 8 + 32
    with pytest.raises(ValueError):
        cov.FrontierCurriculum.from_config(preset, train_seed=kw["seed"] + 1)


# ---- world_size-2 gloo: the table-checksum check ------------------------------------------------------------------------------
def _worker(rank: int, world: int, port: int) -> None:
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from rl_brain_trainer_b200 import distributed as kd

    kd.check_same_on_all_ranks("0123456789abcdef", "table")           # equal on both ranks: passes
    with pytest.raises(RuntimeError, match="differs between ranks"):
        kd.check_same_on_all_ranks(f"checksum-{rank}", "table")      # differs: raises on EVERY rank
    dist.destroy_process_group()


def test_table_checksum_mismatch_raises_on_every_rank():
    import torch.multiprocessing as mp

    from .test_distributed_gloo import _free_port

    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
