"""Whole PPO updates (``PPOTrainer.update`` / ``PPOPopulation.update``, SB3 ``PPO.train()``) replayed minibatch by minibatch against the
fp64 oracle of ``tests/_ppo_oracle.py``, on every update path; and direct tests of the update entry points nothing else calls directly.

The trainer and the population reach the library only through ``self._L``.  The replay swaps that handle for a recorder that forwards
every call unchanged and, around the update-family entry points, clones device state on the current stream: the epoch's tile
permutation and advantage-statistics rows, the parameters / Adam moments / weight image each gradient launch reads, the gradient and
statistics it leaves, and what the optimiser step wrote.  Each recorded run must end bitwise equal to the same run without the recorder.

The replay is teacher-forced: every minibatch is judged from the device's own state before it, so errors do not build up and the
tolerances stay those the single-kernel tests in ``test_gpu_ppo.py`` justify.  Every minibatch of two consecutive ``update()`` calls is
checked: the minibatch's tiles, the advantage statistics the kernel received, the gradient, the bf16 weight image the launch read,
clip + Adam at the step count the oracle expects, the per-minibatch statistics, the running sums and what ``update()`` returns.
"""

from __future__ import annotations

import ctypes
import dataclasses
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from . import _ppo_oracle as oracle
from ._util import env_config

pytestmark = pytest.mark.gpu

GRAD_NORM, SKIP = 5, 7
ROLLOUT = ("act_buf", "adv_buf", "ret_buf", "tile_sums", "rew_buf", "val_buf", "start_buf", "done_buf", "last_val")

# Learning rate of the case that shows the replay tells fresh weights from stale ones: large enough that one Adam step moves the
# oracle gradient of the next minibatch by well over twice the tensor-core tolerance.  Measured on a B200 (1000 W) with one epoch per
# update: the smallest separation over its minibatches (max over tensors of rel. change / tolerance) is 6.3 at 1e-2 (3.1 at 2e-2, 7.5 at
# 3e-2), while its largest gradient error is 0.63 x the tolerance.  A second epoch at such rates revisits samples whose ratios the
# earlier steps pushed far outside the clip range (clip fraction 1): the few unclipped samples then carry bf16 log-prob errors beyond
# the tensor-core bounds (up to 0.16 per tensor), so the multi-epoch regime is covered by the other cases at ordinary rates.
STALE_LR = 1e-2


def _fields(c) -> dict:
    return {f: getattr(c, f) for f, _ in c._fields_}


def _hyper32(hp) -> SimpleNamespace:
    """The hyper-parameters as the kernels receive them (fp32 KinPpoHyper)."""
    return SimpleNamespace(**_fields(hp.c()))


def _pack(params: torch.Tensor, in_dim: int) -> torch.Tensor:
    from rl_brain_trainer_b200 import _lib

    w = torch.empty(36864, dtype=torch.uint8, device=params.device)
    _lib.check(_lib.lib().kin_ppo_pack_weights(params.data_ptr(), in_dim, w.data_ptr(), torch.cuda.current_stream().cuda_stream))
    return w


def _before(t) -> dict:
    return dict(p0=t.params.clone(), w0=t.weight_image.clone(), m0=t.adam_m.clone(), v0=t.adam_v.clone(), acc0=t.stats_accum.clone())


def _after(t) -> dict:
    return dict(grad=t.grad.clone(), stats=t.stats.clone(), p1=t.params.clone(), m1=t.adam_m.clone(), v1=t.adam_v.clone(),
                acc1=t.stats_accum.clone())


class _Recorder:
    """Stands in for the library handle of a trainer (``members = [trainer]``) or a population (its members): every call is forwarded
    unchanged; the hooks below add only stream-ordered clones around the update-family calls."""

    def __init__(self, lib, members):
        self._lib = lib
        self.members = list(members)
        self.runs = [dict(updates=[]) for _ in self.members]

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        hook = getattr(type(self), "_" + name, None)
        return fn if hook is None else (lambda *a: hook(self, fn, *a))

    def begin_update(self) -> None:
        """Snapshot the rollout the next ``update()`` reads (it does not change during the update; the old log-probs may, through
        ``refresh_old_logp``, so they are taken at the first gradient launch)."""
        for t, run in zip(self.members, self.runs):
            obs = t.obs_img if (t._img and not t.is_route) else t.obs_buf
            snap = {k: getattr(t, k).clone() for k in ROLLOUT}
            snap["obs"] = obs.clone()
            run["updates"].append(dict(snap=snap, logp=None, epochs=[], mbs=[], count0=t.update_count))

    def _new_mb(self, k: int, adv_row: int, grad_hp) -> dict:
        t, u = self.members[k], self.runs[k]["updates"][-1]
        if u["logp"] is None:
            u["logp"] = t.logp_buf.clone()
        mb = dict(epoch=len(u["epochs"]) - 1, adv_row=adv_row, grad_hp=grad_hp, **_before(t))
        u["mbs"].append(mb)
        return mb

    # ---- PPOTrainer
    def _kin_ppo_adv_stats(self, fn, *a):
        tr = self.members[0]
        ep = dict(perm=tr._perm.clone(), sample_perm=tr._sample_perm.clone() if tr._use_shadow else None)
        rc = fn(*a)
        ep["table"] = tr._adv_stats.clone()
        self.runs[0]["updates"][-1]["epochs"].append(ep)
        return rc

    def _grad(self, fn, a, adv_i, fused=False):
        tr = self.members[0]
        mb = self._new_mb(0, (a[adv_i] - tr._adv_stats.data_ptr()) // 8, _fields(a[2]._obj))
        rc = fn(*a)
        if fused:        # kin_ppo_grad_tc_update: the optimiser step ran in the kernel's tail
            mb.update(step=a[27], adam_hp=mb["grad_hp"], **_after(tr))
        return rc

    def _kin_ppo_grad(self, fn, *a):
        return self._grad(fn, a, 16)

    def _kin_ppo_grad_tc(self, fn, *a):
        return fn(*a) if a[18] else self._grad(fn, a, 20)       # forward_only: refresh_old_logp

    def _kin_ppo_grad_tc_exchange(self, fn, *a):
        return self._grad(fn, a, 17)

    def _kin_ppo_grad_tc_update(self, fn, *a):
        return self._grad(fn, a, 17, fused=True)

    def _kin_ppo_adam(self, fn, *a):
        tr, mb = self.members[0], self.runs[0]["updates"][-1]["mbs"][-1]
        mb.update(step=a[6], adam_hp=_fields(a[5]._obj))
        rc = fn(*a)
        mb.update(_after(tr))       # (grad and stats: with the peer exchange they are final only once gather has run)
        return rc

    # ---- PPOPopulation
    def _kin_pop_adv_stats(self, fn, *a):
        perm = self._pop._perm.clone()
        rc = fn(*a)
        for k, t in enumerate(self.members):
            self.runs[k]["updates"][-1]["epochs"].append(dict(perm=perm[k], sample_perm=None, table=t._adv_stats.clone()))
        return rc

    def _kin_pop_grad_tc(self, fn, *a):         # (table, K, minibatch, n_tiles, global_batch, grid, stream)
        for k in range(len(self.members)):
            self._new_mb(k, a[2], None)
        return fn(*a)

    def _kin_pop_adam(self, fn, *a):            # (table, K, host_hypers, host_steps, stream)
        mbs = [run["updates"][-1]["mbs"][-1] for run in self.runs]
        for k, mb in enumerate(mbs):
            mb.update(step=int(a[3][k]), adam_hp=_fields(a[2][k]))
        rc = fn(*a)
        for t, mb in zip(self.members, mbs):
            mb.update(_after(t))
        return rc


def _rel(a: torch.Tensor, b: torch.Tensor) -> float:
    return float((a - b).norm() / (b.norm() + 1e-30))


def _tensor_tols(clip_active: bool):
    """Tensor-core kernels: (per-tensor, whole gradient, cosine).  Without clipping, the bf16 bounds of
    test_minibatch_gradient_tc_matches_autograd (the whole-gradient bound is the one the three-stream test needs for the coherent bf16
    bias of large minibatches).  Once clipping is active (later epochs), the bounds that test uses with clipping: the actor gradient then
    comes from fewer samples with more cancellation, and the critic has fitted the returns, so its residuals shrink towards the bf16
    error of the value itself.  The oracle still takes the clip decisions from the device's own ratios (_device_logp): without that, a
    sample whose bf16 ratio sits on the other side of the boundary adds its whole surrogate term to the "error" (up to 0.3 per tensor
    measured on a B200 with clip_range 0.05 - 0.2)."""
    return (0.12, 8e-2, 0.998) if clip_active else (5e-2, 2e-2, 0.9999)


def _device_logp(t, sn, params: torch.Tensor) -> torch.Tensor:
    """Log-probs of every rollout sample by the tensor-core kernel's own forward at ``params`` (the forward-only launch
    ``refresh_old_logp`` uses, on the observations the update reads and the weight image of ``params``)."""
    from rl_brain_trainer_b200 import _lib

    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    if t.is_route:
        obs = torch.empty((t.S // 128, 16384), dtype=torch.uint8, device="cuda")
        _lib.check(L.kin_route_obs_images(sn["obs"][: t.T].contiguous().data_ptr(), t.S, obs.data_ptr(), stream))
    else:
        obs = sn["obs"] if t._img else sn["obs"][: t.T].contiguous()
    tiles = torch.arange(t.S // 64, dtype=torch.int32, device="cuda")
    out = torch.empty(t.S, device="cuda")
    wimg = _pack(params, t.in_dim)
    hp = t.hp.c()
    _lib.check(L.kin_ppo_grad_tc(params.data_ptr(), t.in_dim, ctypes.byref(hp), obs.data_ptr(), sn["act_buf"].data_ptr(), None, None, None, None,
                                 tiles.data_ptr(), int(tiles.numel()), 0, None, t.grad_ctas, None, None, out.data_ptr(), None, 1, int(t._img), None,
                                 wimg.data_ptr(), stream))
    return out


def _check_run(t, run, returned, *, label, stale=False):
    """Every check of one trainer's (or population member's) recorded updates; returns (failures, measured extremes)."""
    from rl_brain_trainer_b200 import ppo

    fails: list[str] = []
    worst: dict[str, float] = {}

    def check(ok, msg):
        if not ok:
            fails.append(f"{label}: {msg}")

    def note(key, val, low=False):
        worst[key] = (min if low else max)(worst.get(key, val), val)

    hp = _hyper32(t.hp)
    tc = t.update_variant == "tc"
    T, S, in_dim = t.T, t.S, t.in_dim
    n_tiles, k = S // 64, t.local_batch // 64
    n_mb = n_tiles // k
    counter = run["updates"][0]["count0"]
    prev_p = None
    n_clipped = 0
    lane = torch.arange(64, device="cuda")
    slices = oracle.param_slices(in_dim)
    for ui, u in enumerate(run["updates"]):
        sn = u["snap"]
        # GAE inputs: advantages, returns and tile sums against an fp64 GAE of the recorded rollout
        ra, rr = ppo.numpy_gae(sn["rew_buf"].cpu().numpy(), sn["val_buf"].cpu().numpy(), sn["start_buf"].cpu().numpy(), sn["last_val"].cpu().numpy(),
                               ((sn["done_buf"][T - 1] & 3) != 0).cpu().numpy(), float(t.hp.gamma), float(t.hp.gae_lambda))
        for name, got, ref in (("advantage", sn["adv_buf"], ra), ("returns", sn["ret_buf"], rr)):
            scale = max(1.0, float(np.abs(ref).max()))
            err = float(np.abs(got.cpu().numpy() - ref).max()) / scale
            note(f"gae_{name}", err)
            check(err < 2e-5, f"update {ui}: GAE {name} off by {err:.3g} (relative to max(1, |ref|))")
        flat = sn["adv_buf"].reshape(-1, 64).double()
        check(torch.allclose(sn["tile_sums"][:, 0], flat.sum(1), rtol=1e-12, atol=1e-9)
              and torch.allclose(sn["tile_sums"][:, 1], (flat * flat).sum(1), rtol=1e-12, atol=1e-9), f"update {ui}: tile sums")
        # what the gradient kernels read, per sample of the rollout order
        if t._img and not t.is_route:
            obs_all = ppo.decode_obs_images(sn["obs"]).reshape(S, 64)[:, :56]
        else:
            obs_all = sn["obs"][:T].reshape(S, in_dim)
        act_all, logp_all, adv_all, ret_all = sn["act_buf"].reshape(S, 7), u["logp"].reshape(S), sn["adv_buf"].reshape(S), sn["ret_buf"].reshape(S)
        n_epochs = int(t.hp.n_epochs)
        check(len(u["epochs"]) == n_epochs and len(u["mbs"]) == n_epochs * n_mb,
              f"update {ui}: {len(u['epochs'])} epochs / {len(u['mbs'])} minibatches recorded, expected {n_epochs} / {n_epochs * n_mb}")
        per_mb_stats = []
        for j, mb in enumerate(u["mbs"]):
            e, m = divmod(j, n_mb)
            where = f"update {ui} epoch {e} minibatch {m}"
            check(mb["epoch"] == e, f"{where}: launched in epoch {mb['epoch']}")
            ep = u["epochs"][e]
            perm = ep["perm"].long()
            sp = ep["sample_perm"]
            if m == 0:          # minibatch composition: a permutation of all tiles, whole (2i, 2i + 1) image pairs on image paths
                check(torch.equal(perm.sort().values, torch.arange(n_tiles, device="cuda")), f"{where}: not a permutation of the tiles")
                if t._img and t.shuffle != "sample":
                    pairs = perm.view(-1, 2)
                    check(bool(((pairs[:, 0] % 2 == 0) & (pairs[:, 1] == pairs[:, 0] + 1)).all()), f"{where}: tiles not in whole image pairs")
                if sp is not None:
                    check(torch.equal(sp.long().sort().values, torch.arange(S, device="cuda")), f"{where}: sample permutation")
            idx = (perm[m * k:(m + 1) * k, None] * 64 + lane[None]).reshape(-1)
            if sp is not None:
                idx = sp.long()[idx]
            args = (obs_all[idx], act_all[idx], logp_all[idx], adv_all[idx], ret_all[idx])
            clip_ratio = torch.exp(_device_logp(t, sn, mb["p0"]).double()[idx] - logp_all[idx].double()) if tc else None
            g_ref, s_ref, (mu, inv) = oracle.minibatch(mb["p0"], hp, *args, clip_ratio=clip_ratio)
            # advantage statistics: the row the kernel was handed
            rows = ep["table"]
            r = mb["adv_row"]
            if not 0 <= r < rows.shape[0]:
                check(False, f"{where}: advantage-statistics row {r} outside the table")
            elif hp.normalize_advantage:
                got_mu, got_inv = float(rows[r, 0]), float(rows[r, 1])
                e_mu, e_inv = abs(got_mu - mu) * inv / (1.0 + abs(mu) * inv), abs(got_inv - inv) / inv
                note("adv_stats", max(e_mu, e_inv))
                check(e_mu < 2e-6 and e_inv < 2e-6, f"{where}: advantage statistics ({got_mu}, {got_inv}) vs ({mu}, {inv})")
            else:
                check((float(rows[r, 0]), float(rows[r, 1])) == (0.0, 1.0), f"{where}: normalize_advantage=False must hand (0, 1)")
            # the gradient, at the device's parameters before this step
            g_dev = mb["grad"].double()
            clip_active = float(s_ref[4]) > 0.0
            whole = _rel(g_dev, g_ref)
            if tc:
                tol_k, tol_all, min_cos = _tensor_tols(clip_active)
                for name, sl in slices:
                    n = sl.stop - sl.start
                    # val_b is one signed sum over every sample with full cancellation: its bf16 noise has no useful relative bound
                    # (the three-stream test compares it with the two-chain kernel instead); it still counts in the whole-gradient bounds
                    if n == 1:
                        continue
                    rel = _rel(g_dev[sl], g_ref[sl])
                    note(f"grad_{'clip' if clip_active else 'noclip'}_tensor/tol", rel / (tol_k if n > 64 else 3 * tol_k))
                    check(rel < (tol_k if n > 64 else 3 * tol_k), f"{where}: {name} gradient rel. error {rel:.3g} (clip fraction {float(s_ref[4]):.3g})")
                cos = float(torch.dot(g_dev, g_ref) / (g_dev.norm() * g_ref.norm()))
                note("grad_cos", cos, low=True)
                check(cos > min_cos and whole < tol_all, f"{where}: gradient cos {cos:.6f}, rel {whole:.3g} (clip fraction {float(s_ref[4]):.3g})")
            else:
                check(whole < 1e-4, f"{where}: fp32 gradient rel. error {whole:.3g}")
            note("grad_whole_rel", whole)
            if stale and prev_p is not None:
                # the oracle gradient one step stale, on the same samples: if the device had read the previous step's weights, its
                # error against g_ref would be at least (separation - 1) x the tolerance of some tensor -- the check above would fail
                g_prev, _, _ = oracle.minibatch(prev_p, hp, *args, clip_ratio=clip_ratio)
                tol_k = _tensor_tols(clip_active)[0]
                sep = max(_rel(g_prev[sl], g_ref[sl]) / (tol_k if sl.stop - sl.start > 64 else 3 * tol_k) for _, sl in slices if sl.stop - sl.start > 1)
                note("stale_separation", sep, low=True)
                check(sep > 2.0, f"{where}: the gradient one step stale is only {sep:.3g} x the tolerance away")
            prev_p = mb["p0"]
            # the weight image this launch read is the bf16 pack of the parameters it read
            check(torch.equal(mb["w0"], _pack(mb["p0"], in_dim)), f"{where}: the weight image the launch read is not pack(params)")
            # clip + Adam at the step count the oracle expects (counting across update() calls)
            counter += 1
            check(mb["step"] == counter, f"{where}: the host passed Adam step {mb['step']}, expected {counter}")
            check(mb["adam_hp"] == _fields(t.hp.c()) and (mb["grad_hp"] is None or mb["grad_hp"] == mb["adam_hp"]),
                  f"{where}: the host passed other hyper-parameters than the run's")
            p1, m1, v1, norm, coef = oracle.adam_step(mb["p0"], mb["m0"], mb["v0"], mb["grad"], hp, counter)
            dev_norm = float(mb["stats"][GRAD_NORM])
            note("grad_norm_rel", abs(dev_norm - norm) / norm)
            check(abs(dev_norm - norm) <= 1e-5 * norm, f"{where}: gradient norm {dev_norm} vs {norm}")
            n_clipped += coef < 1.0
            e_p = float((mb["p1"].double() - p1).abs().max())
            e_m = float((mb["m1"].double() - m1).abs().max()) / (float(m1.abs().max()) + 1e-30)
            e_v = float((mb["v1"].double() - v1).abs().max()) / (float(v1.abs().max()) + 1e-30)
            p_tol = 1e-6 * max(1.0, float(p1.abs().max())) + 1e-5 * hp.learning_rate
            note("adam_p/tol", e_p / p_tol)
            note("adam_m_rel", e_m)
            note("adam_v_rel", e_v)
            check(e_p < p_tol and e_m < 2e-6 and e_v < 1e-5, f"{where}: Adam step p {e_p:.3g} (tol {p_tol:.3g}), m {e_m:.3g}, v {e_v:.3g}")
            # per-minibatch statistics and the running sums
            s_dev = mb["stats"][:5].double()
            tol_s = 3e-2 if tc else 2e-4
            for i, key in enumerate(oracle.STAT_NAMES):
                err = abs(float(s_dev[i]) - float(s_ref[i])) / max(1.0, abs(float(s_ref[i])))
                note(f"stat_{key}", err)
                check(err < tol_s, f"{where}: {key} {float(s_dev[i])} vs {float(s_ref[i])}")
            want = mb["acc0"].clone()
            want[:6] += mb["stats"][:6]
            want[7] += 1.0
            check(float(mb["stats"][SKIP]) == 0.0 and torch.equal(want, mb["acc1"]), f"{where}: stats_accum {mb['acc1'].tolist()} vs {want.tolist()}")
            per_mb_stats.append(mb["stats"][:6].double())
        # what update() returns: the means of the per-minibatch values (grad_norm before the clip)
        mean = torch.stack(per_mb_stats).mean(0)
        got = returned[ui]
        for i, key in enumerate(oracle.STAT_NAMES + ("grad_norm",)):
            check(abs(got[key] - float(mean[i])) <= 1e-5 * max(1.0, abs(float(mean[i]))), f"update {ui}: returned {key} {got[key]} vs mean {float(mean[i])}")
        check(got["minibatches"] == len(per_mb_stats), f"update {ui}: returned {got['minibatches']} minibatches, recorded {len(per_mb_stats)}")
    check(torch.equal(t.weight_image, _pack(t.params, in_dim)), "final weight image is not pack(final params)")
    worst["clipped_step_share"] = n_clipped / max(counter - run["updates"][0]["count0"], 1)
    return fails, worst


def _arm_policy(seed, in_dim=56):
    from rl_brain_trainer_b200 import ppo

    pol = ppo.random_policy(in_dim, seed=seed, log_std_init=-1.0, device="cuda")
    pol.tensors["act_w"].mul_(30.0)         # SB3's 0.01 action gain would hide errors in the actor gradient
    return pol


def _trainer(case):
    from rl_brain_trainer_b200 import ppo

    hp = ppo.PPOHyper(**{"learning_rate": 1e-3, "gamma": 0.98, **case["hp"]})
    if case.get("route"):
        from rl_brain_trainer_b200 import config as kcfg
        from rl_brain_trainer_b200.route import synthetic_route

        route = synthetic_route(160, seed=7)
        renv, seq = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
        tr = ppo.PPOTrainer(renv, _arm_policy(2, 80), num_envs=case["n"], hyper=hp, seed=3, route=route, route_sequence_config=seq, **case.get("kw", {}))
    else:
        tr = ppo.PPOTrainer(env_config("approach_dynamic_scale_big"), _arm_policy(1), num_envs=case["n"], hyper=hp, seed=3, **case.get("kw", {}))
    if "fused_exchange" in case:
        tr.fused_exchange = case["fused_exchange"]
    return tr


# Hyper-parameter corners are spread over the cases: normalize_advantage off, ent_coef 0 / 0.05, vf_coef 0.25 / 1.0, clip_range 0.05
# (active from epoch 2 on), max_grad_norm clipping nearly every step (0.05) and never (1e3), betas (0.8, 0.99) with eps 1e-8, one
# minibatch per epoch, 512 tiles per minibatch (kin_ppo_adv_stats loops twice over its 256 threads), grad_ctas 3 and the default.
CASES = {
    "fp32_tile": dict(n=256, hp=dict(n_steps=16, batch_size=512, n_epochs=2, ent_coef=0.05, vf_coef=0.25, max_grad_norm=0.05),
                      kw=dict(update_variant="fp32", collect_variant="steps", grad_ctas=3)),
    "fp32_sample": dict(n=512, hp=dict(n_steps=16, batch_size=8192, n_epochs=3, normalize_advantage=False, ent_coef=0.0, vf_coef=1.0, max_grad_norm=1e3),
                        kw=dict(update_variant="fp32", collect_variant="steps", shuffle="sample")),
    "tc_steps": dict(n=256, hp=dict(learning_rate=5e-4, n_steps=32, batch_size=1024, n_epochs=3, clip_range=0.05, adam_beta1=0.8, adam_beta2=0.99, adam_eps=1e-8,
                                    ent_coef=0.01), kw=dict(collect_variant="steps")),
    "tc_fused": dict(n=512, hp=dict(n_steps=16, batch_size=1024, n_epochs=1, learning_rate=STALE_LR), kw=dict(collect_variant="fused"), stale=True),
    "tc_fused_update": dict(n=512, hp=dict(n_steps=16, batch_size=2048, n_epochs=2, max_grad_norm=0.05, ent_coef=0.05),
                            kw=dict(fused_update=True, grad_ctas=3)),
    "tc_peer_fused": dict(n=256, hp=dict(n_steps=16, batch_size=1024, n_epochs=2, vf_coef=1.0), kw=dict(grad_exchange="peer"), fused_exchange=True),
    "tc_peer_unfused": dict(n=256, hp=dict(n_steps=16, batch_size=1024, n_epochs=2, vf_coef=0.25), kw=dict(grad_exchange="peer"), fused_exchange=False),
    "tc_sample_once": dict(n=1024, hp=dict(n_steps=32, batch_size=32768, n_epochs=3, clip_range=0.05), kw=dict(shuffle="sample_once")),
    "route": dict(n=256, hp=dict(n_steps=16, batch_size=1024, n_epochs=2, ent_coef=0.01), route=True),
}


def _report(label, fails, worst):
    print(f"\n[{label}] " + ", ".join(f"{k}={v:.3g}" for k, v in sorted(worst.items())))
    assert not fails, f"{len(fails)} failed checks:\n" + "\n".join(fails[:40])


@pytest.mark.parametrize("case", list(CASES))
def test_update_replay(case):
    """Two collect + update rounds recorded through the library proxy, against an identical trainer without it (bitwise), then every
    minibatch replayed through the oracle.  STALE_LR case: smallest stale separation measured on a B200 -- see the printed report."""
    spec = CASES[case]
    tr, twin = _trainer(spec), _trainer(spec)
    rec = _Recorder(tr._L, [tr])
    tr._L = rec
    returned, twin_returned = [], []
    for _ in range(2):
        tr.collect()
        twin.collect()
        rec.begin_update()
        returned.append(tr.update())
        twin_returned.append(twin.update())
    torch.cuda.synchronize()
    # the recorder changes nothing: bitwise on every path
    for name in ("params", "adam_m", "adam_v", "stats_accum", "weight_image"):
        assert torch.equal(getattr(tr, name), getattr(twin, name)), name
    assert returned == twin_returned
    assert tr.update_count == twin.update_count
    fails, worst = _check_run(tr, rec.runs[0], returned, label=case, stale=spec.get("stale", False))
    tr.close()
    twin.close()
    _report(case, fails, worst)


def _population_members():
    from rl_brain_trainer_b200 import ppo

    base = env_config("approach_default")
    out = []
    for i in range(3):      # every member its own PPO and Adam hyper-parameters; member 2 without advantage normalisation
        hp = ppo.PPOHyper(learning_rate=1e-3 * (1 + i), n_steps=16, batch_size=1024, n_epochs=2, gamma=0.98 - 0.01 * i, gae_lambda=0.95 - 0.02 * i,
                          clip_range=(0.2, 0.05, 0.1)[i], ent_coef=(0.0, 0.05, 0.01)[i], vf_coef=(0.5, 1.0, 0.25)[i], max_grad_norm=(0.05, 1e3, 0.5)[i],
                          normalize_advantage=(i != 2), adam_beta1=(0.9, 0.8, 0.85)[i], adam_beta2=(0.999, 0.99, 0.995)[i], adam_eps=(1e-5, 1e-8, 1e-6)[i])
        out.append((base, hp, 100 + 7 * i, 1 + i, i))
    return out


def _population():
    from rl_brain_trainer_b200 import ppo
    from rl_brain_trainer_b200.population import PPOPopulation

    return PPOPopulation([ppo.PPOTrainer(cfg, _arm_policy(ps), num_envs=256, hyper=dataclasses.replace(hp), seed=seed, stage_index=st,
                                         collect_variant="fused", update_variant="tc", shuffle="tile", fused_update=False)
                          for cfg, hp, seed, st, ps in _population_members()])


def test_population_update_replay():
    """PPOPopulation (K = 3): kin_pop_adv_stats / kin_pop_grad_tc / kin_pop_adam, each member replayed with its own hyper-parameters."""
    pop, twin = _population(), _population()
    rec = _Recorder(pop._L, pop.members)
    rec._pop = pop
    pop._L = rec
    returned, twin_returned = [], []
    for _ in range(2):
        pop.collect()
        twin.collect()
        rec.begin_update()
        returned.append(pop.update())
        twin_returned.append(twin.update())
    torch.cuda.synchronize()
    for a, b in zip(pop.members, twin.members):
        for name in ("params", "adam_m", "adam_v", "weight_image", "stats_accum"):
            assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert returned == twin_returned
    fails, worst = [], {}
    for k, t in enumerate(pop.members):
        f, w = _check_run(t, rec.runs[k], [r[k] for r in returned], label=f"member {k}")
        fails += f
        worst.update({f"m{k}.{key}": v for key, v in w.items()})
    _report("population", fails, worst)


# ---------------------------------------------------------------------------------------------------- direct entry-point tests
def test_adv_stats_kernel_matches_fp64():
    """kin_ppo_adv_stats against fp64 torch: 1 and 300 tiles per minibatch, several minibatches per launch, normalize = 0, and
    advantages with a large offset (mean 1e3, std 1e-2), where a one-pass s2 - n mean^2 variance loses its digits."""
    from rl_brain_trainer_b200 import _lib

    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda").manual_seed(21)
    worst = 0.0
    for n_tiles, n_mb, loc, scale, normalize in ((1, 1, 0.3, 1.0, 1), (300, 1, -0.2, 2.0, 1), (40, 7, 0.5, 1.5, 1), (40, 7, 0.5, 1.5, 0),
                                                 (300, 2, 1e3, 1e-2, 1), (7, 5, -1e3, 1e-2, 1)):
        total = n_tiles * n_mb + 9                 # tiles no minibatch uses
        adv = (loc + scale * torch.randn(total * 64, device="cuda", generator=g, dtype=torch.float64)).float()
        t64 = adv.reshape(total, 64).double()
        sums = torch.stack([t64.sum(1), (t64 * t64).sum(1)], dim=1).contiguous()
        ids = torch.randperm(total, device="cuda", generator=g)[: n_tiles * n_mb].to(torch.int32)
        out = torch.full((n_mb, 2), 7.0, device="cuda")
        _lib.check(L.kin_ppo_adv_stats(sums.data_ptr(), ids.data_ptr(), n_tiles, n_mb, normalize, out.data_ptr(), stream))
        torch.cuda.synchronize()
        for m in range(n_mb):
            samples = t64[ids[m * n_tiles:(m + 1) * n_tiles].long()].reshape(-1)
            mu, inv = oracle.adv_stats(samples, bool(normalize))
            got_mu, got_inv = float(out[m, 0]), float(out[m, 1])
            if not normalize:
                assert (got_mu, got_inv) == (0.0, 1.0)
                continue
            e_mu, e_inv = abs(got_mu - mu) / (abs(mu) + 1.0 / inv), abs(got_inv - inv) / inv
            worst = max(worst, e_mu, e_inv)
            assert e_mu < 1e-6 and e_inv < 1e-6, (n_tiles, n_mb, loc, scale, m, (got_mu, got_inv), (mu, inv))
    print(f"\n[adv_stats] worst relative error {worst:.3g}")


def test_adam_kernel_corners():
    """kin_ppo_adam against the oracle with non-default betas / eps over several steps: clip active, inactive and max_grad_norm <= 0
    (no clip, unlike clip_grad_norm_(0)); stats_accum sums with slot 7 counting the calls; the weight image equals a fresh pack after
    every step; stats[KIN_PPO_STAT_SKIP] != 0 leaves parameters, moments, image and stats_accum untouched."""
    from rl_brain_trainer_b200 import _lib, ppo

    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda").manual_seed(31)
    flat = ppo.flatten_policy_(_arm_policy(4))
    P = flat.numel()
    params = flat.clone()
    m, v = torch.zeros(P, device="cuda"), torch.zeros(P, device="cuda")
    wimg = _pack(params, 56)
    acc = torch.zeros(8, device="cuda")
    stats = torch.zeros(8, device="cuda")
    acc_ref = torch.zeros(8, dtype=torch.float64)
    for step, (mx, scale) in enumerate(((0.5, 0.3), (0.5, 1e-3), (0.0, 0.3), (-1.0, 0.05), (1e3, 0.2), (0.05, 0.01)), start=1):
        hp = ppo.PPOHyper(learning_rate=2e-3, max_grad_norm=mx, adam_beta1=0.8, adam_beta2=0.99, adam_eps=1e-8)
        h32 = _hyper32(hp)
        grad = torch.randn(P, device="cuda", generator=g) * scale / math.sqrt(P) * 100
        stats[:5] = torch.randn(5, device="cuda", generator=g)
        stats[5:] = 0.0
        p_ref, m_ref, v_ref, norm, coef = oracle.adam_step(params, m, v, grad, h32, step)
        c_hp = hp.c()
        _lib.check(L.kin_ppo_adam(params.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), P, ctypes.byref(c_hp), step, stats.data_ptr(),
                                  acc.data_ptr(), wimg.data_ptr(), 56, stream))
        torch.cuda.synchronize()
        assert (coef < 1.0) == (mx > 0 and norm > mx), (step, norm, coef)
        assert abs(float(stats[GRAD_NORM]) - norm) <= 1e-5 * norm, step
        assert float((params.double() - p_ref).abs().max()) < 1e-6 * max(1.0, float(p_ref.abs().max())) + 1e-5 * 2e-3, step
        assert float((m.double() - m_ref).abs().max()) < 2e-6 * float(m_ref.abs().max()), step
        assert float((v.double() - v_ref).abs().max()) < 1e-5 * float(v_ref.abs().max()), step
        acc_ref[:6] += stats[:6].double().cpu()
        acc_ref[7] += 1.0
        assert torch.allclose(acc.double().cpu(), acc_ref, rtol=1e-6, atol=1e-6) and float(acc[7]) == step, (acc, acc_ref)
        assert torch.equal(wimg, _pack(params, 56)), step
    # a skipped minibatch (peer exchange timed out) touches nothing
    before = [x.clone() for x in (params, m, v, wimg, acc)]
    stats[SKIP] = 1.0
    grad = torch.randn(P, device="cuda", generator=g)
    c_hp = ppo.PPOHyper(learning_rate=2e-3).c()
    _lib.check(L.kin_ppo_adam(params.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), P, ctypes.byref(c_hp), 7, stats.data_ptr(),
                              acc.data_ptr(), wimg.data_ptr(), 56, stream))
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(before, (params, m, v, wimg, acc)))


@pytest.mark.parametrize("in_dim", [56, 80])
def test_bootstrap_list_matches_fp64_critic(in_dim):
    """kin_ppo_bootstrap_list: reward[boot_index[i]] += gamma * V(boot_obs[i]) for i < min(*boot_count, boot_cap) against the fp64
    critic; a count past the capacity applies only the first boot_cap entries."""
    from rl_brain_trainer_b200 import _lib, ppo

    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda").manual_seed(41 + in_dim)
    pol = _arm_policy(5, in_dim)
    pol.tensors["vf_b1"].normal_(0, 0.2, generator=g)
    pol.tensors["val_w"].mul_(3.0)
    params = ppo.flatten_policy_(pol)
    n_rew, cap, gamma = 3000, 300, 0.97
    for count in (cap + 77, 129, 0):
        boot_obs = (torch.rand((cap, in_dim), device="cuda", generator=g) * 2 - 1).contiguous()
        boot_index = torch.randperm(n_rew, device="cuda", generator=g)[:cap].to(torch.int32)
        reward = torch.randn(n_rew, device="cuda", generator=g)
        want = reward.double().clone()
        n = min(count, cap)
        _, value, _ = oracle.forward(params, boot_obs[:n])
        want[boot_index[:n].long()] += gamma * value
        cnt = torch.tensor([count], dtype=torch.int32, device="cuda")
        _lib.check(L.kin_ppo_bootstrap_list(params.data_ptr(), in_dim, boot_obs.data_ptr(), boot_index.data_ptr(), cnt.data_ptr(), cap,
                                            reward.data_ptr(), gamma, stream))
        torch.cuda.synchronize()
        err = float((reward.double() - want).abs().max())
        assert err < 3e-5 * max(1.0, float(value.abs().max()) if n else 1.0), (count, err)
        untouched = torch.ones(n_rew, dtype=torch.bool, device="cuda")
        untouched[boot_index[:n].long()] = False
        assert torch.equal(reward[untouched], want[untouched].float()), count
