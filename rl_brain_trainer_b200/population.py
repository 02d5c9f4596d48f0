"""A population of independent PPO runs trained together on one GPU: K complete ``PPOTrainer`` members, each phase of all of
them in ONE launch (``kin_pop_*`` in ``include/kin_b200.h``, the member index on a grid dimension).

Seed and hyper-parameter sweeps at the reference's own small batch sizes are bound by launches and host work, not by the GPU: a
minibatch of 512 samples is 4 GEMM tiles.  Independent runs share nothing, so their collection, GAE, minibatch gradients and Adam
steps go through the same launches for about the launch cost of one run.  Member k is bitwise the standalone ``PPOTrainer`` built
with the same arguments: the population kernels are the standalone kernels' bodies reading member k's pointers, seeds and
hyper-parameters, and every host-side draw (the epoch permutations) comes from member k's own generator.

Scope: the 56-input Approach / Finisher policies on the fused path (``collect_variant="fused"``, ``update_variant="tc"``,
``shuffle="tile"``), one rank, no ``target_kl``, no adaptive frontier curriculum.  Members share the env params and policy mode,
``num_envs``, ``n_steps``, ``batch_size``, ``n_epochs`` and the gradient grid; seeds, initial policies, start stages, curriculum
settings and the PPO / Adam hyper-parameters are their own.
"""

from __future__ import annotations

import ctypes
from typing import Any, Sequence

import numpy as np
import torch

from . import _lib
from .env import _D
from .ppo import PPOHyper, PPOTrainer
from .policy import PolicyWeights


class PPOPopulation:
    """K ``PPOTrainer`` members run as one: ``collect()``, ``update()`` and ``learn()`` mirror the trainer's and return one result per
    member.  ``members[k]`` is the unchanged trainer (``save_checkpoint``, ``load_checkpoint``, ``state_dict`` and ``policy`` work per
    member); the population keeps only the device descriptor table of the members and the per-epoch tile permutations it points at."""

    def __init__(self, members: Sequence[PPOTrainer]) -> None:
        self.members = list(members)
        self._validate()
        t0 = self.members[0]
        self.K = len(self.members)
        self.device = t0.device
        self._L = t0._L
        self._Member = _lib.c_struct("KinPopMember")
        self._host = (self._Member * self.K)()
        self._hypers = (_lib.c_struct("KinPpoHyper") * self.K)()
        self._steps = (ctypes.c_int * self.K)()
        n_tiles = t0.S // _D("KIN_PPO_TILE")
        with torch.cuda.device(self.device):
            self._table = torch.zeros(ctypes.sizeof(self._host), dtype=torch.uint8, device=self.device)
            self._perm = torch.zeros((self.K, n_tiles), dtype=torch.int32, device=self.device)     # member k's epoch permutation
        self._uploaded: bytes | None = None

    @classmethod
    def build(cls, config: Any, policies: Sequence[PolicyWeights], hypers: Sequence[PPOHyper], seeds: Sequence[int], num_envs: int, *,
              stage_indices: Sequence[int] | None = None, handoff_states: torch.Tensor | None = None, device: str | torch.device = "cuda",
              grad_ctas: int | None = None) -> "PPOPopulation":
        """One member per (policy, hyper, seed[, stage]).  ``config`` is one ``Phase1EnvConfig`` for all members or one per member (the
        env params must still agree: per-member configs may differ only in host-side settings such as the curriculum tracker's)."""
        k = len(policies)
        configs = list(config) if isinstance(config, (list, tuple)) else [config] * k
        stages = list(stage_indices) if stage_indices is not None else [0] * k
        if not (len(configs) == len(hypers) == len(seeds) == len(stages) == k):
            raise ValueError("PPOPopulation.build: one config (or a shared one), hyper, seed and stage index per policy")
        return cls([PPOTrainer(c, p, num_envs=num_envs, hyper=h, device=device, seed=s, stage_index=st, handoff_states=handoff_states,
                               grad_ctas=grad_ctas, collect_variant="fused", update_variant="tc", shuffle="tile", fused_update=False)
                    for c, p, h, s, st in zip(configs, policies, hypers, seeds, stages)])

    def __len__(self) -> int:
        return len(self.members)

    def __getitem__(self, k: int) -> PPOTrainer:
        return self.members[k]

    # ------------------------------------------------------------------ checks and the descriptor table
    def _validate(self) -> None:
        """Every scope rule, checked on the host before any population launch."""
        ms = self.members
        if not ms:
            raise ValueError("PPOPopulation needs at least one member")
        if len(ms) > _D("KIN_POP_MAX"):
            raise ValueError(f"PPOPopulation: at most KIN_POP_MAX = {_D('KIN_POP_MAX')} members")
        if not all(isinstance(t, PPOTrainer) for t in ms):
            raise TypeError("PPOPopulation members are PPOTrainer instances")
        if len({id(t) for t in ms}) != len(ms):
            raise ValueError("PPOPopulation: a trainer appears twice; members must be independent runs")
        for t in ms:
            if t.is_route or t.in_dim != 56:
                raise ValueError("PPOPopulation: the route policy (80 inputs) is not supported; members train the 56-input Approach / Finisher policies")
            if t.collect_variant != "fused" or t.update_variant != "tc":
                raise ValueError("PPOPopulation: members need collect_variant='fused' and update_variant='tc' (the per-step and strict-fp32 paths are not batched)")
            if t.shuffle != "tile":
                raise ValueError("PPOPopulation: per-sample shuffling is not supported; members need shuffle='tile'")
            if t.world != 1 or t.group is not None or t.peer is not None or t.fused_update:
                raise ValueError("PPOPopulation: members run on one rank with the plain (non-exchange, non-fused) update")
            if t.hp.target_kl is not None:
                raise ValueError("PPOPopulation: target_kl stops a member's epochs early, which breaks the members' lockstep; not supported")
            if getattr(t.env, "_frontier", None) is not None:
                raise ValueError("PPOPopulation: the adaptive frontier curriculum is not supported")
            if t.device != ms[0].device:
                raise ValueError("PPOPopulation: all members must live on one device")
            if t.env._mode_all is None:
                raise _lib.KinError("PPOPopulation: the fused collection runs ONE policy mode for all envs of a member")
        t0 = ms[0]
        shape = lambda t: (t.N, t.T, t.local_batch, int(t.hp.n_epochs), t.grad_ctas, t.env._mode_all)  # noqa: E731
        for t in ms[1:]:
            if shape(t) != shape(t0):
                raise ValueError("PPOPopulation: members run in lockstep and must share num_envs, n_steps, batch_size, n_epochs, grad_ctas "
                                 f"and the policy mode ({shape(t)} != {shape(t0)})")
            same = ctypes.c_int(0)
            _lib.check(t0._L.kin_params_same_env(t0.env._params.handle, t.env._params.handle, ctypes.byref(same)))
            if not same.value:
                raise ValueError("PPOPopulation: members must share the env config (identical KinEnvParams)")

    def _sync(self) -> None:
        """Rebuild the host descriptors from the members' current state and upload them when anything changed (a sampler after a
        promotion, a step counter, a hyper-parameter, a seed)."""
        self._validate()
        for k, t in enumerate(self.members):
            d = self._host[k]
            env = t.env
            sp = ctypes.c_void_p()
            _lib.check(self._L.kin_params_device_sampler(env._params.handle, ctypes.byref(sp)))
            if not sp.value:
                raise _lib.KinError("PPOPopulation: a member's env has no device sampler (kin_params_set_sampler)")
            d.sampler = sp.value
            d.state, d.stride, d.boot_cap = env.state.data_ptr(), env.stride, t.boot_cap
            d.noise_seed, d.reset_seed, d.first_step = t.seed, env._seed, t.global_step & 0xFFFFFFFF
            d.params, d.weight_image, d.obs_tiles = t.params.data_ptr(), t.weight_image.data_ptr(), t.obs_img.data_ptr()
            d.action, d.logp, d.value, d.reward = t.act_buf.data_ptr(), t.logp_buf.data_ptr(), t.val_buf.data_ptr(), t.rew_buf.data_ptr()
            d.done, d.episode_start, d.start_io = t.done_buf.data_ptr(), t.start_buf.data_ptr(), t._next_start.data_ptr()
            d.last_value = t.last_val.data_ptr()
            d.boot_count, d.boot_index, d.boot_obs = t.boot_count.data_ptr(), t.boot_index.data_ptr(), t.boot_obs.data_ptr()
            d.advantage, d.returns, d.tile_sums = t.adv_buf.data_ptr(), t.ret_buf.data_ptr(), t.tile_sums.data_ptr()
            d.tile_ids, d.adv_stats = self._perm[k].data_ptr(), t._adv_stats.data_ptr()
            d.partials, d.grad, d.stats, d.stats_accum = t.partials.data_ptr(), t.grad.data_ptr(), t.stats.data_ptr(), t.stats_accum.data_ptr()
            d.adam_m, d.adam_v = t.adam_m.data_ptr(), t.adam_v.data_ptr()
            d.hyper = t.hp.c()
            self._hypers[k] = d.hyper
        raw = bytes(self._host)
        if raw != self._uploaded:      # a blocking copy: the launches still reading the previous table were enqueued before it
            self._table.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8))
            self._uploaded = raw

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ phases
    def collect(self) -> list[dict[str, float]]:
        """``collect_rollouts`` of every member: one fused collection launch, one bootstrap-list launch and one GAE launch for all."""
        for t in self.members:
            t.env._ensure_sampler()          # a curriculum promotion since the last rollout re-uploads that member's device sampler
        self._sync()
        t0, L, tab = self.members[0], self._L, self._table.data_ptr()
        with torch.cuda.device(self.device):
            stream = self._stream()
            _lib.check(L.kin_pop_collect(t0.env._params.handle, tab, self.K, t0.N, int(t0.env._mode_all), t0.T, stream))
            _lib.check(L.kin_pop_bootstrap_list(tab, self.K, max(t.boot_cap for t in self.members), stream))
            _lib.check(L.kin_pop_gae(tab, self.K, t0.N, t0.T, stream))
        return [t._finish_fused_collect() for t in self.members]

    def update(self) -> list[dict[str, float]]:
        """``PPO.train`` of every member: per epoch one advantage-statistics launch, per minibatch one gradient (+ reduction) and one
        Adam launch for all members; member k's tile permutation comes from member k's own generator."""
        if self._L.kin_ppo_tc3_config(-1, -1) & 1:
            raise _lib.KinError("PPOPopulation: the three-stream gradient kernel is enabled (KIN_PPO_TC3); members would not match standalone trainers")
        self._sync()
        t0, L, tab = self.members[0], self._L, self._table.data_ptr()
        tile = _D("KIN_PPO_TILE")
        n_tiles_total = t0.S // tile
        tiles_per_mb = t0.local_batch // tile
        mb_per_epoch = n_tiles_total // tiles_per_mb
        global_batch = tiles_per_mb * tile
        with torch.cuda.device(self.device):
            stream = self._stream()
            for t in self.members:
                t.stats_accum.zero_()
            for _ in range(int(t0.hp.n_epochs)):
                p2 = torch.stack([torch.randperm(n_tiles_total // 2, generator=t._gen, device=self.device, dtype=torch.int64) for t in self.members])
                self._perm.copy_(torch.stack((2 * p2, 2 * p2 + 1), dim=2).reshape(self.K, n_tiles_total))     # whole 128-sample images
                _lib.check(L.kin_pop_adv_stats(tab, self.K, tiles_per_mb, mb_per_epoch, stream))
                for m in range(mb_per_epoch):
                    _lib.check(L.kin_pop_grad_tc(tab, self.K, m, tiles_per_mb, global_batch, t0.grad_ctas, stream))
                    for k, t in enumerate(self.members):
                        t.update_count += 1
                        self._steps[k] = t.update_count
                    _lib.check(L.kin_pop_adam(tab, self.K, self._hypers, self._steps, stream))
            acc = torch.stack([t.stats_accum for t in self.members]).cpu().numpy().astype(np.float64)
        out = []
        for a in acc:
            n_mb = max(int(round(a[7])), 1)
            a = a / n_mb
            out.append({"policy_loss": float(a[0]), "value_loss": float(a[1]), "entropy": float(a[2]), "approx_kl": float(a[3]),
                        "clip_fraction": float(a[4]), "grad_norm": float(a[5]), "minibatches": n_mb})
        return out

    def learn(self, iterations: int, gates: Sequence[Any] | None = None) -> list[list[dict[str, float]]]:
        """``PPOTrainer.learn`` for every member: iterations of collect + update, per-member curriculum promotion and optional per-member
        eval gates (``gate.EvalGate``, run one member after another).  Returns one log per member; its rows carry ``PPOTrainer.learn``'s
        keys plus ``"member"``."""
        if gates is not None and len(gates) != self.K:
            raise ValueError("PPOPopulation.learn: one gate (or None) per member")
        logs: list[list[dict[str, float]]] = [[] for _ in self.members]
        for _ in range(int(iterations)):
            rs = self.collect()
            us = self.update()
            for k, t in enumerate(self.members):
                if t.curriculum is not None and t.curriculum.record_rollout(t._finished, t._success, t.group, t.num_timesteps):
                    t.env.set_curriculum_stage(t.curriculum.stage_index)
                row = {**rs[k], **us[k], "stage": float(t.env.get_curriculum_stage()), "timesteps": float(t.num_timesteps)}
                if gates is not None and gates[k] is not None:
                    rec = gates[k].maybe_eval(t.num_timesteps, t.policy)
                    if rec is not None:
                        row["gate_score"] = float(rec["score"])
                row["member"] = k
                logs[k].append(row)
        return logs
