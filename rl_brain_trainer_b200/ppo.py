"""PPO training of the Approach / Finisher policies on the GPU env (rollout collection + agent update + grad all-reduce).

Replaces ``model.learn`` of the reference's trainers (``kinematic_phase1/train_workspace_expansion.py:144-270``), whose
arithmetic is stable-baselines3 2.8.0 PPO (third-party, absent from the reference tree; restated in ``csrc/kin_ppo.cu`` and
checked against a PyTorch autograd restatement in ``tests/test_gpu_ppo.py``).  Differences that are deliberate and
documented in DESIGN.md: by default minibatches are random unions of 64-sample tiles (64 consecutive envs of one time step);
``PPOTrainer(shuffle="sample")`` gives SB3's per-sample permutation (``RolloutBuffer.get``, ``kin_ppo_shuffle``); with several ranks
the advantage normalisation is per rank-local minibatch and every minibatch's gradient is summed over the ranks (NVLink peer memory
in the gradient kernel's tail, or NCCL) before the identical clip + Adam step on every rank.
"""

from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Any

import numpy as np
import torch

from . import _lib
from .config import Phase1EnvConfig
from .distributed import CurriculumTracker, PeerGradExchange, allreduce_sum_, check_same_on_all_ranks, world
from .env import BatchedArmKinematicEnv, _D
from .policy import KEYS, PolicyWeights

PARAM_ORDER = ("pi_w0", "pi_b0", "pi_w1", "pi_b1", "act_w", "act_b", "vf_w0", "vf_b0", "vf_w1", "vf_b1", "val_w", "val_b", "log_std")


@dataclass
class PPOHyper:
    """SB3 PPO hyper-parameters (defaults of ``configs/ppo_default.yaml`` + SB3's own)."""

    learning_rate: float = 3e-4
    n_steps: int = 128
    batch_size: int = 256
    n_epochs: int = 10
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    normalize_advantage: bool = True
    adam_beta1: float = 0.9
    adam_beta2: float = 0.999
    adam_eps: float = 1e-5
    target_kl: float | None = None      # SB3's early stop: no further epochs once the mean approx. KL of an epoch exceeds 1.5 x target_kl

    @classmethod
    def from_config(cls, cfg: dict[str, Any]) -> "PPOHyper":
        """``algorithms.ppo`` section of a reference YAML."""
        known = {k: cfg[k] for k in cls.__dataclass_fields__ if k in cfg}
        return cls(**known)

    def c(self):
        h = _lib.c_struct("KinPpoHyper")()
        for f in ("gamma", "gae_lambda", "clip_range", "ent_coef", "vf_coef", "max_grad_norm", "learning_rate", "adam_beta1", "adam_beta2", "adam_eps"):
            setattr(h, f, float(getattr(self, f)))
        h.normalize_advantage = int(self.normalize_advantage)
        return h


def flatten_policy_(policy: PolicyWeights) -> torch.Tensor:
    """Move every parameter of ``policy`` into ONE flat fp32 buffer (``PARAM_ORDER``) and re-point its tensors at views of it."""
    if not policy.has_value or "log_std" not in policy.tensors:
        raise ValueError("training needs actor, critic and log_std")
    sizes = [policy.tensors[k].numel() for k in PARAM_ORDER]
    flat = torch.empty(sum(sizes), dtype=torch.float32, device=policy.device)
    off = 0
    for k, n in zip(PARAM_ORDER, sizes):
        view = flat[off:off + n].view_as(policy.tensors[k])
        view.copy_(policy.tensors[k])
        policy.tensors[k] = view
        off += n
    policy._c = None   # rebuild the C view with the new pointers
    expect = _lib.lib().kin_ppo_param_count(policy.in_dim)
    if expect != flat.numel():
        raise RuntimeError(f"flat parameter count {flat.numel()} != library layout {expect}")
    return flat


def random_policy(in_dim: int = 56, *, seed: int = 0, log_std_init: float = 0.0, device: str | torch.device = "cuda") -> PolicyWeights:
    """Fresh ``MultiInputPolicy``-shaped weights (orthogonal init with SB3's gains: sqrt(2) hidden, 0.01 action, 1 value)."""
    g = torch.Generator().manual_seed(seed)

    def ortho(rows: int, cols: int, gain: float) -> torch.Tensor:
        a = torch.randn(max(rows, cols), min(rows, cols), generator=g)
        q, r = torch.linalg.qr(a)
        q = q * torch.sign(torch.diagonal(r))
        q = q.t() if rows < cols else q
        return (gain * q[:rows, :cols]).contiguous()

    sd = {}
    for net, out_key, out_dim, gain in (("policy_net", "action_net", 7, 0.01), ("value_net", "value_net", 1, 1.0)):
        sd[f"mlp_extractor.{net}.0.weight"] = ortho(64, in_dim, 2 ** 0.5)
        sd[f"mlp_extractor.{net}.0.bias"] = torch.zeros(64)
        sd[f"mlp_extractor.{net}.2.weight"] = ortho(64, 64, 2 ** 0.5)
        sd[f"mlp_extractor.{net}.2.bias"] = torch.zeros(64)
        sd[f"{out_key}.weight"] = ortho(out_dim, 64, gain)
        sd[f"{out_key}.bias"] = torch.zeros(out_dim)
    sd["log_std"] = torch.full((7,), float(log_std_init))
    return PolicyWeights({k: v.numpy() for k, v in sd.items()}, device)


class PPOTrainer:
    """Batched on-device PPO: ``collect()`` fills the rollout buffer, ``update()`` runs the epochs, ``learn()`` loops.

    Two env families: the 56-input Approach / Finisher policies on ``BatchedArmKinematicEnv`` (``config`` = ``Phase1EnvConfig``;
    ``train_workspace_expansion.py:144-270``), and -- with ``route=`` -- the 80-input route policy on ``BatchedRouteKinematicEnv``
    (``config`` = ``RouteEnvConfig``; ``train_route_curriculum.py``): one fused ``kin_route_collect`` launch per rollout (or per
    ``route_chunk_steps`` steps under a prefix curriculum; ``collect_variant="steps"`` is the five-launches-per-step restatement) and the
    tensor-core update on constant-folded observation images.
    """

    def __init__(self, config: Any, policy: PolicyWeights, *, num_envs: int, hyper: PPOHyper, device: str | torch.device = "cuda",
                 seed: int = 0, stage_index: int = 0, process_group: Any = None, grad_ctas: int | None = None,
                 update_variant: str = "tc", collect_variant: str | None = None, handoff_states: torch.Tensor | None = None,
                 grad_exchange: str = "nccl", route: Any = None, route_sequence_config: Any = None, route_curriculum: Any = None,
                 shuffle: str = "tile", fused_update: bool | None = None) -> None:
        if not torch.cuda.is_available():
            raise _lib.KinError("PPOTrainer needs a CUDA device; there is no CPU fallback")
        self.in_dim = int(policy.in_dim)
        self.is_route = route is not None
        if self.in_dim != (80 if self.is_route else 56):
            raise _lib.KinError("PPOTrainer: 56-input policies train on the arm env, the 80-input route policy needs route=<RouteDataset>")
        if self.is_route:
            if update_variant != "tc" or num_envs % 128:
                raise ValueError("route training uses update_variant='tc' (folded bf16 observation images: num_envs must be a multiple of 128)")
            # "fused": ONE kin_route_collect launch per rollout (or per `route_chunk_steps` steps when a prefix curriculum must be able
            # to widen the reset window mid-rollout); "steps": five launches per time step (the restatement the fused kernel is tested against)
            collect_variant = collect_variant or ("fused" if num_envs % 128 == 0 else "steps")
        tile = _D("KIN_PPO_TILE")
        if num_envs % tile:
            raise ValueError(f"num_envs must be a multiple of {tile}")
        if update_variant not in ("tc", "fp32"):
            raise ValueError("update_variant must be 'tc' (tcgen05 bf16 GEMMs, fp32 accumulate) or 'fp32' (strict FP32-pipe kernel)")
        if grad_exchange not in ("nccl", "peer"):
            raise ValueError("grad_exchange must be 'nccl' (torch.distributed all-reduce) or 'peer' (NVLink peer-memory push, one node)")
        # minibatch composition: "tile" = random unions of 64-sample tiles of the rollout order (64 consecutive envs of one time step; no
        # data movement); "sample" = SB3's RolloutBuffer.get -- a fresh permutation of ALL samples every epoch (kin_ppo_shuffle moves the
        # rollout once per epoch, +0.6 ms per 8 M samples); "sample_once" = one per-sample permutation per rollout, tile unions after that
        if shuffle not in ("tile", "sample", "sample_once"):
            raise ValueError("shuffle must be 'tile', 'sample' (SB3: per-sample permutation every epoch) or 'sample_once'")
        if shuffle != "tile" and (num_envs * int(hyper.n_steps)) % 128:
            raise ValueError("per-sample shuffling moves 128-sample blocks: num_envs * n_steps must be a multiple of 128")
        self.shuffle = shuffle
        self._use_shadow = False
        self._shadow = None
        self.update_variant = update_variant
        # "fused": one kin_ppo_collect launch per rollout (tensor-core policy, bf16 observation images, needs the tc update);
        # "steps": one policy / env-step / bootstrap launch per time step (strict fp32, fp32 observation buffer)
        self.collect_variant = collect_variant or ("fused" if update_variant == "tc" and num_envs % 128 == 0 else "steps")
        if self.collect_variant not in ("fused", "steps"):
            raise ValueError("collect_variant must be 'fused' or 'steps'")
        if self.collect_variant == "fused" and (update_variant != "tc" or num_envs % 128):
            raise ValueError("the fused collection runs 128-env GEMM tiles and feeds the tensor-core update: it needs update_variant='tc' and num_envs % 128 == 0")
        self.device = torch.device(device)
        self.group = process_group
        self.rank, self.world = world(process_group)
        self.cfg, self.hp, self.policy = config, hyper, policy
        self.N, self.T = int(num_envs), int(hyper.n_steps)
        self.S = self.N * self.T
        self.local_batch = int(hyper.batch_size)
        if self.local_batch % tile or self.S % self.local_batch:
            raise ValueError("batch_size must be a multiple of 64 and divide num_envs * n_steps (per rank)")
        if update_variant == "tc" and (self.local_batch % (2 * tile) or self.S % (2 * tile)):
            raise ValueError("the tensor-core update pairs 64-sample tiles: batch_size and num_envs * n_steps must be multiples of 128")
        self._L = _lib.lib()
        self.seed = int(seed) + 7919 * self.rank
        with torch.cuda.device(self.device):
            self.params = flatten_policy_(policy)
            self.P = self.params.numel()
            self.adam_m = torch.zeros_like(self.params)
            self.adam_v = torch.zeros_like(self.params)
            # gradient and per-minibatch statistics share one buffer so that several ranks need ONE all-reduce per minibatch
            self._gradstats = torch.zeros(self.P + _D("KIN_PPO_STATS"), dtype=torch.float32, device=self.device)
            self.grad = self._gradstats[: self.P]
            self.stats = self._gradstats[self.P:]
            # bf16 operand image of `params` (the route policy's is constant-folded: rebuilt after every Adam step, not patched in place)
            self.weight_image = torch.zeros(36864, dtype=torch.uint8, device=self.device)
            self.pack_weights()
            self.stats_accum = torch.zeros(_D("KIN_PPO_STATS"), dtype=torch.float32, device=self.device)
            self._adv_stats = torch.zeros((max(self.S // self.local_batch, 1), 2), dtype=torch.float32, device=self.device)
            props = torch.cuda.get_device_properties(self.device)
            self.grad_ctas = int(grad_ctas or props.multi_processor_count)
            self.partials = torch.zeros((self.grad_ctas, self.P + _D("KIN_PPO_STATS") + 8), dtype=torch.float32, device=self.device)
            # several ranks: the per-minibatch gradient sum goes through NCCL or through NVLink peer buffers (distributed.PeerGradExchange)
            self.peer = PeerGradExchange(self.P, self.device, process_group) if grad_exchange == "peer" else None
            # One launch per minibatch (kin_ppo_grad_tc_update): gradient, reduction, rank-ordered exchange, clip + Adam all in the tensor-core
            # gradient kernel's tail.  Default with several ranks on the peer-memory exchange, where the tail already holds the grid barrier
            # and the summed slice (2 x B200: update 19.21 ms vs 19.51 ms with a separate Adam launch, NCCL 19.76 ms).  A single rank can ask
            # for it too (it then owns a one-rank exchange buffer) but gains nothing: 18.6 vs 18.4 ms -- the two grid barriers and the slice
            # reduction cost what the two small launches did.
            if fused_update is None:
                fused_update = update_variant == "tc" and self.peer is not None and self.world > 1
            if fused_update and (update_variant != "tc" or (self.peer is None and self.world > 1)):
                raise ValueError("fused_update needs update_variant='tc' and, with several ranks, grad_exchange='peer'")
            self.fused_update = bool(fused_update)
            if self.fused_update and self.peer is None:
                self.peer = PeerGradExchange(self.P, self.device, None)
            self._norm_scratch = torch.zeros(2 * self.grad_ctas, dtype=torch.float32, device=self.device)
            self._adam_done = False
            self.route_curriculum = None
            if self.is_route:
                from .route import BatchedRouteKinematicEnv

                self.env = BatchedRouteKinematicEnv(route, config, self.N, self.device, sequence_config=route_sequence_config)
                self.route_curriculum = route_curriculum
                if route_curriculum is not None:
                    if self.world > 1:
                        raise _lib.KinError("route prefix curriculum promotion is per process; run route training on one rank or without it")
                    self.env.set_route_window(max_route_index=route_curriculum.prefix_end_index)
            else:
                self.env = BatchedArmKinematicEnv(config, self.N, self.device, auto_reset=True, seed=self.seed, host_sampler=False, with_aux=False)
                self.env.set_curriculum_stage(stage_index)
                if handoff_states is not None:       # Finisher training: dock resets replay Approach handoff states (handoff.py)
                    self.env.set_handoff_states(handoff_states)
            f32 = dict(dtype=torch.float32, device=self.device)
            fused = self.collect_variant == "fused" and not self.is_route      # the arm path's fused collection stores bf16 operand images
            self.obs_buf = None if fused else torch.zeros((self.T + 1, self.N, self.in_dim), **f32)
            if self.collect_variant == "fused":
                base_cfg = config.base_env_config if self.is_route else config
                limit = max(int(getattr(base_cfg.termination_config, "max_episode_steps", base_cfg.episode_length)), 1)
                self.boot_cap = self.N * (self.T // limit + 2)     # an env hits the time limit at most once per `limit` steps
                self.boot_count = torch.zeros(1, dtype=torch.int32, device=self.device)
                self.boot_index = torch.zeros(self.boot_cap, dtype=torch.int32, device=self.device)
                self.boot_obs = torch.zeros((self.boot_cap, self.in_dim), **f32)
            if fused or (self.is_route and self.N % 128 == 0):
                self.obs_img = torch.zeros((self.T, self.N // 128, 128 * 128), dtype=torch.uint8, device=self.device)
            self.act_buf = torch.zeros((self.T, self.N, 7), **f32)
            self.logp_buf = torch.zeros((self.T, self.N), **f32)
            self.val_buf = torch.zeros((self.T, self.N), **f32)
            self.rew_buf = torch.zeros((self.T, self.N), **f32)
            self.done_buf = torch.zeros((self.T, self.N), dtype=torch.uint8, device=self.device)
            self.start_buf = torch.zeros((self.T, self.N), dtype=torch.uint8, device=self.device)
            self.adv_buf = torch.zeros((self.T, self.N), **f32)
            self.ret_buf = torch.zeros((self.T, self.N), **f32)
            self.last_val = torch.zeros(self.N, **f32)
            self.tile_sums = torch.zeros((self.S // tile, 2), dtype=torch.float64, device=self.device)
            self._gen = torch.Generator(device=self.device)
            self._gen.manual_seed(self.seed)
            if self.is_route:
                self.env.reset(seed=self.seed)
            else:
                self.env.reset()
            if not fused:
                self.obs_buf[0].copy_(self.env.obs)
        self._next_start = torch.ones(self.N, dtype=torch.uint8, device=self.device)
        self.tiles_per_cta = 0              # fused collection: 128-env tiles per CTA (0 = fewest that fit one wave)
        # grad_exchange="peer" with the tensor-core update: True runs the exchange inside the gradient kernel's tail
        # (kin_ppo_grad_tc_exchange) instead of the push + gather kernels: two launches per minibatch instead of four, bitwise the same
        # sums (2 x B200, 65 536 envs: update 20.06 vs 20.42 ms; NCCL 19.87 ms; one GPU 18.45 ms)
        self.fused_exchange = True
        # the tensor-core update reads bf16 operand images: written by the fused arm collection, or built from the route observations
        self._img = self.update_variant == "tc" and (self.is_route or self.collect_variant == "fused")
        self.route_chunk_steps = 16         # fused route collection with a prefix curriculum: steps per launch (promotion latency)
        self.num_timesteps = 0
        self.update_count = 0
        self.global_step = 0
        cur = None if self.is_route else config.curriculum_config
        self.curriculum = CurriculumTracker(len(cur.stages), cur.success_rate_threshold, cur.window_episodes, cur.min_episodes_per_stage,
                                            stage_index) if (cur is not None and cur.enabled) else None
        self.last_rollout: dict[str, float] = {}

    def pack_weights(self) -> None:
        """Rebuild the bf16 operand image from ``self.params`` (needed after the parameters were written from outside the trainer)."""
        _lib.check(self._L.kin_ppo_pack_weights(self.params.data_ptr(), self.in_dim, self.weight_image.data_ptr(),
                                                torch.cuda.current_stream(self.device).cuda_stream))

    # ------------------------------------------------------------------ rollout
    def collect(self) -> dict[str, float]:
        """``collect_rollouts``: T steps of (sample action, env step with auto-reset, TimeLimit bootstrap), then GAE."""
        if self.is_route:
            return self._collect_route_fused() if self.collect_variant == "fused" else self._collect_route()
        self.env._ensure_sampler()          # a curriculum promotion since the last rollout re-uploads the device sampler
        if self.collect_variant == "fused":
            return self._collect_fused()
        L, env, hp = self._L, self.env, self.hp
        stream = torch.cuda.current_stream(self.device).cuda_stream
        w = ctypes.byref(self.policy.c)
        done_bits = _D("KIN_DONE_TERMINATED") | _D("KIN_DONE_TRUNCATED")
        with torch.cuda.device(self.device):
            for t in range(self.T):
                env.obs = self.obs_buf[t + 1]      # the step kernel writes the next observation straight into the buffer
                env.reward = self.rew_buf[t]
                env.done = self.done_buf[t]
                self.start_buf[t].copy_(self._next_start)
                _lib.check(L.kin_policy_act(w, self.obs_buf[t].data_ptr(), self.act_buf[t].data_ptr(), self.logp_buf[t].data_ptr(),
                                            self.val_buf[t].data_ptr(), self.N, self.seed, self.global_step, 0, stream))
                env.step_raw(self.act_buf[t])
                _lib.check(L.kin_ppo_bootstrap(w, env.terminal_obs.data_ptr(), self.done_buf[t].data_ptr(), self.rew_buf[t].data_ptr(),
                                               float(hp.gamma), self.N, stream))
                self._next_start = ((self.done_buf[t] & done_bits) != 0).to(torch.uint8)
                self.global_step += 1
            _lib.check(L.kin_policy_act(w, self.obs_buf[self.T].data_ptr(), self._scratch_act().data_ptr(),
                                        self._scratch_logp().data_ptr(), self.last_val.data_ptr(), self.N, self.seed, self.global_step, 1, stream))
            _lib.check(L.kin_ppo_gae(self.rew_buf.data_ptr(), self.val_buf.data_ptr(), self.start_buf.data_ptr(), self.last_val.data_ptr(),
                                     self.done_buf[self.T - 1].data_ptr(), float(hp.gamma), float(hp.gae_lambda), self.T, self.N,
                                     self.adv_buf.data_ptr(), self.ret_buf.data_ptr(), self.tile_sums.data_ptr(), stream))
            self.obs_buf[0].copy_(self.obs_buf[self.T])
        self.num_timesteps += self.S * self.world
        finished = (self.done_buf & done_bits) != 0
        succ = ((self.done_buf & _D("KIN_DONE_SUCCESS")) != 0) & finished
        self._finished, self._success = finished, succ      # [T, N] bool: the rollout's episode outcomes in callback order
        self.last_rollout = {"episodes": float(finished.sum()), "successes": float(succ.sum()), "mean_reward": float(self.rew_buf.mean())}
        return self.last_rollout

    def _collect_route(self) -> dict[str, float]:
        """Route env rollout: per step policy sample -> ``kin_route_step`` -> TimeLimit bootstrap from the terminal observation ->
        sampled route reset of the finished slots in one launch (``kin_route_reset_sampled``), all on the device with no host round trip
        and every kernel writing straight into the rollout buffers.
        The finished episodes' flags are kept per step and fed to the prefix curriculum in time order after the rollout, so a
        promotion widens the reset window from the next rollout on (the reference's callback widens it at the very step)."""
        L, env, hp = self._L, self.env, self.hp
        stream = torch.cuda.current_stream(self.device).cuda_stream
        w = ctypes.byref(self.policy.c)
        done_bits = _D("KIN_DONE_TERMINATED") | _D("KIN_DONE_TRUNCATED")
        if not hasattr(self, "_route_raw"):
            self._route_raw = torch.zeros((self.T, self.N), dtype=torch.int32, device=self.device)      # KIN_RAUX_FLAGS word per step
        flag_row = env.raux[_D("KIN_RAUX_FLAGS"), : self.N].view(torch.int32)
        keep = env.obs, env.reward, env.done
        with torch.cuda.device(self.device):
            self.start_buf[0].copy_(self._next_start)
            for t in range(self.T):       # five launches per step: policy, route step, bootstrap, flag row, sampled reset
                env.obs, env.reward, env.done = self.obs_buf[t + 1], self.rew_buf[t], self.done_buf[t]     # written in place by the kernels
                _lib.check(L.kin_policy_act(w, self.obs_buf[t].data_ptr(), self.act_buf[t].data_ptr(), self.logp_buf[t].data_ptr(),
                                            self.val_buf[t].data_ptr(), self.N, self.seed, self.global_step, 0, stream))
                env.step_raw(self.act_buf[t])
                # env.obs now holds the terminal observation of the slots that just finished (no auto-reset inside the step kernel)
                _lib.check(L.kin_ppo_bootstrap(w, env.obs.data_ptr(), env.done.data_ptr(), env.reward.data_ptr(), float(hp.gamma), self.N, stream))
                self._route_raw[t].copy_(flag_row)
                env.reset_done(seed=self.seed ^ 0x5EED, counter=self.global_step)       # rewrites the finished slots' rows of obs_buf[t + 1]
                self.global_step += 1
            env.obs, env.reward, env.done = keep
            env.obs.copy_(self.obs_buf[self.T])
            finished = (self.done_buf & done_bits) != 0
            self.start_buf[1:].copy_(finished[:-1])
            self._next_start = finished[-1].to(torch.uint8)
            _lib.check(L.kin_policy_act(w, self.obs_buf[self.T].data_ptr(), self._scratch_act().data_ptr(),
                                        self._scratch_logp().data_ptr(), self.last_val.data_ptr(), self.N, self.seed, self.global_step, 1, stream))
            _lib.check(L.kin_ppo_gae(self.rew_buf.data_ptr(), self.val_buf.data_ptr(), self.start_buf.data_ptr(), self.last_val.data_ptr(),
                                     self.done_buf[self.T - 1].data_ptr(), float(hp.gamma), float(hp.gae_lambda), self.T, self.N,
                                     self.adv_buf.data_ptr(), self.ret_buf.data_ptr(), self.tile_sums.data_ptr(), stream))
            self.obs_buf[0].copy_(self.obs_buf[self.T])
            raw = self._route_raw
            flags = torch.stack([finished, (self.done_buf & _D("KIN_DONE_SUCCESS")) != 0, (raw & 1) != 0, (raw & 4) != 0, (raw & 2) != 0],
                                dim=1).cpu().numpy()          # [T, 5, N]: finished, success, route_ready, orientation_hit, regression
        fin = flags[:, 0]
        episodes, successes = float(fin.sum()), float((flags[:, 1] & fin).sum())
        if self.route_curriculum is not None:
            promoted = False
            for t in range(self.T):
                ids = np.nonzero(fin[t])[0]
                if ids.size:
                    promoted |= self.route_curriculum.record(flags[t, 1, ids], flags[t, 2, ids], flags[t, 3, ids], flags[t, 4, ids],
                                                            total_timesteps=self.num_timesteps + (t + 1) * self.N * self.world)
            if promoted:
                env.set_route_window(max_route_index=self.route_curriculum.prefix_end_index)
        self.num_timesteps += self.S * self.world
        self.last_rollout = {"episodes": episodes, "successes": successes, "mean_reward": float(self.rew_buf.mean())}
        return self.last_rollout

    def _collect_route_fused(self) -> dict[str, float]:
        """Route env rollout in fused launches (``kin_route_collect``): policy forward on tcgen05, route step with waypoint advance,
        sampled route resets -- same draws, same arithmetic as the per-step path (``_collect_route``), which the kernel is replayed
        against.  Without a prefix curriculum the whole rollout is ONE launch.  With one, the rollout runs in chunks of
        ``route_chunk_steps`` steps and the finished episodes of each chunk are fed to the curriculum in time order before the next
        chunk starts, so a promotion widens the reset window at most ``route_chunk_steps`` steps after the step that triggered it
        (the reference's callback widens it at that very step, route/route_curriculum.py:85-99; chunk 1 reproduces that)."""
        L, env, hp = self._L, self.env, self.hp
        done_bits = _D("KIN_DONE_TERMINATED") | _D("KIN_DONE_TRUNCATED")
        if not hasattr(self, "_route_raw"):
            self._route_raw = torch.zeros((self.T, self.N), dtype=torch.int32, device=self.device)
        chunk = self.T if self.route_curriculum is None else max(1, min(int(self.route_chunk_steps), self.T))
        seq = env.sequence is not None
        episodes = successes = 0.0
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            t0 = 0
            while t0 < self.T:
                tc = min(chunk, self.T - t0)
                _lib.check(L.kin_route_collect(
                    env._params.handle, ctypes.byref(env.table.c), ctypes.byref(env._reset_params()), env.state.data_ptr(), env.stride, self.N,
                    self.params.data_ptr(), tc, self.seed, self.global_step, self.seed ^ 0x5EED, int(seq),
                    int(bool(env.sequence.reset_ready_streak_on_advance)) if seq else 1, self.obs_buf[t0].data_ptr(), self.act_buf[t0].data_ptr(),
                    self.logp_buf[t0].data_ptr(), self.val_buf[t0].data_ptr(), self.rew_buf[t0].data_ptr(), self.done_buf[t0].data_ptr(),
                    self.start_buf[t0].data_ptr(), self._route_raw[t0].data_ptr(), self._next_start.data_ptr(), self.last_val.data_ptr(),
                    self.boot_count.data_ptr(), self.boot_index.data_ptr(), self.boot_obs.data_ptr(), self.boot_cap, int(self.tiles_per_cta), stream))
                # time-limit episodes of this chunk: r += gamma * V(terminal observation); indices are relative to the chunk's first row
                _lib.check(L.kin_ppo_bootstrap_list(self.params.data_ptr(), 80, self.boot_obs.data_ptr(), self.boot_index.data_ptr(), self.boot_count.data_ptr(),
                                                    self.boot_cap, self.rew_buf[t0].data_ptr(), float(hp.gamma), stream))
                self.global_step += tc
                if self.route_curriculum is not None:
                    d, raw = self.done_buf[t0:t0 + tc], self._route_raw[t0:t0 + tc]
                    fin = (d & done_bits) != 0
                    flags = torch.stack([fin, (d & _D("KIN_DONE_SUCCESS")) != 0, (raw & 1) != 0, (raw & 4) != 0, (raw & 2) != 0], dim=1).cpu().numpy()
                    promoted = False
                    for t in range(tc):
                        ids = np.nonzero(flags[t, 0])[0]
                        if ids.size:
                            promoted |= self.route_curriculum.record(flags[t, 1, ids], flags[t, 2, ids], flags[t, 3, ids], flags[t, 4, ids],
                                                                    total_timesteps=self.num_timesteps + (t0 + t + 1) * self.N * self.world)
                    if promoted:
                        env.set_route_window(max_route_index=self.route_curriculum.prefix_end_index)
                if int(self.boot_count.item()) > self.boot_cap:
                    raise _lib.KinError("TimeLimit bootstrap list overflow in the fused route collection: rebuild the trainer")
                t0 += tc
            _lib.check(L.kin_ppo_gae(self.rew_buf.data_ptr(), self.val_buf.data_ptr(), self.start_buf.data_ptr(), self.last_val.data_ptr(),
                                     self.done_buf[self.T - 1].data_ptr(), float(hp.gamma), float(hp.gae_lambda), self.T, self.N,
                                     self.adv_buf.data_ptr(), self.ret_buf.data_ptr(), self.tile_sums.data_ptr(), stream))
            env.obs.copy_(self.obs_buf[self.T])
        finished = (self.done_buf & done_bits) != 0
        succ = ((self.done_buf & _D("KIN_DONE_SUCCESS")) != 0) & finished
        self._finished, self._success = finished, succ
        self.num_timesteps += self.S * self.world
        self.last_rollout = {"episodes": float(finished.sum()), "successes": float(succ.sum()), "mean_reward": float(self.rew_buf.mean())}
        return self.last_rollout

    def _collect_fused(self) -> dict[str, float]:
        """The whole rollout in one launch (``kin_ppo_collect``), then the TimeLimit bootstrap of the listed episodes and GAE."""
        L, env, hp = self._L, self.env, self.hp
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            if env._mode_all is None:
                raise _lib.KinError("the fused collection runs ONE policy mode for all envs; per-env mixed modes need collect_variant='steps'")
            mode = env._mode_all
            _lib.check(L.kin_ppo_collect(env._params.handle, env.state.data_ptr(), env.stride, self.N, mode, self.params.data_ptr(), self.weight_image.data_ptr(), 56,
                                         self.T,
                                         self.seed, self.global_step, env._seed, self.obs_img.data_ptr(), self.act_buf.data_ptr(),
                                         self.logp_buf.data_ptr(), self.val_buf.data_ptr(), self.rew_buf.data_ptr(), self.done_buf.data_ptr(),
                                         self.start_buf.data_ptr(), self._next_start.data_ptr(), self.last_val.data_ptr(), self.boot_count.data_ptr(),
                                         self.boot_index.data_ptr(), self.boot_obs.data_ptr(), self.boot_cap, int(self.tiles_per_cta), stream))
            _lib.check(L.kin_ppo_bootstrap_list(self.params.data_ptr(), 56, self.boot_obs.data_ptr(), self.boot_index.data_ptr(),
                                                self.boot_count.data_ptr(), self.boot_cap, self.rew_buf.data_ptr(), float(hp.gamma), stream))
            _lib.check(L.kin_ppo_gae(self.rew_buf.data_ptr(), self.val_buf.data_ptr(), self.start_buf.data_ptr(), self.last_val.data_ptr(),
                                     self.done_buf[self.T - 1].data_ptr(), float(hp.gamma), float(hp.gae_lambda), self.T, self.N,
                                     self.adv_buf.data_ptr(), self.ret_buf.data_ptr(), self.tile_sums.data_ptr(), stream))
        return self._finish_fused_collect()

    def _finish_fused_collect(self) -> dict[str, float]:
        """Host bookkeeping after a fused arm collection (this trainer's own launches or a ``PPOPopulation``'s): step counters,
        bootstrap-list overflow check, the rollout's episode outcomes and ``last_rollout``."""
        self.global_step += self.T
        self.num_timesteps += self.S * self.world
        if int(self.boot_count.item()) > self.boot_cap:       # the kernel drops entries past the capacity: returns would be biased
            raise _lib.KinError(f"TimeLimit bootstrap list overflow ({int(self.boot_count.item())} > {self.boot_cap}): the env's episode limit "
                                "changed after the trainer was built; rebuild the trainer")
        done_bits = _D("KIN_DONE_TERMINATED") | _D("KIN_DONE_TRUNCATED")
        finished = (self.done_buf & done_bits) != 0
        succ = ((self.done_buf & _D("KIN_DONE_SUCCESS")) != 0) & finished
        self._finished, self._success = finished, succ      # [T, N] bool: the rollout's episode outcomes in callback order
        self.last_rollout = {"episodes": float(finished.sum()), "successes": float(succ.sum()), "mean_reward": float(self.rew_buf.mean())}
        return self.last_rollout

    def _scratch_act(self) -> torch.Tensor:
        if not hasattr(self, "_sa"):
            self._sa = torch.zeros((self.N, 7), dtype=torch.float32, device=self.device)
            self._sl = torch.zeros(self.N, dtype=torch.float32, device=self.device)
        return self._sa

    def _scratch_logp(self) -> torch.Tensor:
        self._scratch_act()
        return self._sl

    # ------------------------------------------------------------------ update
    def _buffers(self) -> tuple[int, int, int, int, int, int]:
        """Device pointers of (observations, actions, old log-probs, advantages, returns, tile sums) the update reads: the rollout buffers,
        or their per-sample-permuted copies while a ``shuffle="sample"`` epoch runs."""
        if self._use_shadow:
            sh = self._shadow
            return (sh["obs"].data_ptr(), sh["act"].data_ptr(), sh["logp"].data_ptr(), sh["adv"].data_ptr(), sh["ret"].data_ptr(), sh["sums"].data_ptr())
        obs = self.obs_img if (self.update_variant == "tc" and self._img) else self.obs_buf
        return (obs.data_ptr(), self.act_buf.data_ptr(), self.logp_buf.data_ptr(), self.adv_buf.data_ptr(), self.ret_buf.data_ptr(), self.tile_sums.data_ptr())

    def _shuffle_samples(self) -> None:
        """SB3 ``RolloutBuffer.get``: permute ALL samples of the rollout (device permutation from the trainer's generator) into the shadow
        buffers; the epoch's minibatches are then consecutive tile ranges of the permuted order."""
        img = self.update_variant == "tc" and self._img
        if self._shadow is None:
            f32 = dict(dtype=torch.float32, device=self.device)
            self._shadow = {"obs": torch.empty((self.S // 128, 16384), dtype=torch.uint8, device=self.device) if img else torch.empty((self.S, self.in_dim), **f32),
                            "act": torch.empty((self.S, 7), **f32), "logp": torch.empty(self.S, **f32), "adv": torch.empty(self.S, **f32),
                            "ret": torch.empty(self.S, **f32), "sums": torch.empty((self.S // _D("KIN_PPO_TILE"), 2), dtype=torch.float64, device=self.device)}
        sh = self._shadow
        perm = torch.randperm(self.S, generator=self._gen, device=self.device, dtype=torch.int64).to(torch.int32)
        self._use_shadow = False
        obs, act, logp, adv, ret, _ = self._buffers()
        _lib.check(self._L.kin_ppo_shuffle(obs, int(img), self.in_dim, act, logp, adv, ret, perm.data_ptr(), self.S, sh["obs"].data_ptr(), sh["act"].data_ptr(),
                                           sh["logp"].data_ptr(), sh["adv"].data_ptr(), sh["ret"].data_ptr(), sh["sums"].data_ptr(),
                                           torch.cuda.current_stream(self.device).cuda_stream))
        self._sample_perm = perm
        self._use_shadow = True

    def _grad_launch(self, tile_ptr: int, n_tiles: int, adv_ptr: int | None, with_update: bool = False) -> None:
        stream = torch.cuda.current_stream(self.device).cuda_stream
        hp = self._c_hyper
        global_batch = n_tiles * _D("KIN_PPO_TILE") * self.world
        obs, act, logp, adv, ret, sums = self._buffers()
        if self.update_variant == "tc":
            img = self._img
            wimg = self.weight_image.data_ptr()
            if self.peer and self.fused_exchange and self.fused_update and with_update:      # ... and clip + Adam: ONE launch per minibatch
                _lib.check(self._L.kin_ppo_grad_tc_update(self.params.data_ptr(), self.in_dim, ctypes.byref(hp), obs, act, logp, adv, ret, sums,
                                                          tile_ptr, n_tiles, global_batch, self.partials.data_ptr(), self.grad_ctas, self.grad.data_ptr(),
                                                          self.stats.data_ptr(), int(img), adv_ptr, wimg, self.peer.buffers, self.peer.rank, self.peer.world,
                                                          self.peer.next_epoch(), self.peer.timed_out.data_ptr(), self.params.data_ptr(),
                                                          self.adam_m.data_ptr(), self.adam_v.data_ptr(), self.update_count + 1, self.stats_accum.data_ptr(),
                                                          self._norm_scratch.data_ptr(), stream))
                self._adam_done = True
                return
            if self.peer and self.fused_exchange:     # reduce + push + rank-ordered gather inside the gradient kernel's tail
                _lib.check(self._L.kin_ppo_grad_tc_exchange(self.params.data_ptr(), self.in_dim, ctypes.byref(hp), obs, act, logp, adv, ret, sums,
                                                            tile_ptr, n_tiles, global_batch, self.partials.data_ptr(), self.grad_ctas, self.grad.data_ptr(),
                                                            self.stats.data_ptr(), int(img), adv_ptr, wimg, self.peer.buffers, self.peer.rank, self.peer.world,
                                                            self.peer.next_epoch(), self.peer.timed_out.data_ptr(), stream))
                return
            _lib.check(self._L.kin_ppo_grad_tc(self.params.data_ptr(), self.in_dim, ctypes.byref(hp), obs, act, logp, adv, ret, sums, tile_ptr, n_tiles,
                                               global_batch, self.partials.data_ptr(), self.grad_ctas, None if self.peer else self.grad.data_ptr(),
                                               self.stats.data_ptr(), None, None, 0, int(img), adv_ptr, wimg, stream))
            if self.peer:
                self.peer.push(self.partials, min(self.grad_ctas, n_tiles // 2), global_batch)
            return
        _lib.check(self._L.kin_ppo_grad(self.params.data_ptr(), 56, ctypes.byref(hp), obs, act, logp, adv, ret, sums,
                                        tile_ptr, n_tiles, global_batch, self.partials.data_ptr(), self.grad_ctas,
                                        None if self.peer else self.grad.data_ptr(), self.stats.data_ptr(), adv_ptr, stream))
        if self.peer:
            self.peer.push(self.partials, min(self.grad_ctas, n_tiles), global_batch)

    def minibatch_grad(self, tile_ids: torch.Tensor) -> None:
        """Gradient of one minibatch (sum over local samples, already divided by the GLOBAL minibatch size) into ``self.grad``."""
        self._c_hyper = self.hp.c()
        self._grad_launch(tile_ids.data_ptr(), int(tile_ids.numel()), None)

    def refresh_old_logp(self) -> None:
        """Recompute the rollout's log-probs with the tensor-core kernel's own forward (bf16 operands), so that the probability
        ratio of the first epoch is exactly 1 as in SB3 (the rollout sampled with the fp32 policy; the two forwards differ by O(1e-3))."""
        if not hasattr(self, "_all_tiles"):
            self._all_tiles = torch.arange(self.S // _D("KIN_PPO_TILE"), dtype=torch.int32, device=self.device)
        hp = self.hp.c()
        _lib.check(self._L.kin_ppo_grad_tc(self.params.data_ptr(), self.in_dim, ctypes.byref(hp), (self.obs_img if self._img else self.obs_buf).data_ptr(),
                                           self.act_buf.data_ptr(), None, None, None, None, self._all_tiles.data_ptr(), int(self._all_tiles.numel()), 0, None,
                                           self.grad_ctas, None, None, self.logp_buf.data_ptr(), None, 1, int(self._img), None, self.weight_image.data_ptr(),
                                           torch.cuda.current_stream(self.device).cuda_stream))

    def apply_update(self) -> None:
        """All-reduce the gradient (sum over ranks), clip by global norm, Adam step -- identical on every rank."""
        if self._adam_done:          # kin_ppo_grad_tc_update already did all of it in the gradient kernel's tail
            self._adam_done = False
            self.update_count += 1
            if self.is_route:        # the folded bias column mixes three parameters: rebuild the image
                _lib.check(self._L.kin_ppo_pack_weights(self.params.data_ptr(), self.in_dim, self.weight_image.data_ptr(),
                                                        torch.cuda.current_stream(self.device).cuda_stream))
            return
        if self.peer:
            if not (self.fused_exchange and self.update_variant == "tc"):  # (the fused form already left the rank-ordered sum in self.grad)
                self.peer.gather(self.grad, self.stats)                    # waits for every rank's push, rank-ordered sum
        elif self.world > 1:
            allreduce_sum_(self._gradstats[: self.P + 5], self.group)      # gradient + the five loss statistics
        self.update_count += 1
        hp = getattr(self, "_c_hyper", None) or self.hp.c()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self._L.kin_ppo_adam(self.params.data_ptr(), self.grad.data_ptr(), self.adam_m.data_ptr(), self.adam_v.data_ptr(), self.P,
                                        ctypes.byref(hp), self.update_count, self.stats.data_ptr(), self.stats_accum.data_ptr(),
                                        None if self.is_route else self.weight_image.data_ptr(), self.in_dim, stream))
        if self.is_route and self.update_variant == "tc":      # the folded bias column mixes three parameters: rebuild the image
            _lib.check(self._L.kin_ppo_pack_weights(self.params.data_ptr(), self.in_dim, self.weight_image.data_ptr(), stream))

    def _identity_tiles(self, n: int) -> torch.Tensor:
        if getattr(self, "_arange_tiles", None) is None or self._arange_tiles.numel() != n:
            self._arange_tiles = torch.arange(n, dtype=torch.int32, device=self.device)
        return self._arange_tiles

    def update(self) -> dict[str, float]:
        """``PPO.train``: n_epochs passes over the rollout in random minibatches; no host synchronisation until the statistics are read."""
        tile = _D("KIN_PPO_TILE")
        n_tiles_total = self.S // tile
        tiles_per_mb = self.local_batch // tile
        mb_per_epoch = n_tiles_total // tiles_per_mb
        self._c_hyper = self.hp.c()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            self.stats_accum.zero_()
            img = self._img
            if self.is_route and self.update_variant == "tc":      # fp32 route observations -> folded bf16 operand images, once per rollout
                _lib.check(self._L.kin_route_obs_images(self.obs_buf.data_ptr(), self.S, self.obs_img.data_ptr(), stream))
            if self.update_variant == "tc" and not (self.collect_variant == "fused" and not self.is_route):
                self.refresh_old_logp()        # (the arm path's fused collection already sampled with the update's own forward)
            adv = self._adv_stats
            kl_seen = mb_seen = 0.0
            for epoch in range(self.hp.n_epochs):
                if self.shuffle == "sample" or (self.shuffle == "sample_once" and epoch == 0):
                    self._shuffle_samples()
                if self.shuffle == "sample":      # the samples are freshly permuted: minibatch m = tiles [m k, (m + 1) k) of that order
                    perm = self._identity_tiles(n_tiles_total)
                elif img:   # minibatches are unions of whole 128-sample images: permute pairs of 64-sample tiles
                    p2 = torch.randperm(n_tiles_total // 2, generator=self._gen, device=self.device, dtype=torch.int64)
                    perm = torch.stack((2 * p2, 2 * p2 + 1), dim=1).reshape(-1).to(torch.int32)
                else:
                    perm = torch.randperm(n_tiles_total, generator=self._gen, device=self.device, dtype=torch.int64).to(torch.int32)
                self._perm = perm                          # keep the ids alive until the launches that read them have run
                _lib.check(self._L.kin_ppo_adv_stats(self._buffers()[5], perm.data_ptr(), tiles_per_mb, mb_per_epoch,
                                                     int(self.hp.normalize_advantage), adv.data_ptr(), stream))
                for m in range(mb_per_epoch):
                    self._grad_launch(perm.data_ptr() + 4 * m * tiles_per_mb, tiles_per_mb, adv.data_ptr() + 8 * m, with_update=True)
                    self.apply_update()
                if self.peer:
                    self.peer.poll()         # once per epoch, without a host sync: a dead peer surfaces after at most two epochs of skipped updates
                if self.hp.target_kl is not None:
                    # SB3 checks after every minibatch (ppo.py:262-267); here once per epoch, so the rollout stays one host sync per
                    # epoch instead of one per minibatch (the statistics are sums over the minibatches seen so far)
                    acc = self.stats_accum.cpu().numpy().astype(np.float64)
                    kl_epoch = (acc[3] - kl_seen) / max(acc[7] - mb_seen, 1.0)
                    kl_seen, mb_seen = acc[3], acc[7]
                    if kl_epoch > 1.5 * float(self.hp.target_kl):
                        break
            a = self.stats_accum.cpu().numpy().astype(np.float64)
            self._use_shadow = False
            if self.peer:
                self.peer.check()
        n_mb = max(int(round(a[7])), 1)
        a = a / n_mb
        return {"policy_loss": float(a[0]), "value_loss": float(a[1]), "entropy": float(a[2]), "approx_kl": float(a[3]),
                "clip_fraction": float(a[4]), "grad_norm": float(a[5]), "minibatches": n_mb}

    def _frontier_refresh(self, frontier: Any, force: bool) -> dict[str, Any] | None:
        rec = frontier.maybe_refresh(self.num_timesteps, self.policy, self.env, force=force)
        if rec is not None:     # every rank ran the same eval on bitwise-identical parameters: the tables must agree
            check_same_on_all_ranks(rec["table_checksum"], "the adaptive frontier table", self.group)
        return rec

    def learn(self, iterations: int, gate: Any = None, frontier: Any = None) -> list[dict[str, float]]:
        """``model.learn``: iterations of collect + update; curriculum promotion; optional eval gate (``gate.EvalGate``); optional
        adaptive frontier curriculum (``coverage.FrontierCurriculum``: refreshed before the first rollout, then after every update
        once its interval has passed; a row gets ``frontier_<field>`` entries when a refresh ran)."""
        if frontier is not None and self.is_route:
            raise _lib.KinError("the adaptive frontier curriculum draws arm-env goals; the route trainer has no use for it")
        pending = self._frontier_refresh(frontier, force=True) if frontier is not None else None
        log = []
        for _ in range(int(iterations)):
            r = self.collect()
            u = self.update()
            if self.curriculum is not None and self.curriculum.record_rollout(self._finished, self._success, self.group, self.num_timesteps):
                self.env.set_curriculum_stage(self.curriculum.stage_index)
            stage = float(self.route_curriculum.current_stage_index) if (self.is_route and self.route_curriculum is not None) else (
                0.0 if self.is_route else float(self.env.get_curriculum_stage()))
            row = {**r, **u, "stage": stage, "timesteps": float(self.num_timesteps)}
            if gate is not None:
                rec = gate.maybe_eval(self.num_timesteps, self.policy)
                if rec is not None:
                    row["gate_score"] = float(rec["score"])
            if frontier is not None:
                rec = self._frontier_refresh(frontier, force=False) or pending
                pending = None
                if rec is not None:
                    row.update({f"frontier_{k}": float(v) for k, v in rec.items() if isinstance(v, (int, float))})
            log.append(row)
        return log

    def close(self) -> None:
        """Release the peer-exchange buffers (several ranks: call on every rank after the last ``update``)."""
        if self.peer is not None:
            if self.world > 1:
                import torch.distributed as dist

                torch.cuda.synchronize(self.device)
                dist.barrier(group=self.group)       # nobody unmaps a buffer a peer may still be pushing into
            self.peer.close()
            self.peer = None

    def state_dict(self) -> dict[str, torch.Tensor]:
        """SB3 ``policy.pth`` key names, so a trained policy loads back into the reference (and vice versa)."""
        return {KEYS[f]: t.detach().clone() for f, t in self.policy.tensors.items()}

    # SB3's ``policy.parameters()`` order for MultiInputPolicy (= the index of each tensor in ``policy.optimizer.pth``)
    SB3_PARAM_ORDER = ("log_std", "pi_w0", "pi_b0", "pi_w1", "pi_b1", "vf_w0", "vf_b0", "vf_w1", "vf_b1", "act_w", "act_b", "val_w", "val_b")

    def _flat_views(self, flat: torch.Tensor) -> dict[str, torch.Tensor]:
        out, off = {}, 0
        for k in PARAM_ORDER:
            n = self.policy.tensors[k].numel()
            out[k] = flat[off:off + n].view_as(self.policy.tensors[k])
            off += n
        return out

    def save_checkpoint(self, path: str) -> None:
        """Everything a resume needs -- what SB3's ``model.save`` keeps (``train_workspace_expansion.py:187-196`` resumes with
        ``PPO.load``: weights AND Adam state AND the run's own hyper-parameters): ``policy.pth`` (SB3 key names),
        ``policy.optimizer.pth`` (torch-Adam state dict in SB3's parameter order), ``data`` (hyper-parameters, counters) and
        ``trainer_state.json`` (curriculum tracker, step counters)."""
        import io
        import json
        from dataclasses import asdict

        m, v = self._flat_views(self.adam_m), self._flat_views(self.adam_v)
        opt = {"state": {i: {"step": torch.tensor(float(self.update_count)), "exp_avg": m[k].detach().cpu().clone(),
                             "exp_avg_sq": v[k].detach().cpu().clone()} for i, k in enumerate(self.SB3_PARAM_ORDER)},
               "param_groups": [{"lr": self.hp.learning_rate, "betas": (self.hp.adam_beta1, self.hp.adam_beta2), "eps": self.hp.adam_eps,
                                 "weight_decay": 0, "amsgrad": False, "params": list(range(len(self.SB3_PARAM_ORDER)))}]}
        buf = io.BytesIO()
        torch.save(opt, buf)
        state = {"update_count": self.update_count, "num_timesteps": self.num_timesteps, "global_step": self.global_step,
                 "curriculum": None if self.curriculum is None else self.curriculum.state_dict(),
                 "stage_index": None if self.is_route else int(self.env.get_curriculum_stage())}
        data = {"policy_class": "MultiInputPolicy", "n_envs": self.N, "num_timesteps": self.num_timesteps, **asdict(self.hp)}
        self.policy.save_weights_zip(path, data=data, extra={"policy.optimizer.pth": buf.getvalue(), "trainer_state.json": json.dumps(state).encode()})

    def load_checkpoint(self, path: str, *, load_hyper: bool = True, learning_rate: float | None = None) -> None:
        """Resume from ``save_checkpoint`` output or from one of the REFERENCE's own ``model.zip`` files: weights, Adam moments and
        step count, and (``load_hyper``) the checkpoint's own gamma / gae_lambda / clip_range / ent_coef / vf_coef / max_grad_norm /
        n_epochs -- ``PPO.load(path, env, learning_rate=...)`` keeps all of those and only overrides the learning rate
        (``train_workspace_expansion.py:187-196``)."""
        import io
        import json
        import zipfile

        with zipfile.ZipFile(path) as z:
            names = set(z.namelist())
            sd = torch.load(io.BytesIO(z.read("policy.pth")), weights_only=True, map_location="cpu")
            opt = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), weights_only=True, map_location="cpu") if "policy.optimizer.pth" in names else None
            data = json.loads(z.read("data")) if "data" in names else {}
            state = json.loads(z.read("trainer_state.json")) if "trainer_state.json" in names else {}
        for f, key in KEYS.items():
            if f in self.policy.tensors and key in sd:
                self.policy.tensors[f].copy_(sd[key].to(self.device))
        if opt is not None and opt.get("state"):
            m, v = self._flat_views(self.adam_m), self._flat_views(self.adam_v)
            steps = []
            for i, k in enumerate(self.SB3_PARAM_ORDER):
                st = opt["state"].get(i)
                if st is None:
                    continue
                m[k].copy_(st["exp_avg"].to(self.device))
                v[k].copy_(st["exp_avg_sq"].to(self.device))
                steps.append(int(float(st["step"])))
            if steps:
                self.update_count = max(steps)
        if load_hyper:
            for k in ("gamma", "gae_lambda", "ent_coef", "vf_coef", "max_grad_norm", "n_epochs", "normalize_advantage"):
                if isinstance(data.get(k), (int, float, bool)):
                    setattr(self.hp, k, type(getattr(self.hp, k))(data[k]))
            if isinstance(data.get("clip_range"), (int, float)):
                self.hp.clip_range = float(data["clip_range"])
            if isinstance(data.get("learning_rate"), (int, float)):
                self.hp.learning_rate = float(data["learning_rate"])
        if learning_rate is not None:
            self.hp.learning_rate = float(learning_rate)
        self.update_count = int(state.get("update_count", self.update_count))
        self.num_timesteps = int(state.get("num_timesteps", data.get("num_timesteps", self.num_timesteps)) or 0)
        self.global_step = int(state.get("global_step", self.global_step))
        if self.curriculum is not None and state.get("curriculum"):
            self.curriculum.load_state_dict(state["curriculum"])
            self.env.set_curriculum_stage(self.curriculum.stage_index)
        elif state.get("stage_index") is not None and not self.is_route:
            self.env.set_curriculum_stage(int(state["stage_index"]))
        self.pack_weights()


def decode_obs_images(images: torch.Tensor) -> torch.Tensor:
    """``[..., 16384]`` uint8 operand images written by ``kin_ppo_collect`` -> ``[..., 128, 64]`` float32 rows
    (56 observation floats rounded to bf16, a constant 1 that carries the layer-1 bias, zero padding)."""
    lead = images.shape[:-1]
    chunks = images.reshape(*lead, 128, 8, 16)                       # row, 16-byte chunk slot, bytes
    r = torch.arange(128, device=images.device)[:, None]
    c = torch.arange(8, device=images.device)[None, :]
    slot = (c ^ (r & 7)).reshape(*([1] * len(lead)), 128, 8, 1).expand(*lead, 128, 8, 16)
    rows = torch.gather(chunks, -2, slot).reshape(*lead, 128, 128).contiguous()
    return rows.view(torch.bfloat16).float()


def encode_obs_images(obs: torch.Tensor) -> torch.Tensor:
    """``[n, 56]`` float observations (n a multiple of 128) -> ``[n / 128, 16384]`` uint8 operand images in the layout ``kin_ppo_collect``
    writes and ``kin_ppo_grad_tc(obs_is_image=1)`` reads: rows ``[bf16(obs56) | 1 | 0 x 7]``, SWIZZLE_128B (the inverse of
    ``decode_obs_images``; the chunk swizzle is an involution)."""
    n, d = obs.shape
    if n % 128 or d != 56:
        raise ValueError("encode_obs_images: [n, 56] observations, n a multiple of 128")
    rows = torch.zeros((n // 128, 128, 64), dtype=torch.bfloat16, device=obs.device)
    rows[..., :56] = obs.reshape(n // 128, 128, 56).to(torch.bfloat16)
    rows[..., 56] = 1.0
    chunks = rows.view(torch.uint8).reshape(n // 128, 128, 8, 16)
    r = torch.arange(128, device=obs.device)[:, None]
    c = torch.arange(8, device=obs.device)[None, :]
    slot = (c ^ (r & 7)).reshape(1, 128, 8, 1).expand(n // 128, 128, 8, 16)
    return torch.gather(chunks, -2, slot).reshape(n // 128, 16384).contiguous()


def numpy_gae(rewards: np.ndarray, values: np.ndarray, episode_starts: np.ndarray, last_values: np.ndarray, last_dones: np.ndarray,
              gamma: float, gae_lambda: float) -> tuple[np.ndarray, np.ndarray]:
    """Plain restatement of SB3 ``RolloutBuffer.compute_returns_and_advantage`` (host-side reference for tests)."""
    T = rewards.shape[0]
    adv = np.zeros_like(rewards, dtype=np.float64)
    last = np.zeros(rewards.shape[1])
    for step in reversed(range(T)):
        if step == T - 1:
            nnt, nv = 1.0 - last_dones.astype(np.float64), last_values.astype(np.float64)
        else:
            nnt, nv = 1.0 - episode_starts[step + 1].astype(np.float64), values[step + 1].astype(np.float64)
        delta = rewards[step] + gamma * nv * nnt - values[step]
        last = delta + gamma * gae_lambda * nnt * last
        adv[step] = last
    return adv, adv + values
