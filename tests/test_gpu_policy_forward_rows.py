"""Per-row checks of the tensor-core policy forwards against an fp64 MLP.

The fused training rollout (K4, kin_collect.cu), the fused route rollout (kin_route_collect.cu) and the forward-only mode of the
tensor-core update (K3-TC, kin_ppo_tc.cu) each run the SB3 MLP on tcgen05 with bf16 operands (the eval rollout K2-TC with fp16 operands).  A closed loop forgives a small bias
in the actions, so every output here is compared row by row with two references:

  * an emulation of the kernel's operand contract, written from the kernel source: observations, weights and the bias column
    rounded to bf16, folded biases summed in fp32 and then rounded, b1 / output biases in fp32, activations rounded to bf16 after
    tanh.  What remains against it is tanh.approx.f32 (which moves an activation across a bf16 rounding boundary now and then)
    and the fp32 summation order: the TIGHT bound.
  * the plain fp64 MLP on the same observation: the LOOSE bound, the intrinsic error of bf16 operands.

Errors are expressed in "activation units": an output error divided by the sum of |weights| of that output's row (what the output
moves by if every activation in front of it moves by 1), so one bound serves policies whose heads differ in scale by 1000x.
The bounds were set from a B200 run (1000 W power limit) with margin; the measured maxima are next to them.

The K4 actor mean is not written by the kernel.  It is recovered per row from the sampled action: the kernel draws its noise from
Philox(noise_seed, env, first_step + t), and kin_policy_act(seed = noise_seed, step = first_step + t) draws the same noise for row
env, so action_K4 - (action_fp32 - mean_fp32) is the kernel's mean to within an ulp of the action.

K2-TC (kin_rollout_tc16.cu, fp16 operands) writes no per-step output: it is checked through one-step episodes, whose final joint
vector is a function of the first action only.

The fold contract (every constant observation column holds its constant on every path, so folding them into the layer-1 bias is
exact) is checked on the arm step kernel in both modes, the K4 images, the route step kernels with both wrappers, the fused route
rollout and the golden reference traces.
"""

from __future__ import annotations

import ctypes
import dataclasses

import numpy as np
import pytest
import torch

from ._util import env_config, golden

# ---- constant observation columns ------------------------------------------------------------------------------------------
# arm observation (56): mode_flag one-hot 20..29, progress[2] = 39, task_type [1, 0, 0] 47..49, waypoint blocks 50..55
ARM_CONST = np.array(list(range(20, 30)) + [39] + list(range(47, 56)))
# route observation (80): the same blocks; the route mode flag is column 20, task_type[0] column 71
ROUTE_CONST = np.array(list(range(20, 30)) + [39] + list(range(71, 80)))
ROUTE_ONES = (20, 71)
ROUTE_LIVE = np.array([c for c in range(80) if c not in set(ROUTE_CONST.tolist())])
HALF_LOG_2PI = 0.5 * np.log(2.0 * np.pi)


def arm_const_expect(mode: np.ndarray | int) -> np.ndarray:
    """[n, 20] expected values of the arm observation's constant columns for policy mode(s) ``mode``."""
    mode = np.broadcast_to(np.asarray(mode), np.shape(mode) or (1,))
    want = np.zeros((mode.size, ARM_CONST.size), dtype=np.float32)
    want[np.arange(mode.size), np.asarray(mode, dtype=np.int64)] = 1.0        # column 20 + mode
    want[:, list(ARM_CONST).index(47)] = 1.0
    return want


def route_const_expect(n: int) -> np.ndarray:
    want = np.zeros((n, ROUTE_CONST.size), dtype=np.float32)
    for c in ROUTE_ONES:
        want[:, list(ROUTE_CONST).index(c)] = 1.0
    return want


# ---- references ------------------------------------------------------------------------------------------------------------
def bf16(x) -> np.ndarray:
    """fp32 -> nearest-even bf16, returned as fp32 (cvt.rn.bf16x2.f32 on finite inputs)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def _np_params(pol) -> dict[str, np.ndarray]:
    return {k: v.detach().cpu().numpy().astype(np.float32) for k, v in pol.tensors.items()}


def mlp_fp64(p: dict[str, np.ndarray], x: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """SB3 MultiInputPolicy forward in fp64: actor mean [n, 7], critic value [n]."""
    x = np.asarray(x, np.float64)
    f = lambda k: p[k].astype(np.float64)  # noqa: E731
    ha = np.tanh(np.tanh(x @ f("pi_w0").T + f("pi_b0")) @ f("pi_w1").T + f("pi_b1"))
    hc = np.tanh(np.tanh(x @ f("vf_w0").T + f("vf_b0")) @ f("vf_w1").T + f("vf_b1"))
    return ha @ f("act_w").T + f("act_b"), (hc @ f("val_w").T + f("val_b"))[:, 0]


def mlp_bf16_emulated(p: dict[str, np.ndarray], x: np.ndarray, *, fold_route: bool = False) -> tuple[np.ndarray, np.ndarray]:
    """The tensor-core kernels' operand contract (kin_collect.cu::policy_forward_tc and its weight staging, kin_route_collect.cu,
    kin_ppo_tc.cu, kin_ppo.cu::kin_ppo_pack_weights_kernel), products and sums in fp64:
      layer 1  bf16(x) . bf16(W0)^T + bf16(b0)   -- the bias rides on a constant-one column, so it is a bf16 operand too;
               fold_route: x and W0 restricted to the 60 live route columns, bias = bf16(fp32(fp32(b0 + W0[:, 20]) + W0[:, 71])),
               the left-to-right order both the packed image and K3-TC's in-kernel staging use
      layer 2  bf16(tanh(z1)) . bf16(W1)^T + b1   (b1 fp32, added to the accumulator)
      output   bf16(tanh(z2)) . bf16(W_out)^T + b_out (fp32)."""
    x = np.asarray(x, np.float32)
    hs = []
    for net in ("pi", "vf"):
        w0, b0 = p[f"{net}_w0"], p[f"{net}_b0"]
        if fold_route:
            bias = (b0 + w0[:, ROUTE_ONES[0]]).astype(np.float32)
            bias = (bias + w0[:, ROUTE_ONES[1]]).astype(np.float32)
            xs, ws = x[:, ROUTE_LIVE], w0[:, ROUTE_LIVE]
        else:
            bias, xs, ws = b0, x, w0
        z1 = bf16(xs).astype(np.float64) @ bf16(ws).astype(np.float64).T + bf16(bias).astype(np.float64)
        h1 = bf16(np.tanh(z1).astype(np.float32)).astype(np.float64)
        z2 = h1 @ bf16(p[f"{net}_w1"]).astype(np.float64).T + p[f"{net}_b1"].astype(np.float64)
        hs.append(bf16(np.tanh(z2).astype(np.float32)).astype(np.float64))
    mean = hs[0] @ bf16(p["act_w"]).astype(np.float64).T + p["act_b"].astype(np.float64)
    value = (hs[1] @ bf16(p["val_w"]).astype(np.float64).T + p["val_b"].astype(np.float64))[:, 0]
    return mean, value


def gauss_logp(act: np.ndarray, mean: np.ndarray, log_std: np.ndarray) -> np.ndarray:
    z = (np.asarray(act, np.float64) - mean) / np.exp(log_std.astype(np.float64))
    return (-0.5 * z * z - log_std - HALF_LOG_2PI).sum(-1)


def act_units(err: np.ndarray, w: np.ndarray) -> np.ndarray:
    """Output error [n, d] over the row sums |W_out[d, :]|: the error in units of 'every activation moved by 1'."""
    return np.abs(err) / np.abs(w).sum(1)


class Bounds:
    """Collects (name, measured, bound) so a failure reports every margin of the case, not only the first one."""

    def __init__(self, case: str) -> None:
        self.case, self.rows = case, []

    def check(self, name: str, measured: float, bound: float) -> None:
        for i, (n, m, bd) in enumerate(self.rows):
            if n == name:
                self.rows[i] = (n, max(m, float(measured)), bd)
                return
        self.rows.append((name, float(measured), float(bound)))

    def assert_all(self) -> None:
        bad = [r for r in self.rows if not r[1] <= r[2]]
        report = "\n".join(f"  {n:28s} {m:.3e} (bound {b:.1e})" for n, m, b in self.rows)
        print(f"[{self.case}]\n{report}")
        assert not bad, f"{self.case}: {bad}\n{report}"


# tight bounds (against the emulation) and loose bounds (against fp64), activation units; measured maxima on a B200 in comments
TIGHT_MEAN, LOOSE_MEAN = 1.5e-3, 8e-3       # measured 6.4e-4 (K4, saturating policy), 2.9e-3
TIGHT_VALUE, LOOSE_VALUE = 1.5e-3, 8e-3     # measured 5.9e-4 (K4, approach_stage8_11), 3.0e-3
# |mean over rows of (kernel - emulation)| per output: tanh.approx moves activations both ways, a wrong operand moves them one way;
# measured 8.2e-7 (route last value, 384 rows)
TIGHT_BIAS = 1e-5
TIGHT_QUADRANT = 5e-5             # mean |error| of the actor over one 32-row TMEM lane quadrant of one tile; measured 7.5e-6
LOGP_NOISE = 1e-5                 # log-prob from the recovered noise (fp32 sum of seven terms of O(1)); measured 4.0e-6
TIGHT_LOGP, LOOSE_LOGP = 5e-4, 3e-3         # K3-TC log-prob, first-order activation units; measured 1.7e-4, 9.5e-4


def _policy_act(pol, obs: torch.Tensor, seed: int, step: int, deterministic: int):
    from rl_brain_trainer_b200 import _lib

    n = obs.shape[0]
    act, logp, val = torch.zeros((n, 7), device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    _lib.check(_lib.lib().kin_policy_act(ctypes.byref(pol.c), obs.contiguous().data_ptr(), act.data_ptr(), logp.data_ptr(), val.data_ptr(), n, seed,
                                         step, deterministic, torch.cuda.current_stream().cuda_stream))
    return act, logp


def _check_rows(b: Bounds, tag: str, p, obs_np, mean_k, value_k, *, fold_route=False, obs_fp64=None):
    """Per-row actor mean (optional) and value against the emulation (tight) and fp64 (loose)."""
    mean_e, value_e = mlp_bf16_emulated(p, obs_np, fold_route=fold_route)
    mean_r, value_r = mlp_fp64(p, obs_np if obs_fp64 is None else obs_fp64)
    if mean_k is not None:
        e = mean_k - mean_e
        b.check(f"{tag} mean tight", act_units(e, p["act_w"]).max(), TIGHT_MEAN)
        b.check(f"{tag} mean row bias", (np.abs(e.mean(0)) / np.abs(p["act_w"]).sum(1)).max(), TIGHT_BIAS)
        b.check(f"{tag} mean loose", act_units(mean_k - mean_r, p["act_w"]).max(), LOOSE_MEAN)
    if value_k is not None:
        wv = np.abs(p["val_w"]).sum()
        b.check(f"{tag} value tight", np.abs(value_k - value_e).max() / wv, TIGHT_VALUE)
        b.check(f"{tag} value row bias", abs((value_k - value_e).mean()) / wv, TIGHT_BIAS)
        b.check(f"{tag} value loose", np.abs(value_k - value_r).max() / wv, LOOSE_VALUE)


# ---- K4: kin_ppo_collect ---------------------------------------------------------------------------------------------------
def _collect(tr, T: int, wimg: bool) -> dict[str, torch.Tensor]:
    """One kin_ppo_collect launch of T steps on the trainer's env, into fresh buffers (the trainer's own state is advanced)."""
    from rl_brain_trainer_b200 import _lib

    n, env = tr.N, tr.env
    f32 = dict(dtype=torch.float32, device="cuda")
    limit = max(int(tr.cfg.termination_config.max_episode_steps or tr.cfg.episode_length), 1)
    cap = n * (T // limit + 2)
    out = dict(img=torch.zeros((T, n // 128, 16384), dtype=torch.uint8, device="cuda"), act=torch.zeros((T, n, 7), **f32), logp=torch.zeros((T, n), **f32),
               val=torch.zeros((T, n), **f32), rew=torch.zeros((T, n), **f32), done=torch.zeros((T, n), dtype=torch.uint8, device="cuda"),
               start=torch.zeros((T, n), dtype=torch.uint8, device="cuda"), last=torch.zeros(n, **f32))
    boot_count, boot_index, boot_obs = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(cap, dtype=torch.int32, device="cuda"), torch.zeros((cap, 56), **f32)
    _lib.check(tr._L.kin_ppo_collect(env._params.handle, env.state.data_ptr(), env.stride, n, env._mode_all, tr.params.data_ptr(),
                                     tr.weight_image.data_ptr() if wimg else None, 56, T, tr.seed, 0, env._seed, out["img"].data_ptr(),
                                     out["act"].data_ptr(), out["logp"].data_ptr(), out["val"].data_ptr(), out["rew"].data_ptr(), out["done"].data_ptr(),
                                     out["start"].data_ptr(), tr._next_start.data_ptr(), out["last"].data_ptr(), boot_count.data_ptr(),
                                     boot_index.data_ptr(), boot_obs.data_ptr(), cap, int(tr.tiles_per_cta), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return out


def _k4_trainer(kind: str, num_envs: int, tiles: int, T: int):
    from rl_brain_trainer_b200 import ppo
    from rl_brain_trainer_b200.policy import PolicyWeights

    cfg = env_config("finisher_noop_ft" if kind == "finisher_dock" else "approach_dynamic_scale_big")
    cfg = dataclasses.replace(cfg, episode_length=12, termination_config=dataclasses.replace(cfg.termination_config, max_episode_steps=12))
    handoff_rows, stage = None, 3
    if kind == "random":
        pol = ppo.random_policy(56, seed=2, log_std_init=-1.5, device="cuda")
        pol.tensors["act_w"].mul_(40.0)
        pol.tensors["pi_b0"].normal_(0, 0.3)
        pol.tensors["vf_b1"].normal_(0, 0.2)
    elif kind == "saturating":      # |z| of several units: most activations sit on tanh's flat tails, the bias column is large
        pol = ppo.random_policy(56, seed=5, log_std_init=-1.0, device="cuda")
        for net in ("pi", "vf"):
            pol.tensors[f"{net}_w0"].mul_(4.0)
            pol.tensors[f"{net}_b0"].normal_(0, 1.5)
            pol.tensors[f"{net}_w1"].mul_(3.0)
            pol.tensors[f"{net}_b1"].normal_(0, 1.0)
        pol.tensors["act_w"].mul_(100.0)
    elif kind == "stage8_11":
        pol, stage = PolicyWeights.preset("approach_stage8_11", "cuda"), 0
    else:
        from rl_brain_trainer_b200 import handoff
        from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

        acfg = env_config("approach_dynamic_scale_big")
        buf, _ = handoff.build_finisher_handoff_state_buffer(acfg, PolicyWeights.preset("approach_stage8_11", "cuda"), stage_index=5,
                                                             suite=build_curriculum_local_eval_suite(acfg, seed=3, stage_index=5, n_episodes=128))
        handoff_rows = buf.device_rows("cuda")
        pol, stage = PolicyWeights.preset("finisher", "cuda"), 5
    hp = ppo.PPOHyper(n_steps=T, batch_size=num_envs * T // 2, n_epochs=1, learning_rate=0.0)
    tr = ppo.PPOTrainer(cfg, pol, num_envs=num_envs, hyper=hp, seed=11, stage_index=stage, update_variant="tc", collect_variant="fused",
                        handoff_states=handoff_rows)
    tr.tiles_per_cta = tiles
    tr.env._ensure_sampler()
    return tr, pol


# (policy, envs, tiles per CTA, prebuilt weight image): 384 / 640 envs leave the last CTA partial (1 of 2, 1 of 4 tiles live)
K4_CASES = [("random", 256, 1, True), ("random", 384, 2, False), ("saturating", 384, 2, True), ("saturating", 640, 4, False),
            ("stage8_11", 640, 4, True), ("stage8_11", 256, 1, False), ("finisher_dock", 256, 2, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,num_envs,tiles,wimg", K4_CASES, ids=[f"{k}-{n}-t{t}-{'img' if w else 'noimg'}" for k, n, t, w in K4_CASES])
def test_k4_collect_forward_rows(kind, num_envs, tiles, wimg):
    from rl_brain_trainer_b200 import _lib, ppo

    T = 14            # > the 12-step episode limit: auto-reset rows are in the batch
    tr, pol = _k4_trainer(kind, num_envs, tiles, T)
    mode = int(tr.env._mode_all)
    assert mode == (1 if kind == "finisher_dock" else 0)
    p = _np_params(pol)
    n = num_envs
    state0, start0 = tr.env.state.clone(), tr._next_start.clone()
    run = _collect(tr, T, wimg)
    # the same launch one step longer from the same state: last_value of the T-step run is the value of step T of this one
    tr.env.state.copy_(state0)
    tr._next_start.copy_(start0)
    longer = _collect(tr, T + 1, wimg)
    for k in ("img", "act", "logp", "val", "rew", "done", "start"):
        assert torch.equal(run[k], longer[k][:T]), k
    assert torch.equal(run["last"], longer["val"][T])
    assert int(((run["done"] & 3) != 0).sum()) > 0

    obs_rows = ppo.decode_obs_images(longer["img"]).reshape(T + 1, n, 64)
    b = Bounds(f"K4 {kind} n={n} tiles={tiles} wimg={wimg}")
    # fold contract of the images: bias carrier and padding, and the 20 constant observation columns
    assert bool((obs_rows[..., 56] == 1.0).all()) and bool((obs_rows[..., 57:] == 0.0).all())
    const = obs_rows[..., ARM_CONST].reshape(-1, ARM_CONST.size).cpu().numpy()
    assert np.array_equal(const, np.broadcast_to(arm_const_expect(mode), const.shape))
    sigma = np.exp(p["log_std"].astype(np.float64))
    means, values, obs_all = [], [], []
    for t in range(T + 1):
        obs_t = obs_rows[t, :, :56].contiguous()
        a_fp32, lp_fp32 = _policy_act(pol, obs_t, tr.seed, t, 0)
        m_fp32, _ = _policy_act(pol, obs_t, tr.seed, t, 1)
        noise = (a_fp32 - m_fp32).double().cpu().numpy()
        a_k = longer["act"][t].double().cpu().numpy()
        means.append(a_k - noise)
        values.append(longer["val"][t].double().cpu().numpy())
        obs_all.append(obs_t.cpu().numpy())
        # log-prob of the sample under the kernel's own mean: log N(eps) from the recovered noise, and what the fp32 kernel wrote
        eps = noise / sigma
        lp_ref = (-0.5 * eps * eps - p["log_std"] - HALF_LOG_2PI).sum(-1)
        lp_k = longer["logp"][t].double().cpu().numpy()
        b.check("logp vs recovered noise", np.abs(lp_k - lp_ref).max(), LOGP_NOISE)
        b.check("logp vs kin_policy_act", np.abs(lp_k - lp_fp32.double().cpu().numpy()).max(), LOGP_NOISE)
    obs_np = np.concatenate(obs_all)
    _check_rows(b, "rows", p, obs_np, np.concatenate(means), np.concatenate(values))
    # per 32-row TMEM lane quadrant and per tile of a CTA: a bias confined to some rows must not hide in the maximum over all
    mean_e, _ = mlp_bf16_emulated(p, obs_np)
    err = act_units(np.concatenate(means) - mean_e, p["act_w"]).reshape(T + 1, n // 128, 4, 32, 7)
    b.check("worst quadrant mean |err|", err.mean(axis=(0, 3, 4)).max(), TIGHT_QUADRANT)

    # K3-TC forward-only on the rollout's own images: the log-probs the first update epoch recomputes
    tiles_ids = torch.arange(T * n // 64, dtype=torch.int32, device="cuda")
    lp3, v3 = torch.full((T * n,), 123.0, device="cuda"), torch.full((T * n,), 123.0, device="cuda")
    hp = ppo.PPOHyper().c()
    _lib.check(tr._L.kin_ppo_grad_tc(tr.params.data_ptr(), 56, ctypes.byref(hp), run["img"].data_ptr(), run["act"].data_ptr(), None, None, None, None,
                                     tiles_ids.data_ptr(), int(tiles_ids.numel()), 0, None, 148, None, None, lp3.data_ptr(), v3.data_ptr(), 1, 1, None,
                                     tr.weight_image.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    b.check("K3 value == K4 value", float((v3 - run["val"].reshape(-1)).abs().max()), 0.0)
    b.check("K3 logp vs K4 logp", float((lp3 - run["logp"].reshape(-1)).abs().max()), K3_K4_LOGP)
    b.assert_all()


# K3-TC recomputes z = (a - mean) / sigma from the stored action, K4 had eps itself: the sample's rounding to fp32 remains.
# Measured 2.9e-6; the value (no sample involved) is bitwise K4's.
K3_K4_LOGP = 1e-5


# ---- K3-TC forward-only ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("in_dim,is_img", [(56, 0), (56, 1), (80, 1)], ids=["56raw", "56img", "80folded"])
def test_k3_forward_only_rows(in_dim, is_img):
    from rl_brain_trainer_b200 import _lib, ppo

    pol = ppo.random_policy(in_dim, seed=7, log_std_init=-1.2, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(3)
    pol.tensors["act_w"].mul_(40.0)
    pol.tensors["pi_b0"].normal_(0, 0.5, generator=g)
    pol.tensors["vf_b0"].normal_(0, 0.5, generator=g)
    pol.tensors["vf_b1"].normal_(0, 0.3, generator=g)
    pol.tensors["val_b"].fill_(0.7)
    flat = ppo.flatten_policy_(pol)
    p = _np_params(pol)
    S = 128 * 40
    obs = (torch.rand((S, in_dim), device="cuda", generator=g) * 2.4 - 1.2).contiguous()      # beyond the clip range: bf16 of |x| > 1
    if in_dim == 80:
        obs[:, ROUTE_CONST] = 0.0
        obs[:, list(ROUTE_ONES)] = 1.0
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    kobs = obs
    if is_img and in_dim == 56:
        kobs = ppo.encode_obs_images(obs)
    elif is_img:
        kobs = torch.zeros((S // 128, 16384), dtype=torch.uint8, device="cuda")
        _lib.check(L.kin_route_obs_images(obs.data_ptr(), S, kobs.data_ptr(), stream))
    wimg = torch.zeros(36864, dtype=torch.uint8, device="cuda")
    _lib.check(L.kin_ppo_pack_weights(flat.data_ptr(), in_dim, wimg.data_ptr(), stream))
    obs_np = obs.cpu().numpy()
    mean_e, _ = mlp_bf16_emulated(p, obs_np, fold_route=in_dim == 80)
    sigma = np.exp(p["log_std"].astype(np.float64))
    act = torch.as_tensor((mean_e + sigma * np.random.default_rng(4).standard_normal((S, 7))).astype(np.float32), device="cuda").contiguous()
    act_np = act.double().cpu().numpy()
    hp = ppo.PPOHyper().c()
    perm = torch.randperm(S // 128, generator=torch.Generator().manual_seed(1))[:31]      # 31 of 40 images, out of order
    tile_ids = torch.stack((2 * perm, 2 * perm + 1), 1).reshape(-1).to(torch.int32).cuda()
    idx = (tile_ids.long()[:, None] * 64 + torch.arange(64, device="cuda")[None]).reshape(-1).cpu().numpy()
    b = Bounds(f"K3-TC forward in_dim={in_dim} img={is_img}")
    ref = None
    for ctas in (5, 31, 148):                  # below, equal to and above the number of 128-sample GEMM tiles
        for use_wimg in (False, True):
            lp, v = torch.full((S,), 123.0, device="cuda"), torch.full((S,), 123.0, device="cuda")
            _lib.check(L.kin_ppo_grad_tc(flat.data_ptr(), in_dim, ctypes.byref(hp), kobs.data_ptr(), act.data_ptr(), None, None, None, None,
                                         tile_ids.data_ptr(), int(tile_ids.numel()), 0, None, ctas, None, None, lp.data_ptr(), v.data_ptr(), 1, is_img,
                                         None, wimg.data_ptr() if use_wimg else None, stream))
            torch.cuda.synchronize()
            untouched = np.ones(S, dtype=bool)
            untouched[idx] = False
            assert bool((lp.cpu().numpy()[untouched] == 123.0).all()) and bool((v.cpu().numpy()[untouched] == 123.0).all())
            if ref is None:
                ref = (lp.clone(), v.clone())
                lp_k, v_k = lp.double().cpu().numpy()[idx], v.double().cpu().numpy()[idx]
                _check_rows(b, "rows", p, obs_np[idx], None, v_k, fold_route=in_dim == 80)
                mean_r, _ = mlp_fp64(p, obs_np[idx])
                # log-prob error over |z| / sigma-weighted head rows: the mean's error in activation units, to first order
                scale = (np.abs(act_np[idx] - mean_e[idx]) / sigma ** 2 * np.abs(p["act_w"]).sum(1)).sum(1) + 1e-3
                b.check("logp tight", (np.abs(lp_k - gauss_logp(act_np[idx], mean_e[idx], p["log_std"])) / scale).max(), TIGHT_LOGP)
                b.check("logp loose", (np.abs(lp_k - gauss_logp(act_np[idx], mean_r, p["log_std"])) / scale).max(), LOOSE_LOGP)
            else:       # every grid and both weight paths: bitwise the same rows
                assert torch.equal(lp, ref[0]) and torch.equal(v, ref[1]), (ctas, use_wimg)
    b.assert_all()


# ---- K4-route: kin_route_collect -------------------------------------------------------------------------------------------
def _route_setup(sequence: bool, num_envs: int, T: int):
    from rl_brain_trainer_b200 import config as kcfg, ppo
    from rl_brain_trainer_b200.route import synthetic_route

    route = synthetic_route(160, seed=7)
    renv, seq = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    pol = ppo.random_policy(80, seed=3, log_std_init=-1.0, device="cuda")
    pol.tensors["act_w"].mul_(40.0)
    pol.tensors["pi_b0"].normal_(0, 0.3)
    pol.tensors["vf_b1"].normal_(0, 0.2)
    hp = ppo.PPOHyper(n_steps=T, batch_size=num_envs * T // 2, n_epochs=1, learning_rate=0.0)
    tr = ppo.PPOTrainer(renv, pol, num_envs=num_envs, hyper=hp, seed=5, route=route, route_sequence_config=seq if sequence else None)
    return tr, pol, route, renv, seq


@pytest.mark.gpu
@pytest.mark.parametrize("sequence", [False, True], ids=["route", "sequence"])
def test_route_collect_forward_rows(sequence):
    T, n = 12, 384
    tr, pol, *_ = _route_setup(sequence, n, T)
    assert tr.collect_variant == "fused"
    tr.collect()
    torch.cuda.synchronize()
    p = _np_params(pol)
    b = Bounds(f"K4-route sequence={sequence}")
    obs_all = tr.obs_buf.cpu().numpy()                     # [T + 1, n, 80] fp32: the kernel's observations
    const = obs_all[..., ROUTE_CONST].reshape(-1, ROUTE_CONST.size)
    assert np.array_equal(const, np.broadcast_to(route_const_expect(1), const.shape))
    means = []
    for t in range(T):
        obs_t = tr.obs_buf[t].contiguous()
        a_fp32, _ = _policy_act(pol, obs_t, tr.seed, t, 0)
        m_fp32, _ = _policy_act(pol, obs_t, tr.seed, t, 1)
        means.append(tr.act_buf[t].double().cpu().numpy() - (a_fp32 - m_fp32).double().cpu().numpy())
        eps = (a_fp32 - m_fp32).double().cpu().numpy() / np.exp(p["log_std"].astype(np.float64))
        lp_ref = (-0.5 * eps * eps - p["log_std"] - HALF_LOG_2PI).sum(-1)
        b.check("logp vs recovered noise", np.abs(tr.logp_buf[t].double().cpu().numpy() - lp_ref).max(), LOGP_NOISE)
    _check_rows(b, "rows", p, obs_all[:T].reshape(-1, 80), np.concatenate(means), tr.val_buf.double().cpu().numpy().reshape(-1))
    _check_rows(b, "last value", p, obs_all[T], None, tr.last_val.double().cpu().numpy())
    b.assert_all()


# ---- fold contract ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("preset,mode_name", [("approach_dynamic_scale_big", "approach"), ("finisher_noop_ft", "dock")])
def test_arm_step_observations_hold_the_folded_constants(preset, mode_name):
    from rl_brain_trainer_b200.env import MODE_INDEX, BatchedArmKinematicEnv

    cfg = env_config(preset)
    cfg = dataclasses.replace(cfg, episode_length=6, termination_config=dataclasses.replace(cfg.termination_config, max_episode_steps=6))
    n = 512
    env = BatchedArmKinematicEnv(cfg, n, "cuda", auto_reset=True, seed=3, host_sampler=False, with_aux=False)
    env._ensure_sampler()
    env.reset()
    env.set_policy_mode(mode_name)
    want = arm_const_expect(MODE_INDEX[mode_name])
    g = torch.Generator(device="cuda").manual_seed(2)
    seen_reset = False
    for _ in range(14):
        env.step_raw((torch.randn((n, 7), device="cuda", generator=g) * 1.5).contiguous())
        torch.cuda.synchronize()
        fin = ((env.done & 3) != 0).cpu().numpy()           # terminal_obs holds the rows that finished this step
        for name, o, rows in (("obs", env.obs, slice(None)), ("terminal_obs", env.terminal_obs, fin), ("observe", env.current_observation(), slice(None))):
            c = o[:, ARM_CONST].cpu().numpy()[rows]
            assert np.array_equal(c, np.broadcast_to(want, c.shape)), name
        seen_reset |= bool(fin.any())
    assert seen_reset


@pytest.mark.gpu
@pytest.mark.parametrize("sequence", [False, True], ids=["route", "sequence"])
def test_route_step_observations_hold_the_folded_constants(sequence):
    from rl_brain_trainer_b200.route import BatchedRouteKinematicEnv

    T, n = 4, 256
    _, _, route, renv, seq = _route_setup(sequence, 128, 2)
    g = torch.Generator(device="cuda").manual_seed(4)
    for auto in (False, True):
        env = BatchedRouteKinematicEnv(route, renv, n, "cuda", sequence_config=seq if sequence else None, auto_reset=auto, seed=9)
        env.reset(seed=9)
        for _ in range(3 * T):
            obs, *_ = env.step(torch.randn((n, 7), device="cuda", generator=g) * 1.5)
            fin = ((env.done & 3) != 0).cpu().numpy()
            outs = [(obs, slice(None))] + ([(env.terminal_obs, fin)] if auto else [])
            for o, rows in outs:
                c = o[:, ROUTE_CONST].cpu().numpy()[rows]
                assert np.array_equal(c, np.broadcast_to(route_const_expect(1), c.shape)), auto
        env.close()


def test_golden_traces_hold_the_folded_constants():
    """The reference's own observations: what the fold assumes is what the reference env produces."""
    for name in ("trace_approach.npz", "trace_dock.npz"):
        gz = golden(name)
        obs = np.concatenate([gz["obs"], gz["reset_obs"]])
        modes = np.unique(gz["reset_mode"])
        assert modes.size == 1, name
        c = obs[:, ARM_CONST].astype(np.float32)
        assert np.array_equal(c, np.broadcast_to(arm_const_expect(int(modes[0])), c.shape)), name
    gz = golden("trace_route.npz")
    for key in ("seq_obs", "seq_reset_obs", "adv_obs", "adv_reset_obs"):
        c = gz[key][:, ROUTE_CONST].astype(np.float32)
        assert np.array_equal(c, np.broadcast_to(route_const_expect(1), c.shape)), key


def test_emulation_helpers():
    """The reference's own arithmetic: bf16 rounding is nearest-even, the emulation with fp64 rounding hooks is the fp64 MLP."""
    x = np.array([1.0, 1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -1.0 - 2 ** -9, 3.0e-39, 65504.0], dtype=np.float32)
    want = torch.tensor(x).bfloat16().float().numpy()
    assert np.array_equal(bf16(x), want)
    rng = np.random.default_rng(0)
    p = {"pi_w0": rng.normal(0, 0.3, (64, 80)), "pi_b0": rng.normal(0, 0.3, 64), "pi_w1": rng.normal(0, 0.2, (64, 64)), "pi_b1": rng.normal(0, 0.1, 64),
         "act_w": rng.normal(0, 0.3, (7, 64)), "act_b": rng.normal(0, 0.1, 7), "vf_w0": rng.normal(0, 0.3, (64, 80)), "vf_b0": rng.normal(0, 0.3, 64),
         "vf_w1": rng.normal(0, 0.2, (64, 64)), "vf_b1": rng.normal(0, 0.1, 64), "val_w": rng.normal(0, 0.3, (1, 64)), "val_b": rng.normal(0, 0.1, 1)}
    p = {k: bf16(v.astype(np.float32)) for k, v in p.items()}            # operands already on the bf16 grid
    obs = bf16(rng.uniform(-1, 1, (256, 80)).astype(np.float32))
    obs[:, ROUTE_CONST] = 0.0
    obs[:, list(ROUTE_ONES)] = 1.0
    m_e, v_e = mlp_bf16_emulated(p, obs)
    m_r, v_r = mlp_fp64(p, obs)
    # only the activations' bf16 rounding separates them (<= 2^-9 relative per activation)
    assert act_units(m_e - m_r, p["act_w"]).max() < 2 ** -8 and np.abs(v_e - v_r).max() / np.abs(p["val_w"]).sum() < 2 ** -8
    # folding the constant columns is exact when the folded bias is representable
    m_f, v_f = mlp_bf16_emulated(p, obs, fold_route=True)
    fold_ok = np.array_equal(bf16(p["pi_b0"] + p["pi_w0"][:, 20] + p["pi_w0"][:, 71]), (p["pi_b0"] + p["pi_w0"][:, 20] + p["pi_w0"][:, 71]).astype(np.float32))
    assert act_units(m_f - m_e, p["act_w"]).max() < (1e-12 if fold_ok else 2 ** -6)


# ---- K2-TC: kin_rollout_tc16_kernel through one-step episodes ----------------------------------------------------------------
# The eval kernel writes no per-step outputs.  With episode_length = max_episode_steps = 1, no dynamic action scale and no
# finisher, KIN_RES_FINAL_Q is the joint vector after ONE step, a function of the first action only; the oracle env stepped with
# the emulated action gives the same vector.  Errors are converted back to action units per joint (the q gain of the step).
K2_DYN = np.array(list(range(20)) + list(range(30, 39)) + list(range(40, 47)))     # kin_tc16.cuh::dyn_col, X-image order


def k2_fp16_emulated(p: dict[str, np.ndarray], obs: np.ndarray, mode: int) -> np.ndarray:
    """kin_tc16.cuh::load_weights / obs_pack and kin_rollout_tc16.cu::mlp16: fp16 operands, fp32 accumulation (fp64 here).
      layer 1  fp16(obs[dyn]) . fp16(W0[:, dyn])^T + fp16(fp32((b0 + W0[:, 20 + mode]) + W0[:, 47]))   (bias on X column 36)
      layer 2  fp16(tanh(z1)) . fp16(W1)^T + fp16(b1)       (b1 rides on X column 36 times W0-image column 52)
      output   fp16(tanh(z2)) . fp16(W_out)^T + fp16(b_out) (WOB column 36), clipped to [-1, 1]."""
    h = lambda a: np.asarray(a, np.float32).astype(np.float16).astype(np.float64)  # noqa: E731
    w0 = p["pi_w0"]
    bias = (p["pi_b0"] + w0[:, 20 + mode]).astype(np.float32)
    bias = (bias + w0[:, 47]).astype(np.float32)
    z1 = h(obs[:, K2_DYN]) @ h(w0[:, K2_DYN]).T + h(bias)
    z2 = h(np.tanh(z1)) @ h(p["pi_w1"]).T + h(p["pi_b1"])
    out = h(np.tanh(z2)) @ h(p["act_w"]).T + h(p["act_b"])
    return np.clip(out, -1.0, 1.0)


def k2_fp64(p: dict[str, np.ndarray], obs: np.ndarray) -> np.ndarray:
    return np.clip(_actor_fp64(p, obs), -1.0, 1.0)


def _actor_fp64(p, obs):
    f = lambda k: p[k].astype(np.float64)  # noqa: E731
    return np.tanh(np.tanh(np.asarray(obs, np.float64) @ f("pi_w0").T + f("pi_b0")) @ f("pi_w1").T + f("pi_b1")) @ f("act_w").T + f("act_b")


# tight: against the fp16 emulation; loose: against the fp64 actor.  Action units over sum |act_w| of the joint's row.
K2_TIGHT, K2_LOOSE = 3e-4, 1e-3            # measured 9.7e-5 (n = 200 003), 2.4e-4 (n = 65 536)
K2_STRICT = 2e-6                 # strict K2 (variant 0, fp32 FFMA MLP) against the fp64 actor; measured 3.2e-7


def _one_step_cfg(preset: str):
    cfg = env_config(preset)
    return dataclasses.replace(cfg, episode_length=1, dynamic_action_delta_scale_enabled=False,
                               termination_config=dataclasses.replace(cfg.termination_config, max_episode_steps=1))


def _oracle_final_q(params, mode, suite, rows, actions, q_start=None):
    """q after one oracle step from the suite's reset state (or from q_start with zero dq / prev_action) with the given actions."""
    from oracle import kin_oracle as ko

    env, out = ko.OracleEnv(params), np.zeros((len(rows), 7))
    for j, e in enumerate(rows):
        if q_start is None:
            env.reset(mode=mode, initial_q=suite.initial_q[e], goal_q=suite.goal_q[e],
                      initial_dq=None if suite.initial_dq is None else suite.initial_dq[e],
                      initial_prev_action=None if suite.initial_prev_action is None else suite.initial_prev_action[e])
        else:
            env.reset(mode=mode, initial_q=q_start[j], goal_q=suite.goal_q[e], initial_dq=np.zeros(7), initial_prev_action=np.zeros(7))
        env.step(actions[j])
        out[j] = np.array(env.state.q[:7])
    return out


def _oracle_obs(params, mode, suite, rows, q_start=None):
    from oracle import kin_oracle as ko

    env, out = ko.OracleEnv(params), np.zeros((len(rows), 56), np.float32)
    for j, e in enumerate(rows):
        if q_start is None:
            out[j] = env.reset(mode=mode, initial_q=suite.initial_q[e], goal_q=suite.goal_q[e],
                               initial_dq=None if suite.initial_dq is None else suite.initial_dq[e],
                               initial_prev_action=None if suite.initial_prev_action is None else suite.initial_prev_action[e])
        else:
            out[j] = env.reset(mode=mode, initial_q=q_start[j], goal_q=suite.goal_q[e], initial_dq=np.zeros(7), initial_prev_action=np.zeros(7))
    return out


def _q_gain(params, mode, suite, rows, q_start=None):
    """Per-joint q change of one step per unit of action (the largest over rows: rows pinned at a joint limit move less)."""
    dq = _oracle_final_q(params, mode, suite, rows, np.full((len(rows), 7), 0.5), q_start) - (
        suite.initial_q[rows] if q_start is None else q_start)
    return np.abs(dq).max(0) / 0.5


def _k2_check(b, tag, p, final_q, q_emu, q_ref, gain, tight, loose):
    w = np.abs(p["act_w"]).sum(1)
    b.check(f"{tag} tight", (np.abs(final_q - q_emu) / gain / w).max(), tight)
    b.check(f"{tag} loose", (np.abs(final_q - q_ref) / gain / w).max(), loose)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 129, 65536, 200003])
def test_k2_tc_one_step_action_rows(n):
    """Approach phase, approach mode: fold of column 20 + KIN_MODE_APPROACH and 47; one wave with issuer warps (65 536) and a
    multi-wave batch above 148 x 512 (200 003).  Strict K2 runs the same episodes against fp64 at fp32 level."""
    from oracle import kin_oracle as ko
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.rollout import VARIANT_FFMA, VARIANT_TC, ApproachFinisherRollout
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    cfg = _one_step_cfg("approach_dynamic_scale_big")
    pol = PolicyWeights.preset("approach_stage8_11", "cuda")
    p = _np_params(pol)
    suite = build_curriculum_local_eval_suite(cfg, seed=700001 + 5 * 1009, stage_index=5, n_episodes=n)
    res = {v: ApproachFinisherRollout(cfg, pol, variant=v).evaluate_suite(suite) for v in (VARIANT_TC, VARIANT_FFMA)}
    torch.cuda.synchronize()
    assert bool(((res[VARIANT_TC].raw[5, :n] & 0xffff) == 1).all())          # exactly one approach step per episode
    rng = np.random.default_rng(n)
    rows = np.arange(n) if n <= 4096 else np.unique(np.concatenate([np.arange(256), np.arange(n - 300, n), rng.choice(n, 3000, replace=False)]))
    params = ko.params_from_config(cfg)
    obs = _oracle_obs(params, 0, suite, rows)
    a_emu, a_ref = k2_fp16_emulated(p, obs, 0), k2_fp64(p, obs)
    q_emu, q_ref = _oracle_final_q(params, 0, suite, rows, a_emu), _oracle_final_q(params, 0, suite, rows, a_ref)
    gain = _q_gain(params, 0, suite, rows[:256])
    b = Bounds(f"K2-TC one step n={n}")
    _k2_check(b, "TC", p, res[VARIANT_TC].final_q.double().cpu().numpy()[rows], q_emu, q_ref, gain, K2_TIGHT, K2_LOOSE)
    fq0 = res[VARIANT_FFMA].final_q.double().cpu().numpy()[rows]
    b.check("strict K2 vs fp64", (np.abs(fq0 - q_ref) / gain / np.abs(p["act_w"]).sum(1)).max(), K2_STRICT)
    b.assert_all()


@pytest.mark.gpu
def test_k2_tc_finisher_dock_step_after_the_weight_swap():
    """An all-zero approach policy acts exactly 0; episodes start at their goal, so the approach hands off (kind 2) after one step and
    the finisher runs ONE dock-mode step: pins the fold of column 20 + KIN_MODE_DOCK and the swap to the finisher's weights."""
    from oracle import kin_oracle as ko
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.rollout import VARIANT_TC, ApproachFinisherRollout
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    from ._util import policy_weights

    acfg, fcfg = _one_step_cfg("approach_dynamic_scale_big"), _one_step_cfg("finisher_noop_ft")
    zero = PolicyWeights({k: np.zeros_like(v) for k, v in policy_weights("approach_stage8_11").items()}, "cuda")
    fin = PolicyWeights.preset("finisher", "cuda")
    p = _np_params(fin)
    n = 1000
    src = build_curriculum_local_eval_suite(acfg, seed=700001 + 5 * 1009, stage_index=5, n_episodes=n)
    suite = dataclasses.replace(src, initial_q=src.goal_q.copy(), initial_dq=np.zeros((n, 7)), initial_prev_action=np.zeros((n, 7)))
    res = ApproachFinisherRollout(acfg, zero, fcfg, fin, variant=VARIANT_TC, handoff_confirm_steps=1).evaluate_suite(suite)
    torch.cuda.synchronize()
    kind = (res.flags.cpu().numpy() >> 4) & 3
    steps = res.raw[5, :n].cpu().numpy()
    assert (kind == 2).all(), np.unique(kind, return_counts=True)
    assert ((steps & 0xffff) == 1).all() and ((steps >> 16) == 1).all()
    rows = np.arange(n)
    q0 = suite.initial_q.astype(np.float32).astype(np.float64)
    params = ko.params_from_config(fcfg)
    obs = _oracle_obs(params, 1, suite, rows, q0)
    a_emu, a_ref = k2_fp16_emulated(p, obs, 1), k2_fp64(p, obs)
    q_emu, q_ref = _oracle_final_q(params, 1, suite, rows, a_emu, q0), _oracle_final_q(params, 1, suite, rows, a_ref, q0)
    gain = _q_gain(params, 1, suite, rows[:256], q0[:256])
    b = Bounds("K2-TC finisher dock step")
    _k2_check(b, "finisher", p, res.final_q.double().cpu().numpy(), q_emu, q_ref, gain, K2_TIGHT, K2_LOOSE)
    b.assert_all()


K2_CHILD = r"""
import sys, dataclasses
import numpy as np, torch
from rl_brain_trainer_b200 import config as kcfg
from rl_brain_trainer_b200.policy import PolicyWeights
from rl_brain_trainer_b200.rollout import VARIANT_TC, ApproachFinisherRollout
from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite
cfg = kcfg.load_preset("approach_dynamic_scale_big")
cfg = dataclasses.replace(cfg, episode_length=1, dynamic_action_delta_scale_enabled=False,
                          termination_config=dataclasses.replace(cfg.termination_config, max_episode_steps=1))
ro = ApproachFinisherRollout(cfg, PolicyWeights.preset("approach_stage8_11", "cuda"), variant=VARIANT_TC)
rows = {}
for n in (129, 65536):
    res = ro.evaluate_suite(build_curriculum_local_eval_suite(cfg, seed=700001 + 5 * 1009, stage_index=5, n_episodes=n))
    torch.cuda.synchronize()
    rows[str(n)] = res.final_q.cpu().numpy()
np.savez(sys.argv[1], **rows)
"""


@pytest.mark.gpu
def test_k2_tc_one_step_launch_variants(tmp_path):
    """The one-step action under each launch switch (child processes: the kernel reads them once) is bitwise the default's."""
    import os
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    switches = ("KIN_TC16_SMEM_A", "KIN_TC16_NO_ISSUER_WARPS", "KIN_TC_WARPS", "KIN_TC16_EXACT_SINCOS", "KIN_TC16_POLL_HINT")
    got = {}
    for name, extra in (("default", {}), ("smem_a", {"KIN_TC16_SMEM_A": "1"}), ("no_issuer", {"KIN_TC16_NO_ISSUER_WARPS": "1"}),
                        ("warps8", {"KIN_TC_WARPS": "8"})):
        env = {k: v for k, v in os.environ.items() if k not in switches}
        env.update(extra)
        out = tmp_path / f"{name}.npz"
        r = subprocess.run([sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", K2_CHILD, str(out)], cwd=root, env=env,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, f"{name}:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
        with np.load(out) as z:
            got[name] = {k: z[k] for k in z.files}
    for name in ("smem_a", "no_issuer", "warps8"):
        for k, v in got["default"].items():
            assert np.array_equal(v, got[name][k]), (name, k)
