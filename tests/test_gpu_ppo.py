"""GPU tests of the PPO kernels against a PyTorch autograd restatement of stable-baselines3's formulas (test infrastructure)."""

from __future__ import annotations

import ctypes

import numpy as np
import pytest
import torch

from ._util import env_config

pytestmark = pytest.mark.gpu


def _setup(seed=0, log_std=-0.5, in_dim=56):
    from rl_brain_trainer_b200 import ppo

    pol = ppo.random_policy(in_dim, seed=seed, log_std_init=log_std, device="cuda")
    torch.manual_seed(1000 + seed)      # the in-place normal_() below draw from the global generators: pin the problem instance
    # make the action head non-trivial (SB3's 0.01 gain would hide errors in the actor gradient)
    pol.tensors["act_w"].mul_(30.0)
    pol.tensors["pi_b0"].normal_(0, 0.1)
    pol.tensors["vf_b1"].normal_(0, 0.1)
    flat = ppo.flatten_policy_(pol)
    return ppo, pol, flat


def _torch_forward(pol, obs):
    t = pol.tensors
    lin = torch.nn.functional.linear
    h = torch.tanh(lin(torch.tanh(lin(obs, t["pi_w0"], t["pi_b0"])), t["pi_w1"], t["pi_b1"]))
    mean = lin(h, t["act_w"], t["act_b"])
    hv = torch.tanh(lin(torch.tanh(lin(obs, t["vf_w0"], t["vf_b0"])), t["vf_w1"], t["vf_b1"]))
    value = lin(hv, t["val_w"], t["val_b"])[:, 0]
    return mean, value


def test_policy_act_matches_gaussian_policy():
    from rl_brain_trainer_b200 import _lib

    ppo, pol, _ = _setup()
    n = 5000
    obs = (torch.rand((n, 56), device="cuda") * 2 - 1).contiguous()
    act, logp, val = (torch.zeros((n, 7), device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"))
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    _lib.check(L.kin_policy_act(ctypes.byref(pol.c), obs.data_ptr(), act.data_ptr(), logp.data_ptr(), val.data_ptr(), n, 11, 3, 1, s))
    mean, value = _torch_forward(pol, obs)
    assert torch.allclose(act, mean, atol=3e-6) and torch.allclose(val, value, atol=3e-5)
    _lib.check(L.kin_policy_act(ctypes.byref(pol.c), obs.data_ptr(), act.data_ptr(), logp.data_ptr(), val.data_ptr(), n, 11, 3, 0, s))
    dist = torch.distributions.Normal(mean, pol.tensors["log_std"].exp())
    assert torch.allclose(logp, dist.log_prob(act).sum(-1), atol=2e-4)
    z = ((act - mean) / pol.tensors["log_std"].exp()).cpu().numpy()
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1.0) < 0.02 and abs(np.mean(z ** 3)) < 0.06      # standard normal draws
    act2 = torch.zeros_like(act)
    _lib.check(L.kin_policy_act(ctypes.byref(pol.c), obs.data_ptr(), act2.data_ptr(), logp.data_ptr(), val.data_ptr(), n, 11, 4, 0, s))
    assert not torch.equal(act, act2)                                                                 # new step -> new noise


def test_gae_matches_sb3_restatement():
    from rl_brain_trainer_b200 import _lib, ppo

    rng = np.random.default_rng(0)
    T, n = 37, 192
    rew, val = rng.normal(0, 1, (T, n)).astype(np.float32), rng.normal(0, 1, (T, n)).astype(np.float32)
    starts = (rng.random((T, n)) < 0.1).astype(np.uint8)
    last_val = rng.normal(0, 1, n).astype(np.float32)
    last_done_flag = (rng.random(n) < 0.3)
    last_done = np.where(last_done_flag, 2, 0).astype(np.uint8)   # KIN_DONE_TRUNCATED
    d = lambda a: torch.as_tensor(a).cuda().contiguous()  # noqa: E731
    adv, ret = torch.zeros((T, n), device="cuda"), torch.zeros((T, n), device="cuda")
    sums = torch.zeros((T * n // 64, 2), dtype=torch.float64, device="cuda")
    tr, tv, ts, tl, td = d(rew), d(val), d(starts), d(last_val), d(last_done)
    _lib.check(_lib.lib().kin_ppo_gae(tr.data_ptr(), tv.data_ptr(), ts.data_ptr(), tl.data_ptr(), td.data_ptr(), 0.98, 0.95, T, n, adv.data_ptr(),
                                      ret.data_ptr(), sums.data_ptr(), torch.cuda.current_stream().cuda_stream))
    ra, rr = ppo.numpy_gae(rew, val, starts, last_val, last_done_flag, 0.98, 0.95)
    assert np.abs(adv.cpu().numpy() - ra).max() < 2e-5 and np.abs(ret.cpu().numpy() - rr).max() < 2e-5
    flat = adv.reshape(-1, 64).double()
    assert torch.allclose(sums[:, 0], flat.sum(1), atol=1e-9) and torch.allclose(sums[:, 1], (flat * flat).sum(1), atol=1e-9)


def _torch_ppo_loss(pol, hp, obs, act, old_logp, adv, ret):
    mean, value = _torch_forward(pol, obs)
    dist = torch.distributions.Normal(mean, pol.tensors["log_std"].exp().expand_as(mean))
    logp = dist.log_prob(act).sum(-1)
    entropy = dist.entropy().sum(-1)
    a = (adv - adv.mean()) / (adv.std() + 1e-8) if hp.normalize_advantage else adv
    ratio = torch.exp(logp - old_logp)
    pl = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - hp.clip_range, 1 + hp.clip_range)).mean()
    vl = torch.nn.functional.mse_loss(ret, value)
    loss = pl + hp.ent_coef * (-entropy.mean()) + hp.vf_coef * vl
    with torch.no_grad():
        lr = logp - old_logp
        stats = dict(policy_loss=float(pl), value_loss=float(vl), entropy=float(entropy.mean()), approx_kl=float(((torch.exp(lr) - 1) - lr).mean()),
                     clip_fraction=float(((ratio - 1).abs() > hp.clip_range).float().mean()))
    return loss, stats


def test_minibatch_gradient_matches_autograd():
    from rl_brain_trainer_b200 import _lib

    ppo, pol, flat = _setup(seed=3)
    hp = ppo.PPOHyper(clip_range=0.15, ent_coef=0.01, vf_coef=0.5, normalize_advantage=True)
    S = 64 * 40
    g = torch.Generator(device="cuda").manual_seed(1)
    obs = (torch.rand((S, 56), device="cuda", generator=g) * 2 - 1).contiguous()
    with torch.no_grad():
        mean, value = _torch_forward(pol, obs)
    act = (mean + pol.tensors["log_std"].exp() * torch.randn((S, 7), device="cuda", generator=g)).contiguous()
    old_logp = (torch.distributions.Normal(mean, pol.tensors["log_std"].exp()).log_prob(act).sum(-1)
                + 0.3 * torch.randn(S, device="cuda", generator=g)).contiguous()        # ratios well away from 1: clipping is exercised
    adv = torch.randn(S, device="cuda", generator=g).contiguous()
    ret = (value + torch.randn(S, device="cuda", generator=g)).contiguous()
    sums = torch.stack([adv.reshape(-1, 64).double().sum(1), (adv.reshape(-1, 64).double() ** 2).sum(1)], dim=1).contiguous()
    tile_ids = torch.tensor([3, 17, 0, 39, 8, 21, 22, 5, 30, 11, 12, 1], dtype=torch.int32, device="cuda")
    P = flat.numel()
    ctas = 5
    c_hp = hp.c()

    def launch():
        partials = torch.zeros((ctas, P + 16), device="cuda")
        grad, stats = torch.zeros(P, device="cuda"), torch.zeros(8, device="cuda")
        _lib.check(_lib.lib().kin_ppo_grad(flat.data_ptr(), 56, ctypes.byref(c_hp), obs.data_ptr(), act.data_ptr(), old_logp.data_ptr(), adv.data_ptr(),
                                           ret.data_ptr(), sums.data_ptr(), tile_ids.data_ptr(), tile_ids.numel(), tile_ids.numel() * 64,
                                           partials.data_ptr(), ctas, grad.data_ptr(), stats.data_ptr(), None, torch.cuda.current_stream().cuda_stream))
        return grad, stats

    grad, stats = launch()
    grad2, stats2 = launch()
    assert torch.equal(grad, grad2) and torch.equal(stats, stats2)      # every sum in a fixed order: the kernel is deterministic
    idx = (tile_ids.long()[:, None] * 64 + torch.arange(64, device="cuda")[None]).reshape(-1)
    for t in pol.tensors.values():
        t.requires_grad_(True)
    loss, ref_stats = _torch_ppo_loss(pol, hp, obs[idx], act[idx], old_logp[idx], adv[idx], ret[idx])
    grads = torch.autograd.grad(loss, [pol.tensors[k] for k in ppo.PARAM_ORDER])
    ref = torch.cat([gk.reshape(-1) for gk in grads])
    off = 0
    for k, gk in zip(ppo.PARAM_ORDER, grads):
        n = gk.numel()
        got = grad[off:off + n]
        scale = float(gk.abs().max()) + 1e-12
        assert float((got - gk.reshape(-1)).abs().max()) < 2e-4 * scale + 1e-7, (k, float((got - gk.reshape(-1)).abs().max()), scale)
        off += n
    assert float((grad - ref).norm() / ref.norm()) < 1e-4
    got_stats = stats.cpu().numpy()
    for i, key in enumerate(("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction")):
        assert abs(got_stats[i] - ref_stats[key]) < 2e-4 * max(1.0, abs(ref_stats[key])), key
    assert ref_stats["clip_fraction"] > 0.2
    for t in pol.tensors.values():
        t.requires_grad_(False)


@pytest.mark.parametrize("in_dim", [56, 80])
def test_minibatch_gradient_tc_matches_autograd(in_dim):
    """Tensor-core (bf16 operand, fp32 accumulate) variant of the minibatch gradient vs fp32 autograd: bf16-level agreement per
    tensor, near-perfect direction overall; the forward-only pass reproduces log-prob / value to bf16 accuracy.  in_dim 80 is the
    route policy (two K tiles in layer 1, N = 96 weight-gradient GEMM)."""
    from rl_brain_trainer_b200 import _lib

    ppo, pol, flat = _setup(seed=4, in_dim=in_dim)
    hp = ppo.PPOHyper(clip_range=0.15, ent_coef=0.01, vf_coef=0.5, normalize_advantage=True)
    c_hp = hp.c()
    S = 64 * 48
    g = torch.Generator(device="cuda").manual_seed(2)
    obs = (torch.rand((S, in_dim), device="cuda", generator=g) * 2 - 1).contiguous()
    if in_dim == 80:       # the route observation's constant columns (the kernel folds them into the layer-1 bias)
        const = [c for c in range(80) if c in range(20, 30) or c == 39 or c >= 71]
        obs[:, const] = 0.0
        obs[:, [20, 71]] = 1.0
    with torch.no_grad():
        mean, value = _torch_forward(pol, obs)
    sigma = pol.tensors["log_std"].exp()
    act = (mean + sigma * torch.randn((S, 7), device="cuda", generator=g)).contiguous()
    exact_logp = torch.distributions.Normal(mean, sigma).log_prob(act).sum(-1)
    old_logp = (exact_logp + 0.3 * torch.randn(S, device="cuda", generator=g)).contiguous()
    adv = torch.randn(S, device="cuda", generator=g).contiguous()
    ret = (value + torch.randn(S, device="cuda", generator=g)).contiguous()
    sums = torch.stack([adv.reshape(-1, 64).double().sum(1), (adv.reshape(-1, 64).double() ** 2).sum(1)], dim=1).contiguous()
    tile_ids = torch.tensor([3, 17, 0, 39, 8, 21, 22, 5, 30, 11, 12, 1, 47, 40], dtype=torch.int32, device="cuda")
    kobs, is_img = obs, 0
    if in_dim == 80:       # folded bf16 images, whole images per pair of 64-sample tiles
        tile_ids = torch.tensor([2, 3, 16, 17, 0, 1, 38, 39, 8, 9, 20, 21, 46, 47, 10, 11], dtype=torch.int32, device="cuda")
        kobs, is_img = torch.zeros((S // 128, 16384), dtype=torch.uint8, device="cuda"), 1
        _lib.check(_lib.lib().kin_route_obs_images(obs.data_ptr(), S, kobs.data_ptr(), torch.cuda.current_stream().cuda_stream))
    idx = (tile_ids.long()[:, None] * 64 + torch.arange(64, device="cuda")[None]).reshape(-1)
    P = flat.numel()
    c_hp = hp.c()
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    # forward only: log-prob and value of the visited samples
    lp_out, v_out = torch.full((S,), 123.0, device="cuda"), torch.full((S,), 123.0, device="cuda")
    _lib.check(L.kin_ppo_grad_tc(flat.data_ptr(), in_dim, ctypes.byref(c_hp), kobs.data_ptr(), act.data_ptr(), None, None, None, None,
                                 tile_ids.data_ptr(), tile_ids.numel(), 0, None, 3, None, None, lp_out.data_ptr(), v_out.data_ptr(), 1, is_img, None, None, stream))
    torch.cuda.synchronize()
    assert float((v_out[idx] - value[idx]).abs().max()) < 0.03 and float((lp_out[idx] - exact_logp[idx]).abs().max()) < 0.06
    assert float((lp_out[idx] - exact_logp[idx]).abs().mean()) < 0.008
    untouched = torch.ones(S, dtype=torch.bool, device="cuda")
    untouched[idx] = False
    assert bool((lp_out[untouched] == 123.0).all())
    # (clip_range, per-tensor tolerance, whole-gradient tolerance, cosine): without clipping the only error is bf16 rounding; with the
    # 0.3-sigma ratio noise of this case bf16-level log-prob errors flip the clip state of samples at the boundary (0.2 % of them)
    for clip, tol_k, tol_all, min_cos in ((50.0, 5e-2, 1.2e-2, 0.9999), (0.15, 0.12, 8e-2, 0.998)):
        hp = ppo.PPOHyper(clip_range=clip, ent_coef=0.01, vf_coef=0.5, normalize_advantage=True)
        c_hp = hp.c()
        for t in pol.tensors.values():
            t.requires_grad_(True)
        loss, ref_stats = _torch_ppo_loss(pol, hp, obs[idx], act[idx], old_logp[idx], adv[idx], ret[idx])
        grads = torch.autograd.grad(loss, [pol.tensors[k] for k in ppo.PARAM_ORDER])
        ref = torch.cat([gk.reshape(-1) for gk in grads])
        for t in pol.tensors.values():
            t.requires_grad_(False)
        for ctas in (2, 7, 148):      # several GEMM tiles per CTA (TMEM accumulation across tiles), one per CTA, more CTAs than tiles
            partials = torch.zeros((ctas, P + 16), device="cuda")
            grad, stats = torch.zeros(P, device="cuda"), torch.zeros(8, device="cuda")
            _lib.check(L.kin_ppo_grad_tc(flat.data_ptr(), in_dim, ctypes.byref(c_hp), kobs.data_ptr(), act.data_ptr(), old_logp.data_ptr(), adv.data_ptr(),
                                         ret.data_ptr(), sums.data_ptr(), tile_ids.data_ptr(), tile_ids.numel(), tile_ids.numel() * 64,
                                         partials.data_ptr(), ctas, grad.data_ptr(), stats.data_ptr(), None, None, 0, is_img, None, None, stream))
            torch.cuda.synchronize()
            off = 0
            for k, gk in zip(ppo.PARAM_ORDER, grads):
                n = gk.numel()
                rel = float((grad[off:off + n] - gk.reshape(-1)).norm() / (gk.norm() + 1e-12))
                # bias-like tensors are signed sums of bf16-rounded per-sample terms with heavy cancellation: looser bound
                assert rel < (tol_k if n > 64 else 3 * tol_k), (clip, ctas, k, rel)
                off += n
            cos = float(torch.dot(grad, ref) / (grad.norm() * ref.norm()))
            assert cos > min_cos and float((grad - ref).norm() / ref.norm()) < tol_all, (clip, ctas, cos)
            got_stats = stats.cpu().numpy()
            for i, key in enumerate(("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction")):
                assert abs(got_stats[i] - ref_stats[key]) < 3e-2 * max(1.0, abs(ref_stats[key])), (key, got_stats[i], ref_stats[key])
    # odd tile counts are refused (two 64-sample tiles per GEMM tile)
    rc = L.kin_ppo_grad_tc(flat.data_ptr(), in_dim, ctypes.byref(c_hp), kobs.data_ptr(), act.data_ptr(), old_logp.data_ptr(), adv.data_ptr(),
                           ret.data_ptr(), sums.data_ptr(), tile_ids.data_ptr(), 3, 192, partials.data_ptr(), 2, grad.data_ptr(), stats.data_ptr(),
                           None, None, 0, is_img, None, None, stream)
    assert rc != 0
    if in_dim == 80:       # the route policy without folded images is refused, and its folded weight image gives the same gradient
        rc = L.kin_ppo_grad_tc(flat.data_ptr(), in_dim, ctypes.byref(c_hp), obs.data_ptr(), act.data_ptr(), old_logp.data_ptr(), adv.data_ptr(),
                               ret.data_ptr(), sums.data_ptr(), tile_ids.data_ptr(), 4, 256, partials.data_ptr(), 2, grad.data_ptr(), stats.data_ptr(),
                               None, None, 0, 0, None, None, stream)
        assert rc != 0
        wimg = torch.zeros(36864, dtype=torch.uint8, device="cuda")
        _lib.check(L.kin_ppo_pack_weights(flat.data_ptr(), 80, wimg.data_ptr(), stream))
        g2 = torch.zeros(P, device="cuda")
        _lib.check(L.kin_ppo_grad_tc(flat.data_ptr(), in_dim, ctypes.byref(c_hp), kobs.data_ptr(), act.data_ptr(), old_logp.data_ptr(), adv.data_ptr(),
                                     ret.data_ptr(), sums.data_ptr(), tile_ids.data_ptr(), tile_ids.numel(), tile_ids.numel() * 64,
                                     partials.data_ptr(), 148, g2.data_ptr(), stats.data_ptr(), None, None, 0, 1, None, wimg.data_ptr(), stream))
        torch.cuda.synchronize()
        assert torch.equal(g2, grad)


def test_minibatch_gradient_three_stream_kernel_matches_autograd_and_the_two_chain_kernel():
    """kin_ppo_tc3.cu (three tile streams per SM, dO in the spare X columns, one M = 128 GEMM for dW0 | db0 | db1): same tolerances
    against fp32 autograd as the two-chain kernel, agreement with the two-chain kernel on the same inputs to summation-order level,
    bitwise reproducible, for grids where streams idle (more streams than tiles), where every stream has one tile and several."""
    from rl_brain_trainer_b200 import _lib

    ppo, pol, flat = _setup(seed=4, in_dim=56)
    S = 128 * 512
    g = torch.Generator(device="cuda").manual_seed(5)
    obs = (torch.rand((S, 56), device="cuda", generator=g) * 2 - 1).contiguous()
    with torch.no_grad():
        mean, value = _torch_forward(pol, obs)
    sigma = pol.tensors["log_std"].exp()
    act = (mean + sigma * torch.randn((S, 7), device="cuda", generator=g)).contiguous()
    exact_logp = torch.distributions.Normal(mean, sigma).log_prob(act).sum(-1)
    old_logp = (exact_logp + 0.3 * torch.randn(S, device="cuda", generator=g)).contiguous()
    adv = torch.randn(S, device="cuda", generator=g).contiguous()
    ret = (value + torch.randn(S, device="cuda", generator=g)).contiguous()
    sums = torch.stack([adv.reshape(-1, 64).double().sum(1), (adv.reshape(-1, 64).double() ** 2).sum(1)], dim=1).contiguous()
    images = ppo.encode_obs_images(obs)
    P = flat.numel()
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    wimg = torch.zeros(36864, dtype=torch.uint8, device="cuda")
    _lib.check(L.kin_ppo_pack_weights(flat.data_ptr(), 56, wimg.data_ptr(), stream))
    hp = ppo.PPOHyper(clip_range=50.0, ent_coef=0.01, vf_coef=0.5, normalize_advantage=True)
    c_hp = hp.c()
    perm = torch.randperm(S // 128, generator=torch.Generator().manual_seed(9))

    def run(tile_ids, ctas, enabled, pct=-1):
        L.kin_ppo_tc3_config(enabled, pct)
        partials = torch.full((ctas, P + 16), 7.0, device="cuda")      # stale rows must not leak into the sum
        grad, stats = torch.zeros(P, device="cuda"), torch.zeros(8, device="cuda")
        _lib.check(L.kin_ppo_grad_tc(flat.data_ptr(), 56, ctypes.byref(c_hp), images.data_ptr(), act.data_ptr(), old_logp.data_ptr(), adv.data_ptr(),
                                     ret.data_ptr(), sums.data_ptr(), tile_ids.data_ptr(), tile_ids.numel(), tile_ids.numel() * 64,
                                     partials.data_ptr(), ctas, grad.data_ptr(), stats.data_ptr(), None, None, 0, 1, None, wimg.data_ptr(), stream))
        torch.cuda.synchronize()
        return grad, stats

    try:
        # (pairs, CTAs): streams without a tile; exactly one tile per stream; ragged; the trainer's shape (148 CTAs, several tiles per stream)
        for n_pairs, ctas in ((5, 4), (12, 4), (37, 6), (512, 148)):
            img_ids = perm[:n_pairs].to(torch.int32)
            tile_ids = torch.stack((2 * img_ids, 2 * img_ids + 1), dim=1).reshape(-1).contiguous().cuda()
            idx = (tile_ids.long()[:, None] * 64 + torch.arange(64, device="cuda")[None]).reshape(-1)
            for t in pol.tensors.values():
                t.requires_grad_(True)
            loss, ref_stats = _torch_ppo_loss(pol, hp, obs[idx], act[idx], old_logp[idx], adv[idx], ret[idx])
            grads = torch.autograd.grad(loss, [pol.tensors[k] for k in ppo.PARAM_ORDER])
            ref = torch.cat([gk.reshape(-1) for gk in grads])
            for t in pol.tensors.values():
                t.requires_grad_(False)
            g2, s2 = run(tile_ids, ctas, 0)
            for pct in (52, 30, 75):
                g3, s3 = run(tile_ids, ctas, 1, pct)
                off = 0
                for k, gk in zip(ppo.PARAM_ORDER, grads):
                    n = gk.numel()
                    rel = float((g3[off:off + n] - gk.reshape(-1)).norm() / (gk.norm() + 1e-12))
                    # (a single-element tensor -- val_b -- is a signed sum over all samples with full cancellation: its bf16 noise is
                    # checked against the two-chain kernel below, not against fp32 autograd)
                    assert n == 1 or rel < (5e-2 if n > 64 else 0.15), (n_pairs, ctas, pct, k, rel)
                    # against the two-chain kernel: the same per-element arithmetic, sums in another order
                    rel2 = float((g3[off:off + n] - g2[off:off + n]).norm() / (g2[off:off + n].norm() + 1e-12))
                    assert rel2 < (2e-4 if n > 1 else 5e-3), (n_pairs, ctas, pct, k, rel2)
                    off += n
                cos = float(torch.dot(g3, ref) / (g3.norm() * ref.norm()))
                # (65 536 samples: the bf16 rounding of the activations is a coherent bias, not noise -- the two-chain kernel shows the same
                # 1.4e-2 on this case, see rel2 above -- so the whole-gradient bound is looser than in the 900-sample test)
                assert cos > 0.9999 and float((g3 - ref).norm() / ref.norm()) < 2e-2, (n_pairs, ctas, pct, cos)
                assert float((s3[:5] - s2[:5]).abs().max()) < 1e-4 * max(1.0, float(s2[:5].abs().max())), (s3, s2)
                g3b, s3b = run(tile_ids, ctas, 1, pct)
                assert torch.equal(g3, g3b) and torch.equal(s3, s3b)
    finally:
        L.kin_ppo_tc3_config(0, 52)


def test_adam_matches_torch():
    from rl_brain_trainer_b200 import _lib, ppo

    P = 16143
    g = torch.Generator(device="cuda").manual_seed(5)
    params = torch.randn(P, device="cuda", generator=g)
    ref_p = params.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref_p], lr=3e-4, eps=1e-5)
    m, v, stats = torch.zeros(P, device="cuda"), torch.zeros(P, device="cuda"), torch.zeros(8, device="cuda")
    hp = ppo.PPOHyper(learning_rate=3e-4, max_grad_norm=0.5)
    c_hp = hp.c()
    for step in range(1, 6):
        grad = torch.randn(P, device="cuda", generator=g) * (0.001 if step % 2 else 0.1)   # below and above the clip norm
        ref_p.grad = grad.clone()
        norm = torch.nn.utils.clip_grad_norm_([ref_p], 0.5)
        opt.step()
        _lib.check(_lib.lib().kin_ppo_adam(params.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), P, ctypes.byref(c_hp), step, stats.data_ptr(), None, None, 56,
                                           torch.cuda.current_stream().cuda_stream))
        assert abs(float(stats[5]) - float(norm)) < 1e-4 * float(norm)
        assert float((params - ref_p.detach()).abs().max()) < 2e-6


def test_bootstrap_adds_discounted_terminal_value():
    from rl_brain_trainer_b200 import _lib

    ppo, pol, _ = _setup(seed=2)
    n = 300
    obs = (torch.rand((n, 56), device="cuda") * 2 - 1).contiguous()
    done = torch.zeros(n, dtype=torch.uint8, device="cuda")
    done[5] = 2          # truncated
    done[6] = 3          # terminated and truncated -> no bootstrap
    done[200] = 2
    rew = torch.ones(n, device="cuda")
    _lib.check(_lib.lib().kin_ppo_bootstrap(ctypes.byref(pol.c), obs.data_ptr(), done.data_ptr(), rew.data_ptr(), 0.9, n, torch.cuda.current_stream().cuda_stream))
    _, value = _torch_forward(pol, obs)
    exp = torch.ones(n, device="cuda")
    exp[5] += 0.9 * value[5]
    exp[200] += 0.9 * value[200]
    assert torch.allclose(rew, exp, atol=3e-5)


@pytest.mark.parametrize("variant", ["tc", "fp32"])
def test_trainer_runs_and_improves_value_fit(variant):
    """A short on-device PPO run on the Stage-0 shell: finite statistics, parameters move, the critic's loss falls."""
    from rl_brain_trainer_b200 import ppo

    cfg = env_config("approach_dynamic_scale_big")
    pol = ppo.random_policy(56, seed=1, log_std_init=-1.0, device="cuda")
    hp = ppo.PPOHyper(learning_rate=1e-3, n_steps=32, batch_size=2048, n_epochs=4, gamma=0.98, clip_range=0.2)
    tr = ppo.PPOTrainer(cfg, pol, num_envs=1024, hyper=hp, seed=3, update_variant=variant)
    p0 = tr.params.clone()
    log = tr.learn(4)
    assert all(np.isfinite(list(row.values())).all() for row in log)
    assert float((tr.params - p0).abs().max()) > 1e-4
    assert log[-1]["value_loss"] < log[0]["value_loss"]
    assert log[0]["minibatches"] == 4 * (1024 * 32 // 2048)
    sd = tr.state_dict()
    assert "mlp_extractor.policy_net.0.weight" in sd and sd["log_std"].shape == (7,)
    # the bf16 operand image Adam maintains equals a fresh pack of the final parameters
    kept = tr.weight_image.clone()
    tr.pack_weights()
    assert torch.equal(kept, tr.weight_image) and int(kept.count_nonzero()) > 30000
    # lr = 0 leaves the parameters untouched
    tr2 = ppo.PPOTrainer(cfg, ppo.random_policy(56, seed=1, device="cuda"), num_envs=256, hyper=ppo.PPOHyper(learning_rate=0.0, n_steps=8, batch_size=512, n_epochs=1),
                         update_variant=variant)
    q0 = tr2.params.clone()
    tr2.learn(1)
    assert torch.equal(tr2.params, q0)


def test_fused_update_is_the_three_launch_update():
    """kin_ppo_grad_tc_update (gradient + reduction + exchange + clip + Adam in one launch) against the same update as gradient kernel
    + kin_ppo_adam: same parameters, Adam moments, weight image and statistics (the clip norm is summed in another order: a few ulp)."""
    from rl_brain_trainer_b200 import ppo

    cfg = env_config("approach_dynamic_scale_big")
    out = {}
    for fused in (True, False):
        pol = ppo.random_policy(56, seed=1, log_std_init=-1.0, device="cuda")
        hp = ppo.PPOHyper(learning_rate=1e-3, n_steps=32, batch_size=4096, n_epochs=3, gamma=0.98, clip_range=0.2, max_grad_norm=0.05)
        tr = ppo.PPOTrainer(cfg, pol, num_envs=1024, hyper=hp, seed=3, update_variant="tc", fused_update=fused)
        assert tr.fused_update == fused and (tr.peer is not None) == fused
        tr.collect()
        stats = tr.update()
        torch.cuda.synchronize()
        out[fused] = (tr.params.clone(), tr.adam_m.clone(), tr.adam_v.clone(), tr.weight_image.clone(), stats, tr.update_count)
        kept = tr.weight_image.clone()
        tr.pack_weights()
        assert torch.equal(kept, tr.weight_image)
        tr.close()
    (p1, m1, v1, w1, s1, c1), (p0, m0, v0, w0, s0, c0) = out[True], out[False]
    assert c1 == c0 == 3 * (1024 * 32 // 4096)
    assert s1["grad_norm"] > 0.05                      # the clip is active: the coefficient matters
    assert float((p1 - p0).abs().max()) < 2e-6 and float((m1 - m0).abs().max()) < 1e-6 * float(m0.abs().max()) + 1e-9
    assert float((v1 - v0).abs().max()) < 1e-5 * float(v0.abs().max()) + 1e-12
    assert (w1 != w0).float().mean() < 0.01            # bf16 image: at most a few last-bit differences
    for k in ("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction", "grad_norm"):
        assert abs(s1[k] - s0[k]) < 1e-4 * max(1.0, abs(s0[k])), (k, s1[k], s0[k])
    assert s1["minibatches"] == s0["minibatches"]


def test_per_sample_shuffle_is_sb3_rollout_buffer_get():
    """kin_ppo_shuffle = SB3's RolloutBuffer.get: every array of the rollout permuted by one per-sample permutation (bit-exact, operand
    images included: rows move between swizzle phases), tile sums of the new order; PPOTrainer(shuffle="sample") then runs the gradient
    kernels on consecutive tile ranges of the permuted rollout -- the first minibatch's gradient equals the gradient of exactly the samples
    perm[0 : batch] of the rollout order, computed by the strict fp32 kernel's autograd restatement."""
    from rl_brain_trainer_b200 import _lib, ppo

    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda").manual_seed(11)
    S = 128 * 40
    for in_dim, is_img in ((56, 1), (56, 0), (80, 0)):
        obs = (torch.rand((S, in_dim), device="cuda", generator=g) * 2 - 1).contiguous()
        src = ppo.encode_obs_images(obs) if is_img else obs
        act = torch.randn((S, 7), device="cuda", generator=g)
        logp, adv, ret = (torch.randn(S, device="cuda", generator=g) for _ in range(3))
        perm = torch.randperm(S, device="cuda", generator=g).to(torch.int32)
        o2 = torch.zeros_like(src)
        a2, l2, d2, r2 = torch.zeros_like(act), torch.zeros_like(logp), torch.zeros_like(adv), torch.zeros_like(ret)
        sums = torch.zeros((S // 64, 2), dtype=torch.float64, device="cuda")
        _lib.check(L.kin_ppo_shuffle(src.data_ptr(), is_img, in_dim, act.data_ptr(), logp.data_ptr(), adv.data_ptr(), ret.data_ptr(), perm.data_ptr(), S,
                                     o2.data_ptr(), a2.data_ptr(), l2.data_ptr(), d2.data_ptr(), r2.data_ptr(), sums.data_ptr(), stream))
        torch.cuda.synchronize()
        idx = perm.long()
        assert torch.equal(a2, act[idx]) and torch.equal(l2, logp[idx]) and torch.equal(d2, adv[idx]) and torch.equal(r2, ret[idx])
        if is_img:
            assert torch.equal(o2, ppo.encode_obs_images(obs[idx]))
        else:
            assert torch.equal(o2, obs[idx])
        want = torch.stack([adv[idx].reshape(-1, 64).double().sum(1), (adv[idx].reshape(-1, 64).double() ** 2).sum(1)], dim=1)
        assert torch.allclose(sums, want, rtol=1e-13, atol=1e-13)
    # refusals: in place, ragged size
    assert L.kin_ppo_shuffle(src.data_ptr(), 0, 80, act.data_ptr(), logp.data_ptr(), adv.data_ptr(), ret.data_ptr(), perm.data_ptr(), S, src.data_ptr(),
                             a2.data_ptr(), l2.data_ptr(), d2.data_ptr(), r2.data_ptr(), sums.data_ptr(), stream) != 0
    assert L.kin_ppo_shuffle(src.data_ptr(), 0, 80, act.data_ptr(), logp.data_ptr(), adv.data_ptr(), ret.data_ptr(), perm.data_ptr(), S - 64, o2.data_ptr(),
                             a2.data_ptr(), l2.data_ptr(), d2.data_ptr(), r2.data_ptr(), sums.data_ptr(), stream) != 0
    # the trainer: per-sample minibatches (fp32 kernels, so the comparison with autograd is tight)
    cfg = env_config("approach_dynamic_scale_big")
    for mode in ("sample", "sample_once"):
        pol = ppo.random_policy(56, seed=1, log_std_init=-1.0, device="cuda")
        hp = ppo.PPOHyper(learning_rate=0.0, n_steps=16, batch_size=2048, n_epochs=2, gamma=0.98, clip_range=0.2)
        tr = ppo.PPOTrainer(cfg, pol, num_envs=512, hyper=hp, seed=3, update_variant="fp32", shuffle=mode)
        tr.collect()
        tr.update()
        sh, perm = tr._shadow, tr._sample_perm.long()
        flat_obs = tr.obs_buf[: tr.T].reshape(tr.S, 56)
        assert torch.equal(sh["obs"], flat_obs[perm]) and torch.equal(sh["act"], tr.act_buf.reshape(tr.S, 7)[perm])
        assert torch.equal(sh["adv"], tr.adv_buf.reshape(-1)[perm]) and torch.equal(sh["ret"], tr.ret_buf.reshape(-1)[perm])
        assert sorted(perm.tolist()) == list(range(tr.S))
        # gradient of the first minibatch of the permuted order vs autograd on the samples perm[:2048] of the rollout order
        tr._use_shadow = True
        tr.minibatch_grad(torch.arange(2048 // 64, dtype=torch.int32, device="cuda"))
        tr._use_shadow = False
        torch.cuda.synchronize()
        pick = perm[:2048]
        for t in pol.tensors.values():
            t.requires_grad_(True)
        loss, _ = _torch_ppo_loss(pol, hp, flat_obs[pick], tr.act_buf.reshape(tr.S, 7)[pick], tr.logp_buf.reshape(-1)[pick], tr.adv_buf.reshape(-1)[pick],
                                  tr.ret_buf.reshape(-1)[pick])
        ref = torch.cat([gk.reshape(-1) for gk in torch.autograd.grad(loss, [pol.tensors[k] for k in ppo.PARAM_ORDER])])
        for t in pol.tensors.values():
            t.requires_grad_(False)
        assert float((tr.grad - ref).norm() / ref.norm()) < 1e-4
    # it learns with per-sample minibatches and the tensor-core path too (images are shuffled)
    pol = ppo.random_policy(56, seed=1, log_std_init=-1.0, device="cuda")
    hp = ppo.PPOHyper(learning_rate=1e-3, n_steps=32, batch_size=2048, n_epochs=4, gamma=0.98, clip_range=0.2)
    tr = ppo.PPOTrainer(cfg, pol, num_envs=1024, hyper=hp, seed=3, update_variant="tc", shuffle="sample")
    log = tr.learn(4)
    assert all(np.isfinite(list(row.values())).all() for row in log) and log[-1]["value_loss"] < log[0]["value_loss"]
    assert tr._shadow["obs"].dtype == torch.uint8 and tr._shadow["obs"].shape == (1024 * 32 // 128, 16384)


def test_bf16_and_fp32_update_variants_train_equivalently():
    """The tensor-core (bf16 operand) update is accepted at bf16-level gradient tolerances; this is the check that it TRAINS like the strict
    fp32 update: from one random init and seed, the reference's from-scratch config (approach_default, 6 stages, promotion at a windowed
    success rate of 0.8) through the whole curriculum with either variant -- both reach the last stage in a similar number of rollouts and
    the policies they produce score the same (+- 3 points) on every stage under ONE evaluator (the strict-fp32 fused rollout)."""
    from dataclasses import replace

    from rl_brain_trainer_b200 import gate, ppo
    from rl_brain_trainer_b200.rollout import VARIANT_FFMA

    cfg = env_config("approach_default")
    cfg = replace(cfg, curriculum_config=replace(cfg.curriculum_config, window_episodes=2048, min_episodes_per_stage=2048))
    n_stages = len(cfg.curriculum_config.stages)
    envs, n_steps = 8192, 64
    result = {}
    for variant in ("tc", "fp32"):
        pol = ppo.random_policy(56, seed=0, log_std_init=-0.5, device="cuda")
        hp = ppo.PPOHyper(learning_rate=3e-4, n_steps=n_steps, batch_size=envs * n_steps // 16, n_epochs=8, gamma=0.98, gae_lambda=0.95, clip_range=0.2)
        tr = ppo.PPOTrainer(cfg, pol, num_envs=envs, hyper=hp, seed=1, stage_index=0, update_variant=variant)
        iters, rate = 0, 0.0
        while iters < 120:
            row = tr.learn(1)[0]
            iters += 1
            rate = row["successes"] / max(row["episodes"], 1.0)
            assert np.isfinite(list(row.values())).all()
            if int(row["stage"]) >= n_stages - 1 and rate >= 0.95:
                break
        ev = gate.evaluate_workspace_expansion(cfg, pol, None, None, episodes=1024, seed=720001, stage_indices=list(range(n_stages)), variant=VARIANT_FFMA)
        result[variant] = (iters, int(tr.env.get_curriculum_stage()), rate, [ev["stage_metrics"][s]["success_rate"] for s in range(n_stages)])
    (it_tc, st_tc, rate_tc, ev_tc), (it_f, st_f, rate_f, ev_f) = result["tc"], result["fp32"]
    assert st_tc == st_f == n_stages - 1, result
    assert rate_tc >= 0.95 and rate_f >= 0.95, result
    assert abs(it_tc - it_f) <= 0.4 * max(it_tc, it_f) + 2, result
    assert min(ev_tc) > 0.9 and min(ev_f) > 0.9, result
    assert max(abs(a - b) for a, b in zip(ev_tc, ev_f)) < 0.03, result


def test_route_policy_training_runs_end_to_end():
    """train_route_curriculum.py on the device: the 80-input route policy on the batched RouteSequence env -- rollout with sampled
    route resets, TimeLimit bootstrap, tensor-core update (fp32 route observations), prefix curriculum promotion."""
    from rl_brain_trainer_b200 import config as kcfg, ppo
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.route import RouteCurriculumStage, RoutePrefixCurriculum, evaluate_sequential_route, synthetic_route

    route = synthetic_route(160, seed=7)
    renv, seq = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    # (1) a fresh policy: finite statistics, parameters move, the critic's fit improves
    pol = ppo.random_policy(80, seed=2, log_std_init=-1.0, device="cuda")
    hp = ppo.PPOHyper(learning_rate=1e-3, n_steps=32, batch_size=4096, n_epochs=4, gamma=0.98, clip_range=0.2)
    tr = ppo.PPOTrainer(renv, pol, num_envs=512, hyper=hp, seed=3, route=route, route_sequence_config=seq)
    assert tr.is_route and tr.in_dim == 80 and tr.obs_buf.shape == (33, 512, 80) and tr.obs_img.shape == (32, 4, 16384)
    p0 = tr.params.clone()
    log = tr.learn(4)
    assert all(np.isfinite(list(row.values())).all() for row in log)
    assert float((tr.params - p0).abs().max()) > 1e-4
    assert log[-1]["value_loss"] < log[0]["value_loss"]
    assert log[0]["episodes"] > 0 and log[0]["minibatches"] == 4 * (512 * 32 // 4096)
    assert tr.state_dict()["mlp_extractor.policy_net.0.weight"].shape == (64, 80)
    # (2) the bundled route checkpoint under a two-stage prefix curriculum: it already passes the promotion thresholds on the short
    # prefix, so the window opens; a few updates at the reference's learning rate keep the probe's prefix
    pol = PolicyWeights.preset("route_prefix120", "cuda")
    before = evaluate_sequential_route(route, renv, pol, n_replicas=64, start_index=1, end_index=60, start_q_noise_std=0.0008)
    cur = RoutePrefixCurriculum([RouteCurriculumStage("prefix20", 20), RouteCurriculumStage("prefix60", 60)], promotion_success_rate=0.5,
                                promotion_route_ready_hit_rate=0.5, promotion_orientation_hit_rate=0.5, promotion_max_regression_rate=0.6,
                                window_episodes=128, min_episodes_per_stage=128)
    hp = ppo.PPOHyper(learning_rate=4e-6, n_steps=64, batch_size=8192, n_epochs=2, gamma=0.98, clip_range=0.1)
    tr = ppo.PPOTrainer(renv, pol, num_envs=512, hyper=hp, seed=5, route=route, route_sequence_config=seq, route_curriculum=cur)
    assert tr.env.config.reset_config.max_route_index == 20
    log = tr.learn(3)
    assert cur.current_stage_index == 1 and tr.env.config.reset_config.max_route_index == 60 and cur.history[0]["to_prefix_end_index"] == 60
    assert log[-1]["stage"] == 1.0 and log[-1]["approx_kl"] < 0.05
    after = evaluate_sequential_route(route, renv, pol, n_replicas=64, start_index=1, end_index=60, start_q_noise_std=0.0008)
    assert float(after["longest_success_prefix"].float().mean()) >= float(before["longest_success_prefix"].float().mean()) - 6.0


@pytest.mark.parametrize("variant", ["tc", "tc_two_kernel", "fp32"])
def test_peer_gradient_exchange_single_rank_is_the_plain_reduction(variant):
    """The NVLink peer-memory exchange with one rank pushes into its own buffer: the update must be bitwise the one of the plain
    reduction.  "tc" / "fp32": kin_peer_grad_push + kin_peer_grad_gather (csrc/kin_peer.cu); "tc_two_kernel": the opt-in form with the
    exchange inside the gradient kernel's tail (kin_ppo_grad_tc_exchange: grid barrier, per-CTA column slices, per-slice flags).  The N-rank sum is
    checked by tools/peer_check.py under torchrun."""
    from rl_brain_trainer_b200 import ppo

    two_kernel = variant == "tc_two_kernel"
    variant = "tc" if two_kernel else variant

    cfg = env_config("approach_dynamic_scale_big")
    hp = ppo.PPOHyper(learning_rate=1e-3, n_steps=16, batch_size=2048, n_epochs=2, gamma=0.98, clip_range=0.2)
    params = {}
    for ex in ("nccl", "peer"):
        tr = ppo.PPOTrainer(cfg, ppo.random_policy(56, seed=1, log_std_init=-1.0, device="cuda"), num_envs=512, hyper=hp, seed=3, update_variant=variant,
                            grad_exchange=ex)
        assert (tr.peer is not None) == (ex == "peer")
        if two_kernel:
            tr.fused_exchange = False
        tr.learn(2)
        params[ex] = tr.params.clone()
        if tr.peer:
            assert tr.peer.epoch == 2 * 2 * (512 * 16 // 2048)
            tr.peer.close()
    assert torch.equal(params["nccl"], params["peer"])


@pytest.mark.parametrize("tiles_per_cta,num_envs,trained", [(1, 256, False), (2, 512, False), (4, 640, True), (2, 384, "dock")])
def test_fused_collection_replays_through_the_step_kernel(tiles_per_cta, num_envs, trained):
    """kin_ppo_collect (one launch per rollout, tensor-core policy) against the per-step kernels: replaying its recorded actions
    through kin_env_step from the same start state reproduces rewards, done flags, observations (as bf16 images) and the
    auto-reset draws; its sampled actions / log-probs / values agree with the fp32 policy on the recorded observations."""
    import dataclasses

    from rl_brain_trainer_b200 import _lib, ppo
    from rl_brain_trainer_b200.env import BatchedArmKinematicEnv

    cfg = env_config("finisher_noop_ft" if trained == "dock" else "approach_dynamic_scale_big")
    # short episodes: several time-limit truncations per rollout
    cfg = dataclasses.replace(cfg, episode_length=24, termination_config=dataclasses.replace(cfg.termination_config, max_episode_steps=24))
    T = 60
    handoff_rows = None
    if trained == "dock":   # Finisher training set-up: dock mode, dock reward, resets replay Approach handoff states / close buckets
        from rl_brain_trainer_b200 import handoff
        from rl_brain_trainer_b200.policy import PolicyWeights
        from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

        acfg = env_config("approach_dynamic_scale_big")
        buf, _ = handoff.build_finisher_handoff_state_buffer(acfg, PolicyWeights.preset("approach_stage8_11", "cuda"), stage_index=5,
                                                             suite=build_curriculum_local_eval_suite(acfg, seed=3, stage_index=5, n_episodes=256))
        handoff_rows = buf.device_rows("cuda")
        assert len(buf) > 100 and cfg.dock_reset_config.handoff_state_probability > 0.5
        pol, stage = PolicyWeights.preset("finisher", "cuda"), 5
    elif trained:     # the bundled approach checkpoint on the easiest shell: success / near-goal flags and dwell counters are exercised
        from rl_brain_trainer_b200.policy import PolicyWeights

        pol, stage = PolicyWeights.preset("approach_stage8_11", "cuda"), 0
    else:
        pol, stage = ppo.random_policy(56, seed=2, log_std_init=-1.5, device="cuda"), 3
        pol.tensors["act_w"].mul_(40.0)
        pol.tensors["vf_b1"].normal_(0, 0.2)
    hp = ppo.PPOHyper(n_steps=T, batch_size=num_envs * T // 4, n_epochs=1, gamma=0.97, learning_rate=0.0)
    tr = ppo.PPOTrainer(cfg, pol, num_envs=num_envs, hyper=hp, seed=11, stage_index=stage, update_variant="tc", collect_variant="fused",
                        handoff_states=handoff_rows)
    tr.tiles_per_cta = tiles_per_cta
    replay = BatchedArmKinematicEnv(cfg, num_envs, "cuda", auto_reset=True, seed=tr.env._seed, host_sampler=False, with_aux=False)
    replay.set_curriculum_stage(stage)
    if handoff_rows is not None:
        replay.set_handoff_states(handoff_rows)
    replay._ensure_sampler()
    for rollout in range(2):                 # the second rollout starts mid-episode from the state the first one left
        replay.state.copy_(tr.env.state)
        start0 = tr._next_start.clone()
        obs0 = replay.current_observation()
        tr.collect()
        torch.cuda.synchronize()
        obs_img = ppo.decode_obs_images(tr.obs_img).reshape(T, num_envs, 64)
        assert bool((obs_img[..., 56] == 1.0).all()) and bool((obs_img[..., 57:] == 0.0).all())
        raw_rew = torch.zeros((T, num_envs), device="cuda")
        obs_t = obs0
        n_trunc = 0
        for t in range(T):
            # observation image of step t == bf16(observation the step kernel produced)
            assert torch.equal(obs_img[t, :, :56], obs_t.bfloat16().float()), (rollout, t)
            mean, value = _torch_forward(pol, obs_t)
            sigma = pol.tensors["log_std"].exp()
            z = (tr.act_buf[t] - mean) / sigma
            lp = torch.distributions.Normal(mean, sigma).log_prob(tr.act_buf[t]).sum(-1)
            assert float((tr.val_buf[t] - value).abs().max()) < 0.05 * max(1.0, float(value.abs().max()))
            # the buffer holds log N(a) under the SAMPLING (bf16-operand) policy; against the fp32 policy it moves by z * d(mean) / sigma
            smin = float(sigma.min())
            assert float((tr.logp_buf[t] - lp).abs().max()) < 0.08 / smin and float((tr.logp_buf[t] - lp).abs().mean()) < 0.008 / smin
            assert abs(float(z.mean())) < 0.15 and 0.8 < float(z.std()) < 1.2
            replay.step_raw(tr.act_buf[t].contiguous())
            torch.cuda.synchronize()
            assert torch.equal(replay.done, tr.done_buf[t]), (rollout, t)
            raw_rew[t] = replay.reward
            trunc = ((replay.done & 2) != 0) & ((replay.done & 1) == 0)
            expect = replay.reward.clone()
            if bool(trunc.any()):
                _, tv = _torch_forward(pol, replay.terminal_obs)
                expect[trunc] += hp.gamma * tv[trunc]
                n_trunc += int(trunc.sum())
            assert torch.allclose(tr.rew_buf[t], expect, atol=2e-5), (rollout, t, float((tr.rew_buf[t] - expect).abs().max()))
            exp_start = start0 if t == 0 else ((tr.done_buf[t - 1] & 3) != 0).to(torch.uint8)
            assert torch.equal(tr.start_buf[t], exp_start)
            obs_t = replay.obs.clone()
        assert n_trunc == int(tr.boot_count) and n_trunc > 0
        assert not trained or bool(((tr.done_buf & 4) != 0).any())           # the trained policy reaches the success zone
        if trained == "dock":
            assert int(tr.env._mode_all) == 1 and bool(((tr.done_buf & 0x80) != 0).any())
        assert torch.equal(replay.state[:, :num_envs], tr.env.state[:, :num_envs])
        _, v_last = _torch_forward(pol, obs_t)
        assert float((tr.last_val - v_last).abs().max()) < 0.05 * max(1.0, float(v_last.abs().max()))
        assert torch.equal(tr._next_start, ((tr.done_buf[T - 1] & 3) != 0).to(torch.uint8))
        # GAE ran on the bootstrapped rewards
        ra, rr = ppo.numpy_gae(tr.rew_buf.cpu().numpy(), tr.val_buf.cpu().numpy(), tr.start_buf.cpu().numpy(), tr.last_val.cpu().numpy(),
                               ((tr.done_buf[T - 1] & 3) != 0).cpu().numpy(), hp.gamma, hp.gae_lambda)
        assert np.abs(tr.adv_buf.cpu().numpy() - ra).max() < 5e-4
    # the update consumes the images with the arithmetic that sampled them: with frozen parameters the probability ratio is 1
    stats = tr.update()
    assert stats["approx_kl"] < 1e-6 and stats["clip_fraction"] == 0.0 and np.isfinite(list(stats.values())).all()
    assert stats["grad_norm"] > 0


@pytest.mark.parametrize("tiles_per_cta,num_envs,sequence,chunk", [(1, 256, True, 0), (2, 512, True, 8), (4, 640, False, 0)])
def test_fused_route_collection_replays_through_the_step_kernels(tiles_per_cta, num_envs, sequence, chunk):
    """kin_route_collect (fused rollout of the 80-input route policy) against the per-step kernels it replaces: replaying its recorded
    actions through kin_route_step + kin_route_reset_sampled from the same start state reproduces observations, rewards (the TimeLimit
    bootstrap included), done flags, route flags, reset draws and the final SoA state BIT FOR BIT; sampled actions / log-probs / values
    agree with the fp32 policy to bf16 accuracy.  `chunk` > 0 runs the rollout in several launches (the prefix-curriculum mode)."""
    import dataclasses

    from rl_brain_trainer_b200 import config as kcfg, ppo
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.route import BatchedRouteKinematicEnv, RouteCurriculumStage, RoutePrefixCurriculum, synthetic_route

    route = synthetic_route(160, seed=7)
    renv, seq = kcfg.to_route_env_config(kcfg.preset_dict("route_prefix120"), max_route_index=len(route) - 1)
    base = renv.base_env_config       # short episodes: time-limit truncations inside the rollout
    renv = dataclasses.replace(renv, base_env_config=dataclasses.replace(base, episode_length=20, termination_config=dataclasses.replace(
        base.termination_config, max_episode_steps=20)))
    seq = dataclasses.replace(seq, enabled=bool(sequence))
    T = 48
    pol = PolicyWeights.preset("route_prefix120", "cuda")
    hp = ppo.PPOHyper(n_steps=T, batch_size=num_envs * T // 4, n_epochs=1, gamma=0.97, learning_rate=0.0)
    cur = None
    if chunk:   # a curriculum that never promotes: it only switches the chunked launch mode on
        cur = RoutePrefixCurriculum([RouteCurriculumStage("all", len(route) - 1)], promotion_success_rate=2.0, promotion_route_ready_hit_rate=2.0,
                                    promotion_orientation_hit_rate=2.0, promotion_max_regression_rate=-1.0, window_episodes=64, min_episodes_per_stage=64)
    tr = ppo.PPOTrainer(renv, pol, num_envs=num_envs, hyper=hp, seed=11, route=route, route_sequence_config=seq, collect_variant="fused", route_curriculum=cur)
    assert tr.collect_variant == "fused"
    tr.tiles_per_cta = tiles_per_cta
    if chunk:
        tr.route_chunk_steps = chunk
    replay = BatchedRouteKinematicEnv(route, renv, num_envs, "cuda", sequence_config=seq)
    if cur is not None:
        replay.set_route_window(max_route_index=cur.prefix_end_index)
    for rollout in range(2):
        replay.state.copy_(tr.env.state)
        start0 = tr._next_start.clone()
        step0 = tr.global_step
        tr.collect()
        torch.cuda.synchronize()
        obs_t = tr.obs_buf[0]
        n_trunc = 0
        for t in range(T):
            mean, value = _torch_forward(pol, obs_t)
            sigma = pol.tensors["log_std"].exp()
            lp = torch.distributions.Normal(mean, sigma).log_prob(tr.act_buf[t]).sum(-1)
            assert float((tr.val_buf[t] - value).abs().max()) < 0.05 * max(1.0, float(value.abs().max()))
            smin = float(sigma.min())
            assert float((tr.logp_buf[t] - lp).abs().mean()) < 0.01 / smin
            replay.step_raw(tr.act_buf[t].contiguous())
            torch.cuda.synchronize()
            assert torch.equal(replay.done, tr.done_buf[t]), (rollout, t)
            assert torch.equal(replay.raux[_lib_define("KIN_RAUX_FLAGS"), :num_envs].view(torch.int32), tr._route_raw[t]), (rollout, t)
            trunc = ((replay.done & 2) != 0) & ((replay.done & 1) == 0)
            expect = replay.reward.clone()
            if bool(trunc.any()):
                _, tv = _torch_forward(pol, replay.obs)           # the observation after the step IS the terminal observation
                expect[trunc] += hp.gamma * tv[trunc]
                n_trunc += int(trunc.sum())
            assert torch.equal(tr.rew_buf[t][~trunc], replay.reward[~trunc]), (rollout, t)
            assert torch.allclose(tr.rew_buf[t], expect, atol=2e-5), (rollout, t)
            replay.reset_done(seed=tr.seed ^ 0x5EED, counter=step0 + t)
            torch.cuda.synchronize()
            assert torch.equal(replay.obs, tr.obs_buf[t + 1]), (rollout, t)
            exp_start = start0 if t == 0 else ((tr.done_buf[t - 1] & 3) != 0).to(torch.uint8)
            assert torch.equal(tr.start_buf[t], exp_start)
            obs_t = tr.obs_buf[t + 1]
        assert n_trunc > 0 and bool(((tr.done_buf & 4) != 0).any())        # time limits were hit and waypoints were reached
        assert torch.equal(replay.state[:, :num_envs], tr.env.state[:, :num_envs])
        _, v_last = _torch_forward(pol, obs_t)
        assert float((tr.last_val - v_last).abs().max()) < 0.05 * max(1.0, float(v_last.abs().max()))
        ra, rr = ppo.numpy_gae(tr.rew_buf.cpu().numpy(), tr.val_buf.cpu().numpy(), tr.start_buf.cpu().numpy(), tr.last_val.cpu().numpy(),
                               ((tr.done_buf[T - 1] & 3) != 0).cpu().numpy(), hp.gamma, hp.gae_lambda)
        assert np.abs(tr.adv_buf.cpu().numpy() - ra).max() < 5e-4
    stats = tr.update()
    assert np.isfinite(list(stats.values())).all() and stats["approx_kl"] < 1e-5


def _lib_define(name):
    from rl_brain_trainer_b200 import _lib

    return _lib.define(name)


def test_gate_eval_and_finetune_retention():
    """Multi-stage gate evaluation in one launch; a short fine-tune at the reference's learning rate keeps the gate's retention
    (the acceptance SURVEY 8c asks for: a policy touched by the new trainer still passes when evaluated by the ORACLE env)."""
    from oracle import kin_oracle as ko
    from rl_brain_trainer_b200 import gate, ppo
    from rl_brain_trainer_b200.policy import PolicyWeights
    from rl_brain_trainer_b200.samplers import build_curriculum_local_eval_suite

    from ._util import oracle_params

    acfg, fcfg = env_config("approach_dynamic_scale_big"), env_config("finisher_noop_ft")
    pol, fin = PolicyWeights.preset("approach_stage8_11", "cuda"), PolicyWeights.preset("finisher", "cuda")
    gate_cfg = {"score_stage_index": 9, "retention_stage0_4_success": 0.95, "retention_stage5_success": 0.85, "promotion_stage_success": 0.55,
                "promotion_ready_rate": 0.62, "max_mean_position_error_m": 0.024, "max_mean_orientation_error_rad": 0.16}
    before = gate.evaluate_workspace_expansion(acfg, pol, fcfg, fin, episodes=256, seed=720001, gate_config=gate_cfg)
    m = before["stage_metrics"]
    assert set(m) == set(range(12)) and all(m[s]["episode_count"] == 256 for s in m)
    assert m[0]["success_rate"] > 0.98 and m[5]["success_rate"] > 0.9 and m[11]["success_rate"] < m[5]["success_rate"]
    assert before["best_model_selection"]["retention_ok"]
    assert 12 * 256 * 128 <= before["env_steps"] <= 12 * 256 * 164      # episodes without a handoff skip the 36 finisher steps
    hp = ppo.PPOHyper(learning_rate=4e-6, n_steps=128, batch_size=8192, n_epochs=2, gamma=0.995, clip_range=0.1, ent_coef=0.0003)
    tr = ppo.PPOTrainer(acfg, pol, num_envs=1024, hyper=hp, seed=5, stage_index=8)
    g = gate.EvalGate(acfg, fcfg, fin, eval_interval=1024 * 128, episodes=128, seed=720001, stage_indices=list(range(12)), gate_config=gate_cfg)
    log = tr.learn(2, gate=g)
    assert len(g.history) == 2 and "gate_score" in log[-1] and g.best_state is not None
    after = gate.evaluate_workspace_expansion(acfg, pol, fcfg, fin, episodes=256, seed=720001, gate_config=gate_cfg)
    assert after["best_model_selection"]["retention_ok"]
    assert abs(after["stage_metrics"][5]["success_rate"] - m[5]["success_rate"]) < 0.05
    # the fine-tuned weights, evaluated by the CPU oracle env on Stage 5
    suite = build_curriculum_local_eval_suite(acfg, seed=720001 + 5 * 1009, stage_index=5, n_episodes=256)
    w = {k: v.detach().cpu().numpy() for k, v in tr.state_dict().items()}
    fw = {k: v.detach().cpu().numpy() for k, v in fin.state_dict().items()}
    ref, _ = ko.eval_approach_finisher(oracle_params(acfg), oracle_params(fcfg), ko.OracleMlp(w), ko.OracleMlp(fw),
                                       initial_q=suite.initial_q.astype(np.float32).astype(float), goal_q=suite.goal_q.astype(np.float32).astype(float),
                                       n_threads=8)
    assert ref["success"].mean() >= 0.85
    assert abs(ref["success"].mean() - after["stage_metrics"][5]["success_rate"]) < 0.03
