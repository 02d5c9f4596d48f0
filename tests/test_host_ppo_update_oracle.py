"""CPU checks of the fp64 PPO oracle (``tests/_ppo_oracle.py``) the GPU update replays are judged by: its optimiser step is
``clip_grad_norm_`` + ``torch.optim.Adam``, and its loss gradient is the derivative of its loss (central finite differences)."""

from __future__ import annotations

from types import SimpleNamespace

import pytest
import torch

from . import _ppo_oracle as oracle


def _hp(**kw):
    base = dict(learning_rate=3e-4, clip_range=0.2, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, normalize_advantage=True,
                adam_beta1=0.9, adam_beta2=0.999, adam_eps=1e-5)
    base.update(kw)
    return SimpleNamespace(**base)


@pytest.mark.parametrize("betas,eps,lr", [((0.9, 0.999), 1e-5, 3e-4), ((0.8, 0.99), 1e-8, 2e-2)])
def test_adam_step_is_clip_grad_norm_and_torch_adam(betas, eps, lr):
    g = torch.Generator().manual_seed(7)
    P = 301
    hp = _hp(learning_rate=lr, adam_beta1=betas[0], adam_beta2=betas[1], adam_eps=eps, max_grad_norm=0.5)
    p0 = torch.randn(P, dtype=torch.float64, generator=g)
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=lr, betas=betas, eps=eps, foreach=False)
    p, m, v = p0.clone(), torch.zeros(P, dtype=torch.float64), torch.zeros(P, dtype=torch.float64)
    active = []
    for step in range(1, 7):
        grad = torch.randn(P, dtype=torch.float64, generator=g) * (0.004 if step % 2 else 0.3)    # norm ~0.07 (kept) / ~5 (clipped)
        ref.grad = grad.clone()
        norm = float(torch.nn.utils.clip_grad_norm_([ref], hp.max_grad_norm))
        opt.step()
        p, m, v, o_norm, coef = oracle.adam_step(p, m, v, grad, hp, step)
        active.append(coef < 1.0)
        assert abs(o_norm - norm) <= 1e-12 * norm
        st = opt.state[ref]
        assert torch.allclose(p, ref.detach(), rtol=0, atol=1e-13), step
        assert torch.allclose(m, st["exp_avg"], rtol=1e-12, atol=0) and torch.allclose(v, st["exp_avg_sq"], rtol=1e-12, atol=0), step
    assert active == [False, True] * 3


def test_adam_step_without_a_positive_clip_norm_keeps_the_gradient():
    """``max_grad_norm <= 0`` means no clip (``kin_ppo_adam``'s rule), where ``clip_grad_norm_(0)`` would zero the gradient."""
    g = torch.Generator().manual_seed(8)
    grad = torch.randn(50, dtype=torch.float64, generator=g) * 10
    zeros = torch.zeros(50, dtype=torch.float64)
    for mx in (0.0, -1.0):
        p, m, v, norm, coef = oracle.adam_step(zeros, zeros, zeros, grad, _hp(max_grad_norm=mx), 1)
        assert coef == 1.0 and torch.allclose(m, 0.1 * grad, rtol=1e-15, atol=0)
    with pytest.raises(ValueError):
        oracle.adam_step(zeros, zeros, zeros, grad, _hp(), 0)


def _problem(seed, n, ratio_noise, in_dim=12):
    """A tiny random policy (in_dim inputs; the hidden sizes are the kernels') and a minibatch drawn from it."""
    g = torch.Generator().manual_seed(seed)
    P = oracle.param_count(in_dim)
    params = torch.randn(P, dtype=torch.float64, generator=g) * 0.3
    t = oracle.unflatten(params, in_dim)
    t["log_std"].copy_(torch.linspace(-0.8, 0.2, oracle.ACT, dtype=torch.float64))
    obs = torch.rand((n, in_dim), dtype=torch.float64, generator=g) * 2 - 1
    mean, value, log_std = oracle.forward(params, obs)
    act = mean + log_std.exp() * torch.randn((n, oracle.ACT), dtype=torch.float64, generator=g)
    logp = (-0.5 * ((act - mean) / log_std.exp()) ** 2 - log_std - oracle._HALF_LOG_2PI).sum(-1)
    old_logp = logp + ratio_noise * torch.randn(n, dtype=torch.float64, generator=g)
    adv = torch.randn(n, dtype=torch.float64, generator=g) * 2.0 + 0.7
    ret = value + torch.randn(n, dtype=torch.float64, generator=g)
    return params, obs, act, old_logp, adv, ret


@pytest.mark.parametrize("normalize,ent_coef,ratio_noise", [(True, 0.0, 0.0), (False, 0.05, 0.0), (True, 0.05, 0.5), (False, 0.0, 0.5)])
def test_loss_gradient_matches_central_differences(normalize, ent_coef, ratio_noise):
    """ratio_noise 0: every ratio is 1 (inside the clip range); 0.5: log-ratios of std 0.5 put most samples outside clip_range = 0.1."""
    in_dim, n = 12, 48
    params, obs, act, old_logp, adv, ret = _problem(3 + int(normalize) + 10 * int(ratio_noise > 0), n, ratio_noise, in_dim)
    hp = _hp(clip_range=0.1, ent_coef=ent_coef, vf_coef=0.7, normalize_advantage=normalize)
    grad, stats, (mu, inv) = oracle.minibatch(params, hp, obs, act, old_logp, adv, ret)
    if normalize:
        assert abs(mu - float(adv.mean())) < 1e-12 and abs(inv - 1.0 / (float(adv.std(unbiased=True)) + 1e-8)) < 1e-12
    else:
        assert (mu, inv) == (0.0, 1.0)
    clip_fraction = float(stats[4])
    assert (clip_fraction == 0.0) if ratio_noise == 0 else (0.3 < clip_fraction < 0.95)
    if ratio_noise == 0:
        assert abs(float(stats[3])) < 1e-15           # approx_kl of ratio 1
    f = lambda q: float(oracle.loss(q, hp, obs, act, old_logp, adv, ret)[0])  # noqa: E731
    # finite differences on a spread of coordinates: a few of every tensor, every log_std and val_b
    gsel = torch.Generator().manual_seed(99)
    picks = []
    for name, sl in oracle.param_slices(in_dim):
        size = sl.stop - sl.start
        k = size if size <= 7 else 6
        picks += (sl.start + torch.randperm(size, generator=gsel)[:k]).tolist()
    h = 1e-6
    for i in picks:
        e = torch.zeros_like(params)
        e[i] = h
        fd = (f(params + e) - f(params - e)) / (2 * h)
        assert abs(fd - float(grad[i])) < 1e-6 * max(1.0, abs(fd)), (i, fd, float(grad[i]))
    # the entropy term: exactly -ent_coef on every log_std entry, nothing elsewhere
    hp0 = _hp(clip_range=0.1, ent_coef=0.0, vf_coef=0.7, normalize_advantage=normalize)
    g0, _, _ = oracle.minibatch(params, hp0, obs, act, old_logp, adv, ret)
    ls = oracle.param_slices(in_dim)[-1][1]
    assert torch.allclose(grad[ls] - g0[ls], torch.full((oracle.ACT,), -ent_coef, dtype=torch.float64), rtol=0, atol=1e-14)
    assert torch.equal(grad[: ls.start], g0[: ls.start])
    # the clip decided by given ratios: by the oracle's own, it is SB3's min(a r, a clamp(r)); by shifted ones, other samples clip
    mean, _, log_std = oracle.forward(params, obs)
    own = torch.exp((-0.5 * ((act - mean) / log_std.exp()) ** 2 - log_std - oracle._HALF_LOG_2PI).sum(-1) - old_logp)
    g1, s1, _ = oracle.minibatch(params, hp, obs, act, old_logp, adv, ret, clip_ratio=own)
    assert torch.allclose(g1, grad, rtol=1e-12, atol=1e-15) and torch.equal(s1, stats)
    if ratio_noise > 0:
        g2, _, _ = oracle.minibatch(params, hp, obs, act, old_logp, adv, ret, clip_ratio=own * 1.08)
        assert not torch.allclose(g2, grad, rtol=1e-6, atol=1e-9)


def test_forward_layout_is_param_order():
    """The flat layout is the kernels' (``include/kin_b200.h``): 16143 parameters at 56 inputs, 17679 at 80."""
    assert oracle.param_count(56) == 16143 and oracle.param_count(80) == 16143 + 2 * 64 * 24
    params = torch.zeros(oracle.param_count(56), dtype=torch.float64)
    t = oracle.unflatten(params, 56)
    t["act_b"].copy_(torch.arange(7, dtype=torch.float64))
    t["val_b"].fill_(2.5)
    mean, value, log_std = oracle.forward(params, torch.randn(3, 56))
    assert torch.equal(mean, torch.arange(7, dtype=torch.float64).expand(3, 7)) and torch.equal(value, torch.full((3,), 2.5, dtype=torch.float64))
