"""fp64 restatement of one step of stable-baselines3 2.8.0 ``PPO.train()`` (test infrastructure).

Plain torch float64 on whatever device the inputs live on, in the flat ``PARAM_ORDER`` parameter layout of the kernels
(``include/kin_b200.h``): the actor-critic forward, the minibatch loss with its gradient and statistics, and the optimiser step
(``clip_grad_norm_`` + ``torch.optim.Adam``).  ``tests/test_host_ppo_update_oracle.py`` checks it against torch and finite differences;
``tests/test_gpu_ppo_update_oracle.py`` replays whole device updates against it.
"""

from __future__ import annotations

import math

import torch

PARAM_ORDER = ("pi_w0", "pi_b0", "pi_w1", "pi_b1", "act_w", "act_b", "vf_w0", "vf_b0", "vf_w1", "vf_b1", "val_w", "val_b", "log_std")
HIDDEN, ACT = 64, 7
STAT_NAMES = ("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction")
_HALF_LOG_2PI = 0.5 * math.log(2.0 * math.pi)


def param_shapes(in_dim: int) -> list[tuple[str, tuple[int, ...]]]:
    h = HIDDEN
    shapes = {"pi_w0": (h, in_dim), "pi_b0": (h,), "pi_w1": (h, h), "pi_b1": (h,), "act_w": (ACT, h), "act_b": (ACT,),
              "vf_w0": (h, in_dim), "vf_b0": (h,), "vf_w1": (h, h), "vf_b1": (h,), "val_w": (1, h), "val_b": (1,), "log_std": (ACT,)}
    return [(k, shapes[k]) for k in PARAM_ORDER]


def param_count(in_dim: int) -> int:
    return sum(math.prod(s) for _, s in param_shapes(in_dim))


def param_slices(in_dim: int) -> list[tuple[str, slice]]:
    """(name, slice of the flat buffer) in ``PARAM_ORDER``."""
    out, off = [], 0
    for k, s in param_shapes(in_dim):
        n = math.prod(s)
        out.append((k, slice(off, off + n)))
        off += n
    return out


def unflatten(params: torch.Tensor, in_dim: int) -> dict[str, torch.Tensor]:
    if params.numel() != param_count(in_dim):
        raise ValueError(f"{params.numel()} parameters, the in_dim = {in_dim} layout has {param_count(in_dim)}")
    return {k: params[sl].view(s) for (k, sl), (_, s) in zip(param_slices(in_dim), param_shapes(in_dim))}


def forward(params_flat: torch.Tensor, obs: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """SB3 ``MultiInputPolicy`` actor-critic (tanh MLPs 64-64, separate nets) in fp64: (action mean [n, 7], value [n], log_std [7])."""
    t = unflatten(params_flat.double(), obs.shape[-1])
    x = obs.double()
    lin = torch.nn.functional.linear
    h = torch.tanh(lin(torch.tanh(lin(x, t["pi_w0"], t["pi_b0"])), t["pi_w1"], t["pi_b1"]))
    hv = torch.tanh(lin(torch.tanh(lin(x, t["vf_w0"], t["vf_b0"])), t["vf_w1"], t["vf_b1"]))
    return lin(h, t["act_w"], t["act_b"]), lin(hv, t["val_w"], t["val_b"])[:, 0], t["log_std"]


def adv_stats(adv: torch.Tensor, normalize: bool) -> tuple[float, float]:
    """SB3's per-minibatch advantage normalisation as (mean, 1 / (std + 1e-8)), unbiased std; (0, 1) when it is off."""
    if not normalize:
        return 0.0, 1.0
    a = adv.double()
    return float(a.mean()), float(1.0 / (a.std() + 1e-8))


def loss(params: torch.Tensor, hp, obs, act, old_logp, adv, ret, clip_ratio=None) -> tuple[torch.Tensor, torch.Tensor, tuple[float, float]]:
    """SB3 loss of one minibatch: clipped surrogate + vf_coef * MSE(returns, value) - ent_coef * entropy.  Returns (loss, the five
    statistics [policy_loss, value_loss, entropy, approx_kl, clip_fraction], advantage (mean, 1 / (std + 1e-8))).
    clip_ratio (optional, [n]): decide which samples the clip takes by these ratios instead of the oracle's own -- a clipped sample
    contributes the constant a * (1 +- clip_range), as in SB3.  A replay passes the device's own ratios, so that samples whose bf16
    ratio sits on the other side of the clip boundary do not count as gradient error; the statistics keep the oracle's ratios."""
    mean, value, log_std = forward(params, obs)
    act, old_logp, ret = act.double(), old_logp.double(), ret.double()
    logp = (-0.5 * ((act - mean) * torch.exp(-log_std)) ** 2 - log_std - _HALF_LOG_2PI).sum(-1)
    entropy = (0.5 + _HALF_LOG_2PI + log_std).sum().expand(logp.shape[0])
    mu, inv = adv_stats(adv, bool(hp.normalize_advantage))
    a = (adv.double() - mu) * inv
    log_ratio = logp - old_logp
    ratio = torch.exp(log_ratio)
    clip = float(hp.clip_range)
    if clip_ratio is None:
        policy_loss = -torch.min(a * ratio, a * torch.clamp(ratio, 1.0 - clip, 1.0 + clip)).mean()
    else:
        r = clip_ratio.double()
        policy_loss = -torch.where((a > 0) & (r > 1.0 + clip), a * (1.0 + clip),
                                   torch.where((a < 0) & (r < 1.0 - clip), a * (1.0 - clip), a * ratio)).mean()
    value_loss = ((ret - value) ** 2).mean()
    total = policy_loss - float(hp.ent_coef) * entropy.mean() + float(hp.vf_coef) * value_loss
    with torch.no_grad():
        stats = torch.stack([policy_loss, value_loss, entropy.mean(), ((ratio - 1.0) - log_ratio).mean(),
                             ((ratio - 1.0).abs() > clip).double().mean()]).detach()
    return total, stats, (mu, inv)


def minibatch(params: torch.Tensor, hp, obs, act, old_logp, adv, ret, clip_ratio=None) -> tuple[torch.Tensor, torch.Tensor, tuple[float, float]]:
    """(d loss / d params [P] fp64, the five statistics, advantage (mean, 1 / (std + 1e-8))) of one minibatch (``loss``)."""
    p = params.detach().double().clone().requires_grad_(True)
    total, stats, ms = loss(p, hp, obs, act, old_logp, adv, ret, clip_ratio)
    (g,) = torch.autograd.grad(total, [p])
    return g.detach(), stats, ms


def adam_step(p, m, v, grad, hp, step: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, float, float]:
    """``clip_grad_norm_(max_grad_norm)`` (coefficient max / (norm + 1e-6), capped at 1) then one ``torch.optim.Adam`` step (lr, betas, eps
    of ``hp``; ``step`` counts from 1), all in fp64.  ``max_grad_norm <= 0`` skips the clip, as ``kin_ppo_adam`` does (torch would zero
    the gradient).  Returns (p, m, v, pre-clip norm, clip coefficient)."""
    if step < 1:
        raise ValueError("Adam steps count from 1")
    g = grad.double()
    norm = float(torch.linalg.vector_norm(g))
    mx = float(hp.max_grad_norm)
    coef = min(mx / (norm + 1e-6), 1.0) if mx > 0.0 else 1.0
    g = g * coef
    b1, b2, lr, eps = float(hp.adam_beta1), float(hp.adam_beta2), float(hp.learning_rate), float(hp.adam_eps)
    m = b1 * m.double() + (1.0 - b1) * g
    v = b2 * v.double() + (1.0 - b2) * g * g
    bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
    p = p.double() - (lr / bc1) * (m / (v.sqrt() / math.sqrt(bc2) + eps))
    return p, m, v, norm, coef
