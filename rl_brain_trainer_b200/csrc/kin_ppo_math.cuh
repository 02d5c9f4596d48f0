// kin_ppo_math.cuh -- the arithmetic of one PPO update, defined once for every kernel that runs it: the Gaussian policy's log-density
// and entropy terms, the minibatch advantage normalisation, the clipped-surrogate / value / entropy loss of one sample with its
// derivatives, and clip_grad_norm_ + Adam of one parameter.
//
// Third-party arithmetic restated here: stable-baselines3 2.8.0 (ppo.py train(), distributions.py DiagGaussianDistribution) and torch
// (nn.utils.clip_grad_norm_, optim.Adam).  tests/_ppo_oracle.py is the independent fp64 restatement every update path is replayed
// against, and the paths are checked bitwise against each other, so the expression order is part of the definition.  The helpers take
// values and leave the loads and stores to the kernels (which stage their inputs differently), except for the tile-sum gather and the
// normaliser's two plain stores.
#pragma once

#include "kin_internal.h"

namespace kin {

constexpr float kHalfLog2Pi = 0.91893853320467274178f;   // 0.5 * log(2 pi): the normalising term of the policy's Gaussian log-density

// log N(a; mean, sigma) of one action dimension, z = (a - mean) / sigma, ls = log sigma
__device__ __forceinline__ float gauss_logp_term(float z, float ls) { return -0.5f * z * z - ls - kHalfLog2Pi; }
// entropy of one action dimension
__device__ __forceinline__ float gauss_entropy_term(float ls) { return 0.5f + kHalfLog2Pi + ls; }

// (sum adv, sum adv^2) of a minibatch from the per-tile fp64 sums of its tiles ids[first], ids[first + stride], ..., ids[n - 1],
// summed over the 32 lanes of the warp: every lane returns the warp's total
__device__ __forceinline__ double2 warp_tile_sums(const double* tile_sums, const int* ids, int n, int first, int stride) {
    double s1 = 0.0, s2 = 0.0;
    for (int j = first; j < n; j += stride) {
        const int t = ids[j];
        s1 += tile_sums[2 * t];
        s2 += tile_sums[2 * t + 1];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, off);
        s2 += __shfl_xor_sync(0xffffffffu, s2, off);
    }
    return make_double2(s1, s2);
}

// the advantage normaliser of a minibatch, A = (adv - out[0]) * out[1], from the fp64 sums of its nsamp advantages (torch: mean,
// unbiased std): out[0] = mean, out[1] = 1 / (std + 1e-8); 0 and 1 when normalize is off.  One plain store each, in that order.
__device__ __forceinline__ void adv_normaliser(double s1, double s2, double nsamp, int normalize, float* out) {
    const double mean = s1 / nsamp;
    const double var = nsamp > 1.0 ? fmax((s2 - nsamp * mean * mean) / (nsamp - 1.0), 0.0) : 0.0;
    out[0] = normalize ? (float)mean : 0.0f;
    out[1] = normalize ? (float)(1.0 / (sqrt(var) + 1e-8)) : 1.0f;
}

// the clipped surrogate of one sample, -min(r A, clip(r, 1 - clip_range, 1 + clip_range) A) with r = exp(logp - old_logp) and A the
// advantage normalised by (adv_mean, adv_scale).  The members give what the update takes from it; each kernel evaluates them where it
// uses them.
struct Surrogate {
    float adv_n, log_ratio, ratio, pl1, pl2;
    __device__ __forceinline__ float dpl_dlp() const { return (pl1 <= pl2) ? -adv_n * ratio : 0.0f; }      // d(policy loss) / d logp
    __device__ __forceinline__ float loss() const { return -fminf(pl1, pl2); }
    __device__ __forceinline__ float approx_kl() const { return (ratio - 1.0f) - log_ratio; }
    __device__ __forceinline__ float clipped(const KinPpoHyper& hp) const { return fabsf(ratio - 1.0f) > hp.clip_range ? 1.0f : 0.0f; }
};
__device__ __forceinline__ Surrogate clipped_surrogate(float adv, float adv_mean, float adv_scale, float logp, float old_logp, const KinPpoHyper& hp) {
    Surrogate s;
    s.adv_n = (adv - adv_mean) * adv_scale;
    s.log_ratio = logp - old_logp;
    s.ratio = expf(s.log_ratio);
    s.pl1 = s.adv_n * s.ratio;
    s.pl2 = s.adv_n * fminf(fmaxf(s.ratio, 1.0f - hp.clip_range), 1.0f + hp.clip_range);
    return s;
}

// one sample's share of dL/dmean_d and of dL/dlog_std_d (the surrogate through logp, and the entropy bonus), inv_batch = 1 / minibatch size
__device__ __forceinline__ float dloss_dmean(float inv_batch, float dpl_dlp, float z, float inv_sig) { return inv_batch * dpl_dlp * z * inv_sig; }
__device__ __forceinline__ float dloss_dlog_std(float inv_batch, float dpl_dlp, float z, const KinPpoHyper& hp) {
    return inv_batch * dpl_dlp * (z * z - 1.0f) - inv_batch * hp.ent_coef;
}

// the value loss of one sample, (ret - v)^2, and its share of dL/dvalue = vf_coef * d mse / dv
__device__ __forceinline__ float value_loss(float v, float ret) { return (ret - v) * (ret - v); }
__device__ __forceinline__ float dloss_dvalue(float inv_batch, float v, float ret, const KinPpoHyper& hp) { return inv_batch * hp.vf_coef * 2.0f * (v - ret); }

// clip_grad_norm_'s coefficient for the global gradient norm; max_grad_norm <= 0 turns the clip off
__device__ __forceinline__ float clip_coef(float norm, const KinPpoHyper& hp) {
    const float c = hp.max_grad_norm > 0.0f ? hp.max_grad_norm / (norm + 1e-6f) : 1.0f;
    return c < 1.0f ? c : 1.0f;
}

// Adam on one parameter, in the two steps the kernels store: the moments (m, v) from the gradient grad scaled by the clip coefficient cf,
// then the parameter w from them, with the bias corrections bc1 / bc2 of adam_bias_corrections
struct AdamMoments {
    float m, v;
};
__device__ __forceinline__ AdamMoments adam_moments(float grad, float cf, float m, float v, const KinPpoHyper& hp) {
    const float g = grad * cf;
    return {fmaf(hp.adam_beta1, m, (1.0f - hp.adam_beta1) * g), fmaf(hp.adam_beta2, v, (1.0f - hp.adam_beta2) * g * g)};
}
__device__ __forceinline__ float adam_param(float w, AdamMoments mv, float bc1, float bc2, const KinPpoHyper& hp) {
    const float denom = sqrtf(mv.v) / sqrtf(bc2) + hp.adam_eps;
    return w - (hp.learning_rate / bc1) * (mv.m / denom);
}

// (1 - beta1^step, 1 - beta2^step), computed on the host; step counts optimiser steps from 1
inline float2 adam_bias_corrections(const KinPpoHyper& hp, int step) {
    const auto bc = [step](float beta) { return 1.0f - powf(beta, (float)step); };
    return make_float2(bc(hp.adam_beta1), bc(hp.adam_beta2));
}

}  // namespace kin
