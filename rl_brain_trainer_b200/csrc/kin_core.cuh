// kin_core.cuh -- per-env device arithmetic of the kinematic env, fp32, registers only.
//
// Everything here works on ONE env held in registers (EnvRegs) so the same code serves the
// standalone fused step kernel (kin_step.cu: load SoA -> step_core -> store) and the fused
// policy-in-loop rollout (kin_rollout.cu: T steps per launch without touching HBM).
//
// Reference (behaviour only; paths under hrl_ws/src/hrl_trainer/hrl_trainer/):
//   v5_1/ee_fk.py:98-134, kinematic_phase1/kinematics/pose_utils.py:11-26,
//   kinematic_phase1/kinematics/joint_limits.py:140-174,
//   kinematic_phase1/envs/arm_kinematic_env.py:213-365,425-444,489-542 ("AKE"),
//   kinematic_phase1/envs/observation_builder.py:29-94, envs/termination.py:20-57,
//   envs/reward_approach.py:75-373, envs/reward_dock.py:105-484.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>

#include "kin_b200.h"

namespace kin {

constexpr int NJ = KIN_NJ;
constexpr float kPi = 3.14159265358979323846f;
constexpr float kTwoPi = 6.28318530717958647692f;
constexpr float kInvTwoPi = 0.15915494309189533577f;

struct EnvRegs {
    float q[NJ];
    float dq[NJ];
    float pa[NJ];    // prev_action
    float goal[6];   // goal pose6
    float ee[6];     // cached FK(q)
    float min_pos;
    float entry[4];  // entry pos err, ori err, action l2, dq norm
    int step;
    int dwell;
    int entry_cnt;
    int drift_cnt;
    unsigned flags;  // KIN_FLAG_*
};

struct StepOut {
    float reward;
    float pos, ori;          // position / orientation error norms after the step
    float action_l2, dq_l2;  // ||clipped action||, ||executed dq||
    float dq_change_l2;
    float dock_limit, dqc_scale;
    float margin_min;
    float pe[3], oe[3];      // pose error components after the step (reused by the observation)
    float margin[NJ];        // per-joint limit margins after the step (reused by the observation)
    float qn[NJ];            // FAST flavour only: normalised joint positions 2(q-lo)/span-1 after the step (observation "q")
    unsigned done;           // KIN_DONE_* bits
};

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }
// Quotients of the rewards' shaping terms (value / configured radius or threshold): MUFU reciprocal + multiply (2 ulp) instead of
// the IEEE division sequence -- reward terms only, never a predicate, so flags and counters are untouched and the reward stays inside
// its 2e-4 relative tolerance by three orders of magnitude.  (The approach reward gets the same saving from host-side reciprocals.)
__device__ __forceinline__ float qdiv(float x, float y) { return __fdividef(x, y); }

__device__ __forceinline__ float norm3(float a, float b, float c) { return sqrtf(fmaf(a, a, fmaf(b, b, c * c))); }
__device__ __forceinline__ float norm7(const float* v) {
    float acc = v[0] * v[0];
#pragma unroll
    for (int i = 1; i < NJ; ++i) acc = fmaf(v[i], v[i], acc);
    return sqrtf(acc);
}

// ---- FAST flavour (the tensor-core rollout / collection kernels) -----------------------------------------------------
// Same formulas, cheaper instruction sequences: single-MUFU sqrt / reciprocal (relative error 2^-23, no slow path), a
// branch-free atan2 (minimax polynomial, |error| < 5e-7 rad), margins from the normalised joint position, and the previous
// step's pose-error norms carried instead of recomputed.  Measured FK differences from the strict flavour (B200): with the
// polynomial sine / cosine (FAST = 1) the same position and Euler angles within 3.2e-7 rad; with the MUFU ones (FAST = 2, the
// default of the tensor-core rollout) 4.8e-7 m and 8.7e-6 rad (an Euler angle near pitch +-pi/2; 1.4e-6 rad elsewhere on the
// joint limits) -- inside the 1e-5 m / 1e-5 rad pose tolerance (tests/test_gpu_fast_env_math.py).  The strict kernels (K1,
// kin_rollout_ffma) do not use it.
__device__ __forceinline__ float sqrt_approx(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
template <int FAST>
__device__ __forceinline__ float sqrt_sel(float x) {
    if constexpr (FAST) return sqrt_approx(x);
    else return sqrtf(x);
}
template <int FAST>
__device__ __forceinline__ float norm3_sel(float a, float b, float c) { return sqrt_sel<FAST>(fmaf(a, a, fmaf(b, b, c * c))); }

// atan2 for the Euler extraction: t = min/max in [0, 1], atan(t) = t + t^3 Q(t^2) (Remez fit, max |error| 7.5e-8 in fp32),
// then the octant / quadrant / sign fixes.  |error| < 5e-7 rad (the fit, rcp.approx and the rounding of pi/2 - r, pi - r) for
// max(|x|, |y|) in [2^-126, 2^126]: the guard of the reciprocal is the smallest normal float, so t is the true ratio for every
// normal input (rcp.approx flushes a subnormal operand); with both inputs subnormal the octant and sign are still right.
// atan2(+-0, +0) = +-0 and atan2(+-0, x < 0) = +-pi like math.atan2, but atan2(+-0, -0) = +-0 where math.atan2 gives +-pi:
// the x < 0 test does not see the sign of a zero.
__device__ __forceinline__ float atan2_fast(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float t = mn * rcp_approx(fmaxf(mx, 1.17549435e-38f));
    const float s = t * t;
    float p = 0.0026222446467727423f;
    p = fmaf(p, s, -0.015132537111639977f);
    p = fmaf(p, s, 0.04112186282873154f);
    p = fmaf(p, s, -0.07366706430912018f);
    p = fmaf(p, s, 0.10573931783437729f);
    p = fmaf(p, s, -0.1418597549200058f);
    p = fmaf(p, s, 0.1999039649963379f);
    p = fmaf(p, s, -0.33332985639572144f);
    float r = fmaf(t * s, p, t);
    r = (ay > ax) ? 1.57079632679489661923f - r : r;
    r = (x < 0.0f) ? kPi - r : r;
    return copysignf(r, y);
}

// pose_utils.py:11-12: (v + pi) mod 2pi - pi with a floored modulo.  Written as v - 2pi*floor((v+pi)/2pi)
// so that |v| < pi (every in-shell step) returns v bit-exactly instead of losing bits in (v + pi) - pi.
__device__ __forceinline__ float wrap_to_pi(float v) {
    float k = floorf((v + kPi) * kInvTwoPi);
    return fmaf(-k, kTwoPi, v);
}

// sin and cos of a joint angle.  Joint values are clipped to their limits (|q| <= pi), so the argument reduction is
// a 3-term Cody-Waite by k*pi/2 with |k| <= 2 and no large-argument path; minimax polynomials on [-pi/4, pi/4]
// (errors ~1 ulp, the same polynomials the fast path of sinf/cosf uses).
__device__ __forceinline__ void sincos_joint(float x, float* sp, float* cp) {
    const float kf = rintf(x * 0.63661977236758134f);
    const int k = (int)kf;
    float r = fmaf(kf, -1.57079601287841796875f, x);
    r = fmaf(kf, -3.1391647326017846353e-07f, r);
    r = fmaf(kf, -5.3903029534742383927e-15f, r);
    const float r2 = r * r;
    float ps = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(ps, r2, -1.6666654611e-1f);
    ps = fmaf(ps * r2, r, r);
    float pc = fmaf(r2, 2.4433157117e-5f, -1.3887316255e-3f);
    pc = fmaf(pc, r2, 4.1666645683e-2f);
    pc = fmaf(pc, r2, -0.5f);
    pc = fmaf(pc, r2, 1.0f);
    const float s0 = (k & 1) ? pc : ps;
    const float c0 = (k & 1) ? ps : pc;
    *sp = (k & 2) ? -s0 : s0;
    *cp = ((k + 1) & 2) ? -c0 : c0;
}

// FAST flavour: two-term Cody-Waite (|k| <= 2, the third term is 5e-15 * k).
__device__ __forceinline__ void sincos_joint_fast(float x, float* sp, float* cp) {
    const float kf = rintf(x * 0.63661977236758134f);
    const int k = (int)kf;
    float r = fmaf(kf, -1.57079601287841796875f, x);
    r = fmaf(kf, -3.1391647326017846353e-07f, r);
    const float r2 = r * r;
    float ps = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(ps, r2, -1.6666654611e-1f);
    ps = fmaf(ps * r2, r, r);
    float pc = fmaf(r2, 2.4433157117e-5f, -1.3887316255e-3f);
    pc = fmaf(pc, r2, 4.1666645683e-2f);
    pc = fmaf(pc, r2, -0.5f);
    pc = fmaf(pc, r2, 1.0f);
    const float s0 = (k & 1) ? pc : ps;
    const float c0 = (k & 1) ? ps : pc;
    *sp = (k & 2) ? -s0 : s0;
    *cp = ((k + 1) & 2) ? -c0 : c0;
}
// FAST: 0 strict, 1 fast, 2 fast with the MUFU sine / cosine (sin.approx / cos.approx: |error| <= 2^-20.9 on [-pi, pi], ~5e-7)
template <int FAST>
__device__ __forceinline__ void sincos_sel(float x, float* sp, float* cp) {
    if constexpr (FAST == 2) {
        *sp = __sinf(x);
        *cp = __cosf(x);
    } else if constexpr (FAST == 1) {
        sincos_joint_fast(x, sp, cp);
    } else {
        sincos_joint(x, sp, cp);
    }
}

// ee_fk.py:98-134 with the constant transforms folded on the host (see KinEnvParams::fk_*):
// one sincos + 12 flops per revolute joint for the Rz, 27 for the constant 3x3, 9 for the offset.
template <int FAST = 0>
__device__ __forceinline__ void fk_pose6(const KinEnvParams& P, const float* q, float* pose) {
    float s, c;
    float R[9], M[9];
    sincos_sel<FAST>(q[1], &s, &c);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        float m0 = P.fk_C[3 * r], m1 = P.fk_C[3 * r + 1];
        R[3 * r] = fmaf(c, m0, s * m1);
        R[3 * r + 1] = fmaf(c, m1, -s * m0);
        R[3 * r + 2] = P.fk_C[3 * r + 2];
    }
    float p0 = fmaf(P.fk_pq0[0], q[0], P.fk_pbase[0]);
    float p1 = fmaf(P.fk_pq0[1], q[0], P.fk_pbase[1]);
    float p2 = fmaf(P.fk_pq0[2], q[0], P.fk_pbase[2]);
#pragma unroll
    for (int j = 2; j < NJ; ++j) {
        const float* t = P.fk_t + 3 * (j - 2);
        const float* C = P.fk_C + 9 * (j - 1);
        p0 = fmaf(R[0], t[0], fmaf(R[1], t[1], fmaf(R[2], t[2], p0)));
        p1 = fmaf(R[3], t[0], fmaf(R[4], t[1], fmaf(R[5], t[2], p1)));
        p2 = fmaf(R[6], t[0], fmaf(R[7], t[1], fmaf(R[8], t[2], p2)));
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int k = 0; k < 3; ++k)
                M[3 * r + k] = fmaf(R[3 * r], C[k], fmaf(R[3 * r + 1], C[3 + k], R[3 * r + 2] * C[6 + k]));
        sincos_sel<FAST>(q[j], &s, &c);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            R[3 * r] = fmaf(c, M[3 * r], s * M[3 * r + 1]);
            R[3 * r + 1] = fmaf(c, M[3 * r + 1], -s * M[3 * r]);
            R[3 * r + 2] = M[3 * r + 2];
        }
    }
    const float* A = P.fk_AT;
    float r00 = fmaf(R[0], A[0], fmaf(R[1], A[3], R[2] * A[6]));
    float r10 = fmaf(R[3], A[0], fmaf(R[4], A[3], R[5] * A[6]));
    float r20 = fmaf(R[6], A[0], fmaf(R[7], A[3], R[8] * A[6]));
    float r21 = fmaf(R[6], A[1], fmaf(R[7], A[4], R[8] * A[7]));
    float r22 = fmaf(R[6], A[2], fmaf(R[7], A[5], R[8] * A[8]));
    pose[0] = p0;
    pose[1] = p1;
    pose[2] = p2;
    if constexpr (FAST) {
        pose[3] = atan2_fast(r21, r22);
        pose[4] = atan2_fast(-r20, sqrt_approx(fmaf(r00, r00, r10 * r10)));
        pose[5] = atan2_fast(r10, r00);
    } else {
        pose[3] = atan2f(r21, r22);
        pose[4] = atan2f(-r20, sqrtf(fmaf(r00, r00, r10 * r10)));
        pose[5] = atan2f(r10, r00);
    }
}

// pose_utils.py:15-26 -> (|pos_err|, |ori_err|) and the components
__device__ __forceinline__ void pose_error(const float* curr, const float* goal, float* pe, float* oe) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        pe[k] = goal[k] - curr[k];
        oe[k] = wrap_to_pi(goal[3 + k] - curr[3 + k]);
    }
}

// joint_limits.py:165-174
__device__ __forceinline__ float joint_margin(const KinEnvParams& P, float q, int i) {
    float nearest = fminf(q - P.joint_lower[i], P.joint_upper[i] - q);
    return clampf(2.0f * nearest * P.k_inv_span[i], 0.0f, 1.0f);
}

// FAST flavour: the normalised joint position 2 (q - lo) / span - 1 of a q inside its limits.  It is >= -1 (q - lo >= 0), but
// 2 k_inv_span (hi - lo) may round above 1 for limits whose span is not representable (up to 1 + 3e-5 for a short span far from
// zero): the upper clamp keeps qn <= 1 and so the margin 1 - |qn| >= 0, which the observation relies on without clipping again.
__device__ __forceinline__ float qnorm(const KinEnvParams& P, float q, int i) {
    return fminf(fmaf(2.0f * P.k_inv_span[i], q - P.joint_lower[i], -1.0f), 1.0f);
}

// AKE:432-444 -- thresholds always come from reward_config (ar_*), also in dock mode
__device__ __forceinline__ bool is_near_goal(const KinEnvParams& P, float pos, float ori) {
    return !(pos > P.ar_near_goal_pos_threshold_m) && !(P.ar_use_orientation_gate && ori > P.ar_near_goal_ori_threshold_rad);
}
__device__ __forceinline__ bool is_pre_near_goal(const KinEnvParams& P, float pos, float ori) {
    return !(pos > P.ar_pre_near_goal_pos_threshold_m) && !(P.ar_use_orientation_gate && ori > P.ar_near_goal_ori_threshold_rad);
}

// AKE:489-507
__device__ __forceinline__ float interp_control(float pos, float near_thr, float far_thr, float near_v, float far_v, float fallback) {
    if (near_thr <= 0.0f || far_thr <= near_thr) return fallback;
    if (pos <= near_thr) return near_v;
    if (pos >= far_thr) return far_v;
    float alpha = (pos - near_thr) / fmaxf(far_thr - near_thr, 1e-9f);
    return fmaf(alpha, far_v - near_v, near_v);
}

// FAST flavour: the division becomes a multiplication by a loop-invariant reciprocal
__device__ __forceinline__ float interp_control_fast(float pos, float near_thr, float far_thr, float near_v, float far_v, float fallback) {
    if (near_thr <= 0.0f || far_thr <= near_thr) return fallback;
    const float alpha = clampf((pos - near_thr) * rcp_approx(fmaxf(far_thr - near_thr, 1e-9f)), 0.0f, 1.0f);
    return fmaf(alpha, far_v - near_v, near_v);
}
template <int FAST>
__device__ __forceinline__ float interp_sel(float pos, float near_thr, float far_thr, float near_v, float far_v, float fallback) {
    if constexpr (FAST) return interp_control_fast(pos, near_thr, far_thr, near_v, far_v, fallback);
    else return interp_control(pos, near_thr, far_thr, near_v, far_v, fallback);
}

// AKE:425-430
__device__ __forceinline__ void capture_entry_metrics(EnvRegs& s) {
    float pe[3], oe[3];
    pose_error(s.ee, s.goal, pe, oe);
    s.entry[0] = norm3(pe[0], pe[1], pe[2]);
    s.entry[1] = norm3(oe[0], oe[1], oe[2]);
    s.entry[2] = norm7(s.pa);
    s.entry[3] = norm7(s.dq);
}

// AKE:102-211 (explicit-options branch): clip q, FK, goal, counters, entry metrics.
// goal_pose == nullptr -> goal pose = FK(clip(goal_q)); gq_out receives the stored goal_q.
__device__ __forceinline__ void reset_core(const KinEnvParams& P, EnvRegs& s, int mode, const float* iq, const float* idq,
                                           const float* ipa, const float* gq, const float* gpose, float* gq_out) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        s.q[i] = clampf(iq[i], P.joint_lower[i], P.joint_upper[i]);
        s.dq[i] = idq ? idq[i] : 0.0f;
        s.pa[i] = ipa ? ipa[i] : 0.0f;
    }
    fk_pose6(P, s.q, s.ee);
    if (gpose) {
#pragma unroll
        for (int k = 0; k < 6; ++k) s.goal[k] = gpose[k];
#pragma unroll
        for (int i = 0; i < NJ; ++i) gq_out[i] = gq ? gq[i] : 0.0f;
    } else {
#pragma unroll
        for (int i = 0; i < NJ; ++i) gq_out[i] = clampf(gq[i], P.joint_lower[i], P.joint_upper[i]);
        fk_pose6(P, gq_out, s.goal);
    }
    s.min_pos = CUDART_INF_F;
    s.step = 0;
    s.dwell = 0;
    s.entry_cnt = 0;
    s.drift_cnt = 0;
    s.flags = (s.flags & ~(KIN_FLAG_PRE_NEAR_HIT | KIN_FLAG_NEAR_HIT | (3u << KIN_FLAG_MODE_SHIFT))) |
              ((unsigned)mode << KIN_FLAG_MODE_SHIFT);
    capture_entry_metrics(s);
}

// observation_builder.py:29-94 in SB3's alphabetical flattening (SURVEY 8a row a6):
// dq 0:7 | goal_ori_err 7:10 | goal_pos_err 10:13 | joint_limit_margin 13:20 | mode_flag 20:24 |
// next_wp_ori_err 24:27 | next_wp_pos_err 27:30 | prev_action 30:37 | progress 37:40 | q 40:47 |
// task_type 47:50 | wp_ori_err 50:53 | wp_pos_err 53:56
// pe/oe = pose error of the CURRENT state, margin = per-joint limit margins (both already computed by the step)
__device__ __forceinline__ void build_obs_from(const KinEnvParams& P, const EnvRegs& s, int mode, const float* pe, const float* oe,
                                               const float* margin, float* o) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        o[i] = clampf(s.dq[i] * P.k_inv_delta_limit[i], -1.0f, 1.0f);
        o[13 + i] = margin[i];
        o[30 + i] = clampf(s.pa[i], -1.0f, 1.0f);
        o[40 + i] = clampf(fmaf(2.0f * P.k_inv_span[i], s.q[i] - P.joint_lower[i], -1.0f), -1.0f, 1.0f);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        o[7 + k] = clampf(oe[k] * P.k_inv_ori_err_scale, -1.0f, 1.0f);
        o[10 + k] = clampf(pe[k] * P.k_inv_pos_err_scale, -1.0f, 1.0f);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) o[20 + k] = (k == mode) ? 1.0f : 0.0f;
#pragma unroll
    for (int k = 24; k < 30; ++k) o[k] = 0.0f;
    o[37] = clampf((float)s.step * P.k_inv_episode_length, 0.0f, 1.0f);
    o[38] = clampf((float)s.dwell * P.k_inv_dwell_steps_target, 0.0f, 1.0f);
    o[39] = 0.0f;
    o[47] = 1.0f;
    o[48] = 0.0f;
    o[49] = 0.0f;
#pragma unroll
    for (int k = 50; k < 56; ++k) o[k] = 0.0f;
}

__device__ __forceinline__ void build_obs(const KinEnvParams& P, const EnvRegs& s, int mode, float* o) {
    float pe[3], oe[3], margin[NJ];
    pose_error(s.ee, s.goal, pe, oe);
#pragma unroll
    for (int i = 0; i < NJ; ++i) margin[i] = joint_margin(P, s.q[i], i);
    build_obs_from(P, s, mode, pe, oe, margin, o);
}

struct RewardIn {
    float prev_pos, prev_ori, curr_pos, curr_ori;
    float act_msq, act_dmsq;          // mean(a^2), mean((a - prev_a)^2)
    float action_norm, prev_action_norm;
    float dq_norm, prev_dq_norm, dq_change_l2;
    float margin_min;
    bool pre, pn, cn, success;
    int dwell, entry_cnt, drift_cnt;
};

__device__ __forceinline__ float ipowf(float base, int n) {
    float r = 1.0f;
    while (n > 0) {
        if (n & 1) r *= base;
        base *= base;
        n >>= 1;
    }
    return r;
}

#define KIN_C(idx, val)                \
    do {                               \
        if constexpr (COMP) c[idx] = (val); \
    } while (0)

// reward_approach.py:75-373; c[] (COMP only) in the reference's dict order.
template <bool COMP>
__device__ __forceinline__ float approach_reward(const KinEnvParams& P, const RewardIn& in, float* c) {
    const float prev_pos = in.prev_pos, curr_pos = in.curr_pos, prev_ori = in.prev_ori, curr_ori = in.curr_ori;
    const bool pre = in.pre, cn = in.cn, pn = in.pn;
    const int dwell = in.dwell;
    const float dpos = prev_pos - curr_pos, dori = prev_ori - curr_ori;
    const float regress = fmaxf(-dpos, 0.0f) + fmaxf(-dori, 0.0f);

    float position_progress = P.ar_position_progress_weight * dpos;
    float global_ori = P.ar_orientation_progress_weight * dori;
    float near_field_ori = pre ? P.ar_near_field_orientation_progress_weight * dori : 0.0f;
    float orientation_progress = global_ori + near_field_ori;
    float milestone = 0.0f;
    if (pre) {
#pragma unroll
        for (int i = 0; i < KIN_MAX_MILESTONES; ++i)
            if (i < P.ar_n_milestones && curr_ori <= P.ar_orientation_milestone_thresholds_rad[i]) milestone += P.ar_orientation_milestone_bonuses[i];
    }
    float nf_center = pre ? -P.ar_near_field_orientation_center_weight * curr_ori : 0.0f;
    float pre_near_goal = (pre && !cn) ? P.ar_pre_near_goal_bonus : 0.0f;
    float bonus_scale = 0.0f, near_goal = 0.0f;
    if (cn && !pn) {
        bonus_scale = ipowf(P.ar_near_goal_bonus_decay, max(in.entry_cnt - 1, 0));
        near_goal = P.ar_near_goal_bonus * bonus_scale;
    }
    float inner_progress = (pre && !cn) ? P.ar_pre_near_to_near_progress_weight * fmaxf(dpos, 0.0f) : 0.0f;
    float coarse_bonus = (pre && curr_ori <= P.ar_coarse_orientation_bonus_threshold_rad) ? P.ar_coarse_orientation_bonus : 0.0f;

    const bool ho_en = P.ar_handover_pos_threshold_m > 0.0f;
    const bool curr_ho = ho_en && curr_pos <= P.ar_handover_pos_threshold_m && (P.ar_handover_ori_threshold_rad <= 0.0f || curr_ori <= P.ar_handover_ori_threshold_rad);
    const bool prev_ho = ho_en && prev_pos <= P.ar_handover_pos_threshold_m && (P.ar_handover_ori_threshold_rad <= 0.0f || prev_ori <= P.ar_handover_ori_threshold_rad);
    float ho_bonus = (curr_ho && !prev_ho) ? P.ar_handover_bonus : 0.0f;
    float ho_ret = (curr_ho && prev_ho) ? P.ar_handover_retention_bonus : 0.0f;
    float ho_dwell = (curr_ho && dwell >= 2) ? P.ar_handover_dwell_bonus : 0.0f;
    float ho_leave = (prev_ho && !curr_ho) ? -P.ar_handover_leave_penalty : 0.0f;
    float ho_regr = (prev_ho || curr_ho) ? -P.ar_handover_regression_weight * regress : 0.0f;
    float dwell_b = (cn && dwell >= 2) ? P.ar_dwell_bonus : 0.0f;
    float drift_scale = fmaf(P.ar_drift_penalty_escalation_per_count, (float)max(in.drift_cnt - P.ar_drift_penalty_escalation_start, 0), 1.0f);
    float drift_pen = pn ? -(P.ar_drift_penalty_weight * drift_scale) * fmaxf(-dpos, 0.0f) : 0.0f;
    float leave_pen = (pn && !cn) ? -P.ar_near_goal_leave_penalty : 0.0f;
    const float an = in.action_norm, pan = in.prev_action_norm, dqn = in.dq_norm, pdqn = in.prev_dq_norm;

    const bool dc_en = P.ar_dock_coarse_ready_pos_threshold_m > 0.0f && P.ar_dock_coarse_ready_ori_threshold_rad > 0.0f;
    const bool curr_dc_pose = dc_en && curr_pos <= P.ar_dock_coarse_ready_pos_threshold_m && curr_ori <= P.ar_dock_coarse_ready_ori_threshold_rad;
    const bool prev_dc_pose = dc_en && prev_pos <= P.ar_dock_coarse_ready_pos_threshold_m && prev_ori <= P.ar_dock_coarse_ready_ori_threshold_rad;
    const bool curr_dc_motion = (P.ar_dock_coarse_ready_action_threshold <= 0.0f || an <= P.ar_dock_coarse_ready_action_threshold) &&
                                (P.ar_dock_coarse_ready_dq_threshold <= 0.0f || dqn <= P.ar_dock_coarse_ready_dq_threshold);
    const bool prev_dc_motion = (P.ar_dock_coarse_ready_action_threshold <= 0.0f || pan <= P.ar_dock_coarse_ready_action_threshold) &&
                                (P.ar_dock_coarse_ready_dq_threshold <= 0.0f || pdqn <= P.ar_dock_coarse_ready_dq_threshold);
    const bool curr_dc = curr_dc_pose && curr_dc_motion, prev_dc = prev_dc_pose && prev_dc_motion;

    const bool fr_en = P.ar_finisher_ready_pos_threshold_m > 0.0f && P.ar_finisher_ready_ori_threshold_rad > 0.0f;
    const bool curr_fr_pose = fr_en && curr_pos <= P.ar_finisher_ready_pos_threshold_m && curr_ori <= P.ar_finisher_ready_ori_threshold_rad;
    const bool prev_fr_pose = fr_en && prev_pos <= P.ar_finisher_ready_pos_threshold_m && prev_ori <= P.ar_finisher_ready_ori_threshold_rad;
    const bool curr_fr_motion = (P.ar_finisher_ready_action_threshold <= 0.0f || an <= P.ar_finisher_ready_action_threshold) &&
                                (P.ar_finisher_ready_dq_threshold <= 0.0f || dqn <= P.ar_finisher_ready_dq_threshold);
    const bool prev_fr_motion = (P.ar_finisher_ready_action_threshold <= 0.0f || pan <= P.ar_finisher_ready_action_threshold) &&
                                (P.ar_finisher_ready_dq_threshold <= 0.0f || pdqn <= P.ar_finisher_ready_dq_threshold);
    const bool curr_fr = curr_fr_pose && curr_fr_motion, prev_fr = prev_fr_pose && prev_fr_motion;

    const bool nh_en = P.ar_near_handoff_pos_threshold_m > 0.0f && P.ar_near_handoff_ori_threshold_rad > 0.0f;
    const bool nh = nh_en && curr_pos <= P.ar_near_handoff_pos_threshold_m && curr_ori <= P.ar_near_handoff_ori_threshold_rad;
    const bool prev_nh = nh_en && prev_pos <= P.ar_near_handoff_pos_threshold_m && prev_ori <= P.ar_near_handoff_ori_threshold_rad;

    float dc_bonus = (curr_dc && !prev_dc) ? P.ar_dock_coarse_ready_bonus : 0.0f;
    float dc_ret = (curr_dc && prev_dc) ? P.ar_dock_coarse_ready_retention_bonus : 0.0f;
    float dc_dwell = (curr_dc && dwell >= 2) ? P.ar_dock_coarse_ready_dwell_bonus : 0.0f;
    float dc_leave = (prev_dc && !curr_dc) ? -P.ar_dock_coarse_ready_leave_penalty : 0.0f;
    float dc_regr = (nh || prev_nh || curr_dc_pose || prev_dc_pose) ? -P.ar_dock_coarse_ready_regression_weight * regress : 0.0f;
    float fr_bonus = (curr_fr && !prev_fr) ? P.ar_finisher_ready_bonus : 0.0f;
    float fr_ret = (curr_fr && prev_fr) ? P.ar_finisher_ready_retention_bonus : 0.0f;
    float fr_dwell = (curr_fr && dwell >= 2) ? P.ar_finisher_ready_dwell_bonus : 0.0f;
    float fr_leave = (prev_fr && !curr_fr) ? -P.ar_finisher_ready_leave_penalty : 0.0f;
    float fr_regr = (nh || prev_nh || curr_fr_pose || prev_fr_pose) ? -P.ar_finisher_ready_regression_weight * regress : 0.0f;

    const bool nh_any = nh || curr_dc_pose || curr_fr_pose;
    float nh_action_pen = 0.0f, nh_dq_pen = 0.0f, nh_motion = 0.0f, nh_settle = 0.0f;
    if (nh_any) {
        nh_action_pen = -P.ar_near_handoff_action_weight * in.act_msq;
        nh_dq_pen = -P.ar_near_handoff_dq_weight * dqn;
        // python `a or b` fallbacks (reward_approach.py:253-254)
        float a_thr = P.ar_finisher_ready_action_threshold != 0.0f ? P.ar_finisher_ready_action_threshold : P.ar_dock_coarse_ready_action_threshold;
        float d_thr = P.ar_finisher_ready_dq_threshold != 0.0f ? P.ar_finisher_ready_dq_threshold : P.ar_dock_coarse_ready_dq_threshold;
        float a_clean = a_thr > 0.0f ? fmaxf(1.0f - qdiv(an, fmaxf(a_thr, 1e-9f)), 0.0f) : 0.0f;
        float d_clean = d_thr > 0.0f ? fmaxf(1.0f - qdiv(dqn, fmaxf(d_thr, 1e-9f)), 0.0f) : 0.0f;
        nh_motion = P.ar_near_handoff_motion_bonus_weight * (0.5f * a_clean + 0.5f * d_clean);
        nh_settle = P.ar_near_handoff_settle_bonus_weight * (0.5f * fmaxf(pan - an, 0.0f) + 0.5f * fmaxf(pdqn - dqn, 0.0f));
    }
    float same_step = (curr_pos < prev_pos && curr_ori < prev_ori && (pre || nh)) ? P.ar_same_step_alignment_bonus : 0.0f;
    float smooth_mult = (curr_ho || prev_ho) ? P.ar_handover_smoothness_multiplier : 1.0f;
    float smooth = smooth_mult * (-P.ar_action_magnitude_weight * in.act_msq - P.ar_action_delta_weight * in.act_dmsq);
    float jl_pen = -P.ar_joint_limit_penalty_weight * (fmaxf(0.25f - in.margin_min, 0.0f) / 0.25f);
    float succ = in.success ? P.ar_success_bonus : 0.0f;

    KIN_C(0, position_progress); KIN_C(1, global_ori); KIN_C(2, near_field_ori); KIN_C(3, orientation_progress);
    KIN_C(4, milestone); KIN_C(5, nf_center); KIN_C(6, pre_near_goal); KIN_C(7, near_goal); KIN_C(8, inner_progress);
    KIN_C(9, bonus_scale); KIN_C(10, coarse_bonus);
    KIN_C(11, ho_bonus); KIN_C(12, ho_ret); KIN_C(13, ho_dwell); KIN_C(14, ho_leave); KIN_C(15, ho_regr);
    KIN_C(16, dc_bonus); KIN_C(17, dc_ret); KIN_C(18, dc_dwell); KIN_C(19, dc_leave); KIN_C(20, dc_regr);
    KIN_C(21, fr_bonus); KIN_C(22, fr_ret); KIN_C(23, fr_dwell); KIN_C(24, fr_leave); KIN_C(25, fr_regr);
    KIN_C(26, nh_action_pen); KIN_C(27, nh_dq_pen); KIN_C(28, nh_motion); KIN_C(29, nh_settle);
    KIN_C(30, same_step); KIN_C(31, dwell_b); KIN_C(32, drift_pen); KIN_C(33, leave_pen); KIN_C(34, drift_scale);
    KIN_C(35, (float)in.entry_cnt); KIN_C(36, (float)in.drift_cnt); KIN_C(37, smooth); KIN_C(38, smooth_mult);
    KIN_C(39, jl_pen); KIN_C(40, succ); KIN_C(41, curr_pos); KIN_C(42, curr_ori); KIN_C(43, an); KIN_C(44, dqn);
    KIN_C(45, (float)dwell); KIN_C(46, pre ? 1.0f : 0.0f); KIN_C(47, cn ? 1.0f : 0.0f); KIN_C(48, curr_ho ? 1.0f : 0.0f);
    KIN_C(49, curr_dc ? 1.0f : 0.0f); KIN_C(50, curr_dc_pose ? 1.0f : 0.0f); KIN_C(51, curr_fr ? 1.0f : 0.0f);
    KIN_C(52, curr_fr_pose ? 1.0f : 0.0f); KIN_C(53, nh ? 1.0f : 0.0f);

    // same summation order as the reference (reward_approach.py:333-371)
    float r = position_progress;
    r += orientation_progress; r += milestone; r += nf_center; r += pre_near_goal; r += near_goal; r += inner_progress;
    r += coarse_bonus; r += ho_bonus; r += ho_ret; r += ho_dwell; r += ho_leave; r += ho_regr;
    r += dc_bonus; r += dc_ret; r += dc_dwell; r += dc_leave; r += dc_regr;
    r += fr_bonus; r += fr_ret; r += fr_dwell; r += fr_leave; r += fr_regr;
    r += nh_action_pen; r += nh_dq_pen; r += nh_motion; r += nh_settle; r += same_step; r += dwell_b; r += drift_pen;
    r += leave_pen; r += smooth; r += jl_pen; r += succ;
    return r;
}

// reward_dock.py:105-120
__device__ __forceinline__ float entry_penalty_scale(float pos, float near_thr, float far_thr, float near_m, float far_m) {
    if (near_thr <= 0.0f || far_thr <= near_thr) return 1.0f;
    if (pos <= near_thr) return near_m;
    if (pos >= far_thr) return far_m;
    float alpha = qdiv(pos - near_thr, fmaxf(far_thr - near_thr, 1e-9f));
    return fmaf(alpha, far_m - near_m, near_m);
}

// reward_dock.py:123-484; c[] (COMP only) in the reference's dict order.
template <bool COMP>
__device__ __forceinline__ float dock_reward(const KinEnvParams& P, const RewardIn& in, const float* entry, float* c) {
    const float prev_pos = in.prev_pos, curr_pos = in.curr_pos, prev_ori = in.prev_ori, curr_ori = in.curr_ori;
    const bool cn = in.cn, pn = in.pn;
    const int dwell = in.dwell;
    const float dqn = in.dq_norm;
    const float dpos = prev_pos - curr_pos, dori = prev_ori - curr_ori;
    const float worse_pos = fmaxf(-dpos, 0.0f), worse_ori = fmaxf(-dori, 0.0f);
    const float dm1 = (float)max(dwell - 1, 0);

    float position_progress = P.dr_position_progress_weight * dpos;
    float orientation_progress = P.dr_orientation_progress_weight * dori;
    float stay = cn ? P.dr_stay_in_zone_bonus : 0.0f;
    float dwell_bonus = cn ? P.dr_dwell_bonus * dm1 : 0.0f;
    float wr_bonus = cn ? P.dr_working_range_bonus : 0.0f;
    float wr_dwell = (cn && dwell >= P.dr_working_range_dwell_start) ? P.dr_working_range_dwell_bonus * (float)max(dwell - P.dr_working_range_dwell_start + 1, 0) : 0.0f;
    const float tp = P.dr_tight_pose_pos_threshold_m, to = P.dr_tight_pose_ori_threshold_rad;
    const bool curr_tight = curr_pos <= tp && curr_ori <= to;
    const bool prev_tight = prev_pos <= tp && prev_ori <= to;
    const float ns_pos = P.dr_near_strict_pos_threshold_m != 0.0f ? P.dr_near_strict_pos_threshold_m : tp * 2.0f;
    const float ns_ori = P.dr_near_strict_ori_threshold_rad != 0.0f ? P.dr_near_strict_ori_threshold_rad : to * 3.0f;
    const bool curr_ns = curr_pos <= ns_pos && curr_ori <= ns_ori;
    const bool prev_ns = prev_pos <= ns_pos && prev_ori <= ns_ori;
    const float r_p = qdiv(curr_pos, fmaxf(tp, 1e-9f)), r_o = qdiv(curr_ori, fmaxf(to, 1e-9f));
    float s_close = 0.8f * fmaxf(1.0f - r_p, 0.0f) + 0.2f * fmaxf(1.0f - r_o, 0.0f);
    s_close *= s_close;
    float tight_bonus = curr_tight ? P.dr_tight_pose_bonus : 0.0f;
    float tight_dwell = curr_tight ? P.dr_tight_pose_dwell_bonus * dm1 : 0.0f;
    float strict_leave = (prev_tight && !curr_tight) ? -P.dr_strict_pose_leave_penalty : 0.0f;
    float sc_reward = curr_tight ? P.dr_strict_center_reward_weight * s_close : 0.0f;
    float sc_pos_pen = P.dr_strict_center_position_weight > 0.0f ? -P.dr_strict_center_position_weight * (r_p * r_p) : 0.0f;
    float sc_ori_pen = P.dr_strict_center_orientation_weight > 0.0f ? -P.dr_strict_center_orientation_weight * (r_o * r_o) : 0.0f;
    const float action_rms = sqrtf(in.act_msq);
    float sc_small = 0.0f;
    if (curr_tight && P.dr_strict_center_small_action_bonus_weight > 0.0f && P.dr_strict_center_small_action_pos_radius_m > 0.0f &&
        P.dr_strict_center_small_action_ori_radius_rad > 0.0f && P.dr_strict_center_small_action_scale > 0.0f) {
        float cpc = fmaxf(1.0f - qdiv(curr_pos, P.dr_strict_center_small_action_pos_radius_m), 0.0f);
        float coc = fmaxf(1.0f - qdiv(curr_ori, P.dr_strict_center_small_action_ori_radius_rad), 0.0f);
        float cc = powf(0.8f * cpc + 0.2f * coc, P.dr_strict_center_small_action_power);
        float smallness = fmaxf(1.0f - qdiv(action_rms, P.dr_strict_center_small_action_scale), 0.0f);
        sc_small = P.dr_strict_center_small_action_bonus_weight * cc * smallness;
    }
    float sc_dwell = 0.0f;
    if (curr_tight && P.dr_strict_center_dwell_bonus_weight > 0.0f && dwell >= P.dr_strict_center_dwell_start) {
        float dscale = fmaf(P.dr_strict_center_dwell_escalation_per_step, (float)max(dwell - P.dr_strict_center_dwell_escalation_start, 0), 1.0f);
        sc_dwell = P.dr_strict_center_dwell_bonus_weight * s_close * dscale;
    }
    float tp_shape = P.dr_tight_position_shaping_radius_m > 0.0f
                         ? P.dr_tight_position_shaping_weight * fmaxf(1.0f - qdiv(curr_pos, fmaxf(P.dr_tight_position_shaping_radius_m, 1e-9f)), 0.0f) : 0.0f;
    float to_shape = P.dr_tight_orientation_shaping_radius_rad > 0.0f
                         ? P.dr_tight_orientation_shaping_weight * fmaxf(1.0f - qdiv(curr_ori, fmaxf(P.dr_tight_orientation_shaping_radius_rad, 1e-9f)), 0.0f) : 0.0f;
    float conv_pos = (P.dr_convergence_position_radius_m > 0.0f && fminf(prev_pos, curr_pos) <= P.dr_convergence_position_radius_m)
                         ? P.dr_convergence_position_progress_weight * dpos : 0.0f;
    float gate_scale = (P.dr_position_first_orientation_pos_threshold_m > 0.0f && curr_pos > P.dr_position_first_orientation_pos_threshold_m)
                           ? P.dr_position_first_orientation_pre_scale : 1.0f;
    float conv_ori = (P.dr_convergence_orientation_radius_rad > 0.0f && fminf(prev_ori, curr_ori) <= P.dr_convergence_orientation_radius_rad)
                         ? gate_scale * P.dr_convergence_orientation_progress_weight * dori : 0.0f;
    float leave_zone = (pn && !cn) ? -P.dr_leave_zone_penalty : 0.0f;
    float wr_exit = (pn && !cn) ? -P.dr_working_range_exit_penalty : 0.0f;
    float drift = -P.dr_drift_penalty_position_weight * worse_pos;
    drift += -P.dr_drift_penalty_orientation_weight * worse_ori;
    if (curr_tight || prev_tight) drift *= P.dr_strict_zone_drift_penalty_multiplier;

    const float action_l2 = in.action_norm;
    float e_scale = entry_penalty_scale(fmaxf(prev_pos, curr_pos), P.dr_entry_action_penalty_near_pos_threshold_m,
                                        P.dr_entry_action_penalty_far_pos_threshold_m, P.dr_entry_action_penalty_near_multiplier,
                                        P.dr_entry_action_penalty_far_multiplier);
    float smooth = -P.dr_action_magnitude_weight * in.act_msq;
    smooth += -P.dr_action_delta_weight * in.act_dmsq;
    if (curr_tight) smooth *= P.dr_strict_zone_action_penalty_multiplier;
    smooth *= e_scale;
    const float ad_rms = sqrtf(in.act_dmsq);
    float adv_pen = (P.dr_action_delta_violation_weight > 0.0f && P.dr_action_delta_violation_threshold > 0.0f)
                        ? -P.dr_action_delta_violation_weight * e_scale * fmaxf(ad_rms - P.dr_action_delta_violation_threshold, 0.0f) : 0.0f;
    float dqc_pen = (P.dr_delta_q_change_penalty_weight > 0.0f && P.dr_delta_q_change_penalty_threshold > 0.0f)
                        ? -P.dr_delta_q_change_penalty_weight * e_scale * fmaxf(in.dq_change_l2 - P.dr_delta_q_change_penalty_threshold, 0.0f) : 0.0f;
    const float entry_pos = entry[0], entry_ori = entry[1], entry_action = entry[2], entry_dq = entry[3];
    float preserve = 0.0f;
    if (P.dr_preserve_state_bonus > 0.0f && (curr_ns || curr_tight) && curr_pos <= entry_pos + P.dr_preserve_position_tolerance_m &&
        curr_ori <= entry_ori + P.dr_preserve_orientation_tolerance_rad)
        preserve = P.dr_preserve_state_bonus;
    float strict_hold = curr_tight ? P.dr_strict_hold_bonus * dm1 : 0.0f;
    float low_motion = 0.0f;
    if (P.dr_low_motion_bonus > 0.0f && curr_ns && (P.dr_low_motion_action_threshold <= 0.0f || action_l2 <= P.dr_low_motion_action_threshold) &&
        (P.dr_low_motion_dq_threshold <= 0.0f || dqn <= P.dr_low_motion_dq_threshold))
        low_motion = P.dr_low_motion_bonus;
    float tiny = 0.0f;
    if (P.dr_tiny_correction_bonus > 0.0f && curr_ns && !curr_tight && curr_pos <= prev_pos && curr_ori <= prev_ori &&
        (P.dr_tiny_correction_action_threshold <= 0.0f || action_l2 <= P.dr_tiny_correction_action_threshold))
        tiny = P.dr_tiny_correction_bonus;
    float worse = -P.dr_worse_than_entry_position_weight * fmaxf(curr_pos - entry_pos - P.dr_worse_than_entry_position_tolerance_m, 0.0f);
    worse += -P.dr_worse_than_entry_orientation_weight * fmaxf(curr_ori - entry_ori - P.dr_worse_than_entry_orientation_tolerance_rad, 0.0f);
    float ns_regr = 0.0f;
    if (curr_ns || prev_ns)
        ns_regr = -P.dr_near_strict_regression_multiplier * (P.dr_drift_penalty_position_weight * worse_pos + P.dr_drift_penalty_orientation_weight * worse_ori);
    float aggr = (P.dr_aggressive_action_weight > 0.0f && P.dr_aggressive_action_threshold > 0.0f)
                     ? -P.dr_aggressive_action_weight * (curr_ns ? P.dr_near_strict_action_penalty_multiplier : 1.0f) * fmaxf(action_l2 - P.dr_aggressive_action_threshold, 0.0f) : 0.0f;
    float dq_pen = (P.dr_dq_penalty_weight > 0.0f && P.dr_dq_penalty_threshold > 0.0f)
                       ? -P.dr_dq_penalty_weight * (curr_ns ? P.dr_near_strict_dq_penalty_multiplier : 1.0f) * fmaxf(dqn - P.dr_dq_penalty_threshold, 0.0f) : 0.0f;
    float jl_pen = -P.dr_joint_limit_penalty_weight * (fmaxf(0.25f - in.margin_min, 0.0f) / 0.25f);
    float succ = in.success ? P.dr_success_bonus : 0.0f;

    float b_outer = 0.0f, b_inner = 0.0f, b_dwell = 0.0f, b_outer_exit = 0.0f, b_inner_exit = 0.0f, b_break = 0.0f, b_drift = 0.0f;
    int zone = 0;
    if (P.dr_basin_outer_radius_m > 0.0f && P.dr_basin_inner_radius_m > 0.0f && P.dr_basin_dwell_radius_m > 0.0f) {
        const float outer_r = fmaxf(P.dr_basin_outer_radius_m, 1e-9f), inner_r = fmaxf(P.dr_basin_inner_radius_m, 1e-9f), dwell_r = fmaxf(P.dr_basin_dwell_radius_m, 1e-9f);
        const bool po = prev_pos <= outer_r, pi = prev_pos <= inner_r, pd = prev_pos <= dwell_r;
        const bool co = curr_pos <= outer_r, ci = curr_pos <= inner_r, cd = curr_pos <= dwell_r;
        zone = cd ? 3 : (ci ? 2 : (co ? 1 : 0));
        if (co) b_outer = P.dr_basin_outer_bonus * (1.0f + fmaxf(1.0f - qdiv(curr_pos, outer_r), 0.0f));
        if (ci) b_inner = P.dr_basin_inner_bonus * (1.0f + fmaxf(1.0f - qdiv(curr_pos, inner_r), 0.0f));
        if (cd) b_dwell = P.dr_basin_dwell_bonus * (1.0f + fmaxf(1.0f - qdiv(curr_pos, dwell_r), 0.0f));
        b_outer_exit = (po && !co) ? -P.dr_basin_outer_exit_penalty : 0.0f;
        b_inner_exit = (pi && !ci) ? -P.dr_basin_inner_exit_penalty : 0.0f;
        b_break = (pd && !cd) ? -P.dr_basin_dwell_break_penalty : 0.0f;
        b_drift = (po || co) ? -P.dr_basin_drift_penalty_weight * worse_pos : 0.0f;
    }

    KIN_C(0, position_progress); KIN_C(1, orientation_progress); KIN_C(2, stay); KIN_C(3, dwell_bonus); KIN_C(4, wr_bonus);
    KIN_C(5, wr_dwell); KIN_C(6, tight_bonus); KIN_C(7, tight_dwell); KIN_C(8, strict_leave); KIN_C(9, sc_reward);
    KIN_C(10, sc_pos_pen); KIN_C(11, sc_ori_pen); KIN_C(12, sc_small); KIN_C(13, sc_dwell); KIN_C(14, tp_shape);
    KIN_C(15, to_shape); KIN_C(16, conv_pos); KIN_C(17, conv_ori); KIN_C(18, gate_scale); KIN_C(19, e_scale);
    KIN_C(20, leave_zone); KIN_C(21, wr_exit); KIN_C(22, drift); KIN_C(23, smooth); KIN_C(24, adv_pen); KIN_C(25, dqc_pen);
    KIN_C(26, preserve); KIN_C(27, strict_hold); KIN_C(28, low_motion); KIN_C(29, tiny); KIN_C(30, worse); KIN_C(31, ns_regr);
    KIN_C(32, aggr); KIN_C(33, dq_pen); KIN_C(34, jl_pen); KIN_C(35, succ); KIN_C(36, b_outer); KIN_C(37, b_inner);
    KIN_C(38, b_dwell); KIN_C(39, b_outer_exit); KIN_C(40, b_inner_exit); KIN_C(41, b_break); KIN_C(42, b_drift);
    KIN_C(43, (float)zone); KIN_C(44, curr_pos); KIN_C(45, curr_ori); KIN_C(46, (float)dwell);
    KIN_C(47, curr_tight ? 1.0f : 0.0f); KIN_C(48, curr_ns ? 1.0f : 0.0f); KIN_C(49, entry_pos); KIN_C(50, entry_ori);
    KIN_C(51, entry_action); KIN_C(52, entry_dq); KIN_C(53, curr_pos - entry_pos); KIN_C(54, curr_ori - entry_ori);
    KIN_C(55, action_l2 - entry_action); KIN_C(56, dqn - entry_dq); KIN_C(57, (float)in.entry_cnt);
    KIN_C(58, (float)in.drift_cnt); KIN_C(59, cn ? 1.0f : 0.0f);

    // reference summation order (reward_dock.py:437-482)
    float r = position_progress;
    r += orientation_progress; r += stay; r += dwell_bonus; r += wr_bonus; r += wr_dwell; r += tight_bonus; r += tight_dwell;
    r += strict_leave; r += sc_reward; r += sc_pos_pen; r += sc_ori_pen; r += sc_small; r += sc_dwell; r += tp_shape;
    r += to_shape; r += conv_pos; r += conv_ori; r += leave_zone; r += wr_exit; r += drift; r += smooth; r += adv_pen;
    r += dqc_pen; r += preserve; r += strict_hold; r += low_motion; r += tiny; r += worse; r += ns_regr; r += aggr;
    r += dq_pen; r += jl_pen; r += succ; r += b_outer; r += b_inner; r += b_dwell; r += b_outer_exit; r += b_inner_exit;
    r += b_break; r += b_drift;
    return r;
}
#undef KIN_C

// AKE:213-365.  MODE: KIN_MODE_APPROACH / KIN_MODE_DOCK compile the other reward away;
// KIN_MODE_PER_ENV reads the mode bits of s.flags.  c[] receives info["reward_components"] (COMP only).
// FAST (tensor-core rollout / collection kernels): `out` must hold the previous step's (or the reset's) pos / ori on entry --
// they are the "previous" pose-error norms the reference recomputes from the cached ee pose -- and s.ee is not maintained.
template <int MODE, bool COMP, int FAST = 0>
__device__ __forceinline__ void step_core(const KinEnvParams& P, EnvRegs& s, const float* action_in, StepOut& out, float* c) {
    const int mode = (MODE == KIN_MODE_PER_ENV) ? (int)((s.flags >> KIN_FLAG_MODE_SHIFT) & 3u) : MODE;
    const bool dock = (mode == KIN_MODE_DOCK);
    float a[NJ];
#pragma unroll
    for (int i = 0; i < NJ; ++i) a[i] = clampf(action_in[i], -1.0f, 1.0f);
    float pe[3], oe[3];
    float prev_pos, prev_ori;
    if constexpr (FAST) {
        prev_pos = out.pos;
        prev_ori = out.ori;
    } else {
        pose_error(s.ee, s.goal, pe, oe);
        prev_pos = norm3(pe[0], pe[1], pe[2]);
        prev_ori = norm3(oe[0], oe[1], oe[2]);
    }
    float dock_limit = clampf(P.dock_residual_action_limit, 0.0f, 1.0f);
    float dqc_scale = fmaxf(P.dock_delta_q_change_limit_scale, 0.0f);
    if (dock) {
        dock_limit = clampf(interp_sel<FAST>(prev_pos, P.dock_dynamic_action_limit_near_pos_threshold_m, P.dock_dynamic_action_limit_far_pos_threshold_m,
                                           P.dock_dynamic_residual_action_limit_near, P.dock_dynamic_residual_action_limit_far,
                                           P.dock_residual_action_limit), 0.0f, 1.0f);
        dqc_scale = fmaxf(interp_sel<FAST>(prev_pos, P.dock_dynamic_action_limit_near_pos_threshold_m, P.dock_dynamic_action_limit_far_pos_threshold_m,
                                         P.dock_dynamic_delta_q_change_limit_scale_near, P.dock_dynamic_delta_q_change_limit_scale_far,
                                         P.dock_delta_q_change_limit_scale), 0.0f);
#pragma unroll
        for (int i = 0; i < NJ; ++i) a[i] = clampf(a[i], -dock_limit, dock_limit);
    }
    const bool prev_in_near = is_near_goal(P, prev_pos, prev_ori);
    float scale = P.action_delta_scale;
    if (dock) {
        if (P.dock_action_delta_scale > 0.0f) scale = P.dock_action_delta_scale;
    } else if (P.dynamic_action_delta_scale_enabled) {
        float mult = interp_sel<FAST>(prev_pos, P.dynamic_action_delta_scale_near_pos_threshold_m, P.dynamic_action_delta_scale_far_pos_threshold_m,
                                    P.dynamic_action_delta_scale_near_multiplier, P.dynamic_action_delta_scale_far_multiplier, 1.0f);
        scale = P.action_delta_scale * fmaxf(mult, 0.0f);
    }
    RewardIn in;
    in.prev_action_norm = FAST ? sqrt_approx(fmaf(s.pa[0], s.pa[0], fmaf(s.pa[1], s.pa[1], fmaf(s.pa[2], s.pa[2], fmaf(s.pa[3], s.pa[3], fmaf(s.pa[4], s.pa[4], fmaf(s.pa[5], s.pa[5], s.pa[6] * s.pa[6])))))))
                               : norm7(s.pa);
    in.prev_dq_norm = FAST ? sqrt_approx(fmaf(s.dq[0], s.dq[0], fmaf(s.dq[1], s.dq[1], fmaf(s.dq[2], s.dq[2], fmaf(s.dq[3], s.dq[3], fmaf(s.dq[4], s.dq[4], fmaf(s.dq[5], s.dq[5], s.dq[6] * s.dq[6])))))))
                           : norm7(s.dq);
    float msq = 0.0f, dmsq = 0.0f, dq_sq = 0.0f, dchg_sq = 0.0f, margin = 1.0f;
    float qn[NJ];
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        float max_dq = P.joint_delta_limit[i] * scale;
        float cmd = a[i] * max_dq;
        if (dock && dqc_scale > 0.0f) {
            float lim = max_dq * dqc_scale;
            cmd = s.dq[i] + clampf(cmd - s.dq[i], -lim, lim);
            cmd = clampf(cmd, -max_dq, max_dq);
        }
        qn[i] = clampf(s.q[i] + cmd, P.joint_lower[i], P.joint_upper[i]);
        float dqi = qn[i] - s.q[i];
        float dch = dqi - s.dq[i];
        float da = a[i] - s.pa[i];
        msq = fmaf(a[i], a[i], msq);
        dmsq = fmaf(da, da, dmsq);
        dq_sq = fmaf(dqi, dqi, dq_sq);
        dchg_sq = fmaf(dch, dch, dchg_sq);
        if constexpr (FAST) {   // margin = clip(2 min(q - lo, hi - q) / span, 0, 1) = 1 - |2 (q - lo) / span - 1| for q inside its limits
            out.qn[i] = qnorm(P, qn[i], i);
            out.margin[i] = 1.0f - fabsf(out.qn[i]);
        } else {
            out.margin[i] = joint_margin(P, qn[i], i);
        }
        margin = fminf(margin, out.margin[i]);
        s.q[i] = qn[i];
        s.dq[i] = dqi;
        s.pa[i] = a[i];
    }
    if constexpr (FAST) {
        float ee[6];
        fk_pose6<FAST>(P, s.q, ee);
        pose_error(ee, s.goal, pe, oe);
    } else {
        fk_pose6(P, s.q, s.ee);
        pose_error(s.ee, s.goal, pe, oe);
    }
    const float curr_pos = norm3_sel<FAST>(pe[0], pe[1], pe[2]), curr_ori = norm3_sel<FAST>(oe[0], oe[1], oe[2]);
    const bool curr_pre = is_pre_near_goal(P, curr_pos, curr_ori);
    const bool curr_near = is_near_goal(P, curr_pos, curr_ori);
    s.min_pos = fminf(s.min_pos, curr_pos);
    if (curr_pre) s.flags |= KIN_FLAG_PRE_NEAR_HIT;
    if (curr_near && !prev_in_near) s.entry_cnt += 1;
    s.dwell = curr_near ? s.dwell + 1 : 0;
    if (prev_in_near && curr_pos > prev_pos) s.drift_cnt += 1;

    // termination.py:20-57
    const int step_count = s.step + 1;
    bool terminated = false, truncated = false, success = false;
    unsigned reason = 0;
    const bool finite_ok = isfinite(curr_pos) && isfinite(curr_ori);
    const bool met = curr_pos <= P.term_success_pos_threshold_m && (!P.term_require_orientation || curr_ori <= P.term_success_ori_threshold_rad) &&
                     s.dwell >= P.term_success_dwell_steps;
    if (!finite_ok) {
        terminated = true;
        reason = 3;
    } else if (met) {
        success = true;
        if (P.term_terminate_on_success) {
            terminated = true;
            reason = 1;
        }
    }
    if (!terminated && step_count >= P.term_max_episode_steps) {
        truncated = true;
        reason = 2;
    }

    in.prev_pos = prev_pos; in.prev_ori = prev_ori; in.curr_pos = curr_pos; in.curr_ori = curr_ori;
    in.act_msq = msq * (1.0f / NJ); in.act_dmsq = dmsq * (1.0f / NJ);
    in.action_norm = sqrt_sel<FAST>(msq);
    in.dq_norm = sqrt_sel<FAST>(dq_sq);
    in.dq_change_l2 = sqrt_sel<FAST>(dchg_sq);
    in.margin_min = margin;
    in.pre = curr_pre; in.pn = prev_in_near; in.cn = curr_near; in.success = success;
    in.dwell = s.dwell; in.entry_cnt = s.entry_cnt; in.drift_cnt = s.drift_cnt;
    out.reward = dock ? dock_reward<COMP>(P, in, s.entry, c) : approach_reward<COMP>(P, in, c);

    s.step = step_count;
    if (curr_near) s.flags |= KIN_FLAG_NEAR_HIT;
    out.pos = curr_pos; out.ori = curr_ori;
#pragma unroll
    for (int k = 0; k < 3; ++k) { out.pe[k] = pe[k]; out.oe[k] = oe[k]; }
    out.action_l2 = in.action_norm; out.dq_l2 = in.dq_norm; out.dq_change_l2 = in.dq_change_l2;
    out.dock_limit = dock_limit; out.dqc_scale = dqc_scale; out.margin_min = margin;
    out.done = (terminated ? KIN_DONE_TERMINATED : 0u) | (truncated ? KIN_DONE_TRUNCATED : 0u) | (success ? KIN_DONE_SUCCESS : 0u) |
               (curr_pre ? KIN_DONE_PRE_NEAR : 0u) | (curr_near ? KIN_DONE_NEAR : 0u) | (reason << KIN_DONE_REASON_SHIFT);
}

}  // namespace kin
