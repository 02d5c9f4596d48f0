// kin_fast_env_harness.cu -- device test harness for the env arithmetic of kin_core.cuh / kin_tc16.cuh, in particular the FAST
// flavour that only the tensor-core rollout (kin_rollout_tc16.cu) runs.  It calls the library's own device functions; the tests
// (tests/test_gpu_fast_env_math.py) compile it with the library's nvcc flags into a temporary directory and load it with ctypes.
//
// Every pointer argument is a device pointer except the KinEnvParams, which are host structs passed on by value.  Each entry point
// launches, synchronises and returns the CUDA error code (0 = success).
#include <cuda_fp16.h>

#include "kin_tc16.cuh"

using namespace kin;

namespace {

constexpr int REC = 112;   // floats per (row, env) of the episode record; the layout is documented in the test module
constexpr int IREC = 8;    // ints per (row, env)

__global__ void scalar_kernel(int op, const float* x, const float* y, float* o0, float* o1, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float a = 0.0f, b = 0.0f;
    switch (op) {
        case 0: a = atan2_fast(y[i], x[i]); break;
        case 1: sincos_joint(x[i], &a, &b); break;
        case 2: sincos_joint_fast(x[i], &a, &b); break;
        case 3: sincos_sel<2>(x[i], &a, &b); break;
        case 4: a = wrap_to_pi(x[i]); break;
        case 5: a = sqrt_approx(x[i]); break;
        case 6: a = rcp_approx(x[i]); break;
        default: a = b = __int_as_float(0x7fc00000); break;
    }
    o0[i] = a;
    if (o1) o1[i] = b;
}

// args [n][6] = (pos, near_thr, far_thr, near_v, far_v, fallback) -> out [n][2] = (interp_control, interp_control_fast)
__global__ void interp_kernel(const float* args, float* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* a = args + 6 * i;
    out[2 * i] = interp_control(a[0], a[1], a[2], a[3], a[4], a[5]);
    out[2 * i + 1] = interp_control_fast(a[0], a[1], a[2], a[3], a[4], a[5]);
}

template <int FAST>
__global__ void fk_kernel(const __grid_constant__ KinEnvParams P, const float* q, float* pose, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float qq[NJ], p[6];
#pragma unroll
    for (int j = 0; j < NJ; ++j) qq[j] = q[(size_t)i * NJ + j];
    fk_pose6<FAST>(P, qq, p);
#pragma unroll
    for (int k = 0; k < 6; ++k) pose[(size_t)i * 6 + k] = p[k];
}

__global__ void dyn_col_kernel(int* out) {
    if (threadIdx.x < tc16::X_DYN) out[threadIdx.x] = tc16::dyn_col(threadIdx.x);
}

// One row of the episode record: the state the next step (and the policy) sees.
// rec: q 0:7 | dq 7:14 | prev_action 14:21 | pose 21:27 | pe 27:30 | oe 30:33 | pos, ori (as carried to the next step) 33:35 |
//      pos, ori recomputed from the pose 35:37 | margin 37:44 | qn 44:51 | reward 51 | min_pos 52 | action_l2 53 | dq_l2 54 |
//      observation 56:112 (FAST: the 36 obs_pack columns decoded; strict: build_obs_from, 56 columns)
// irec: done, step, dwell, entry_cnt, drift_cnt, flags, mode
template <int FAST>
__device__ void record(const KinEnvParams& P, const EnvRegs& s, const StepOut& so, int mode, bool primed, float* r, int* ir) {
    float ee[6], pe[3], oe[3];
    if (FAST && !primed) fk_pose6<FAST>(P, s.q, ee);   // a FAST step does not maintain s.ee
    else
        for (int k = 0; k < 6; ++k) ee[k] = s.ee[k];
    pose_error(ee, s.goal, pe, oe);
    for (int i = 0; i < NJ; ++i) {
        r[i] = s.q[i];
        r[7 + i] = s.dq[i];
        r[14 + i] = s.pa[i];
        r[37 + i] = so.margin[i];
        r[44 + i] = FAST ? so.qn[i] : 0.0f;
    }
    for (int k = 0; k < 6; ++k) r[21 + k] = ee[k];
    for (int k = 0; k < 3; ++k) { r[27 + k] = so.pe[k]; r[30 + k] = so.oe[k]; }
    r[33] = so.pos;
    r[34] = so.ori;
    if (FAST && !primed) { r[35] = norm3_sel<FAST>(pe[0], pe[1], pe[2]); r[36] = norm3_sel<FAST>(oe[0], oe[1], oe[2]); }
    else { r[35] = norm3(pe[0], pe[1], pe[2]); r[36] = norm3(oe[0], oe[1], oe[2]); }
    r[51] = so.reward;
    r[52] = s.min_pos;
    r[53] = so.action_l2;
    r[54] = so.dq_l2;
    r[55] = 0.0f;
    float* o = r + 56;
    if constexpr (FAST) {
        unsigned w[tc16::X_DYN / 2];
        tc16::obs_pack(P, s, so, w);
        for (int i = 0; i < tc16::X_DYN / 2; ++i) {
            const __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
            o[2 * i] = __low2float(h);
            o[2 * i + 1] = __high2float(h);
        }
        for (int k = tc16::X_DYN; k < KIN_OBS_DIM; ++k) o[k] = 0.0f;
    } else {
        build_obs_from(P, s, mode, so.pe, so.oe, so.margin, o);
    }
    ir[0] = (int)so.done; ir[1] = s.step; ir[2] = s.dwell; ir[3] = s.entry_cnt; ir[4] = s.drift_cnt; ir[5] = (int)s.flags; ir[6] = mode; ir[7] = 0;
}

// What the tensor-core rollout does after a reset: FAST primes the carried StepOut (prime_step_out); the strict flavour's StepOut
// fields are filled here from the reset state only so that the record has the same shape.
template <int FAST>
__device__ void prime(const KinEnvParams& P, const EnvRegs& s, StepOut& so) {
    if constexpr (FAST) {
        tc16::prime_step_out(P, s, so);
    } else {
        so.done = 0u;
        pose_error(s.ee, s.goal, so.pe, so.oe);
        so.pos = norm3(so.pe[0], so.pe[1], so.pe[2]);
        so.ori = norm3(so.oe[0], so.oe[1], so.oe[2]);
        so.dq_l2 = 0.0f;
        for (int i = 0; i < NJ; ++i) { so.margin[i] = joint_margin(P, s.q[i], i); so.qn[i] = 0.0f; }
    }
    so.reward = 0.0f;
    so.action_l2 = 0.0f;
}

// reset_core (mode), prime, T steps of step_core<mode, FAST> over the action tape [T][n][7].  handoff in [1, T): after step
// `handoff` the episode is re-reset in dock mode with P2 from its current q / dq / prev_action and goal pose, as the rollout's
// finisher phase does; the primed state of that re-reset is record row T + 1.  Records: [T + 2][n][REC] / [IREC].
template <int FAST>
__global__ void episode_kernel(const __grid_constant__ KinEnvParams P, const __grid_constant__ KinEnvParams P2, int mode, int handoff,
                               const float* iq, const float* idq, const float* ipa, const float* gq, const float* gp, const float* act,
                               int T, int n, float* rec, int* irec) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    auto row = [&](int t) { return rec + ((size_t)t * n + e) * REC; };
    auto irow = [&](int t) { return irec + ((size_t)t * n + e) * IREC; };
    EnvRegs s;
    s.flags = 0u;
    float goal_q[NJ];
    reset_core(P, s, mode, iq + (size_t)e * NJ, idq ? idq + (size_t)e * NJ : nullptr, ipa ? ipa + (size_t)e * NJ : nullptr,
               gq + (size_t)e * NJ, gp ? gp + (size_t)e * 6 : nullptr, goal_q);
    StepOut so;
    prime<FAST>(P, s, so);
    record<FAST>(P, s, so, mode, true, row(0), irow(0));
    bool second = false;
    for (int t = 1; t <= T; ++t) {
        const KinEnvParams& Q = second ? P2 : P;
        const float* a = act + ((size_t)(t - 1) * n + e) * NJ;
        float av[NJ];
        for (int i = 0; i < NJ; ++i) av[i] = a[i];
        if (mode == KIN_MODE_DOCK) step_core<KIN_MODE_DOCK, false, FAST>(Q, s, av, so, nullptr);
        else step_core<KIN_MODE_APPROACH, false, FAST>(Q, s, av, so, nullptr);
        record<FAST>(Q, s, so, mode, false, row(t), irow(t));
        if (t == handoff) {
            float r_iq[NJ], r_idq[NJ], r_ipa[NJ], gq_out[NJ], r_gp[6];
            for (int i = 0; i < NJ; ++i) { r_iq[i] = s.q[i]; r_idq[i] = s.dq[i]; r_ipa[i] = s.pa[i]; }
            for (int k = 0; k < 6; ++k) r_gp[k] = s.goal[k];
            mode = KIN_MODE_DOCK;
            second = true;
            reset_core(P2, s, KIN_MODE_DOCK, r_iq, r_idq, r_ipa, goal_q, r_gp, gq_out);
            prime<FAST>(P2, s, so);
            record<FAST>(P2, s, so, mode, true, row(T + 1), irow(T + 1));
        }
    }
}

int finish() {
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    return (int)e;
}

constexpr int BLK = 128;
int blocks(int n) { return (n + BLK - 1) / BLK; }

}  // namespace

extern "C" {

int kfh_rec_sizes(int* rec, int* irec) {
    *rec = REC;
    *irec = IREC;
    return 0;
}

int kfh_scalar(int op, const float* x, const float* y, float* o0, float* o1, int n) {
    scalar_kernel<<<blocks(n), BLK>>>(op, x, y, o0, o1, n);
    return finish();
}

int kfh_interp(const float* args, float* out, int n) {
    interp_kernel<<<blocks(n), BLK>>>(args, out, n);
    return finish();
}

int kfh_fk(const KinEnvParams* P, int fast, const float* q, float* pose, int n) {
    if (fast == 0) fk_kernel<0><<<blocks(n), BLK>>>(*P, q, pose, n);
    else if (fast == 1) fk_kernel<1><<<blocks(n), BLK>>>(*P, q, pose, n);
    else fk_kernel<2><<<blocks(n), BLK>>>(*P, q, pose, n);
    return finish();
}

int kfh_dyn_col(int* out) {
    dyn_col_kernel<<<1, 64>>>(out);
    return finish();
}

int kfh_episode(const KinEnvParams* P, const KinEnvParams* P2, int fast, int mode, int handoff, const float* iq, const float* idq,
                const float* ipa, const float* gq, const float* gp, const float* act, int T, int n, float* rec, int* irec) {
    const KinEnvParams& Q2 = P2 ? *P2 : *P;
    if (fast == 0) episode_kernel<0><<<blocks(n), BLK>>>(*P, Q2, mode, handoff, iq, idq, ipa, gq, gp, act, T, n, rec, irec);
    else if (fast == 1) episode_kernel<1><<<blocks(n), BLK>>>(*P, Q2, mode, handoff, iq, idq, ipa, gq, gp, act, T, n, rec, irec);
    else episode_kernel<2><<<blocks(n), BLK>>>(*P, Q2, mode, handoff, iq, idq, ipa, gq, gp, act, T, n, rec, irec);
    return finish();
}

}  // extern "C"
