// kin_route.cu -- the dense holder-route wrappers on the GPU: RouteKinematicEnv / RouteSequenceKinematicEnv step with
// the in-episode waypoint advance, and the fused sequential route probe with the 80-input route policy in the loop.
//
// The route wrapper's bookkeeping is per-lane predicated logic on top of step_core: route-ready (5 thresholds), ready
// streak, success, target advance (goal swap + entry metrics), nearest-waypoint scan over the whole route (table of
// waypoint joint vectors staged in shared memory, warp-uniform reads), 13-term route reward, +24 observation floats.
// Two things the reference recomputes every step are reused instead: FK(prev_q) is the cached ee pose and FK(curr_q)
// is the pose the base step just produced (route/route_env.py:127,137 call FK a second and third time).
//
// Replaces route/route_env.py:49-212, route/route_sequence_env.py:96-278, route/reward_route.py:36-143,
// route/route_observation.py:31-61, eval/eval_route_curriculum.py:55-136,188-218 (paths under kinematic_phase1/).
#include "kin_internal.h"
#include "kin_mlp.cuh"
#include "kin_route_core.cuh"
#include "kin_state.cuh"

namespace kin {

// AUTORESET: a slot whose step finishes its episode (terminated or truncated) is re-seeded in the same launch with the draw
// kin_route_reset_sampled makes for it, Philox(seed, env, state[KIN_ROW_EPISODE] + 1), and the counter is written back.
// reward / done / raux / rcomp describe the step just taken; terminal_obs (nullable) receives the finished episode's last
// observation, obs the next episode's first.  The trailing parameters are unused by the AUTORESET = false instances.
template <bool SEQ, bool COMP, bool AUTORESET>
__global__ void __launch_bounds__(RT_THREADS)
kin_route_step_kernel(const __grid_constant__ KinEnvParams P, RouteView R, float* __restrict__ state, int stride, int n,
                      const float* __restrict__ action, float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ done,
                      float* __restrict__ raux, float* __restrict__ rcomp, int reset_streak, const __grid_constant__ KinRouteResetParams C,
                      uint64_t seed, float* __restrict__ terminal_obs) {
    extern __shared__ __align__(128) float smem[];
    float* tiles = smem;                                        // [RT_WARPS][ROBS_TILE_FLOATS]
    float* q_table = smem + RT_WARPS * ROBS_TILE_FLOATS;        // [min(n_wp, 1024)][7]
    load_q_table(q_table, R, threadIdx.x, RT_THREADS);
    __syncthreads();
    const int lane = threadIdx.x & (WARP - 1), warp = threadIdx.x >> 5;
    const int env0 = (blockIdx.x * RT_WARPS + warp) * WARP;
    if (env0 >= n) return;
    const int env = env0 + lane;
    const bool active = env < n;
    const int envc = active ? env : n - 1;
    float* tile = tiles + warp * ROBS_TILE_FLOATS;
    float a[NJ];
    load_action_tile(action, env0, n, tile, lane, a);
    EnvRegs s;
    load_env<true>(state, stride, envc, s);
    RouteRegs rr;
    {
        const unsigned r0 = ld_row_u(state, stride, KIN_ROW_ROUTE, envc), r1 = ld_row_u(state, stride, KIN_ROW_ROUTE2, envc);
        rr.index = (int)(r0 & 0xffffu); rr.streak = (int)(r0 >> 16); rr.last = (int)(r1 & 0xffffu); rr.completed = (int)(r1 >> 16);
    }
    StepOut so;
    RouteOut ro;
    float rc[COMP ? 17 : 1];
    const float* table = R.n <= ROUTE_MAX_SMEM_WP ? q_table : R.q;
    route_step_core<SEQ, COMP>(P, R, table, s, rr, a, reset_streak != 0, so, ro, rc);
    const bool finished = AUTORESET && active && (ro.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED));
    if (active) {
        if (!finished) {   // a finished slot's state rows are written by its reset below
            store_env_step(state, stride, env, s);
            if (SEQ) {   // the advance rewrote goal pose + entry metrics
#pragma unroll
                for (int k = 0; k < 6; ++k) st_row(state, stride, KIN_ROW_GOAL_POSE + k, env, s.goal[k]);
#pragma unroll
                for (int k = 0; k < 4; ++k) st_row(state, stride, KIN_ROW_ENTRY + k, env, s.entry[k]);
                const float* gq = R.q + (size_t)wp_clamp(R, rr.index) * NJ;
#pragma unroll
                for (int i = 0; i < NJ; ++i) st_row(state, stride, KIN_ROW_GOAL_Q + i, env, __ldg(gq + i));
            }
            st_row_u(state, stride, KIN_ROW_ROUTE, env, (unsigned)rr.index | ((unsigned)min(rr.streak, 0xffff) << 16));
            st_row_u(state, stride, KIN_ROW_ROUTE2, env, (unsigned)rr.last | ((unsigned)min(rr.completed, 0xffff) << 16));
        }
        reward[env] = ro.reward;
        done[env] = (uint8_t)(ro.done | (finished ? KIN_DONE_AUTORESET : 0u));
        if (raux) {
            raux[(size_t)KIN_RAUX_Q_ERR * stride + env] = ro.q_err;
            raux[(size_t)KIN_RAUX_NEAREST * stride + env] = ro.nearest;
            raux[(size_t)KIN_RAUX_POS_ERR * stride + env] = so.pos;
            raux[(size_t)KIN_RAUX_ORI_ERR * stride + env] = so.ori;
            raux[(size_t)KIN_RAUX_FLAGS * stride + env] = __uint_as_float(ro.flags);
            raux[(size_t)KIN_RAUX_ROUTE_INDEX * stride + env] = __uint_as_float((unsigned)rr.index);
            raux[(size_t)KIN_RAUX_STREAK * stride + env] = __uint_as_float((unsigned)rr.streak);
            raux[(size_t)KIN_RAUX_COMPLETED * stride + env] = __uint_as_float((unsigned)rr.completed);
        }
        if (COMP) {
#pragma unroll
            for (int k = 0; k < 17; ++k) rcomp[(size_t)k * stride + env] = rc[k];
        }
    }
    float o56[OBS], o[ROBS];
    if (AUTORESET && __ballot_sync(0xffffffffu, finished)) {
        if (terminal_obs) {   // the whole warp's pre-reset rows through the tile; only the finished rows are meaningful to callers
            build_obs(P, s, KIN_MODE_APPROACH, o56);
            build_route_obs(P, R, s, rr.index, o56, o);
            stage_route_obs_row(tile, lane, o);
            bulk_store_tile(terminal_obs + (size_t)env0 * ROBS, tile, min(WARP, n - env0) * ROBS * 4, lane);
            bulk_store_wait_read(lane);
        }
        if (finished) {
            const unsigned episode = ld_row_u(state, stride, KIN_ROW_EPISODE, env) + 1u;
            Philox rng(seed, (uint32_t)env, episode);
            float gq[NJ];
            sample_route_reset_dev(P, R, C, rng, s, rr, gq);
            store_env_reset(state, stride, env, s, gq);
            st_row_u(state, stride, KIN_ROW_ROUTE, env, (unsigned)rr.index);
            st_row_u(state, stride, KIN_ROW_ROUTE2, env, (unsigned)rr.last);
            st_row_u(state, stride, KIN_ROW_EPISODE, env, episode);
        }
    }
    build_obs(P, s, KIN_MODE_APPROACH, o56);   // after an advance the goal changed, so recompute the goal errors
    build_route_obs(P, R, s, rr.index, o56, o);
    stage_route_obs_row(tile, lane, o);
    bulk_store_tile(obs + (size_t)env0 * ROBS, tile, min(WARP, n - env0) * ROBS * 4, lane);
    bulk_store_wait_read(lane);
}

__global__ void __launch_bounds__(128)
kin_route_reset_kernel(const __grid_constant__ KinEnvParams P, RouteView R, float* __restrict__ state, int stride, int n_envs,
                       const int* __restrict__ env_ids, int n_reset, const int* __restrict__ route_index, const int* __restrict__ start_index,
                       const int* __restrict__ last_index, const float* __restrict__ iq, const float* __restrict__ idq,
                       const float* __restrict__ ipa, float* __restrict__ obs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_reset) return;
    const int env = env_ids ? env_ids[i] : i;
    if (env < 0 || env >= n_envs) return;
    const int ri = route_index[i];
    if (ri < 0) return;           // masked reset: a negative waypoint leaves this slot (state and observation row) untouched
    const int st = start_index ? start_index[i] : max(ri - 1, 0);
    float r_iq[NJ], r_idq[NJ], r_ipa[NJ], r_gq[NJ], gq_out[NJ];
    const float* sq = R.q + (size_t)wp_clamp(R, st) * NJ;
    const float* gq = R.q + (size_t)wp_clamp(R, ri) * NJ;
#pragma unroll
    for (int k = 0; k < NJ; ++k) {
        r_iq[k] = iq ? iq[(size_t)i * NJ + k] : __ldg(sq + k);
        r_idq[k] = idq ? idq[(size_t)i * NJ + k] : 0.0f;
        r_ipa[k] = ipa ? ipa[(size_t)i * NJ + k] : 0.0f;
        r_gq[k] = __ldg(gq + k);
    }
    EnvRegs s;
    s.flags = 0u;
    reset_core(P, s, KIN_MODE_APPROACH, r_iq, r_idq, r_ipa, r_gq, nullptr, gq_out);
    store_env_reset(state, stride, env, s, gq_out);
    st_row_u(state, stride, KIN_ROW_ROUTE, env, (unsigned)ri);
    st_row_u(state, stride, KIN_ROW_ROUTE2, env, (unsigned)(last_index ? last_index[i] : ri));
    if (obs) {
        float o56[OBS], o[ROBS];
        build_obs(P, s, KIN_MODE_APPROACH, o56);
        build_route_obs(P, R, s, ri, o56, o);
        float4* dst = reinterpret_cast<float4*>(obs + (size_t)i * ROBS);
#pragma unroll
        for (int k = 0; k < ROBS / 4; ++k) dst[k] = make_float4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
    }
}

// sample_route_reset + reset for the finished slots (route/route_reset_samplers.py:43-117, route/route_env.py:60-97)
__global__ void __launch_bounds__(128)
kin_route_reset_sampled_kernel(const __grid_constant__ KinEnvParams P, RouteView R, const __grid_constant__ KinRouteResetParams C,
                               float* __restrict__ state, int stride, int n_envs, const uint8_t* __restrict__ done, uint64_t seed,
                               uint32_t counter, float* __restrict__ obs) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= n_envs) return;
    if (done && !(done[env] & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED))) return;
    Philox rng(seed, (uint32_t)env, counter);
    EnvRegs s;
    RouteRegs rr;
    float gq_out[NJ];
    sample_route_reset_dev(P, R, C, rng, s, rr, gq_out);
    const int ri = rr.index, last = rr.last;
    store_env_reset(state, stride, env, s, gq_out);
    st_row_u(state, stride, KIN_ROW_ROUTE, env, (unsigned)ri);
    st_row_u(state, stride, KIN_ROW_ROUTE2, env, (unsigned)last);
    if (obs) {
        float o56[OBS], o[ROBS];
        build_obs(P, s, KIN_MODE_APPROACH, o56);
        build_route_obs(P, R, s, ri, o56, o);
        float4* dst = reinterpret_cast<float4*>(obs + (size_t)env * ROBS);
#pragma unroll
        for (int k = 0; k < ROBS / 4; ++k) dst[k] = make_float4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
    }
}

struct DevPolicyR {
    const float *w0, *b0, *w1, *b1, *wo, *bo;
};

// evaluate_sequential_route for one replica per thread, policy in the loop (strict fp32 MLP).  DETAIL: the first detail_n replicas also
// write the per-waypoint row of _roll_one (eval_route_curriculum.py:111-131), KIN_ROUTE_ROW_FIELDS floats each
template <bool DETAIL>
__global__ void __launch_bounds__(RT_THREADS)
kin_route_probe_kernel(const __grid_constant__ KinEnvParams P, RouteView R, DevPolicyR pol, const float* __restrict__ start_q, int start_index,
                       int end_index, int n, int* __restrict__ prefix_out, uint32_t* __restrict__ success_bits, int words,
                       unsigned long long* __restrict__ env_steps, float* __restrict__ rows, int detail_n) {
    extern __shared__ __align__(16) float smem[];
    float* sw = smem;
    float* scratch = smem + MlpSmem<ROBS>::FLOATS + threadIdx.x;
    const int tid = threadIdx.x;
    const int rep = blockIdx.x * RT_THREADS + tid;
    const bool active = rep < n;
    const int repc = active ? rep : n - 1;
    mlp_load_smem<ROBS>(sw, pol.w0, pol.b0, pol.w1, pol.b1, pol.wo, pol.bo, ACT, tid, RT_THREADS);
    __syncthreads();
    float cq[NJ], cdq[NJ], cpa[NJ];
    {
        const float* q0 = start_q ? start_q + (size_t)repc * NJ : R.q + (size_t)wp_clamp(R, max(start_index - 1, 0)) * NJ;
#pragma unroll
        for (int i = 0; i < NJ; ++i) { cq[i] = q0[i]; cdq[i] = 0.0f; cpa[i] = 0.0f; }
    }
    const int final_end = min(end_index, R.n - 1);
    int prefix = 0;
    bool broken = false;
    unsigned long long steps = 0;
    unsigned word = 0u;
    for (int idx = start_index; idx <= final_end; ++idx) {
        EnvRegs s;
        s.flags = 0u;
        float gq_out[NJ], gq[NJ];
        const float* g = R.q + (size_t)wp_clamp(R, idx) * NJ;
#pragma unroll
        for (int i = 0; i < NJ; ++i) gq[i] = __ldg(g + i);
        reset_core(P, s, KIN_MODE_APPROACH, cq, cdq, cpa, gq, nullptr, gq_out);
        RouteRegs rr{idx, 0, idx, 0};
        RouteOut ro;
        ro.done = 0u;
        ro.q_err = 0.0f;
        bool running = active;
        // _roll_one's running minima start from the reset state (eval_route_curriculum.py:88-90)
        float d_min_pos = s.entry[0], d_min_ori = s.entry[1], d_min_q = dist7(gq, cq), d_pos = s.entry[0], d_ori = s.entry[1], d_act = 0.0f, d_dq = 0.0f;
        int d_first = -1, d_max_streak = 0, d_steps = 0;
        while (__any_sync(0xffffffffu, running)) {
            if (running) {
                float o56[OBS], o[ROBS], act[ACT];
                StepOut so;
                build_obs(P, s, KIN_MODE_APPROACH, o56);
                build_route_obs(P, R, s, rr.index, o56, o);
                mlp_forward<ROBS, ACT, RT_THREADS>(sw, o, act, scratch);
#pragma unroll
                for (int i = 0; i < ACT; ++i) act[i] = clampf(act[i], -1.0f, 1.0f);
                route_step_core<false, false>(P, R, nullptr, s, rr, act, true, so, ro, nullptr);   // eval needs no off-route term
                steps += 1;
                running = !(ro.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED));
                if (DETAIL) {
                    d_steps += 1;
                    d_pos = so.pos; d_ori = so.ori; d_act = so.action_l2; d_dq = so.dq_l2;
                    d_min_pos = fminf(d_min_pos, so.pos); d_min_ori = fminf(d_min_ori, so.ori); d_min_q = fminf(d_min_q, ro.q_err);
                    if ((ro.flags & 1u) && d_first < 0) d_first = d_steps;
                    d_max_streak = max(d_max_streak, rr.streak);
                }
            }
        }
        const bool ok = (ro.done & KIN_DONE_SUCCESS) != 0;
        if (DETAIL && active && rep < detail_n) {
            float* row = rows + ((size_t)rep * (final_end - start_index + 1) + (idx - start_index)) * KIN_ROUTE_ROW_FIELDS;
            row[KIN_ROUTE_ROW_SUCCESS] = ok ? 1.0f : 0.0f;
            row[KIN_ROUTE_ROW_READY_HIT] = d_first >= 0 ? 1.0f : 0.0f;
            row[KIN_ROUTE_ROW_READY_DWELL] = d_max_streak >= P.term_success_dwell_steps ? 1.0f : 0.0f;
            row[KIN_ROUTE_ROW_FIRST_READY_STEP] = (float)d_first;
            row[KIN_ROUTE_ROW_MAX_READY_STREAK] = (float)d_max_streak;
            row[KIN_ROUTE_ROW_STEPS] = (float)d_steps;
            row[KIN_ROUTE_ROW_FINAL_POS] = d_pos;
            row[KIN_ROUTE_ROW_FINAL_ORI] = d_ori;
            row[KIN_ROUTE_ROW_FINAL_Q_ERR] = ro.q_err;
            row[KIN_ROUTE_ROW_MIN_POS] = d_min_pos;
            row[KIN_ROUTE_ROW_MIN_ORI] = d_min_ori;
            row[KIN_ROUTE_ROW_MIN_Q_ERR] = d_min_q;
            row[KIN_ROUTE_ROW_FINAL_ACTION_L2] = d_act;
            row[KIN_ROUTE_ROW_FINAL_DQ_L2] = d_dq;
        }
        if (ok && !broken) prefix += 1; else broken = true;
        const int k = idx - start_index;
        if (ok) word |= 1u << (k & 31);
        if (success_bits && active && ((k & 31) == 31 || idx == final_end)) {
            success_bits[(size_t)rep * words + (k >> 5)] = word;
            word = 0u;
        }
#pragma unroll
        for (int i = 0; i < NJ; ++i) { cq[i] = s.q[i]; cdq[i] = s.dq[i]; cpa[i] = s.pa[i]; }
    }
    if (active) prefix_out[rep] = prefix;
    if (env_steps) {
        unsigned long long mine = active ? steps : 0ull;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
        if ((tid & 31) == 0 && mine) atomicAdd(env_steps, mine);
    }
}


}  // namespace kin

using namespace kin;

// every reset mode's target-waypoint range lies inside the route
static bool reset_ranges_ok(const KinRouteResetParams& C, int n_waypoints) {
    for (int m = 0; m < 5; ++m)
        if (C.index_lo[m] < 0 || C.index_hi[m] < C.index_lo[m] || C.index_hi[m] >= n_waypoints) return false;
    return true;
}

extern "C" int kin_route_reset(void* handle, const KinRouteTable* host_route, float* state, int stride, int n_envs, const int* env_ids,
                               int n_reset, const int* route_index, const int* start_route_index, const int* last_route_index,
                               const float* initial_q, const float* initial_dq, const float* initial_prev_action, float* obs, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h || !route_ok(host_route)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset: bad handle or route table");
    if (!state || !route_index || n_envs <= 0 || stride < n_envs || (stride % 32) != 0 || n_reset < 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset: bad sizes");
    if (obs && ((uintptr_t)obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset: obs must be 16-byte aligned");
    if (n_reset == 0) return KIN_OK;
    kin_route_reset_kernel<<<(n_reset + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->params, view_of(host_route), state, stride, n_envs, env_ids, n_reset,
                                                                                    route_index, start_route_index, last_route_index, initial_q,
                                                                                    initial_dq, initial_prev_action, obs);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_route_reset");
}

extern "C" int kin_route_reset_sampled(void* handle, const KinRouteTable* host_route, const KinRouteResetParams* host_reset, float* state, int stride,
                                       int n_envs, const uint8_t* done, uint64_t seed, uint32_t counter, float* obs, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h || !route_ok(host_route) || !host_reset) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset_sampled: bad handle, route table or reset parameters");
    if (!state || n_envs <= 0 || stride < n_envs || (stride % 32) != 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset_sampled: bad sizes");
    if (obs && ((uintptr_t)obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset_sampled: obs must be 16-byte aligned");
    if (!reset_ranges_ok(*host_reset, host_route->n_waypoints)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_reset_sampled: waypoint range outside the route");
    kin_route_reset_sampled_kernel<<<(n_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->params, view_of(host_route), *host_reset, state, stride, n_envs,
                                                                                          done, seed, counter, obs);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_route_reset_sampled");
}

// argument checks + launch shared by kin_route_step and kin_route_step_autoreset (C is only read by the AUTORESET instances)
#define KIN_RMSG(what) (AUTORESET ? "kin_route_step_autoreset: " what : "kin_route_step: " what)
template <bool AUTORESET>
static int launch_route_step(void* handle, const KinRouteTable* host_route, const KinRouteResetParams& C, float* state,
                             int stride, int n_envs, const float* action, float* obs, float* reward, uint8_t* done, float* raux, float* rcomp,
                             int sequence_mode, int reset_ready_streak_on_advance, uint64_t seed, float* terminal_obs, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h || !route_ok(host_route)) return kin_fail(KIN_ERR_INVALID_ARG, KIN_RMSG("bad handle or route table"));
    if (!state || !action || !obs || !reward || !done || n_envs <= 0 || stride < n_envs || (stride % 32) != 0) return kin_fail(KIN_ERR_INVALID_ARG, KIN_RMSG("bad buffers / sizes"));
    if (((uintptr_t)obs & 15u) || ((uintptr_t)terminal_obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, KIN_RMSG("obs must be 16-byte aligned"));
    const RouteView R = view_of(host_route);
    const size_t smem = (size_t)(RT_WARPS * ROBS_TILE_FLOATS + min(R.n, ROUTE_MAX_SMEM_WP) * NJ) * sizeof(float);
    const int blocks = (n_envs + RT_THREADS - 1) / RT_THREADS;
    cudaStream_t st = (cudaStream_t)stream;
#define KIN_RLAUNCH(SEQ, COMP)                                                                                                                  \
    do {                                                                                                                                        \
        cudaError_t ea = cudaFuncSetAttribute(kin_route_step_kernel<SEQ, COMP, AUTORESET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (ea != cudaSuccess) return kin_fail_cuda(ea, KIN_RMSG("smem attribute"));                                                     \
        kin_route_step_kernel<SEQ, COMP, AUTORESET><<<blocks, RT_THREADS, smem, st>>>(h->params, R, state, stride, n_envs, action, obs, reward,  \
                                                                                     done, raux, rcomp, reset_ready_streak_on_advance, C, seed, \
                                                                                     terminal_obs);                                             \
    } while (0)
    if (sequence_mode) { if (rcomp) KIN_RLAUNCH(true, true); else KIN_RLAUNCH(true, false); }
    else { if (rcomp) KIN_RLAUNCH(false, true); else KIN_RLAUNCH(false, false); }
#undef KIN_RLAUNCH
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, AUTORESET ? "kin_route_step_autoreset" : "kin_route_step");
}
#undef KIN_RMSG

extern "C" int kin_route_step(void* handle, const KinRouteTable* host_route, float* state, int stride, int n_envs, const float* action,
                              float* obs, float* reward, uint8_t* done, float* raux, float* rcomp, int sequence_mode,
                              int reset_ready_streak_on_advance, void* stream) {
    return launch_route_step<false>(handle, host_route, KinRouteResetParams{}, state, stride, n_envs, action, obs, reward, done,
                                    raux, rcomp, sequence_mode, reset_ready_streak_on_advance, 0, nullptr, stream);
}

extern "C" int kin_route_step_autoreset(void* handle, const KinRouteTable* host_route, const KinRouteResetParams* host_reset, float* state,
                                        int stride, int n_envs, const float* action, float* obs, float* reward, uint8_t* done, float* raux,
                                        float* rcomp, int sequence_mode, int reset_ready_streak_on_advance, uint64_t seed, float* terminal_obs,
                                        void* stream) {
    if (!host_reset) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_step_autoreset: reset parameters are required");
    if (route_ok(host_route) && !reset_ranges_ok(*host_reset, host_route->n_waypoints))
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_step_autoreset: waypoint range outside the route");
    return launch_route_step<true>(handle, host_route, *host_reset, state, stride, n_envs, action, obs, reward, done,
                                   raux, rcomp, sequence_mode, reset_ready_streak_on_advance, seed, terminal_obs, stream);
}

extern "C" int kin_route_probe_rows(void* handle, const KinRouteTable* host_route, const KinPolicyWeights* w, const float* start_q, int start_index,
                                    int end_index, int n, int* prefix, uint32_t* success_bits, unsigned long long* env_steps, float* rows,
                                    int detail_replicas, void* stream);

extern "C" int kin_route_probe(void* handle, const KinRouteTable* host_route, const KinPolicyWeights* w, const float* start_q, int start_index,
                               int end_index, int n, int* prefix, uint32_t* success_bits, unsigned long long* env_steps, void* stream) {
    return kin_route_probe_rows(handle, host_route, w, start_q, start_index, end_index, n, prefix, success_bits, env_steps, nullptr, 0, stream);
}

extern "C" int kin_route_probe_rows(void* handle, const KinRouteTable* host_route, const KinPolicyWeights* w, const float* start_q, int start_index,
                                    int end_index, int n, int* prefix, uint32_t* success_bits, unsigned long long* env_steps, float* rows,
                                    int detail_replicas, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h || !route_ok(host_route)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe: bad handle or route table");
    if (detail_replicas < 0 || detail_replicas > n || (detail_replicas > 0 && !rows)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe_rows: bad detail arguments");
    if (!w || w->in_dim != ROBS || !w->pi_w0 || !w->pi_b0 || !w->pi_w1 || !w->pi_b1 || !w->act_w || !w->act_b) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe: need an 80-input actor");
    if (!prefix || n <= 0 || start_index < 1 || end_index < start_index) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe: bad sizes / indices");
    const size_t smem = (size_t)(MlpSmem<ROBS>::FLOATS + HID * RT_THREADS) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(kin_route_probe_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kin_route_probe_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_route_probe: smem attribute");
    const int final_end = end_index < host_route->n_waypoints - 1 ? end_index : host_route->n_waypoints - 1;
    const int words = (final_end - start_index + 1 + 31) / 32;
    DevPolicyR p{w->pi_w0, w->pi_b0, w->pi_w1, w->pi_b1, w->act_w, w->act_b};
    if (detail_replicas > 0)
        kin_route_probe_kernel<true><<<(n + RT_THREADS - 1) / RT_THREADS, RT_THREADS, smem, (cudaStream_t)stream>>>(
            h->params, view_of(host_route), p, start_q, start_index, end_index, n, prefix, success_bits, words, env_steps, rows, detail_replicas);
    else
        kin_route_probe_kernel<false><<<(n + RT_THREADS - 1) / RT_THREADS, RT_THREADS, smem, (cudaStream_t)stream>>>(
            h->params, view_of(host_route), p, start_q, start_index, end_index, n, prefix, success_bits, words, env_steps, nullptr, 0);
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_route_probe");
}
