// kin_route_collect.cu -- K4-route: the fused PPO rollout collection of the 80-input route policy.  ONE launch runs n_steps of
//   actor + critic forward (tcgen05 kind::f16, K = 96) -> Gaussian action sample + log-prob -> route wrapper step (base env step,
//   route-ready streak, in-episode waypoint advance, 13-term route reward) -> in-register sampled route reset of finished slots
//   -> rollout-buffer writes
// for every replica, the env + route state in registers for the whole rollout and the waypoint table in shared memory.
//
// Replaces SB3's collect_rollouts over a VecEnv of RouteSequenceKinematicEnv / RouteKinematicEnv (call site
// kinematic_phase1/train_route_curriculum.py:113-145; env: route/route_sequence_env.py:96-278, route/route_env.py:49-212, reset:
// route/route_reset_samplers.py:43-117).  The per-step-launch path of ppo.py (_collect_route: kin_policy_act -> kin_route_step ->
// kin_ppo_bootstrap -> kin_route_reset_sampled, five launches per time step) stays as the restatement this kernel is replayed
// against (tests/test_gpu_ppo.py::test_fused_route_collection_replays_through_the_step_kernels).
//
// The policy half is kin_collect_policy.cuh, shared with K4; here X = [obs80 | 1 | 0] spans two K tiles (K = 96, 6 layer-1 MMAs)
// and the second one is reused for the critic's activations.  The observation goes to the rollout buffer as fp32 rows
// ([T + 1][n][80]: what kin_ppo_grad_tc<80> consumes).  Episodes that hit the time limit append their terminal observation to a
// list; kin_ppo_bootstrap_list adds gamma * V(terminal_obs) afterwards.
#include "kin_collect_policy.cuh"
#include "kin_route_core.cuh"

namespace kin {

using namespace umma;

constexpr int RC_IN = KIN_ROUTE_OBS_DIM;      // 80

template <int TILES>
struct __align__(1024) RouteCollectSmem {
    unsigned char XH[TILES][2][AC_TILE_BYTES];   // [.][0]: X columns 0..63, then actor H1 / H2; [.][1]: X columns 64..127, then critic H1 / H2
    AcWeights<2> w;
    unsigned long long mbar[TILES][1];
    unsigned tmem_base;
    alignas(16) float q_table[ROUTE_MAX_SMEM_WP * KIN_NJ];   // waypoint joint vectors for the nearest-waypoint scan (n <= 1024)
};

struct RouteCollectOut {
    float* obs;               // [T + 1][n][80]
    float* action;            // [T][n][7]
    float* logp;              // [T][n]
    float* value;             // [T][n]
    float* reward;            // [T][n]
    uint8_t* done;            // [T][n]
    uint8_t* episode_start;   // [T][n]
    int* flags;               // [T][n]  route flags of the step (bit0 ready, bit1 regression, bit2 orientation hit, bit3 waypoint success)
    uint8_t* start_io;        // [n]
    float* last_value;        // [n]
    int* boot_count;
    int* boot_index;          // [cap]  t * n + env
    float* boot_obs;          // [cap][80]
    int boot_cap;
};

template <int TILES, bool SEQ>
__global__ void __launch_bounds__(TILES * AC_ROWS, 1)
kin_route_collect_kernel(const __grid_constant__ KinEnvParams P, RouteView R, const __grid_constant__ KinRouteResetParams C, float* __restrict__ state,
                         int stride, int n, const float* __restrict__ params, int T, uint64_t noise_seed, uint32_t step0, uint64_t reset_seed,
                         int reset_streak, RouteCollectOut out) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    RouteCollectSmem<TILES>& S = *reinterpret_cast<RouteCollectSmem<TILES>*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x;
    constexpr int NT = TILES * AC_ROWS;

    convert_weights<RC_IN, 2, NT>(S.w, params, tid);
    load_vectors<RC_IN>(S.w, params, tid);
    load_q_table(S.q_table, R, tid, NT);
    init_tiles<TILES, 1>(S, tid);
    AcTile<2> c = tile_of<2, 1>(S, tid);

    const int gtile = blockIdx.x * TILES + c.tile;
    const int n_tiles = n / AC_ROWS;
    const bool live = gtile < n_tiles;                        // tile-uniform
    const int env = (live ? gtile : 0) * AC_ROWS + c.row;
    const float* table = R.n <= ROUTE_MAX_SMEM_WP ? S.q_table : R.q;

    EnvRegs s;
    load_env<true>(state, stride, env, s);
    RouteRegs rr;
    {
        const unsigned r0 = ld_row_u(state, stride, KIN_ROW_ROUTE, env), r1 = ld_row_u(state, stride, KIN_ROW_ROUTE2, env);
        rr.index = (int)(r0 & 0xffffu); rr.streak = (int)(r0 >> 16); rr.last = (int)(r1 & 0xffffu); rr.completed = (int)(r1 >> 16);
    }
    unsigned start = live ? out.start_io[env] : 0u;

    if (live) {
        // observation of the current (env, route) registers -- what kin_route_step / kin_route_reset_sampled leave in their obs rows
        auto observe = [&](float* o) {
            float o56[OBS];
            build_obs(P, s, KIN_MODE_APPROACH, o56);
            build_route_obs(P, R, s, rr.index, o56, o);
        };
        bool goal_dirty = false;       // an in-episode waypoint advance rewrote goal pose / entry metrics since the last reset
        for (int t = 0; t < T; ++t) {
            const size_t idx = (size_t)t * n + env;
            float mv[8];
            {
                float o[RC_IN];
                observe(o);
                store_row<RC_IN>(out.obs + idx * RC_IN, o);
                policy_forward<RC_IN, false>(S.w, c, o, nullptr, mv);
            }
            float a[NJ];
            const float lp = sample_action(S.w, noise_seed, (unsigned)env, step0 + (uint32_t)t, mv, a, out.action + idx * NJ);
            out.logp[idx] = lp;
            out.value[idx] = mv[7];
            out.episode_start[idx] = (uint8_t)start;
            // ---- route wrapper step (warp-collective: every lane of a live tile is here)
            StepOut so;
            RouteOut ro;
            const int index_before = rr.index;
            route_step_core<SEQ, false>(P, R, table, s, rr, a, reset_streak != 0, so, ro, nullptr);
            if (SEQ && rr.index != index_before) goal_dirty = true;
            const bool finished = (ro.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED)) != 0u;
            if (finished) {
                push_truncated<RC_IN>(out, ro.done, idx, observe);      // the terminal observation
                Philox rng(reset_seed, (uint32_t)env, step0 + (uint32_t)t);
                float gq[NJ];
                sample_route_reset_dev(P, R, C, rng, s, rr, gq);
                store_env_reset(state, stride, env, s, gq);       // goal pose / goal_q / entry rows are only written at resets and advances
                goal_dirty = false;
            }
            out.reward[idx] = ro.reward;
            out.done[idx] = (uint8_t)ro.done;
            out.flags[idx] = (int)ro.flags;
            start = finished ? 1u : 0u;
        }
        // ---- value of the observation after the last step (GAE bootstrap), final observation row, state write-back
        {
            float o[RC_IN], mv[8];
            observe(o);
            store_row<RC_IN>(out.obs + ((size_t)T * n + env) * RC_IN, o);
            policy_forward<RC_IN, false>(S.w, c, o, nullptr, mv);
            out.last_value[env] = mv[7];
        }
        out.start_io[env] = (uint8_t)start;
        store_env_step(state, stride, env, s);
        if (goal_dirty) {      // the last in-episode advance since the last reset: goal pose, entry metrics and goal_q rows
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
    release_tiles<TILES>(S, tid);
}

template <int TILES>
static cudaError_t launch_route_collect(const KinHandle* h, const RouteView& R, const KinRouteResetParams& C, float* state, int stride, int n, const float* params,
                                        int T, uint64_t noise_seed, uint32_t step0, uint64_t reset_seed, int seq, int reset_streak, const RouteCollectOut& out,
                                        cudaStream_t st) {
    auto kernel = seq ? kin_route_collect_kernel<TILES, true> : kin_route_collect_kernel<TILES, false>;
    return launch_tiles<TILES>(kernel, sizeof(RouteCollectSmem<TILES>) + 1024, n, st, h->params, R, C, state, stride, n, params, T, noise_seed, step0,
                               reset_seed, reset_streak, out);
}

}  // namespace kin

using namespace kin;

extern "C" int kin_route_collect(void* handle, const KinRouteTable* host_route, const KinRouteResetParams* host_reset, float* state, int stride, int n_envs,
                                 const float* params, int n_steps, uint64_t noise_seed, uint32_t first_step, uint64_t reset_seed, int sequence_mode,
                                 int reset_ready_streak_on_advance, float* obs, float* action, float* logp, float* value, float* reward, uint8_t* done,
                                 uint8_t* episode_start, int* route_flags, uint8_t* start_io, float* last_value, int* boot_count, int* boot_index,
                                 float* boot_obs, int boot_cap, int tiles_per_cta, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h || !route_ok(host_route) || !host_reset) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_collect: bad handle, route table or reset parameters");
    if (!state || !params || !obs || !action || !logp || !value || !reward || !done || !episode_start || !route_flags || !start_io || !last_value ||
        !boot_count || !boot_index || !boot_obs || boot_cap <= 0 || n_steps <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_collect: null buffer or bad sizes");
    if (n_envs <= 0 || (n_envs % AC_ROWS) != 0 || stride < n_envs || (stride % 32) != 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_collect: n_envs must be a positive multiple of 128 (one GEMM tile), stride % 32 == 0");
    if (((uintptr_t)obs & 15u) || ((uintptr_t)boot_obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_collect: obs / boot_obs must be 16-byte aligned");
    for (int m = 0; m < 5; ++m)
        if (host_reset->index_lo[m] < 0 || host_reset->index_hi[m] >= host_route->n_waypoints || host_reset->index_lo[m] > host_reset->index_hi[m])
            return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_collect: waypoint range outside the route");
    cudaStream_t st = (cudaStream_t)stream;
    const int tiles = collect_tiles_per_cta(tiles_per_cta, n_envs);
    RouteCollectOut out{obs, action, logp, value, reward, done, episode_start, route_flags, start_io, last_value, boot_count, boot_index, boot_obs, boot_cap};
    cudaError_t e = cudaMemsetAsync(boot_count, 0, sizeof(int), st);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_route_collect: memset");
    const RouteView R = view_of(host_route);
    if (tiles == 1) e = launch_route_collect<1>(h, R, *host_reset, state, stride, n_envs, params, n_steps, noise_seed, first_step, reset_seed, sequence_mode, reset_ready_streak_on_advance, out, st);
    else if (tiles == 2) e = launch_route_collect<2>(h, R, *host_reset, state, stride, n_envs, params, n_steps, noise_seed, first_step, reset_seed, sequence_mode, reset_ready_streak_on_advance, out, st);
    else if (tiles == 4) e = launch_route_collect<4>(h, R, *host_reset, state, stride, n_envs, params, n_steps, noise_seed, first_step, reset_seed, sequence_mode, reset_ready_streak_on_advance, out, st);
    else return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_collect: tiles_per_cta must be 0 (auto), 1, 2 or 4");
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_route_collect");
}
